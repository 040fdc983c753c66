#!/usr/bin/env python
"""rr_multi on compressed read files: FASTQ.gz (one gzip member, inflated on the host), bgzip'd FASTQ and unaligned BAM
(BGZF blocks inflated on the device by cfk_bgzf_inflate).
    python tools/rr_bgzf_bench.py [--gbases 0.5] [--units 1,8] [--gpus 1,8] [--dir DIR] [--out FILE]
The reads are tools/rr_stream_bench.py's (log-normal lengths around 20 kb, 10 % carrying a DXZ1 copy), written once as
FASTQ and compressed three ways at zlib level 6.  Recorded:
  * the inflate kernel alone on one 64 MiB chunk's worth of blocks of each BGZF file: GB/s of inflated output (CUDA
    events over 20 launches after 3 of warm-up), next to one host thread of zlib inflating the same blocks;
  * rr_multi (recruit_file_units) wall time and stage seconds at U = 1 and 8 units, threshold 350, for each format, on
    one GPU and on G GPUs where that many are visible; every run is a process of its own, warmed up on a small file;
  * the SHA-256 of every output, which must be equal across the three formats;
  * the GPU's name and power limit, read in the same run."""
import argparse
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from rr_stream_bench import sha256, write_reads  # noqa: E402
from rr_units_bench import THRESHOLD, UNIT_NAMES  # noqa: E402

_CHILD = r"""
import json, sys, time
sys.path.insert(0, {root!r})
import torch
from centroflye_b200 import read_recruitment as rr
path, warm, jobs, devices = sys.argv[1], sys.argv[2], json.loads(sys.argv[3]), json.loads(sys.argv[4])
jobs = [(next(rr.read_sequences(unit_fn))[1], out, {thr}) for unit_fn, out in jobs]
rr.recruit_file_units(jobs, warm, devices=devices)
torch.cuda.synchronize()
stats = {{}}
t = time.perf_counter()
rr.recruit_file_units(jobs, path, devices=devices, stats=stats)
for d in range(torch.cuda.device_count()):
    torch.cuda.synchronize(d)
stats["wall_s"] = time.perf_counter() - t
print("RESULT " + json.dumps(stats))
"""


def run(path, warm, jobs, devices):
    code = _CHILD.format(root=ROOT, thr=THRESHOLD)
    res = subprocess.run([sys.executable, "-c", code, path, warm, json.dumps(jobs), json.dumps(devices)],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(res.stdout[-2000:] + res.stderr[-4000:])
    st = json.loads(res.stdout.split("RESULT ", 1)[1])
    return {"wall_s": round(st["wall_s"], 3),
            "stages_host_s": {k[:-2]: round(st[k], 3) for k in ("read_s", "assemble_s", "scan_s", "plan_s", "wait_s",
                                                                "write_s")},
            "inflate_device_s": round(st["inflate_s"], 3), "bgzf_blocks": st["bgzf_blocks"],
            "stages_device_s": {k: round(v, 3) for k, v in st["device_s"].items()},
            "chunks": st["chunks"], "records": st["records"], "fallback": st["fallback"],
            "sha256": [sha256(out) for _, out in jobs]}


def write_formats(d, fastq, seed_bam_flags=7):
    """fastq.gz (gzip, one member), fastq.bgz (bgzip) and bam, from one FASTQ file."""
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200 import synth
    paths = {"fastq.gz": os.path.join(d, "reads.fastq.gz"), "fastq.bgz": os.path.join(d, "reads.fastq.bgz"),
             "bam": os.path.join(d, "reads.bam")}
    data = open(fastq, "rb").read()
    with gzip.open(paths["fastq.gz"], "wb", compresslevel=6) as f:
        f.write(data)
    synth.write_bgzf(paths["fastq.bgz"], data, level=6)
    del data
    rng = np.random.default_rng(seed_bam_flags)
    comp = str.maketrans(synth.BAM_CODES, "=TGKCYSBAWRDMHVN")
    recs = []
    for name, seq in rr.read_sequences(fastq):
        flag = 0x10 if rng.random() < 0.5 else 0
        stored = seq[::-1].translate(comp) if flag else seq  # BAM stores a reverse-strand read reverse-complemented
        recs.append(synth.bam_record(name, stored, flag=flag, qual=bytes([20]) * len(seq), tags=b"RGZbench\0"))
    with open(paths["bam"], "wb") as f:
        f.write(synth.bgzf_compress(synth.bam_bytes(recs), level=6))
    return paths


def kernel_rate(path, reps=20, warmup=3):
    """The inflate kernel alone on the first 64 MiB of inflated output of a BGZF file, and one zlib thread on it."""
    import torch
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    comp = np.fromfile(path, dtype=np.uint8, count=(64 << 20) + (1 << 16))
    max_blocks = (64 << 20) // 65536
    rows = np.zeros((max_blocks, 5), dtype=np.int64)
    n, consumed, total, flags = rr._bgzf_blocks(comp, max_blocks, rows)
    d_comp = torch.from_numpy(comp[:consumed].copy()).cuda()
    d_rows = torch.from_numpy(rows[:n].copy()).cuda()
    d_out = torch.empty(total, dtype=torch.uint8, device="cuda")
    d_status = torch.empty(n, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    launch = lambda: _lib.call("cfk_bgzf_inflate", d_comp.data_ptr(), d_rows.data_ptr(), n, d_out.data_ptr(),  # noqa
                               d_status.data_ptr(), stream)
    for _ in range(warmup):
        launch()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        launch()
    b.record()
    torch.cuda.synchronize()
    kernel_s = a.elapsed_time(b) / 1e3 / reps
    assert not d_status.any().item()
    out = d_out.cpu().numpy()
    t = time.perf_counter()
    host = [zlib.decompress(comp[o:o + L].tobytes(), -15) for o, L in rows[:n, :2].tolist()]
    host_s = time.perf_counter() - t
    assert b"".join(host) == out.tobytes()
    return {"blocks": n, "inflated_bytes": total, "compressed_bytes": consumed,
            "kernel_ms": round(kernel_s * 1e3, 3), "kernel_gb_per_s": round(total / kernel_s / 1e9, 2),
            "zlib_1_thread_ms": round(host_s * 1e3, 1), "zlib_1_thread_gb_per_s": round(total / host_s / 1e9, 3)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbases", type=float, default=0.5)
    ap.add_argument("--units", default="1,8")
    ap.add_argument("--gpus", default="1,8")
    ap.add_argument("--dir", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from centroflye_b200 import synth
    d = tempfile.mkdtemp(prefix="rr_bgzf_bench_", dir=args.dir)
    units = []
    for name in UNIT_NAMES:
        units.append(os.path.join(d, name + ".fasta"))
        with open(units[-1], "w") as f:
            f.write(f">{name}\n{synth.load_genome(name)[3]}\n")
    dxz1 = synth.load_genome(UNIT_NAMES[0])[3]
    t = time.perf_counter()
    fastq = os.path.join(d, "reads.fastq")
    bases = write_reads(fastq, "fastq", dxz1, args.gbases * 1e9, 1)
    warm_dir = os.path.join(d, "warm")
    os.makedirs(warm_dir)
    warm = os.path.join(warm_dir, "warm.fastq")
    write_reads(warm, "fastq", dxz1, 2e6, 99)
    paths = write_formats(d, fastq)
    warm_paths = write_formats(warm_dir, warm)
    os.remove(fastq)
    res = {"gpu": gpu_info(), "bases": bases, "threshold": THRESHOLD, "write_inputs_s": round(time.perf_counter() - t, 1),
           "file_bytes": {k: os.path.getsize(p) for k, p in paths.items()}, "kernel": {}, "runs": []}
    for fmt in ("fastq.bgz", "bam"):
        res["kernel"][fmt] = kernel_rate(paths[fmt])
        print(fmt, res["kernel"][fmt], flush=True)
    n_vis = torch.cuda.device_count()
    for G in [int(x) for x in args.gpus.split(",")]:
        if G > n_vis:
            res["runs"].append({"gpus": G, "skipped": f"{n_vis} GPU(s) visible"})
            continue
        for U in [int(x) for x in args.units.split(",")]:
            hashes = {}
            for fmt, path in paths.items():
                jobs = [(units[i], os.path.join(d, f"out_{fmt}_{i}.fa")) for i in range(U)]
                r = run(path, warm_paths[fmt], jobs, list(range(G)) if G > 1 else None)
                r.update(format=fmt, units=U, gpus=G, gbases_per_s=round(bases / r["wall_s"] / 1e9, 3))
                hashes[fmt] = r["sha256"]
                res["runs"].append(r)
                print(json.dumps({k: r[k] for k in ("format", "units", "gpus", "wall_s", "stages_host_s",
                                                    "inflate_device_s")}), flush=True)
            assert len({json.dumps(h) for h in hashes.values()}) == 1, hashes
            res["runs"][-1]["outputs_equal_across_formats"] = True
    res["gpu_after"] = gpu_info()
    shutil.rmtree(d)
    text = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
