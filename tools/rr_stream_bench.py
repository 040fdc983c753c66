#!/usr/bin/env python
"""rr from a read file to an output file: the streaming path (read_recruitment.recruit_file, what main() runs) against
the in-memory path (read_sequences + recruit + one join) on the same seeded input.
    python tools/rr_stream_bench.py [--gbases 2] [--gz-gbases 1] [--large-gbases 10] [--dir DIR] [--out FILE]
The reads are tools/rr_bench.py's mix (log-normal lengths around 20 kb, 90 % random, 10 % carrying a DXZ1 copy with
12 % substitutions), threshold 350, written as single-line FASTQ, 80-column FASTA and FASTQ.gz.  Every run is a process
of its own (peak RSS is per process), warmed up on a small file first; the wall clock ends after the output is written
and the device synchronised.  Then the streaming path alone runs on a FASTA of --large-gbases (scaled down to what the
disk holds) to show that its peak RSS does not grow with the input."""
import argparse
import gzip
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
THRESHOLD = 350

_CHILD = r"""
import json, resource, sys, time
sys.path.insert(0, {root!r})
import torch
from centroflye_b200 import read_recruitment as rr
unit, path, out, warm, mode = sys.argv[1:6]
unit = next(rr.read_sequences(unit))[1]
rr.recruit_file(unit, warm, out, {thr})   # CUDA context, module load, allocator warm-up
rr._write_in_memory(unit, warm, out, {thr})
torch.cuda.synchronize()
stats = {{}}
t = time.perf_counter()
if mode == "stream":
    rr.recruit_file(unit, path, out, {thr}, stats=stats)
else:
    rr._write_in_memory(unit, path, out, {thr})
torch.cuda.synchronize()
wall = time.perf_counter() - t
stats["wall_s"] = wall
stats["peak_rss_mib"] = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024
print("RESULT " + json.dumps(stats))
"""


def _records(rng, unit, n_bases):
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    u0 = np.frombuffer(unit.encode(), dtype=np.uint8)
    total, i = 0, 0
    while total < n_bases:
        n = int(np.clip(np.exp(rng.normal(np.log(20000), 0.5)), 2000, 200000))
        s = lut[rng.integers(0, 4, size=n, dtype=np.uint8)]
        if rng.random() < 0.1:
            u = u0.copy()
            hit = rng.random(u.size) < 0.12
            u[hit] = lut[rng.integers(0, 4, size=int(hit.sum()))]
            at = int(rng.integers(0, max(1, n - u.size)))
            s[at:at + u.size] = u[: max(0, min(u.size, n - at))]
        yield f"read{i}", s.tobytes()
        total += n
        i += 1


def write_reads(path, fmt, unit, n_bases, seed):
    rng = np.random.default_rng(seed)
    opener = (lambda p: gzip.open(p, "wb", compresslevel=1)) if fmt.endswith(".gz") else (lambda p: open(p, "wb"))
    bases = 0
    with opener(path) as f:
        buf = []
        for name, s in _records(rng, unit, n_bases):
            if fmt.startswith("fastq"):
                buf.append(b"@%s len=%d\n%s\n+\n%s\n" % (name.encode(), len(s), s, b"5" * len(s)))
            else:
                full = len(s) // 80 * 80
                rows = np.frombuffer(s[:full], dtype=np.uint8).reshape(-1, 80)
                lines = np.hstack([rows, np.full((rows.shape[0], 1), 10, dtype=np.uint8)]).tobytes()
                buf.append(b">%s len=%d\n" % (name.encode(), len(s)) + lines + (s[full:] + b"\n" if full < len(s) else b""))
            bases += len(s)
            if len(buf) >= 256:
                f.write(b"".join(buf))
                buf = []
        f.write(b"".join(buf))
    return bases


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        while True:
            b = f.read(1 << 24)
            if not b:
                return h.hexdigest()
            h.update(b)


def run(mode, unit_fn, path, out, warm):
    code = _CHILD.format(root=ROOT, thr=THRESHOLD)
    res = subprocess.run([sys.executable, "-c", code, unit_fn, path, out, warm, mode], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(res.stdout[-2000:] + res.stderr[-4000:])
    stats = json.loads(res.stdout.split("RESULT ", 1)[1])
    stats["sha256"], stats["out_bytes_file"] = sha256(out), os.path.getsize(out)
    return stats


def summarize(stats, bases, fmt_bytes):
    out = {"wall_s": round(stats["wall_s"], 3), "gbases_per_s": round(bases / stats["wall_s"] / 1e9, 3),
           "file_gbytes_per_s": round(fmt_bytes / stats["wall_s"] / 1e9, 3), "peak_rss_mib": round(stats["peak_rss_mib"]),
           "sha256": stats["sha256"], "out_bytes": stats["out_bytes_file"]}
    if "chunks" in stats:
        out["stages_host_s"] = {k[:-2]: round(stats[k], 3) for k in ("read_s", "assemble_s", "scan_s", "plan_s", "wait_s",
                                                                     "write_s")}
        out["stages_device_s"] = {k: round(v, 3) for k, v in stats["device_s"].items()}
        out["chunks"], out["fallback"] = stats["chunks"], stats["fallback"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbases", type=float, default=2.0, help="FASTQ and FASTA size for the two-path comparison")
    ap.add_argument("--gz-gbases", type=float, default=1.0)
    ap.add_argument("--large-gbases", type=float, default=10.0)
    ap.add_argument("--dir", default=None, help="scratch directory for the generated files (default: the temp dir)")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    from centroflye_b200 import synth
    unit = synth.load_genome("cenx_dxz1_m1500_s1")[3]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    result = {"gpu": gpu[0] if gpu else None, "threshold": THRESHOLD, "host_cpus": os.cpu_count(), "formats": {}}
    with tempfile.TemporaryDirectory(dir=args.dir) as tmp:
        unit_fn, warm, out = os.path.join(tmp, "unit.fasta"), os.path.join(tmp, "warm.fastq"), os.path.join(tmp, "out.fa")
        with open(unit_fn, "w") as f:
            f.write(">DXZ1\n" + unit + "\n")
        write_reads(warm, "fastq", unit, 2e6, 99)
        for fmt, gb in (("fastq", args.gbases), ("fasta", args.gbases), ("fastq.gz", args.gz_gbases)):
            path = os.path.join(tmp, "reads." + fmt)
            bases = write_reads(path, fmt, unit, gb * 1e9, 1)
            size = os.path.getsize(path)
            entry = {"bases": bases, "file_bytes": size}
            for mode in ("stream", "in_memory"):
                entry[mode] = summarize(run(mode, unit_fn, path, out, warm), bases, size)
            entry["sha256_equal"] = entry["stream"]["sha256"] == entry["in_memory"]["sha256"]
            entry["speedup"] = round(entry["in_memory"]["wall_s"] / entry["stream"]["wall_s"], 2)
            result["formats"][fmt] = entry
            print(json.dumps({fmt: entry}), flush=True)
            os.remove(path)
        free = shutil.disk_usage(tmp).free
        gb = min(args.large_gbases, 0.8 * free / 1.02e9)
        path = os.path.join(tmp, "large.fasta")
        bases = write_reads(path, "fasta", unit, gb * 1e9, 2)
        result["large_fasta_stream_only"] = dict(bases=bases, file_bytes=os.path.getsize(path), disk_free_bytes=free,
                                                 **summarize(run("stream", unit_fn, path, out, warm), bases,
                                                             os.path.getsize(path)))
        print(json.dumps({"large": result["large_fasta_stream_only"]}), flush=True)
    print(json.dumps(result), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
