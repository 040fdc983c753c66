#!/usr/bin/env python
"""rr for U units: one pass over the read file (read_recruitment.recruit_file_units) against U sequential recruit_file
runs, one per unit, on the seeded inputs of tools/rr_stream_bench.py.
    python tools/rr_units_bench.py [--gbases 0.5] [--gz-gbases 0.25] [--units 1,2,4,8] [--dir DIR] [--out FILE]
The units are DXZ1 and the committed cenx_like_u2..u8, threshold 350; U = 1, 2, 4, 8 takes the first U of them.  The
reads are rr_stream_bench's (log-normal lengths around 20 kb, 10 % carrying a DXZ1 copy), as FASTQ, FASTA and FASTQ.gz.
Every run is a process of its own, warmed up on a small file first; its wall clock ends after the outputs are written
and the device synchronised.  The sequential time for U units is the sum of the single runs of the first U units (each
single run is made once and shared by every U).  Per run: wall time, host and device stage seconds, peak RSS and the
SHA-256 of every output; the one-pass and the sequential hashes must be equal."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from rr_stream_bench import sha256, write_reads  # noqa: E402

THRESHOLD = 350
UNIT_NAMES = ["cenx_dxz1_m1500_s1"] + [f"cenx_like_u{i}_m1500_s{i}" for i in range(2, 9)]

_CHILD = r"""
import json, resource, sys, time
sys.path.insert(0, {root!r})
import torch
from centroflye_b200 import read_recruitment as rr
path, warm, jobs, mode = sys.argv[1], sys.argv[2], json.loads(sys.argv[3]), sys.argv[4]
jobs = [(next(rr.read_sequences(unit_fn))[1], out, {thr}) for unit_fn, out in jobs]
rr.recruit_file_units(jobs, warm)   # CUDA context, module load, allocator warm-up
torch.cuda.synchronize()
stats = {{}}
t = time.perf_counter()
if mode == "single":
    (unit, out, thr), = jobs
    rr.recruit_file(unit, path, out, thr, stats=stats)
else:
    rr.recruit_file_units(jobs, path, stats=stats)
torch.cuda.synchronize()
stats["wall_s"] = time.perf_counter() - t
stats["peak_rss_mib"] = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024
print("RESULT " + json.dumps(stats))
"""


def run(mode, path, warm, jobs):
    """One process: recruit_file for one job (mode "single"), or recruit_file_units.  jobs = [(unit_fn, out_fn)]."""
    code = _CHILD.format(root=ROOT, thr=THRESHOLD)
    res = subprocess.run([sys.executable, "-c", code, path, warm, json.dumps(jobs), mode], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(res.stdout[-2000:] + res.stderr[-4000:])
    st = json.loads(res.stdout.split("RESULT ", 1)[1])
    return {"wall_s": round(st["wall_s"], 3), "peak_rss_mib": round(st["peak_rss_mib"]),
            "stages_host_s": {k[:-2]: round(st[k], 3) for k in ("read_s", "assemble_s", "scan_s", "plan_s", "wait_s",
                                                                "write_s")},
            "stages_device_s": {k: round(v, 3) for k, v in st["device_s"].items()},
            "chunks": st["chunks"], "fallback": st["fallback"],
            "outputs": [{"sha256": sha256(out), "bytes": os.path.getsize(out)} for _, out in jobs]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbases", type=float, default=0.5, help="FASTQ and FASTA size")
    ap.add_argument("--gz-gbases", type=float, default=0.25)
    ap.add_argument("--units", default="1,2,4,8")
    ap.add_argument("--dir", default=None, help="scratch directory for the generated files (default: the temp dir)")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    counts = [int(u) for u in args.units.split(",")]
    assert max(counts) <= len(UNIT_NAMES)
    from centroflye_b200 import synth
    units = [synth.load_genome(n)[3] for n in UNIT_NAMES]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    result = {"gpu": gpu[0] if gpu else None, "threshold": THRESHOLD, "units": UNIT_NAMES[:max(counts)],
              "host_cpus": os.cpu_count(), "formats": {}}
    with tempfile.TemporaryDirectory(dir=args.dir) as tmp:
        unit_fns = []
        for name, unit in zip(UNIT_NAMES, units):
            unit_fns.append(os.path.join(tmp, name + ".fasta"))
            with open(unit_fns[-1], "w") as f:
                f.write(f">{name}\n{unit}\n")
        warm = os.path.join(tmp, "warm.fastq")
        write_reads(warm, "fastq", units[0], 2e6, 99)
        for fmt, gb in (("fastq", args.gbases), ("fasta", args.gbases), ("fastq.gz", args.gz_gbases)):
            path = os.path.join(tmp, "reads." + fmt)
            bases = write_reads(path, fmt, units[0], gb * 1e9, 1)
            entry = {"bases": bases, "file_bytes": os.path.getsize(path),
                     "single": [run("single", path, warm, [(unit_fns[u], os.path.join(tmp, f"single{u}.fa"))])
                                for u in range(max(counts))]}
            for U in counts:
                one = run("one_pass", path, warm, [(unit_fns[u], os.path.join(tmp, f"multi{u}.fa")) for u in range(U)])
                seq_wall = sum(s["wall_s"] for s in entry["single"][:U])
                entry[f"U{U}"] = {
                    "one_pass": one, "sequential_wall_s": round(seq_wall, 3),
                    "sequential_peak_rss_mib": max(s["peak_rss_mib"] for s in entry["single"][:U]),
                    "speedup": round(seq_wall / one["wall_s"], 2),
                    "sha256_equal": [o["sha256"] for o in one["outputs"]] == [s["outputs"][0]["sha256"]
                                                                             for s in entry["single"][:U]]}
                print(json.dumps({fmt: {f"U{U}": entry[f"U{U}"]}}), flush=True)
            result["formats"][fmt] = entry
            os.remove(path)
    result["all_sha256_equal"] = all(e[f"U{U}"]["sha256_equal"] for e in result["formats"].values() for U in counts)
    print(json.dumps(result), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    return 0 if result["all_sha256_equal"] else 1


if __name__ == "__main__":
    sys.exit(main())
