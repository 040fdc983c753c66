#!/usr/bin/env python
"""rr_multi on G devices: recruit_file_units(devices=...) for U units against the one-device run (G = 1), on the seeded
inputs of tools/rr_stream_bench.py.
    python tools/rr_gpus_bench.py [--gbases 0.5] [--gz-gbases 0.25] [--units 1,8,16,24] [--gpus 1,2,4,8]
                                  [--formats fastq,fasta,fastq.gz] [--dir DIR] [--out FILE]
Units: DXZ1, cenx_like_u2..u8 and D6Z1 (the committed genomes); beyond those nine, seeded copies of them with 5 %
substitutions.  The filter's cost depends only on a unit's word class, and every copy keeps its own output distinct.
Threshold 350.  G runs on cuda:0 .. G-1.  When fewer than G GPUs are visible, the G workers share cuda:0 instead
(devices=[0] * G) and the run is marked "one_gpu": it then measures what dealing records out costs, not what more GPUs
gain.  Every run is a process of its own, warmed up on a small file with the same devices first; its wall clock ends
after the outputs are written and the devices synchronised.  Per run: wall time, host stage seconds, device stage
seconds per device, peak RSS and the SHA-256 of every output; every G > 1 must equal G = 1 hash for hash."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from rr_stream_bench import sha256, write_reads  # noqa: E402

THRESHOLD = 350
UNIT_NAMES = ["cenx_dxz1_m1500_s1"] + [f"cenx_like_u{i}_m1500_s{i}" for i in range(2, 9)] + ["cen6_d6z1_m1000_s4"]

_CHILD = r"""
import json, resource, sys, time
sys.path.insert(0, {root!r})
import torch
from centroflye_b200 import read_recruitment as rr
path, warm, jobs, devices = sys.argv[1], sys.argv[2], json.loads(sys.argv[3]), json.loads(sys.argv[4])
jobs = [(next(rr.read_sequences(unit_fn))[1], out, {thr}) for unit_fn, out in jobs]
rr.recruit_file_units(jobs, warm, devices=devices)   # CUDA contexts, module load, allocator warm-up
for d in set(devices):
    torch.cuda.synchronize(d)
stats = {{}}
t = time.perf_counter()
rr.recruit_file_units(jobs, path, stats=stats, devices=devices)
for d in set(devices):
    torch.cuda.synchronize(d)
stats["wall_s"] = time.perf_counter() - t
stats["peak_rss_mib"] = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024
print("RESULT " + json.dumps(stats))
"""


def units_for(count):
    """(name, unit) of the first `count` units: the committed ones, then seeded 5 %-mutated copies of them."""
    from centroflye_b200 import synth
    base = [(n, synth.load_genome(n)[3]) for n in UNIT_NAMES]
    out = base[:count]
    rng = np.random.default_rng(2024)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    for i in range(count - len(out)):
        name, unit = base[i % len(base)]
        u = np.frombuffer(unit.encode(), dtype=np.uint8).copy()
        hit = rng.random(u.size) < 0.05
        u[hit] = lut[rng.integers(0, 4, size=int(hit.sum()))]
        out.append((f"{name}_copy{i // len(base) + 1}", u.tobytes().decode()))
    return out


def run(path, warm, jobs, devices):
    """One process: recruit_file_units(jobs, path, devices=devices).  jobs = [(unit_fn, out_fn)]."""
    code = _CHILD.format(root=ROOT, thr=THRESHOLD)
    res = subprocess.run([sys.executable, "-c", code, path, warm, json.dumps(jobs), json.dumps(devices)],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(res.stdout[-2000:] + res.stderr[-4000:])
    st = json.loads(res.stdout.split("RESULT ", 1)[1])
    return {"wall_s": round(st["wall_s"], 3), "peak_rss_mib": round(st["peak_rss_mib"]),
            "stages_host_s": {k[:-2]: round(st[k], 3) for k in ("read_s", "assemble_s", "scan_s", "plan_s", "wait_s",
                                                                "write_s")},
            "stages_device_s": {k: round(v, 3) for k, v in st["device_s"].items()},
            "stages_device_s_per_device": [{k: round(v, 3) for k, v in d.items()} for d in st["device_s_per_device"]],
            "chunks": st["chunks"], "fallback": st["fallback"],
            "outputs": [{"sha256": sha256(out), "bytes": os.path.getsize(out)} for _, out in jobs]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbases", type=float, default=0.5, help="FASTQ and FASTA size")
    ap.add_argument("--gz-gbases", type=float, default=0.25)
    ap.add_argument("--units", default="1,8,16,24")
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--formats", default="fastq,fasta,fastq.gz")
    ap.add_argument("--dir", default=None, help="scratch directory for the generated files (default: the temp dir)")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    import torch
    counts = [int(u) for u in args.units.split(",")]
    gpus = [int(g) for g in args.gpus.split(",")]
    assert gpus[0] == 1, "G = 1 is the reference every other G is compared with"
    visible = torch.cuda.device_count()
    units = units_for(max(counts))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    result = {"gpus": smi, "visible_gpus": visible, "threshold": THRESHOLD, "units": [n for n, _ in units],
              "host_cpus": os.cpu_count(), "formats": {}}
    ok = True
    with tempfile.TemporaryDirectory(dir=args.dir) as tmp:
        unit_fns = []
        for name, unit in units:
            unit_fns.append(os.path.join(tmp, name + ".fasta"))
            with open(unit_fns[-1], "w") as f:
                f.write(f">{name}\n{unit}\n")
        warm = os.path.join(tmp, "warm.fastq")
        write_reads(warm, "fastq", units[0][1], 2e6, 99)
        for fmt in args.formats.split(","):
            path = os.path.join(tmp, "reads." + fmt)
            bases = write_reads(path, fmt, units[0][1], (args.gz_gbases if fmt.endswith(".gz") else args.gbases) * 1e9, 1)
            entry = result["formats"][fmt] = {"bases": bases, "file_bytes": os.path.getsize(path)}
            for U in counts:
                jobs = [(unit_fns[u], os.path.join(tmp, f"out{u}.fa")) for u in range(U)]
                rows = entry[f"U{U}"] = {}
                for G in gpus:
                    devices = list(range(G)) if G <= visible else [0] * G
                    r = run(path, warm, jobs, devices)
                    r["one_gpu"] = G > 1 and G > visible
                    if G > 1:
                        r["sha256_equal_G1"] = [o["sha256"] for o in r["outputs"]] == [o["sha256"] for o in
                                                                                      rows["G1"]["outputs"]]
                        r["speedup_vs_G1"] = round(rows["G1"]["wall_s"] / r["wall_s"], 2)
                        ok = ok and r["sha256_equal_G1"]
                    rows[f"G{G}"] = r
                    print(json.dumps({fmt: {f"U{U}": {f"G{G}": {k: r[k] for k in r if k != "outputs"}}}}), flush=True)
            os.remove(path)
    result["all_sha256_equal"] = ok
    print(json.dumps(result), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
