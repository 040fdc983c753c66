#!/usr/bin/env python
"""rr's device filter for units longer than 3328 bases (cfk_rr_filter_long, rr_filter_warp_kernel<W>) on one GPU.
    python tools/rr_long_bench.py [--mbases 300] [--reps 3] [--out profiles/rr_long_bench.json]
About 300 Mbases of random reads (lengths log-normal around 20 kb) are planned into segments as read_recruitment plans
them for the unit and threshold (overlap m + t; step max(SEGMENT, overlap rounded up to 16) for a long unit) and
filtered for one unit at a time; random reads hold no unit, so both strands of every segment are scanned to the end, the
filter's worst case.  Unit lengths 3328 (the longest of rr_filter_kernel<52>; both kernels, alternated in one loop, and
their keep bits must be equal: 10 % of the reads carry a copy of that unit with 5 % substitutions), 4110 (DXZ1 dimer),
5814 (34-monomer HOR), 6444 (D6Z1 dimer), 12000 and 32768; thresholds 350 and 10 % of m.  Filter time by CUDA events
around each launch, after one warm-up launch; rates are read bases (not segment bases) per second.  The card's name and
power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

UNIT_LENGTHS = (3328, 4110, 5814, 6444, 12000, 32768)


def _card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mbases", type=float, default=300.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200.engine import default_engine
    eng = default_engine()
    p, stream = eng._p, eng._stream()
    rng = np.random.default_rng(0)
    lens = []
    while sum(lens) < args.mbases * 1e6:
        lens.append(int(np.clip(np.exp(rng.normal(np.log(20000), 0.5)), 2000, 200000)))
    lens = np.array(lens, dtype=np.int64)
    offs = np.zeros(lens.size, dtype=np.int64)
    np.cumsum(((lens + 15) & ~15)[:-1], out=offs[1:])
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    text = lut[rng.integers(0, 4, size=int(offs[-1] + lens[-1]) + 32, dtype=np.uint8)]
    units = {m: "".join("ACGT"[c] for c in rng.integers(0, 4, size=m)) for m in UNIT_LENGTHS}
    u = np.frombuffer(units[3328].encode(), dtype=np.uint8)
    for r in np.flatnonzero(rng.random(lens.size) < 0.1):  # copies of the 3328-base unit, 5 % substitutions
        c = u.copy()
        hit = rng.random(c.size) < 0.05
        c[hit] = lut[rng.integers(0, 4, size=int(hit.sum()))]
        at = offs[r] + int(rng.integers(0, max(1, lens[r] - c.size)))
        n = int(min(c.size, offs[r] + lens[r] - at))
        text[at:at + n] = c[:n]
    d_text = eng._to_dev(text)
    total = int(lens.sum())
    results = []
    for m in UNIT_LENGTHS:
        unit = units[m]
        for threshold in (350, m // 10):
            overlap = m + threshold
            _, seg_read, start, seg_len = rr._segment_plan(lens, overlap, m > rr.MAX_SHORT_UNIT)
            order = np.argsort(-seg_len, kind="stable").astype(np.int32)
            S = int(seg_read.size)
            d_off, d_len, d_order = eng._to_dev(offs[seg_read] + start), eng._to_dev(seg_len), eng._to_dev(order)
            m_t = np.array([m, threshold], dtype=np.int32)
            kernels = {}
            if m <= rr.MAX_SHORT_UNIT:  # the same unit through both kernels; the long plan is the same below SEGMENT
                peq, sym_of, _ = rr.build_masks(unit)
                kernels["rr_filter_kernel"] = ("cfk_rr_filter_units", eng._to_dev(peq.reshape(-1).view(np.int64)),
                                               eng._to_dev(sym_of))
            peq_l, sym_l, w = rr.build_long_masks(unit)
            kernels["rr_filter_warp_kernel"] = ("cfk_rr_filter_long", eng._to_dev(peq_l.reshape(-1).view(np.int64)),
                                                eng._to_dev(sym_l))
            keeps, times = {}, {k: [] for k in kernels}
            for rep in range(args.reps + 1):  # rep 0 warms up
                for name, (entry, d_peq, d_sym) in kernels.items():
                    d_keep = eng._zeros(S, torch.uint8)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    if entry == "cfk_rr_filter_units":
                        _lib.call(entry, p(d_text), p(d_off), p(d_len), p(d_order), S, 1, p(d_peq), p(d_sym),
                                  m_t.ctypes.data, m_t[1:].ctypes.data, p(d_keep), stream)
                    else:
                        _lib.call(entry, p(d_text), p(d_off), p(d_len), p(d_order), S, 1, p(d_peq), p(d_sym),
                                  m_t.ctypes.data, m_t[1:].ctypes.data, 0, None, p(d_keep), stream)
                    b.record()
                    b.synchronize()
                    if rep:
                        times[name].append(a.elapsed_time(b) / 1e3)
                    keeps[name] = d_keep[:S].cpu().numpy()
            row = {"m": m, "threshold": threshold, "W": int(w), "segments": S,
                   "segment_bases": int(seg_len.sum()), "kept_segments": int(keeps["rr_filter_warp_kernel"].sum())}
            for name, ts in times.items():
                best = min(ts)
                row[name] = {"seconds": ts, "gbases_per_s": total / best / 1e9,
                             "word_steps_per_s": 2 * int(seg_len.sum()) * (32 * w if "warp" in name else -(-m // 64)) / best}
            if len(kernels) == 2:
                row["keep_equal"] = bool(np.array_equal(keeps["rr_filter_kernel"], keeps["rr_filter_warp_kernel"]))
                row["warp_over_thread_time"] = min(times["rr_filter_warp_kernel"]) / min(times["rr_filter_kernel"])
            results.append(row)
            print(json.dumps(row), flush=True)
            del d_off, d_len, d_order, kernels
    out = {"card": _card(), "reads": int(lens.size), "bases": total, "reps": args.reps, "results": results,
           "word_steps": "lane-word steps for the warp kernel (32 W per character and strand, idle lanes included), "
                         "unit words for rr_filter_kernel"}
    ok = all(r.get("keep_equal", True) for r in results)
    out["keep_equal_at_3328"] = ok
    print(json.dumps({"card": out["card"], "keep_equal_at_3328": ok}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
