#!/usr/bin/env python
"""What the reference's read recruitment filter (scripts/read_recruitment/rr.cpp) writes for the seeded inputs of
tests/test_gpu_read_recruitment.py (TEST INFRASTRUCTURE).

    python oracle/make_rr_golden.py [--rr path/to/reference/rr]

rr.cpp:73-90 keeps a read when edlib finds the unit or its reverse complement in it (HW mode: the whole unit against
any infix of the read) within `threshold` edits, -1 meaning no limit, and writes ">name\\nsequence\\n" for the kept
reads in input order.  Here the two infix edit distances of every read come from the test's plain dynamic programming
(exact, no device code), the output bytes from that rule.  With --rr the reference binary is run on the same files
and must write the same bytes.  Stored: tests/golden/rr/outputs.json -- per input format the SHA-256 of the read
text, the distances, and per threshold the kept read names, the size and the SHA-256 of the output file.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
OUT = os.path.join(ROOT, "tests", "golden", "rr", "outputs.json")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rr", help="the reference's rr binary, to confirm every output file")
    args = ap.parse_args()
    import test_gpu_read_recruitment as t
    from centroflye_b200.read_recruitment import reverse_complement
    golden = {"source": "exact infix edit distances (dynamic programming) under rr.cpp:73-90's rule"
                        + (", confirmed byte for byte by the reference binary" if args.rr else "")}
    for fmt in t.FORMATS:
        with tempfile.TemporaryDirectory() as tmp:
            unit_fn, read_fn, reads, text = t.write_inputs(tmp, fmt)
            unit = "".join(ln.strip() for ln in open(unit_fn) if not ln.startswith(">"))
            rc = reverse_complement(unit)
            dist = {n: [t._infix_distance(unit, s), t._infix_distance(rc, s)] for n, s in reads}
            outputs = {}
            for threshold in t.THRESHOLDS:
                kept = [(n, s) for n, s in reads if threshold < 0 or min(dist[n]) <= threshold]
                data = "".join(f">{n}\n{s}\n" for n, s in kept).encode()
                if args.rr:
                    ref_fn = os.path.join(tmp, f"ref{threshold}.fasta")
                    subprocess.check_call([args.rr, unit_fn, read_fn, ref_fn, str(threshold)])
                    assert open(ref_fn, "rb").read() == data, f"{fmt}, threshold {threshold}: the reference differs"
                outputs[str(threshold)] = {"kept": [n for n, _ in kept], "bytes": len(data),
                                           "sha256": hashlib.sha256(data).hexdigest()}
        golden[fmt] = {"reads_sha256": hashlib.sha256(text.encode()).hexdigest(), "distances": dist, "outputs": outputs}
        print(fmt, {th: len(o["kept"]) for th, o in outputs.items()})
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as f:
        json.dump(golden, f, indent=1)
        f.write("\n")
    print(OUT)


if __name__ == "__main__":
    main()
