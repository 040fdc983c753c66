"""Row f rank 4, second half: the read recruitment pre-filter (scripts/read_recruitment/rr.cpp) on the device.

* against the output file the REFERENCE BINARY writes for the same command line -- rr.cpp's rule on exact infix edit
  distances, stored as kept read names, size and SHA-256 in tests/golden/rr/outputs.json by oracle/make_rr_golden.py,
  which also checks it against the binary when given one: byte-identical output file, for several thresholds,
  FASTA / FASTQ / gzip input;
* exact infix edit distances on both strands against a plain dynamic-programming restatement of edlib's HW mode, for
  unit lengths on every side of the 64-bit word boundaries and of the kernel's template sizes (incl. DXZ1 and D6Z1)."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu
RR_GOLDEN = os.path.join(GOLDEN, "rr", "outputs.json")
FORMATS = ["fasta", "fastq", "fasta.gz"]
THRESHOLDS = (0, 100, 350, 700, -1)


def _rnd(rng, n):
    return "".join("ACGT"[c] for c in rng.integers(0, 4, size=n))


def _mutate(rng, s, rate):
    out = []
    for c in s:
        x = rng.random()
        if x < rate / 3:
            out.append("ACGT"[rng.integers(4)])
        elif x < 2 * rate / 3:
            continue
        elif x < rate:
            out.append(c)
            out.append("ACGT"[rng.integers(4)])
        else:
            out.append(c)
    return "".join(out)


def _infix_distance(unit, text):
    """min over infixes of the edit distance (edlib HW): row-wise DP, the in-row dependency by a running minimum."""
    t = np.frombuffer(text.encode(), dtype=np.uint8)
    prev, ar = np.zeros(t.size + 1, dtype=np.int64), np.arange(t.size + 1)
    for i, c in enumerate(unit.encode()):
        cur = np.empty_like(prev)
        cur[0] = i + 1
        cur[1:] = np.minimum(prev[:-1] + (t != c), prev[1:] + 1)
        prev = np.minimum.accumulate(cur - ar) + ar
    return int(prev.min())


def _read_set(rng, unit):
    from centroflye_b200.read_recruitment import reverse_complement
    reads = []
    for i in range(14):
        core = unit if i % 2 == 0 else reverse_complement(unit)
        rate = [0.0, 0.05, 0.1, 0.15, 0.17, 0.2, 0.3][i // 2]
        reads.append((f"cen{i}", _rnd(rng, int(rng.integers(0, 3000))) + _mutate(rng, core, rate) + _rnd(rng, int(rng.integers(0, 3000)))))
    reads += [(f"rnd{i}", _rnd(rng, int(rng.integers(100, 9000)))) for i in range(6)]
    reads += [("half", _rnd(rng, 500) + unit[:1000] + _rnd(rng, 500)), ("tiny", "ACGT"), ("with_n", unit[:900] + "NNNN" + unit[900:])]
    return reads


def write_inputs(tmp_dir, fmt):
    """The unit (DXZ1) and the seeded read set of one input format as files -> (unit_fn, read_fn, reads, read text)."""
    from centroflye_b200 import synth
    rng = np.random.default_rng({"fasta": 1, "fastq": 2, "fasta.gz": 3}[fmt])
    unit = synth.load_genome("cenx_dxz1_m1500_s1")[3]
    reads = _read_set(rng, unit)
    unit_fn, read_fn = os.path.join(tmp_dir, "unit.fasta"), os.path.join(tmp_dir, "reads." + fmt)
    with open(unit_fn, "w") as f:
        f.write(">DXZ1 rc\n" + "\n".join(unit[i:i + 70] for i in range(0, len(unit), 70)) + "\n")
    if fmt == "fastq":
        text = "".join(f"@{n} some comment\n{s}\n+\n{'I' * len(s)}\n" for n, s in reads)
    else:
        text = "".join(f">{n} some comment\n" + "\n".join(s[i:i + 80] for i in range(0, len(s), 80)) + "\n" for n, s in reads)
    if fmt.endswith(".gz"):
        with gzip.open(read_fn, "wt") as f:
            f.write(text)
    else:
        with open(read_fn, "w") as f:
            f.write(text)
    return unit_fn, read_fn, reads, text


@pytest.mark.parametrize("fmt", FORMATS)
def test_rr_output_equals_reference_binary(tmp_path, fmt):
    from centroflye_b200 import read_recruitment as rr
    with open(RR_GOLDEN) as f:
        golden = json.load(f)[fmt]
    unit_fn, read_fn, reads, text = write_inputs(str(tmp_path), fmt)
    assert hashlib.sha256(text.encode()).hexdigest() == golden["reads_sha256"], \
        "the seeded read set is not the one the golden outputs were made from"
    kept_counts = []
    for threshold in THRESHOLDS:
        want = golden["outputs"][str(threshold)]
        got_fn = str(tmp_path / f"got{threshold}.fasta")
        assert rr.main([unit_fn, read_fn, got_fn, str(threshold)]) == 0
        got = open(got_fn, "rb").read()
        assert [ln[1:].decode() for ln in got.split(b"\n") if ln.startswith(b">")] == want["kept"]
        assert len(got) == want["bytes"] and hashlib.sha256(got).hexdigest() == want["sha256"]
        kept_counts.append(len(want["kept"]))
    assert kept_counts[0] >= 2 and kept_counts[0] < kept_counts[2] < kept_counts[4] == len(reads)


@pytest.mark.parametrize("m", [1, 5, 63, 64, 65, 200, 257, 600, 1100, 2055, 3222])
def test_rr_exact_distances_match_dp(m):
    from centroflye_b200 import read_recruitment as rr
    rng = np.random.default_rng(m)
    unit = _rnd(rng, m)
    rc = rr.reverse_complement(unit)
    seqs = [_rnd(rng, int(rng.integers(1, 1200))) for _ in range(6)]
    seqs += [_rnd(rng, 40) + _mutate(rng, unit, 0.1) + _rnd(rng, 33), _mutate(rng, rc, 0.2), unit, rc[: max(1, m // 2)], "A"]
    keep, dist = rr.recruit(unit, seqs, threshold=max(1, m // 5), exact=True)
    for s, d, k in zip(seqs, dist.tolist(), keep.tolist()):
        want = (_infix_distance(unit, s), _infix_distance(rc, s))
        assert tuple(d) == want
        assert k == (min(want) <= max(1, m // 5))
    assert rr.recruit(unit, seqs, threshold=-1).all()                     # edlib's k = -1: no limit
    early = rr.recruit(unit, seqs, threshold=max(1, m // 5))              # early exit gives the same decisions
    assert np.array_equal(early, keep)


def test_rr_unit_checks():
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200._lib import CfkError
    with pytest.raises(AssertionError):
        rr.reverse_complement("ACGN")                                     # complement() asserts in the reference
    with pytest.raises(CfkError):
        rr.build_masks("A" * 4000)
