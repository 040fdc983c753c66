"""The streaming rr filter (read_recruitment.recruit_file: native scanner, rr_gather_kernel, rr_filter_kernel over
segments, rr_emit_kernel) against the reference binary's outputs (tests/golden/rr/outputs.json) at many chunk sizes,
against the in-memory path (read_sequences + recruit + one join) on a fuzz corpus, on the edge cases of rr's command
line, and for memory that does not grow with the input."""
import gzip
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_read_recruitment import FORMATS, RR_GOLDEN, THRESHOLDS, _mutate, _rnd, write_inputs

pytestmark = pytest.mark.gpu


def _unit_of(unit_fn):
    from centroflye_b200 import read_recruitment as rr
    return next(rr.read_sequences(unit_fn))[1]


def _in_memory(unit, read_fn, path, threshold):
    from centroflye_b200 import read_recruitment as rr
    rr._write_in_memory(unit, read_fn, path, threshold)
    return open(path, "rb").read()


@pytest.mark.parametrize("fmt", FORMATS)
def test_goldens_at_many_chunk_sizes(tmp_path, fmt):
    from centroflye_b200 import read_recruitment as rr
    with open(RR_GOLDEN) as f:
        golden = json.load(f)[fmt]
    unit_fn, read_fn, reads, _ = write_inputs(str(tmp_path), fmt)
    unit = _unit_of(unit_fn)
    assert sum(len(s) > 700 for _, s in reads) >= 15      # chunk 700 is smaller than most records
    for chunk in (700, 5000, 1 << 16, 1 << 26):
        for threshold in THRESHOLDS:
            want = golden["outputs"][str(threshold)]
            out = str(tmp_path / f"got_{chunk}_{threshold}.fasta")
            stats = {}
            rr.recruit_file(unit, read_fn, out, threshold, chunk_bytes=chunk, stats=stats)
            got = open(out, "rb").read()
            assert len(got) == want["bytes"] and hashlib.sha256(got).hexdigest() == want["sha256"], (chunk, threshold)
            assert stats["fallback"] is None and stats["records"] == len(reads)
            assert stats["chunks"] >= (2 if chunk < 1 << 16 else 1)


def _fuzz_reads(rng, unit):
    reads = []
    for i in range(60):
        kind = i % 5
        if kind == 0:
            s = _rnd(rng, int(rng.integers(0, 400))) + _mutate(rng, unit, 0.08) + _rnd(rng, int(rng.integers(0, 400)))
        elif kind == 1:  # longer than SEGMENT, the unit near a segment boundary
            s = _rnd(rng, 8192 - int(rng.integers(0, 200))) + _mutate(rng, unit, 0.05) + _rnd(rng, int(rng.integers(0, 20000)))
        elif kind == 2:
            s = _rnd(rng, int(rng.integers(0, 30)))
        else:
            s = _rnd(rng, int(rng.integers(100, 3000)))
        reads.append((f"r{i}" + (" desc" if i % 3 else ""), s))
    # exact copies, so that threshold 0 keeps reads too: one inside a short read, one across the first segment boundary
    from centroflye_b200.read_recruitment import reverse_complement
    reads.append(("exact", _rnd(rng, 50) + unit + _rnd(rng, 70)))
    reads.append(("exact_rc across", _rnd(rng, 8192 - len(unit) // 2) + reverse_complement(unit) + _rnd(rng, 9000)))
    reads.append(("empty", ""))
    return reads


def _fuzz_files(tmp_path, rng, reads):
    fq = "".join(f"@{n}\n{s}\n+\n{'#' * len(s)}\n" for n, s in reads).encode()
    fa = "".join(f">{n}\r\n" + "\r\n".join(s[i:i + 61] for i in range(0, len(s), 61)) + "\r\n" for n, s in reads).encode()
    files = {}
    for name, data in (("fastq", fq), ("fasta", fa)):
        files[name] = str(tmp_path / f"reads.{name}")
        open(files[name], "wb").write(data)
    files["fastq.gz"] = str(tmp_path / "reads.fastq.gz")
    with gzip.open(files["fastq.gz"], "wb") as f:
        f.write(fq)
    # several gzip members and zero padding behind them, as gzip.open reads them
    cut = len(fa) // 3
    files["multi.gz"] = str(tmp_path / "reads.multi.gz")
    with open(files["multi.gz"], "wb") as f:
        f.write(gzip.compress(fa[:cut]) + gzip.compress(fa[cut:]) + b"\0" * 1000)
    return files


def test_fuzz_corpus_equals_in_memory_path(tmp_path):
    from centroflye_b200 import read_recruitment as rr
    rng = np.random.default_rng(11)
    unit = _rnd(rng, 300)
    reads = _fuzz_reads(rng, unit)
    for fmt, path in _fuzz_files(tmp_path, rng, reads).items():
        for threshold in (0, 40, -1):
            want = _in_memory(unit, path, str(tmp_path / "want"), threshold)
            assert want.count(b">") > (0 if threshold == 0 else 10)
            for chunk in (1000, 9000, 50000, 1 << 24):
                out = str(tmp_path / "got")
                stats = {}
                rr.recruit_file(unit, path, out, threshold, chunk_bytes=chunk, stats=stats)
                assert open(out, "rb").read() == want, (fmt, threshold, chunk)
                assert stats["fallback"] is None


def _dir_listing(d):
    return sorted(os.listdir(d))


def test_edge_cases(tmp_path):
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200._lib import CfkError
    good = "ACGTTGCA" * 20
    empty = tmp_path / "empty.fa"
    empty.write_bytes(b"junk only\n\n")
    out = tmp_path / "out.fa"
    for unit in (good, "ACGN", "A" * 4000):  # no records: an empty output, the unit is not checked
        rr.recruit_file(unit, str(empty), str(out), 10)
        assert out.read_bytes() == b""
        out.unlink()
    reads = tmp_path / "reads.fq"
    reads.write_bytes(b"@a\n" + good.encode() + b"\n+\n" + b"I" * len(good) + b"\n")
    before = _dir_listing(tmp_path)
    with pytest.raises(AssertionError):
        rr.recruit_file("ACGN", str(reads), str(out), 10)
    with pytest.raises(CfkError):
        rr.recruit_file("A" * 4000, str(reads), str(out), 10)
    assert _dir_listing(tmp_path) == before  # no output, no temporary file left behind
    # a non-ASCII header: the in-memory path writes the output, byte for byte as before
    utf = tmp_path / "utf.fa"
    utf.write_bytes(">r\xc3\xa9ad x\n".encode("latin-1") + good.encode() + b"\n>b\nTTTT\n")
    stats = {}
    rr.recruit_file(good, str(utf), str(out), 0, stats=stats)
    assert stats["fallback"] is not None
    assert out.read_bytes() == _in_memory(good, str(utf), str(tmp_path / "want"), 0) == ">réad\n".encode() + good.encode() + b"\n"
    # main(): same command line, same file
    unit_fn = tmp_path / "unit.fa"
    unit_fn.write_bytes(b">u\n" + good.encode() + b"\n")
    assert rr.main([str(unit_fn), str(reads), str(out), "3x"]) == 0
    assert out.read_bytes() == b">a\n" + good.encode() + b"\n"


_RSS_CHILD = r"""
import os, resource, sys
sys.path.insert(0, {root!r})
from centroflye_b200 import read_recruitment as rr
stats = {{}}
rr.recruit_file({unit!r}, sys.argv[1], sys.argv[2], 350, chunk_bytes=32 << 20, stats=stats)
print(resource.getrusage(resource.RUSAGE_SELF).ru_maxrss, stats["bases"], stats["chunks"])
"""


def test_memory_does_not_grow_with_the_input(tmp_path):
    """Peak RSS of a >= 512 MiB FASTQ through recruit_file (32 MiB chunks) against the same process on a one-record
    file: at most 256 MiB more."""
    rng = np.random.default_rng(3)
    unit = _rnd(rng, 1500)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    block = b"".join(b"@r%d\n" % i + lut[rng.integers(0, 4, size=20000)].tobytes() + b"\n+\n" + b"I" * 20000 + b"\n"
                     for i in range(64))
    big = tmp_path / "big.fq"
    with open(big, "wb") as f:
        for _ in range((512 << 20) // len(block) + 1):
            f.write(block)
    assert big.stat().st_size >= 512 << 20
    small = tmp_path / "small.fq"
    small.write_bytes(block[:block.index(b"@r1\n")])
    code = _RSS_CHILD.format(root=ROOT, unit=unit)
    rss = {}
    for name, path in (("small", small), ("big", big)):
        res = subprocess.run([sys.executable, "-c", code, str(path), str(tmp_path / f"{name}.out")], capture_output=True,
                             text=True, check=True)
        kib, bases, chunks = map(int, res.stdout.split()[-3:])
        rss[name] = kib << 10
        if name == "big":
            assert bases >= 256 << 20 and chunks >= 16
    print(f"peak RSS: one record {rss['small'] >> 20} MiB, {big.stat().st_size >> 20} MiB FASTQ {rss['big'] >> 20} MiB")
    assert rss["big"] - rss["small"] <= 256 << 20
