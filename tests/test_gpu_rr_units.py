"""rr for several units in one pass over the read file (read_recruitment.recruit_file_units, cfk_rr_filter_units):
every output equals what rr writes for that job alone -- the reference binary's outputs (tests/golden/rr/outputs.json)
and recruit_file on a fuzz corpus with units of every word class -- plus the edge cases of the run, the command line,
the entry point against cfk_rr_filter, and memory that does not grow with the input."""
import ctypes
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_read_recruitment import FORMATS, RR_GOLDEN, THRESHOLDS, _mutate, _rnd, write_inputs
from test_gpu_rr_stream import _fuzz_files, _fuzz_reads

gpu = pytest.mark.gpu


def _units_of_every_class(rng):
    """(name, unit): DXZ1, D6Z1, cenx_like_u2..u8 and random units of 1, 63, 65, 300, 600 and 1100 bases -- every
    word class of rr_filter_kernel (4, 9, 17, 33, 52 words)."""
    from centroflye_b200 import synth
    units = [("dxz1", synth.load_genome("cenx_dxz1_m1500_s1")[3]), ("d6z1", synth.load_genome("cen6_d6z1_m1000_s4")[3])]
    units += [(f"u{i}", synth.load_genome(f"cenx_like_u{i}_m1500_s{i}")[3]) for i in range(2, 9)]
    units += [(f"rnd{m}", _rnd(rng, m)) for m in (1, 63, 65, 300, 600, 1100)]
    return units


def _run_single(jobs, read_fn, chunk):
    from centroflye_b200 import read_recruitment as rr
    out = []
    for unit, path, threshold in jobs:
        rr.recruit_file(unit, read_fn, path + ".single", threshold, chunk_bytes=chunk)
        out.append(open(path + ".single", "rb").read())
    return out


@gpu
@pytest.mark.parametrize("fmt", FORMATS)
def test_goldens_in_one_pass(tmp_path, fmt):
    from centroflye_b200 import read_recruitment as rr
    with open(RR_GOLDEN) as f:
        golden = json.load(f)[fmt]
    unit_fn, read_fn, reads, _ = write_inputs(str(tmp_path), fmt)
    unit = next(rr.read_sequences(unit_fn))[1]
    for chunk in (700, 5000, 1 << 16, 1 << 26):
        jobs = [(unit, str(tmp_path / f"got_{chunk}_{t}.fasta"), t) for t in THRESHOLDS]
        stats = {}
        assert rr.recruit_file_units(jobs, read_fn, chunk_bytes=chunk, stats=stats) == 0
        assert stats["fallback"] is None and stats["records"] == len(reads)
        for (_, path, threshold), n in zip(jobs, stats["job_out_bytes"]):
            want = golden["outputs"][str(threshold)]
            got = open(path, "rb").read()
            assert [ln[1:].decode() for ln in got.split(b"\n") if ln.startswith(b">")] == want["kept"], (chunk, threshold)
            assert len(got) == want["bytes"] == n and hashlib.sha256(got).hexdigest() == want["sha256"], (chunk, threshold)


@gpu
def test_mixed_units_equal_single_runs(tmp_path):
    from centroflye_b200 import read_recruitment as rr
    rng = np.random.default_rng(21)
    units = _units_of_every_class(rng)
    assert sorted({int(rr._lib.load().cfk_rr_words(len(u))) for _, u in units}) == [4, 9, 17, 33, 52]
    reads = _fuzz_reads(rng, units[0][1])
    for name, unit in units:  # mutated copies of every unit, and an exact copy for threshold 0
        reads.append((f"{name}_mut", _rnd(rng, 200) + _mutate(rng, unit, 0.05) + _rnd(rng, 300)))
        reads.append((f"{name}_rc", _rnd(rng, 8100) + _mutate(rng, rr.reverse_complement(unit), 0.03) + _rnd(rng, 500)))
        reads.append((f"{name}_exact", _rnd(rng, 30) + unit + _rnd(rng, 30)))
    thresholds = [350, 500, 0, -1, 120, 200, 60, 0, 150, 0, 6, -1, 30, 60, 0]
    assert len(thresholds) == len(units)
    for fmt, path in _fuzz_files(tmp_path, rng, reads).items():
        for chunk in (2000, 1 << 24):  # 2000 bytes: smaller than most records
            jobs = [(unit, str(tmp_path / f"{fmt}_{chunk}_{name}.fa"), t) for (name, unit), t in zip(units, thresholds)]
            stats = {}
            rr.recruit_file_units(jobs, path, chunk_bytes=chunk, stats=stats)
            assert stats["fallback"] is None
            got = [open(p, "rb").read() for _, p, _ in jobs]
            assert got == _run_single(jobs, path, chunk), (fmt, chunk)
            # every filtered unit keeps its own exact copy, so a mix-up of units between blocks cannot pass
            for ((name, _), t, out) in zip(units, thresholds, got):
                if t >= 0:
                    assert f">{name}_exact\n".encode() in out, (fmt, chunk, name)
            filtered = [out for t, out in zip(thresholds, got) if t >= 0]
            assert len(set(filtered)) == len(filtered)


@gpu
def test_repeated_jobs(tmp_path):
    from centroflye_b200 import read_recruitment as rr
    unit_fn, read_fn, _, _ = write_inputs(str(tmp_path), "fastq")
    unit = next(rr.read_sequences(unit_fn))[1]
    jobs = [(unit, str(tmp_path / "a.fa"), 100), (unit, str(tmp_path / "b.fa"), 700), (unit, str(tmp_path / "c.fa"), 350),
            (unit, str(tmp_path / "d.fa"), 350)]
    rr.recruit_file_units(jobs, read_fn, chunk_bytes=5000)
    got = [open(p, "rb").read() for _, p, _ in jobs]
    assert got == _run_single(jobs, read_fn, 5000)
    assert got[0] != got[1] and got[2] == got[3]


def _dir_listing(d):
    return sorted(os.listdir(d))


@gpu
def test_edge_cases(tmp_path):
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200._lib import CfkError
    good = "ACGTTGCA" * 20
    empty = tmp_path / "empty.fa"
    empty.write_bytes(b"junk only\n\n")
    outs = [str(tmp_path / f"out{i}.fa") for i in range(3)]
    # no records: empty outputs, no unit is checked
    rr.recruit_file_units(list(zip((good, "ACGN", "A" * 4000), outs, (10, 0, -1))), str(empty))
    assert [open(p, "rb").read() for p in outs] == [b""] * 3
    for p in outs:
        os.remove(p)
    reads = tmp_path / "reads.fq"
    reads.write_bytes(b"@a\n" + good.encode() + b"\n+\n" + b"I" * len(good) + b"\n")
    before = _dir_listing(tmp_path)
    for bad, error in (("ACGN", AssertionError), ("A" * 4000, CfkError)):
        with pytest.raises(error):
            rr.recruit_file_units([(good, outs[0], 10), (bad, outs[1], 10), (good, outs[2], -1)], str(reads))
        assert _dir_listing(tmp_path) == before  # no output, no temporary file left behind
    # non-ASCII: the in-memory path writes every output, byte for byte as a single run
    utf = tmp_path / "utf.fa"
    utf.write_bytes(">r\xc3\xa9ad x\n".encode("latin-1") + good.encode() + b"\n>b\nTTTT\n")
    jobs = [(good, outs[0], 0), (good[:40], outs[1], 2), ("TTTT", outs[2], -1)]
    stats = {}
    rr.recruit_file_units(jobs, str(utf), stats=stats)
    assert stats["fallback"] is not None
    got = [open(p, "rb").read() for _, p, _ in jobs]
    assert got == _run_single(jobs, str(utf), 1 << 26)
    assert got[0] == ">réad\n".encode() + good.encode() + b"\n" and got[2].count(b">") == 2
    # the command line: one triple per job
    unit_fn = tmp_path / "unit.fa"
    unit_fn.write_bytes(b">u\n" + good.encode() + b"\n")
    other_fn = tmp_path / "other.fa"
    other_fn.write_bytes(b">v some\nGGGGGGGGGGGG\n>w\nACGT\n")
    assert rr.main_units([str(reads), str(unit_fn), outs[0], "3x", str(other_fn), outs[1], "2"]) == 0
    assert open(outs[0], "rb").read() == b">a\n" + good.encode() + b"\n"
    assert open(outs[1], "rb").read() == b""


def test_job_list_is_checked_first(tmp_path):
    """Zero jobs and two jobs with one output file (after realpath) raise ValueError before anything is read."""
    from centroflye_b200 import read_recruitment as rr
    missing = str(tmp_path / "no_such_reads.fq")
    with pytest.raises(ValueError):
        rr.recruit_file_units([], missing)
    os.symlink(str(tmp_path), str(tmp_path / "link"))
    with pytest.raises(ValueError):
        rr.recruit_file_units([("ACGT", str(tmp_path / "o.fa"), 1), ("ACGT", str(tmp_path / "link" / "o.fa"), 2)], missing)
    with pytest.raises(ValueError):
        rr.recruit_file_units([("ACGT", "o.fa", 1), ("ACGT", os.path.join(os.getcwd(), "o.fa"), 2)], missing)
    assert _dir_listing(tmp_path) == ["link"]


@pytest.mark.parametrize("argv", [[], ["r.fq"], ["r.fq", "u.fa", "o.fa"], ["r.fq", "u.fa", "o.fa", "3", "v.fa"],
                                  ["r.fq", "u.fa", "o.fa", "3", "v.fa", "p.fa"]])
def test_command_line_usage(argv):
    script = os.path.join(ROOT, "scripts", "rr_multi.py")
    res = subprocess.run([sys.executable, script] + argv, capture_output=True, text=True)
    assert res.returncode == 2 and res.stdout == "" and res.stderr.startswith("Usage: rr_multi.py reads")


def test_filter_units_argument_validation():
    """cfk_rr_filter_units checks every unit length and the sizes before any CUDA call (so this runs without a GPU)."""
    from centroflye_b200 import _lib
    _lib.load()

    def call(n_seg, unit_m, n_units=None):
        m = (ctypes.c_int32 * max(1, len(unit_m)))(*unit_m)
        t = (ctypes.c_int32 * max(1, len(unit_m)))(*([5] * len(unit_m)))
        _lib.call("cfk_rr_filter_units", None, None, None, None, n_seg, len(unit_m) if n_units is None else n_units,
                  None, None, m, t, None, None)

    for unit_m in ([0], [100, 3329], [4000, 5], [-1]):
        with pytest.raises(_lib.CfkError, match="1..3328"):
            call(10, unit_m)
    with pytest.raises(_lib.CfkError, match="1..3328"):
        call(0, [5, 0])  # checked even when there is nothing to filter
    with pytest.raises(_lib.CfkError, match="bad sizes"):
        call(-1, [5])
    with pytest.raises(_lib.CfkError, match="bad sizes"):
        call(10, [5], n_units=-1)
    with pytest.raises(_lib.CfkError, match="bad sizes"):
        _lib.call("cfk_rr_filter_units", None, None, None, None, 10, 2, None, None, None, None, None, None)
    call(0, [1, 3328, 64, 65])  # valid and empty: nothing is launched
    call(10, [])


@gpu
def test_filter_units_equals_filter_per_unit():
    """cfk_rr_filter_units against cfk_rr_filter once per unit on the same segments, for units of three word classes
    and more units of one class than one launch takes (64)."""
    import torch
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200.engine import default_engine
    eng = default_engine()
    rng = np.random.default_rng(5)
    units = [_rnd(rng, int(m)) for m in rng.integers(1, 257, size=70)] + [_rnd(rng, 500), _rnd(rng, 2000)]
    thresholds = [int(t) for t in rng.integers(-1, 20, size=len(units))]
    reads = []
    for i in range(400):
        u = units[i % len(units)]
        core = _mutate(rng, u if i % 2 else rr.reverse_complement(u), 0.05)
        reads.append(_rnd(rng, int(rng.integers(0, 300))) + core + _rnd(rng, int(rng.integers(0, 300))))
    lens = np.array([len(s) for s in reads], dtype=np.int64)
    offs = np.zeros(len(reads), dtype=np.int64)
    np.cumsum(((lens + 15) & ~15)[:-1], out=offs[1:])
    text = np.zeros(int(offs[-1] + lens[-1]) + 32, dtype=np.uint8)
    for o, s in zip(offs.tolist(), reads):
        text[o:o + len(s)] = np.frombuffer(s.encode(), dtype=np.uint8)
    order = np.argsort(-lens, kind="stable").astype(np.int32)
    d_text, d_off, d_len, d_order = (eng._to_dev(a) for a in (text, offs, lens, order))
    masks = [rr.build_masks(u) for u in units]
    R, U, p, st = len(reads), len(units), eng._p, eng._stream()
    want = np.zeros((U, R), dtype=np.uint8)
    for u, (unit, (peq, sym_of, _)) in enumerate(zip(units, masks)):
        d_keep = eng._zeros(R, torch.uint8)
        d_peq, d_sym = eng._to_dev(peq.reshape(-1).view(np.int64)), eng._to_dev(sym_of)
        _lib.call("cfk_rr_filter", p(d_text), p(d_off), p(d_len), p(d_order), R, p(d_peq), p(d_sym), len(unit),
                  thresholds[u], 0, None, p(d_keep), st)
        want[u] = d_keep[:R].cpu().numpy()
    d_peq = eng._to_dev(np.concatenate([peq.reshape(-1) for peq, _, _ in masks]).view(np.int64))
    d_sym = eng._to_dev(np.concatenate([sym_of for _, sym_of, _ in masks]))
    unit_m = np.array([len(u) for u in units], dtype=np.int32)
    unit_t = np.array(thresholds, dtype=np.int32)
    d_keep = eng._zeros(U * R, torch.uint8)
    _lib.call("cfk_rr_filter_units", p(d_text), p(d_off), p(d_len), p(d_order), R, U, p(d_peq), p(d_sym),
              unit_m.ctypes.data, unit_t.ctypes.data, p(d_keep), st)
    got = d_keep[:U * R].cpu().numpy().reshape(U, R)
    assert np.array_equal(got, want)
    assert 0 < want.sum() < want.size and len({row.tobytes() for row in want}) > U // 2


_RSS_CHILD = r"""
import os, resource, sys
sys.path.insert(0, {root!r})
from centroflye_b200 import read_recruitment as rr
stats = {{}}
jobs = [(u, sys.argv[2] + str(i), 350) for i, u in enumerate({units!r})]
rr.recruit_file_units(jobs, sys.argv[1], chunk_bytes=32 << 20, stats=stats)
print(resource.getrusage(resource.RUSAGE_SELF).ru_maxrss, stats["bases"], stats["chunks"], min(stats["job_out_bytes"]))
"""


@gpu
def test_memory_does_not_grow_with_the_input(tmp_path):
    """Peak RSS of a >= 512 MiB FASTQ through recruit_file_units with four jobs (32 MiB chunks) against the same
    process on a one-record file: at most 256 MiB more, as for one job.  Every job keeps an eighth of the reads, so each
    job's output buffers are in use and its output (>= 16 MiB) is far larger than what one chunk gives it."""
    rng = np.random.default_rng(3)
    units = [_rnd(rng, m) for m in (1500, 700, 2000, 300)]
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = []
    for i in range(64):
        s = lut[rng.integers(0, 4, size=20000)].tobytes()
        if i % 8 < 4:  # a copy of unit i % 4
            u = units[i % 4].encode()
            s = s[:5000] + u + s[5000 + len(u):]
        seqs.append(s)
    block = b"".join(b"@r%d\n" % i + s + b"\n+\n" + b"I" * len(s) + b"\n" for i, s in enumerate(seqs))
    big = tmp_path / "big.fq"
    with open(big, "wb") as f:
        for _ in range((512 << 20) // len(block) + 1):
            f.write(block)
    small = tmp_path / "small.fq"
    small.write_bytes(block[:block.index(b"@r1\n")])
    code = _RSS_CHILD.format(root=ROOT, units=units)
    rss = {}
    for name, path in (("small", small), ("big", big)):
        res = subprocess.run([sys.executable, "-c", code, str(path), str(tmp_path / f"{name}.out")], capture_output=True,
                             text=True, check=True)
        kib, bases, chunks, least_out = map(int, res.stdout.split()[-4:])
        rss[name] = kib << 10
        if name == "big":
            assert bases >= 256 << 20 and chunks >= 16 and least_out >= 16 << 20
    print(f"peak RSS, four jobs: one record {rss['small'] >> 20} MiB, {big.stat().st_size >> 20} MiB FASTQ "
          f"{rss['big'] >> 20} MiB")
    assert rss["big"] - rss["small"] <= 256 << 20
