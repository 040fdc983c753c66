"""rr_multi on several devices (read_recruitment.recruit_file_units(devices=...), rr_multi.py --gpus N): every chunk's
records are dealt out in contiguous ranges (_split_records), one worker per device, and every output is byte for byte
what the one-device run writes.  Repeated entries ([0, 0, 0]) are separate workers on one GPU, so the dealing, the
rebasing of each range and the ordering of the parts are tested on a single GPU; with two or more visible GPUs the
comparisons are repeated across devices."""
import hashlib
import json
import subprocess
import sys
import threading

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_read_recruitment import FORMATS, RR_GOLDEN, THRESHOLDS, _mutate, _rnd, write_inputs
from test_gpu_rr_stream import _fuzz_files, _fuzz_reads
from test_gpu_rr_units import _dir_listing, _units_of_every_class

gpu = pytest.mark.gpu


# ---- the range split (no GPU) ----------------------------------------------------------------------------------------

def _check_split(seq_len, n):
    from centroflye_b200.read_recruitment import _split_records
    seq_len = np.asarray(seq_len, dtype=np.int64)
    R = len(seq_len)
    b = _split_records(seq_len, n)
    assert b.shape == (n + 1,) and b[0] == 0 and b[-1] == R
    assert np.all(np.diff(b) >= 0)  # contiguous ranges in order: every record exactly once
    if R >= n:
        assert np.all(np.diff(b) >= 1), (seq_len.tolist(), n, b.tolist())
    else:
        assert np.count_nonzero(np.diff(b)) == R
    if R:
        sums = np.add.reduceat(np.append(seq_len, 0), b[:-1])[:n] * (np.diff(b) > 0)
        assert np.all(np.abs(sums - seq_len.sum() / n) <= seq_len.max()), (seq_len.tolist(), n, b.tolist())
    return b


def test_split_records_limits():
    for n in (1, 2, 3, 8):
        assert _check_split([], n).tolist() == [0] * (n + 1)
    assert _check_split([5, 7, 9], 1).tolist() == [0, 3]
    assert _check_split([5, 7], 4).tolist() == [0, 1, 2, 2, 2]
    assert _check_split([10] * 8, 4).tolist() == [0, 2, 4, 6, 8]
    assert _check_split([0] * 5, 3).tolist() == [0, 1, 2, 5]  # no bases: every range still gets a record
    _check_split([1, 1000, 1, 1], 4)
    _check_split([100000, 3, 3, 3, 3, 3], 3)  # one record longer than the others together
    _check_split([3, 3, 3, 3, 3, 100000], 3)
    _check_split([0, 0, 50, 0, 0], 2)


def test_split_records_random():
    rng = np.random.default_rng(8)
    for _ in range(3000):
        R = int(rng.integers(0, 40))
        kind = rng.integers(0, 3)
        if kind == 0:
            seq_len = rng.integers(0, 50, size=R)
        elif kind == 1:  # log-normal, like real read lengths
            seq_len = rng.lognormal(9, 1.2, size=R).astype(np.int64)
        else:  # a few huge records among short ones, and empty ones
            seq_len = np.where(rng.random(R) < 0.1, rng.integers(10 ** 5, 10 ** 6, size=R), rng.integers(0, 3, size=R))
        _check_split(seq_len, int(rng.integers(1, 10)))


# ---- --gpus (no GPU) --------------------------------------------------------------------------------------------------

def test_gpus_option(tmp_path, monkeypatch, capsys):
    import torch
    from centroflye_b200 import read_recruitment as rr
    unit_fn = tmp_path / "u.fa"
    unit_fn.write_bytes(b">u\nACGTACGTTT\n")
    calls = []
    monkeypatch.setattr(rr, "recruit_file_units", lambda jobs, reads, **kw: calls.append((jobs, reads, kw)) or 0)
    triple = [str(unit_fn), str(tmp_path / "o.fa"), "3"]
    monkeypatch.setattr(torch.cuda, "device_count", lambda: 4)
    assert rr.main_units(["r.fq"] + triple) == 0
    assert rr.main_units(["--gpus", "3", "r.fq"] + triple + triple[:2] + ["x"]) == 0
    assert rr.main_units(["--gpus", "4", "r.fq"] + triple) == 0
    assert [kw["devices"] for _, _, kw in calls] == [None, [0, 1, 2], [0, 1, 2, 3]]
    assert calls[1][0] == [("ACGTACGTTT", triple[1], 3), ("ACGTACGTTT", triple[1], 0)] and calls[1][1] == "r.fq"
    capsys.readouterr()
    bad_n = [["--gpus", n, "r.fq"] + triple for n in ("0", "-1", "x", "1.5", "", "5")]  # 5: more than visible
    bad_count = [["--gpus"], ["--gpus", "2"], ["--gpus", "2", "r.fq"] + triple[:2],
                 ["--gpus", "2", "r.fq"] + triple + ["v.fa"], ["--gpus", "2"] + triple, ["r.fq", "--gpus", "2"] + triple]
    for argv in bad_n + bad_count:
        assert rr.main_units(argv) == 2, argv
        out = capsys.readouterr()
        assert out.out == "" and out.err.startswith("Usage: rr_multi.py reads") and "--gpus N" in out.err, argv
    assert len(calls) == 3


def test_gpus_option_beyond_the_visible_devices(tmp_path):
    """The real device count (0 here when no GPU is visible): one more is refused by the script itself."""
    import torch
    script = f"{ROOT}/scripts/rr_multi.py"
    argv = ["--gpus", str(torch.cuda.device_count() + 1), "r.fq", "u.fa", "o.fa", "3"]
    res = subprocess.run([sys.executable, script] + argv, capture_output=True, text=True)
    assert res.returncode == 2 and res.stdout == "" and res.stderr.startswith("Usage: rr_multi.py reads")
    assert not (tmp_path / "o.fa").exists()


# ---- one GPU, repeated entries ----------------------------------------------------------------------------------------

def _rr_threads():
    return [t.name for t in threading.enumerate() if t.name.startswith("rr-")]


def _compare(jobs, read_fn, chunk, devices):
    """recruit_file_units with `devices` against devices=None -> the outputs (bytes per job) and the stats."""
    from centroflye_b200 import read_recruitment as rr
    one = [(u, p + ".one", t) for u, p, t in jobs]
    rr.recruit_file_units(one, read_fn, chunk_bytes=chunk)
    stats = {}
    assert rr.recruit_file_units(jobs, read_fn, chunk_bytes=chunk, stats=stats, devices=devices) == 0
    got = [open(p, "rb").read() for _, p, _ in jobs]
    assert got == [open(p, "rb").read() for _, p, _ in one], (read_fn, chunk, devices)
    assert stats["fallback"] is None and stats["devices"] == len(devices)
    assert stats["job_out_bytes"] == [len(out) for out in got] and stats["out_bytes"] == sum(map(len, got))
    per = stats["device_s_per_device"]
    assert len(per) == len(devices)
    for name, total in stats["device_s"].items():
        assert total == pytest.approx(sum(d.get(name, 0.0) for d in per))
    assert _rr_threads() == []
    return got, stats


def _goldens(tmp_path, devices):
    from centroflye_b200 import read_recruitment as rr
    for fmt in FORMATS:
        with open(RR_GOLDEN) as f:
            golden = json.load(f)[fmt]
        unit_fn, read_fn, reads, _ = write_inputs(str(tmp_path), fmt)
        unit = next(rr.read_sequences(unit_fn))[1]
        for chunk in (700, 5000, 1 << 16, 1 << 26):
            jobs = [(unit, str(tmp_path / f"got_{fmt}_{chunk}_{t}.fasta"), t) for t in THRESHOLDS]
            got, stats = _compare(jobs, read_fn, chunk, devices)
            assert stats["records"] == len(reads)
            for t, out in zip(THRESHOLDS, got):
                want = golden["outputs"][str(t)]
                assert len(out) == want["bytes"] and hashlib.sha256(out).hexdigest() == want["sha256"], (fmt, chunk, t)


def _fuzz(tmp_path, devices):
    """The corpus of test_gpu_rr_units.test_mixed_units_equal_single_runs (seed 21): 15 units of every word class."""
    from centroflye_b200 import read_recruitment as rr
    rng = np.random.default_rng(21)
    units = _units_of_every_class(rng)
    reads = _fuzz_reads(rng, units[0][1])
    for name, unit in units:
        reads.append((f"{name}_mut", _rnd(rng, 200) + _mutate(rng, unit, 0.05) + _rnd(rng, 300)))
        reads.append((f"{name}_rc", _rnd(rng, 8100) + _mutate(rng, rr.reverse_complement(unit), 0.03) + _rnd(rng, 500)))
        reads.append((f"{name}_exact", _rnd(rng, 30) + unit + _rnd(rng, 30)))
    thresholds = [350, 500, 0, -1, 120, 200, 60, 0, 150, 0, 6, -1, 30, 60, 0]
    for fmt, path in _fuzz_files(tmp_path, rng, reads).items():
        for chunk in (2000, 16 << 20):
            jobs = [(unit, str(tmp_path / f"{fmt}_{chunk}_{name}.fa"), t) for (name, unit), t in zip(units, thresholds)]
            got, stats = _compare(jobs, path, chunk, devices)
            assert stats["records"] == len(reads)
            for (name, _), t, out in zip(units, thresholds, got):
                if t >= 0:
                    assert f">{name}_exact\n".encode() in out, (fmt, chunk, name)


@gpu
def test_goldens_on_repeated_devices(tmp_path):
    _goldens(tmp_path, [0, 0, 0])


@gpu
def test_fuzz_corpus_on_repeated_devices(tmp_path):
    _fuzz(tmp_path, [0, 0, 0])


@gpu
def test_edge_cases_on_repeated_devices(tmp_path):
    from centroflye_b200 import read_recruitment as rr
    rng = np.random.default_rng(4)
    unit = _rnd(rng, 400)
    # records longer than the chunk: every chunk holds one record, so two of the three workers get empty ranges
    seqs = [_rnd(rng, 3000) + _mutate(rng, unit, 0.05) + _rnd(rng, 2000) if i % 2 else _rnd(rng, 6000) for i in range(6)]
    big = tmp_path / "big.fq"
    big.write_bytes(b"".join(b"@b%d\n%s\n+\n%s\n" % (i, s.encode(), b"I" * len(s)) for i, s in enumerate(seqs)))
    jobs = [(unit, str(tmp_path / "big50.fa"), 50), (unit, str(tmp_path / "big_all.fa"), -1)]
    got, stats = _compare(jobs, str(big), 4000, [0, 0, 0])
    assert stats["chunks"] == stats["records"] == 6 and got[0].count(b">") == 3 and got[1].count(b">") == 6
    # one record in the whole file
    one = tmp_path / "one.fa"
    one.write_bytes(b">only\n" + seqs[1].encode() + b"\n")
    got, stats = _compare([(unit, str(tmp_path / "one.out"), 50)], str(one), 1 << 20, [0, 0, 0])
    assert stats["records"] == 1 and got[0].startswith(b">only\n")
    # every threshold -1: no filter runs, every read is kept
    got, stats = _compare([(unit, str(tmp_path / "all1.fa"), -1), ("ACGT", str(tmp_path / "all2.fa"), -1)],
                          str(big), 9000, [0, 0, 0])
    assert got[0] == got[1] and got[0].count(b">") == 6
    # no records: empty outputs, no unit checked, no device touched
    empty = tmp_path / "empty.fa"
    empty.write_bytes(b"junk only\n\n")
    outs = [str(tmp_path / f"e{i}.fa") for i in range(2)]
    stats = {}
    rr.recruit_file_units([(unit, outs[0], 10), ("A" * 4000, outs[1], 3)], str(empty), stats=stats, devices=[0, 0, 0])
    assert [open(p, "rb").read() for p in outs] == [b"", b""]
    assert stats["devices"] == 3 and stats["device_s_per_device"] == [{}, {}, {}] and stats["chunks"] == 0
    assert _rr_threads() == []
    with pytest.raises(ValueError):
        rr.recruit_file_units([(unit, outs[0], 1)], str(big), devices=[])


@gpu
def test_failures_leave_nothing_behind(tmp_path, monkeypatch):
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200._lib import CfkError
    unit_fn, read_fn, _, _ = write_inputs(str(tmp_path), "fastq")
    unit = next(rr.read_sequences(unit_fn))[1]
    outs = [str(tmp_path / f"out{i}.fa") for i in range(3)]
    before = _dir_listing(tmp_path)
    for bad, error in (("ACGN", AssertionError), ("A" * 4000, CfkError)):
        with pytest.raises(error):
            rr.recruit_file_units([(unit, outs[0], 10), (bad, outs[1], 10), (unit, outs[2], -1)], read_fn,
                                  chunk_bytes=5000, devices=[0, 0])
        assert _dir_listing(tmp_path) == before and _rr_threads() == []
    step = rr._Worker.step
    calls = []

    def failing_step(self, *args):
        calls.append(self.index)
        if self.index == 1 and calls.count(1) == 3:
            raise RuntimeError("injected into worker 1")
        return step(self, *args)

    monkeypatch.setattr(rr._Worker, "step", failing_step)
    with pytest.raises(RuntimeError, match="injected into worker 1"):
        rr.recruit_file_units([(unit, outs[0], 350), (unit, outs[1], -1)], read_fn, chunk_bytes=5000, devices=[0, 0])
    assert calls.count(1) == 3 and calls.count(0) >= 3
    assert _dir_listing(tmp_path) == before and _rr_threads() == []


_RSS_CHILD = r"""
import os, resource, sys
sys.path.insert(0, {root!r})
from centroflye_b200 import read_recruitment as rr
stats = {{}}
jobs = [(u, sys.argv[2] + str(i), 350) for i, u in enumerate({units!r})]
rr.recruit_file_units(jobs, sys.argv[1], chunk_bytes=32 << 20, stats=stats, devices=[0, 0])
print(resource.getrusage(resource.RUSAGE_SELF).ru_maxrss, stats["bases"], stats["chunks"], min(stats["job_out_bytes"]))
"""


@gpu
def test_memory_on_two_workers(tmp_path):
    """test_gpu_rr_units.test_memory_does_not_grow_with_the_input with devices=[0, 0]: the workers' buffers follow
    their ranges, so peak RSS over a >= 512 MiB FASTQ stays within 256 MiB of a one-record file, as for one device."""
    rng = np.random.default_rng(3)
    units = [_rnd(rng, m) for m in (1500, 700, 2000, 300)]
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = []
    for i in range(64):
        s = lut[rng.integers(0, 4, size=20000)].tobytes()
        if i % 8 < 4:
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
    print(f"peak RSS, four jobs, two workers: one record {rss['small'] >> 20} MiB, {big.stat().st_size >> 20} MiB FASTQ "
          f"{rss['big'] >> 20} MiB")
    assert rss["big"] - rss["small"] <= 256 << 20


# ---- several GPUs -----------------------------------------------------------------------------------------------------

def _all_devices():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"{n} GPU visible; the dealing itself is covered on one GPU by the repeated-device tests")
    return list(range(n))


@gpu
def test_goldens_on_all_devices(tmp_path):
    _goldens(tmp_path, _all_devices())


@gpu
def test_fuzz_corpus_on_all_devices(tmp_path):
    _fuzz(tmp_path, _all_devices())
