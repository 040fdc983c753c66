"""rr for units of more than 3328 bases: cfk_rr_filter_long (rr_filter_warp_kernel<W>, one warp per segment and strand,
W words of the unit per lane) and the host paths that select it by unit length.

The reference is the whole-read DP of test_gpu_read_recruitment._infix_distance, as in test_gpu_rr_decisions.  Checked:
* on the host: cfk_rr_long_words at the limits of every W, the entry point's argument checks, build_long_masks'
  lane-minor layout, the streaming form's long_units switch, and the segment plan of a run with a long unit (its step, 16-byte aligned starts, the overlap bound m + t - 1
  restated against whole-read decisions);
* exact distances on both strands at the first and last unit length of every W, with the bottom word on a lane boundary
  and at m = 0, 1, 63 (mod 64), for reads shorter than the wavefront (32 bases), than the unit, of 0 and 1 bases, and with
  N and lowercase bytes; and at the word classes of rr_filter_kernel<NW>, against that kernel;
* keep decisions of recruit(), recruit_file and recruit_file_units (mixed with a short unit, one worker and three) for
  the DXZ1 and D6Z1 dimers, a 34-monomer HOR with reads from its simulated array and a random unit near 32768 bases, with
  hits one base before a segment boundary, at thresholds d - 1, d and d + 1, from FASTA, FASTQ and gzip FASTQ;
* rr.py and rr_multi.py on a long unit."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_read_recruitment import _mutate, _rnd
from test_gpu_rr_decisions import (WORD_CLASS_LIMITS, _Case, _class_corpus, _distances, _expected, _formats, _keep, _n_seg,
                                   _planted, _Segments, _whole_reads_on_device)

gpu = pytest.mark.gpu

# unit length -> W of rr_filter_warp_kernel<W> (cfk_rr_long_words): the first and last length of every W
LONG_WORDS = {1: 2, 3328: 2, 3329: 2, 4096: 2, 4097: 4, 8192: 4, 8193: 8, 16384: 8, 16385: 16, 32768: 16}
# exact distances: the limits of every W above 3328, the bottom word first (5121: word 80 of W = 4 opens lane 20) and
# last (5376) in its lane, and m = 0, 1, 63 (mod 64)
EXACT_UNITS = sorted(set(LONG_WORDS) - {1, 3328} | {5121, 5376, 6400, 6401, 6463})


# ---- 1. on the host -----------------------------------------------------------------------------------------------------

def test_long_word_classes():
    from centroflye_b200 import _lib
    lib = _lib.load()
    assert {m: lib.cfk_rr_long_words(m) for m in LONG_WORDS} == LONG_WORDS
    assert [lib.cfk_rr_long_words(m) for m in (0, -1, 32769, 1 << 30)] == [-1] * 4
    assert [lib.cfk_rr_words(m) for m in (3328, 3329)] == [52, -1]  # the short kernels keep their limit


def test_filter_long_argument_validation():
    """cfk_rr_filter_long checks every unit length and the sizes before any CUDA call (so this runs without a GPU)."""
    from centroflye_b200 import _lib
    _lib.load()

    def call(n_seg, unit_m, n_units=None, text=None):
        m = (ctypes.c_int32 * max(1, len(unit_m)))(*unit_m)
        t = (ctypes.c_int32 * max(1, len(unit_m)))(*([5] * len(unit_m)))
        _lib.call("cfk_rr_filter_long", text, None, None, None, n_seg, len(unit_m) if n_units is None else n_units,
                  None, None, m, t, 1, None, None, None)

    for unit_m in ([0], [100, 32769], [40000, 5], [-1]):
        with pytest.raises(_lib.CfkError, match="1..32768"):
            call(10, unit_m)
    with pytest.raises(_lib.CfkError, match="1..32768"):
        call(0, [5, 0])  # checked even when there is nothing to filter
    for n_seg, n_units in ((-1, None), (1 << 30, None), (10, -1)):
        with pytest.raises(_lib.CfkError, match="bad sizes"):
            call(n_seg, [5], n_units)
    with pytest.raises(_lib.CfkError, match="bad sizes"):
        _lib.call("cfk_rr_filter_long", None, None, None, None, 10, 2, None, None, None, None, 0, None, None, None)
    with pytest.raises(_lib.CfkError, match="16-byte aligned"):
        call(10, [5], text=8)
    call(0, [1, 3328, 3329, 32768])  # valid and empty: nothing is launched
    call(10, [])


def test_long_masks_are_the_short_layout_lane_minor():
    """build_long_masks: entry [strand][symbol][k][lane] is word lane * W + k of cfk_rr_filter's layout, the words past
    the unit are zero; build_masks keeps its layout and its 3328-base limit."""
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200._lib import CfkError
    rng = np.random.default_rng(5)
    for m in (1, 3328, 3329, 4097, 9000, 32768):
        unit = _rnd(rng, m)
        peq, sym_of, w = rr.build_long_masks(unit)
        assert peq.shape == (2, 8, w, 32) and w == LONG_WORDS[min(k for k in LONG_WORDS if k >= m)]
        assert rr.is_long(unit) == (m > 3328)
        flat, want_sym = rr._masks(unit, 32 * w)[:2]
        nw = -(-m // 64)
        assert np.array_equal(sym_of, want_sym)
        for lane in range(32):
            for k in range(w):
                assert np.array_equal(peq[:, :, k, lane], flat[:, :, lane * w + k])
        assert flat[:, :, :nw].any(axis=(0, 1)).all() and not flat[:, :, nw:].any()
        if m <= 3328:
            short, short_sym, short_nw = rr.build_masks(unit)
            assert np.array_equal(short, flat[:, :, :short_nw]) and np.array_equal(short_sym, sym_of)
        else:
            with pytest.raises(CfkError, match="1..3328"):
                rr.build_masks(unit)
    for bad in ("", "A" * 32769):
        with pytest.raises(CfkError, match="1..32768"):
            rr.build_long_masks(bad)


def test_streaming_form_takes_long_units_on_request(tmp_path):
    """recruit_file and recruit_file_units keep refusing a unit of more than 3328 bases unless long_units is set (the
    command lines set it); past 32768 bases they refuse it either way.  The check comes before any output or device
    work, so this runs without a GPU."""
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200._lib import CfkError
    reads = tmp_path / "reads.fa"
    reads.write_bytes(b">a\nACGTTGCA\n")
    out = str(tmp_path / "out.fa")
    long_unit = _rnd(np.random.default_rng(1), 4110)
    with pytest.raises(CfkError, match="long_units"):
        rr.recruit_file(long_unit, str(reads), out, 10)
    with pytest.raises(CfkError, match="long_units"):
        rr.recruit_file_units([("ACGT", out, 1), (long_unit, out + "2", 10)], str(reads))
    with pytest.raises(CfkError, match="1..32768"):
        rr.recruit_file("A" * 32769, str(reads), out, 10, long_units=True)
    assert sorted(os.listdir(tmp_path)) == ["reads.fa"]


def test_long_plan_step_and_alignment(monkeypatch):
    """_segment_plan: without a long unit, recruit()'s restated plan at SEGMENT; with one, the step is the overlap
    rounded up to 16 when that exceeds SEGMENT, every segment starts on a 16-byte boundary of its read, consecutive
    segments overlap by the overlap, and together they cover the read."""
    from centroflye_b200 import read_recruitment as rr
    rng = np.random.default_rng(3)
    lens = np.concatenate([[0, 1, 15, 16, 8192, 40000, 65536], rng.integers(0, 200000, 200)]).astype(np.int64)
    for segment in (64, 8192):
        monkeypatch.setattr(rr, "SEGMENT", segment)
        for overlap in (3330, 8191, 8193, 32768 + 350, 32768 + 3276):
            n_seg, _, start, _ = rr._segment_plan(lens, overlap, False)
            assert np.array_equal(n_seg, _n_seg(lens, overlap, segment))
            assert np.array_equal(start % segment, np.zeros_like(start))
            n_seg, seg_read, start, seg_len = rr._segment_plan(lens, overlap, True)
            step = max(segment, -(-overlap // 16) * 16)
            assert np.array_equal(n_seg, _n_seg(lens, overlap, step)) and np.all(start % 16 == 0)
            assert np.all(seg_len <= step + overlap) and np.all(seg_len >= 0)
            ends = start + seg_len
            first = np.cumsum(n_seg) - n_seg
            assert np.all(start[first] == 0) and np.all(ends[np.cumsum(n_seg) - 1] == lens)
            inner = np.setdiff1d(np.arange(seg_read.size), first)
            assert np.all(ends[inner - 1] - start[inner] >= overlap)


_LONG_PLAN = (3335, 5)  # (m, t): rr.SEGMENT = 64 leaves the step at ceil16(m + t) = 3344 for every threshold <= t + 3


def test_long_overlap_bound_on_the_host():
    """The plan of a long unit restated with step ceil16(m + t): overlaps m + th - 1 and m + th reproduce every
    whole-read decision, m + th - 2 loses a planted copy."""
    m, t = _LONG_PLAN
    step = -(-(m + t) // 16) * 16
    c = _Case(m, t, step)
    assert t in c.thresholds and max(c.thresholds) == t
    dist = _distances(c.unit, c.seqs)
    segs = _Segments(c.unit, c.seqs, step, m + min(c.thresholds) - 2, m + t)
    for threshold in c.thresholds:
        want = _keep(dist, threshold)
        for o in (m + threshold - 1, m + threshold):
            got = segs.keep(o, threshold)
            assert np.array_equal(got, want), (threshold, o, [c.reads[r][0] for r in np.flatnonzero(got != want)])
        short = segs.keep(m + threshold - 2, threshold)
        assert not (short & ~want).any()
        if threshold == t:
            assert (want & ~short).any(), "no planted copy needs its whole span"
    assert _n_seg(segs.lens, m + t, step).max() >= 4


# ---- 2. exact distances ---------------------------------------------------------------------------------------------------

def _exact_corpus(m):
    """A seeded unit of m bases and reads: a mutated copy in a random flank, two thirds of the reverse complement with
    Ns and a lowercase stretch, the unit's first half, reads of 0, 1, 5 and 31 bases (inside the pipeline fill)."""
    from centroflye_b200.read_recruitment import reverse_complement
    rng = np.random.default_rng(m + 11)
    unit = _rnd(rng, m)
    rc = reverse_complement(unit)[m // 3:]
    h = len(rc) // 2
    reads = [_rnd(rng, 20) + _mutate(rng, unit, 0.03) + _rnd(rng, 40),
             rc[:h] + "NNNNN" + rc[h + 5:h + 60].lower() + rc[h + 60:] + "N" * 7,
             unit[:m // 2], "", "A", _rnd(rng, 5), _rnd(rng, 31)]
    return unit, reads


def _filter_long(eng, units, thresholds, reads, exact):
    """cfk_rr_filter_long over whole reads for every unit -> (keep bool[U, R], out_dist int32[U, R, 2])."""
    import torch
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    masks = [rr.build_long_masks(u)[:2] for u in units]  # also for units the short kernels take
    d_text, d_off, d_len, d_order = _whole_reads_on_device(eng, reads)
    d_peq = eng._to_dev(np.concatenate([p.reshape(-1) for p, _ in masks]).view(np.int64))
    d_sym = eng._to_dev(np.concatenate([s for _, s in masks]))
    unit_m = np.array([len(u) for u in units], dtype=np.int32)
    unit_t = np.array(thresholds, dtype=np.int32)
    R, U, p = len(reads), len(units), eng._p
    d_keep, d_dist = eng._zeros(U * R, torch.uint8), eng._zeros(2 * U * R, torch.int32)
    _lib.call("cfk_rr_filter_long", p(d_text), p(d_off), p(d_len), p(d_order), R, U, p(d_peq), p(d_sym),
              unit_m.ctypes.data, unit_t.ctypes.data, int(exact), p(d_dist), p(d_keep), eng._stream())
    return (d_keep[:U * R].cpu().numpy().reshape(U, R).astype(bool),
            d_dist[:2 * U * R].cpu().numpy().reshape(U, R, 2))


@gpu
@pytest.mark.parametrize("m", EXACT_UNITS)
def test_exact_distances_long(m):
    from centroflye_b200 import read_recruitment as rr
    unit, reads = _exact_corpus(m)
    want = _distances(unit, reads)
    threshold = max(3, m // 50)
    keep, dist = rr.recruit(unit, reads, threshold, exact=True)
    assert np.array_equal(dist, want), (m, dist.tolist(), want.tolist())
    assert np.array_equal(keep, _keep(want, threshold))
    assert np.array_equal(rr.recruit(unit, reads, threshold), keep)  # the early exit decides alike
    assert want[2, 0] == m - m // 2 and want[3].tolist() == [m, m] and want[0, 0] > 0


@gpu
def test_long_kernel_equals_short_kernel_at_the_word_classes():
    """Both kernels on the units of every class limit of rr_filter_kernel<NW> in one launch of each: equal exact
    distances; without exact, equal keep bits and equal out_dist (both stop after the same 16 characters)."""
    import torch
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200.engine import default_engine
    eng = default_engine()
    units, reads = [], []
    for m in sorted(WORD_CLASS_LIMITS):
        unit, rs = _class_corpus(m)
        units.append(unit)
        reads += rs
    reads += ["", "C", _rnd(np.random.default_rng(1), 17)]
    p, R = eng._p, len(reads)
    d_text, d_off, d_len, d_order = _whole_reads_on_device(eng, reads)
    for exact in (1, 0):
        th = [max(3, len(u) // 50) for u in units]
        keep_l, dist_l = _filter_long(eng, units, th, reads, exact)
        for i, unit in enumerate(units):
            peq, sym_of, _ = rr.build_masks(unit)
            d_peq, d_sym = eng._to_dev(peq.reshape(-1).view(np.int64)), eng._to_dev(sym_of)
            d_keep, d_dist = eng._zeros(R, torch.uint8), eng._zeros(2 * R, torch.int32)
            _lib.call("cfk_rr_filter", p(d_text), p(d_off), p(d_len), p(d_order), R, p(d_peq), p(d_sym), len(unit), th[i],
                      exact, p(d_dist), p(d_keep), eng._stream())
            assert np.array_equal(dist_l[i], d_dist[:2 * R].cpu().numpy().reshape(R, 2)), (len(unit), exact)
            assert np.array_equal(keep_l[i], d_keep[:R].cpu().numpy().astype(bool)), (len(unit), exact)
        assert keep_l.sum() >= len(units)


# ---- 3. keep decisions of long units --------------------------------------------------------------------------------------

def _t_plant(m):
    """Insertions of the planted copies: 6 for the unit near 32768, so that m + t - 1 .. m + t + 1 round up to one step."""
    return 6 if m > 32000 else 20


def _units():
    """name -> (unit, genome codes of its array or None)."""
    from centroflye_b200 import synth
    out = {}
    for name, genome in (("dxz1_dimer", "cenx_dxz1_m1500_s1"), ("d6z1_dimer", "cen6_d6z1_m1000_s4")):
        g, a0, alen, unit = synth.load_genome(genome)
        out[name] = (unit + unit, g[a0:a0 + alen])
    hor = synth.hor_unit(34, 171, 0.25, seed=34)
    g, a0, alen = synth.simulate_genome(hor, 8, 0.02, 35, flank_len=3000)
    out["hor34"] = (hor, g[a0 - 2000:a0 + alen + 2000])
    out["random32752"] = (_rnd(np.random.default_rng(32752), 32752), None)  # m + 5 .. m + 7 round up to 32768
    return out


_CORPORA = {}


def _corpus(name):
    """(unit, [(read name, sequence)], thresholds): copies with exactly _t_plant(m) insertions one base before the first
    (and second) segment boundary of the plan and on one, reads from the unit's array, a mutated copy, reads shorter
    than the unit, of 0, 1 and 30 bases, N and lowercase; thresholds d - 1, d, d + 1 around the planted and mutated
    copies' distances."""
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200.synth import codes_to_ascii
    if name in _CORPORA:
        return _CORPORA[name]
    unit, array = _units()[name]
    m = len(unit)
    rng = np.random.default_rng([m, 7])
    rc = rr.reverse_complement(unit)
    t = _t_plant(m)
    step = max(rr.SEGMENT, -(-(m + t + 1) // 16) * 16)  # the plan's step at thresholds t - 1 .. t + 1
    reads = [("before_boundary_1", _rnd(rng, step - 1) + _planted(rng, unit, t) + _rnd(rng, 100)),
             ("mutated_rc", _rnd(rng, 50) + _mutate(rng, rc, 0.04) + _rnd(rng, 70)),
             ("empty", ""), ("one", "G"), ("tiny", _rnd(rng, 30))]
    if m < 32000:
        h = m // 2
        reads += [("short_unit", unit[:m - 40]),
                  ("before_boundary_2_rc", _rnd(rng, 2 * step - 1) + _planted(rng, rc, t) + _rnd(rng, 10)),
                  ("on_boundary", _rnd(rng, step) + _planted(rng, unit, t)),
                  ("n_lower", _rnd(rng, 10) + unit[:h] + "NN" + unit[h + 2:h + 30].lower() + unit[h + 30:] + "n" * 5),
                  ("random", _rnd(rng, 5000))]
    if array is not None:
        for i in range(3):
            a = int(rng.integers(0, max(1, array.size - m - 3000)))
            reads.append((f"array_{i}", _mutate(rng, codes_to_ascii(array[a:a + m + 3000]), 0.02)))
    dist = _distances(unit, [s for _, s in reads]).min(axis=1)
    near = [d for (n, _), d in zip(reads, dist.tolist()) if n.startswith(("before", "on_", "mutated", "array"))]
    thresholds = sorted({x for d in near for x in (d - 1, d, d + 1) if 0 <= x <= max(near)} | {t - 1, t})
    _CORPORA[name] = (unit, reads, thresholds)
    return _CORPORA[name]


LONG_UNITS = ["dxz1_dimer", "d6z1_dimer", "hor34", "random32752"]


@gpu
@pytest.mark.parametrize("name", LONG_UNITS)
def test_recruit_long_decisions_equal_whole_read_dp(name):
    from centroflye_b200 import read_recruitment as rr
    unit, reads, thresholds = _corpus(name)
    seqs = [s for _, s in reads]
    dist = _distances(unit, seqs)
    assert rr.is_long(unit) and len(unit) == {"dxz1_dimer": 4110, "d6z1_dimer": 6444, "hor34": 5814}.get(name, 32752)
    for threshold in thresholds + [-1]:
        got = rr.recruit(unit, seqs, threshold)
        assert np.array_equal(got, _keep(dist, threshold)), (name, threshold, [reads[r][0] for r in np.flatnonzero(got != _keep(dist, threshold))])
    keep, exact = rr.recruit(unit, seqs, thresholds[0], exact=True)
    assert np.array_equal(exact, dist)
    kept = [_keep(dist, th).sum() for th in thresholds]
    assert kept[0] < kept[-1]  # the thresholds straddle decisions


def _file_jobs(names):
    """Reads of the named corpora (names prefixed) and jobs: every unit at the planted copies' distance and at its
    largest threshold, DXZ1 (2055 bases, the short kernels) at 300, one job that keeps every read."""
    from centroflye_b200 import synth
    reads, jobs = [], []
    for name in names:
        unit, rs, thresholds = _corpus(name)
        reads += [(f"{name}_{n}", s) for n, s in rs]
        jobs += [(unit, _t_plant(len(unit))), (unit, thresholds[-1])]
    dxz1 = synth.load_genome("cenx_dxz1_m1500_s1")[3]
    jobs += [(dxz1, 300), (dxz1, -1)]
    return reads, jobs


@gpu
@pytest.mark.parametrize("names", [["dxz1_dimer", "d6z1_dimer", "hor34"], ["random32752"]], ids=["hor", "random32752"])
def test_long_output_files_equal_whole_read_dp(tmp_path, names):
    from centroflye_b200 import read_recruitment as rr
    reads, jobs = _file_jobs(names)
    seqs = [s for _, s in reads]
    want = [_expected(reads, _keep(_distances(u, seqs), th)) for u, th in jobs]
    assert all(w.count(b">") >= 1 for w in want[:-2]) and want[-1].count(b">") == len(reads)
    for fmt, path in _formats(tmp_path, reads).items():
        for chunk in (20000, 1 << 24):  # 20000 bytes: less than one record for the long reads
            where = f"{fmt}_{chunk}"
            for i, (unit, th) in enumerate(jobs[:2]):
                out = str(tmp_path / f"{where}_single{i}.fa")
                stats = {}
                rr.recruit_file(unit, path, out, th, chunk_bytes=chunk, stats=stats, long_units=True)
                assert stats["fallback"] is None
                assert open(out, "rb").read() == want[i], (where, len(unit), th)
            for devices in (None, [0, 0, 0]):
                outs = [str(tmp_path / f"{where}_{devices is not None}_{i}.fa") for i in range(len(jobs))]
                stats = {}
                rr.recruit_file_units([(u, o, th) for (u, th), o in zip(jobs, outs)], path, chunk_bytes=chunk,
                                      stats=stats, devices=devices, long_units=True)
                assert stats["fallback"] is None
                for i, (o, (unit, th)) in enumerate(zip(outs, jobs)):
                    assert open(o, "rb").read() == want[i], (where, devices, len(unit), th)


@gpu
def test_command_lines_take_long_units(tmp_path):
    reads, jobs = _file_jobs(["dxz1_dimer", "hor34"])
    seqs = [s for _, s in reads]
    read_fn = _formats(tmp_path, reads)["fastq.gz"]
    unit_fns = []
    for i, (unit, _) in enumerate(jobs):
        unit_fns.append(str(tmp_path / f"unit{i}.fa"))
        with open(unit_fns[-1], "w") as f:
            f.write(f">u{i} x\n" + "".join(unit[k:k + 70] + "\n" for k in range(0, len(unit), 70)))
    want = [_expected(reads, _keep(_distances(u, seqs), th)) for u, th in jobs]
    out = str(tmp_path / "rr.fa")
    subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "rr.py"), unit_fns[0], read_fn, out, str(jobs[0][1])],
                   check=True)
    assert open(out, "rb").read() == want[0]
    argv = [read_fn]
    outs = [str(tmp_path / f"multi{i}.fa") for i in range(len(jobs))]
    for fn, o, (_, th) in zip(unit_fns, outs, jobs):
        argv += [fn, o, str(th)]
    subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "rr_multi.py")] + argv, check=True)
    assert [open(o, "rb").read() for o in outs] == want
