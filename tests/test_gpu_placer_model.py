"""Row f rank 2, the read placer (read_placer.py + csrc/placer.cu), against ``py_oracle.PlacerModel``: the greedy loop
restated over plain dicts and sets of k-mer strings.

The restatement first checks itself, with no GPU, against read_positions_<tag>.csv that the unmodified reference wrote
for the three golden reports.  The device then runs against it where the goldens never go: tie-breaks at every level
and across blocks of placer_best_kernel, min_cloud_kmer_freq 0..3, the initial pair list of a later call, score
tables that overflow partway through a call, reads of 2^16 - 1 units and contig positions past 2^24."""
import contextlib
import io
import json
import os
import random

import numpy as np
import pytest

from conftest import golden_cases
from oracle import py_oracle

VARIANTS = ("default", "loose")


def _split(lines):
    placed = [ln for ln in lines if not ln.endswith(" None")]
    return placed, sorted(ln for ln in lines if ln.endswith(" None"))


def golden_inputs(g, tag):
    """(params, prefix, internal, suffix, clouds) of ReadPlacer.run on golden case `g`, rebuilt on the CPU."""
    from centroflye_b200.encode import ints_to_kmers
    from centroflye_b200.ncrf_parser import NCRF_Report
    with open(os.path.join(g.dir, f"read_positions_{tag}.json")) as f:
        v = json.load(f)
    selected = set(ints_to_kmers(np.load(os.path.join(g.dir, "p0.npz"))["selected"], v["k_cloud"]))
    rep = NCRF_Report(g.report_path)
    clouds = py_oracle.filter_clouds(py_oracle.reads_kmer_clouds(rep.records, v["n_motif"], v["k_cloud"], selected),
                                     min_mult=v["min_kmer_mult"])
    prefix, internal, suffix = rep.classify(large_threshold=v["prefix_threshold"])
    return v, prefix, internal, suffix, clouds


# which level of the selection rule decided the picks of each golden file (see the docstring below)
_decided = {}


@pytest.mark.parametrize("case", golden_cases())
@pytest.mark.parametrize("tag", VARIANTS)
def test_restatement_reproduces_reference_files(golden, case, tag):
    """The restatement writes what the unmodified reference wrote: placed lines in order, `None` lines as a set.

    What the goldens reach, by which level of the rule decided each pick (`test_golden_tie_break_counts`): only
    dxz1_small places reads beyond its 3 prefix reads (31 picks in each variant: 60 decided by (distinct positions,
    total), one by the larger offset, one without a rival); d6z1_noisy and rand311 place none.  The smaller-r_id level
    is never reached, min_cloud_kmer_freq is only 1 or 2, and min_prop only 3.  Those rules are restated from the
    documentation of read_placer.py and placer.cu, without the reference to confirm them; the device tests below hold
    the kernels to them."""
    g = golden(case)
    v, prefix, internal, suffix, clouds = golden_inputs(g, tag)
    model = py_oracle.place_reads(prefix, internal, suffix, clouds, v["min_cloud_kmer_freq"], v["min_unit"],
                                  v["min_inters"])
    want = open(os.path.join(g.dir, f"read_positions_{tag}.csv")).read().splitlines()
    assert _split(model.lines) == _split(want)
    _decided[(case, tag)] = dict(model.decided)


def test_golden_tie_break_counts(golden):
    """Keeps the counts quoted above true."""
    total = {}
    for case in golden_cases():
        for tag in VARIANTS:
            if (case, tag) not in _decided:
                v, prefix, internal, suffix, clouds = golden_inputs(golden(case), tag)
                _decided[(case, tag)] = dict(py_oracle.place_reads(prefix, internal, suffix, clouds,
                                                                   v["min_cloud_kmer_freq"], v["min_unit"],
                                                                   v["min_inters"]).decided)
            for level, n in _decided[(case, tag)].items():
                total[level] = total.get(level, 0) + n
    assert total == {"score": 60, "offset": 1, "alone": 1}


# ---- the device against the restatement ------------------------------------------------------------------------
class _Cloud:
    """What the placer reads of a foreign cloud object: ``.kmers``, one iterable of k-mer strings per unit."""

    def __init__(self, kmers):
        self.kmers = kmers


class _Clouds(dict):
    """A foreign ``r_id -> cloud`` dict (not a CloudDict): the placer converts it once through state_from_sets."""


def _kmer_pool(n, k, seed):
    rng = random.Random(seed)
    out = set()
    while len(out) < n:
        out.add("".join(rng.choice("ACGT") for _ in range(k)))
    return sorted(out)


def _placer(tmp_path, min_freq):
    """A ReadPlacer without a report: what add_prefix_reads / add_reads need, and nothing else."""
    import argparse
    from centroflye_b200.read_placer import CloudContig, ReadPlacer
    pl = ReadPlacer.__new__(ReadPlacer)
    pl.params = argparse.Namespace(min_cloud_kmer_freq=min_freq)
    pl.cloud_contig = CloudContig(min_freq)
    pl.position_outfile = str(tmp_path / "read_positions.csv")
    return pl


def _run(tmp_path, clouds, prefix, calls, min_freq):
    """Runs prefix -> every (reads, min_unit, min_inters, min_prop) of `calls` on the device and on the restatement;
    compares the files and the contigs' host state.  Returns (placer, model, lines)."""
    pl = _placer(tmp_path, min_freq)
    dev_clouds = _Clouds((r, _Cloud(u)) for r, u in clouds.items())
    model = py_oracle.PlacerModel(min_freq)
    with contextlib.redirect_stdout(io.StringIO()):
        pl.add_prefix_reads(prefix, dev_clouds)
        for reads, min_unit, min_inters, min_prop in calls:
            pl.add_reads(reads, dev_clouds, min_unit, min_inters, min_prop)
    model.add_prefix_reads(prefix, clouds)
    for reads, min_unit, min_inters, min_prop in calls:
        model.add_reads(reads, clouds, min_unit, min_inters, min_prop)
    lines = open(pl.position_outfile).read().splitlines()
    assert _split(lines) == _split(model.lines)
    cc = pl.cloud_contig
    assert cc.read_positions == model.contig.read_positions
    assert dict(cc.coverage) == dict(model.contig.coverage)
    assert cc.max_pos == model.contig.max_pos
    return pl, model, lines


def fuzz_case(seed, n_reads, G, n_universe, width=(0, 3)):
    """A true contig of G positions whose clouds (`width` bounds their sizes) come from `n_universe` k-mers, so k-mers
    repeat at many positions and scores tie, and reads r0, r1, ... (string order is not record order) of four kinds:
    windows of it with k-mers and whole clouds dropped, decoys whose k-mers are never on the contig, and reads of zero
    units.  Prefix reads are windows at position 0, suffix reads mostly windows at the end."""
    rng = random.Random(seed)
    pool = _kmer_pool(n_universe + 12, 11, seed)
    universe, decoy = pool[:n_universe], pool[n_universe:]
    truth = [rng.sample(universe, rng.randint(*width)) for _ in range(G)]

    def window(s, n):
        return [{kmer for kmer in truth[p] if rng.random() > 0.25} if p < G and rng.random() > 0.1 else set()
                for p in range(s, s + n)]

    clouds, prefix, internal, suffix = {}, [], [], []
    for i in range(n_reads):
        r_id = f"r{i}"
        x = rng.random()
        n = rng.randint(1, 40)
        if i % 3 == 0 and len(prefix) < max(3, n_reads // 25):
            clouds[r_id] = window(0, n)
            prefix.append(r_id)
            continue
        if x < 0.04:
            clouds[r_id] = []
        elif x < 0.1:
            clouds[r_id] = [set(rng.sample(decoy, rng.randint(0, 3))) for _ in range(rng.randint(1, 12))]
        elif x < 0.2:
            clouds[r_id] = window(max(G - n + rng.randint(0, 5), 0), n)
            suffix.append(r_id)
            continue
        else:
            clouds[r_id] = window(rng.randint(0, G - 1), n)
        (suffix if rng.random() < 0.1 else internal).append(r_id)
    return clouds, prefix, internal, suffix


FUZZ = [  # seed, reads, contig length, k-mer universe, min_cloud_kmer_freq, min_prop, min_unit, min_inters
    (1, 6, 30, 6, 0, 1, 1, 1),
    (2, 20, 60, 8, 1, 3, 1, 3),
    (3, 60, 100, 10, 2, 1, 2, 4),
    (4, 150, 150, 12, 3, 1, 1, 2),
    (5, 400, 200, 16, 1, 3, 2, 6),
    (6, 800, 300, 40, 2, 3, 2, 8),
    (7, 2000, 400, 40, 1, 1, 3, 6),
    (8, 2000, 400, 60, 0, 3, 2, 10),
]


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n_reads,G,n_universe,min_freq,min_prop,min_unit,min_inters", FUZZ)
def test_fuzz_matches_restatement(tmp_path, seed, n_reads, G, n_universe, min_freq, min_prop, min_unit, min_inters):
    # min_prop 3 needs three hits per unit on average: wider clouds
    clouds, prefix, internal, suffix = fuzz_case(seed, n_reads, G, n_universe, (0, 3) if min_prop == 1 else (3, 7))
    _, model, lines = _run(tmp_path, clouds, prefix, [(internal, min_unit, min_inters, min_prop),
                                                      (suffix, min_unit, min_inters, min_prop)], min_freq)
    placed = [ln for ln in lines[len(prefix):] if not ln.endswith(" None")]
    assert placed


def _mix64(x):
    m = (1 << 64) - 1
    x ^= x >> 33
    x = (x * 0xff51afd7ed558ccd) & m
    x ^= x >> 33
    x = (x * 0xc4ceb9fe1a85ec53) & m
    return x ^ (x >> 33)


@pytest.mark.gpu
@pytest.mark.parametrize("min_freq", [1, 2])
def test_ties_by_construction(tmp_path, min_freq):
    """Identical clouds under different r_ids (the smaller string wins: r10 before r9), a periodic read scoring
    equally at ten offsets (the largest wins), and 300 tied reads whose (read, offset) slots fall in different blocks
    of placer_best_kernel -- decoy reads with many entries make the score table span all of its blocks."""
    uniq = _kmer_pool(48 + 2 + 80 * 6, 11, 99)
    a, (p, q), pad = uniq[:48], uniq[48:50], uniq[50:]
    contig = [{a[i]} for i in range(20)] + [{p} if i % 2 == 0 else {q} for i in range(20)] + [{a[20 + i]} for i in range(8)]
    clouds = {"P1": contig, "P2": [set(c) for c in contig]}  # two copies: every contig pair reaches count 2
    clouds["r10"] = [{a[3]}, {a[4]}, {a[5]}]
    clouds["r9"] = [{a[3]}, {a[4]}, {a[5]}]
    clouds["periodic"] = [{p}, {q}]
    tied = [f"t{i}" for i in range(300)]
    for r_id in tied:
        clouds[r_id] = [{a[20]}, {a[21]}, {a[22]}]  # contig positions 40..42
    decoys = [f"d{i}" for i in range(80)]
    for i, r_id in enumerate(decoys):
        clouds[r_id] = [set(pad[6 * i:6 * i + 6])] * 40  # 240 entries each, never on the contig
    internal = ["r9", "periodic", "r10"] + tied[::-1] + decoys
    pl, model, lines = _run(tmp_path, clouds, ["P1", "P2"], [(internal, 1, 1, 1)], min_freq)
    assert lines[2:] == ([f"{r} 40 3 3" for r in sorted(tied)] + ["r10 3 3 3", "r9 3 3 3", "periodic 38 2 2"]
                         + [f"{r} None" for r in decoys])
    assert model.decided["r_id"] >= 300 and model.decided["offset"] >= 1
    # the tied winners' home slots in the score table, as the device hashes them
    n_sel = sum(len(u) for r in internal for u in clouds[r])
    cap2 = max(1 << 14, 4 * n_sel)
    index = {r: i for i, r in enumerate(clouds)}
    blocks = {((_mix64((index[r] << 32) | 40) * cap2) >> 64) // 256 % 296 for r in tied}
    assert cap2 > 296 * 256 and len(blocks) > 100


@pytest.mark.gpu
def test_score_tables_overflow_partway_and_restore(tmp_path, monkeypatch):
    """One k-mer in every unit makes the (read, offset, position) triples grow quadratically with the contig.  Each
    read, placed at offset 0, extends the contig by 8 positions, so the triple set outgrows cap1 = 16 x entries only
    after some reads were placed: the call restores the contig it started from and repeats itself with larger tables.
    It happens in the internal call (from the prefix contig) and in the suffix call (from a contig that already holds
    every internal read, with the suffix reads' k-mer on its first 8 positions only)."""
    from centroflye_b200.read_placer import ReadPlacer
    K, K2 = _kmer_pool(2, 11, 7)
    clouds = {"P": [{K, K2}] * 8}
    internal = [f"a{i:02d}" for i in range(40)]
    suffix = [f"b{i:02d}" for i in range(30)]
    for i, r_id in enumerate(internal):
        clouds[r_id] = [{K}] * (16 + 8 * i)
    for i, r_id in enumerate(suffix):
        clouds[r_id] = [{K2}] * (16 + 8 * i)
    once = ReadPlacer._add_reads_once
    log = []

    def recording(self, reads, state, min_unit, min_inters, min_prop, grow):
        before = len(self.cloud_contig.read_positions)
        out = once(self, reads, state, min_unit, min_inters, min_prop, grow)
        log.append((reads[0][0], grow, out is None, len(self.cloud_contig.read_positions) - before))
        return out
    monkeypatch.setattr(ReadPlacer, "_add_reads_once", recording)
    _, model, lines = _run(tmp_path, clouds, ["P"], [(internal, 1, 1, 1), (suffix, 1, 1, 1)], 1)
    assert lines == (["P 0"] + [f"{r} 0 {8 + 8 * i} {8 + 8 * i}" for i, r in enumerate(internal)]
                     + [f"{r} 0 {8 + 8 * i} {8 + 8 * i}" for i, r in enumerate(suffix)])
    for call in "ab":
        failed = [e for e in log if e[0] == call and e[2]]
        assert failed and all(e[3] > 0 for e in failed), log  # overflowed after placing reads
        assert [e[1] for e in log if e[0] == call][-1] > 1 and not [e for e in log if e[0] == call][-1][2]


EMPTY = ()


@pytest.mark.gpu
def test_read_of_65535_units(tmp_path):
    """The last position a read can have, 2^16 - 2, in the triple key; one more unit is refused."""
    from centroflye_b200._lib import CfkError
    A, B, C = _kmer_pool(3, 11, 5)
    clouds = {"P": [EMPTY] * 65534 + [{A}],
              "L": [EMPTY] * 65534 + [{A}],
              "M": [{A}, {B}],
              "N": [{B}] + [EMPTY] * 65533 + [{C}]}
    _, _, lines = _run(tmp_path, clouds, ["P"], [(["L", "M", "N"], 1, 1, 1)], 1)
    assert lines == ["P 0", "M 65534 1 1", "N 65535 1 1", "L 0 1 1"]
    big = _Clouds({"P": _Cloud([{A}]), "X": _Cloud([{A}] + [EMPTY] * 65535)})
    pl = _placer(tmp_path, 1)
    with contextlib.redirect_stdout(io.StringIO()):
        pl.add_prefix_reads(["P"], big)
        with pytest.raises(CfkError):
            pl.add_reads(["X"], big, 1, 1, 1)


CHAIN = 257  # reads of 65535 units, each placed 65534 positions after the previous one: the last reaches past 2^24


@pytest.mark.gpu
def test_offsets_past_2_to_24(tmp_path):
    """Offsets of 2^24 and more.  A chain of 257 reads of 65535 mostly empty units, each sharing one k-mer with the
    previous read's last unit, drives the contig past 2^24.  Then read A (state index r) scores at offset 2^24 + 5 and
    read B (state index r + 1) at offset 5, both at position 1 in the read: packing (read, offset, position) as
    read << 40 | offset << 16 | position gives both triples one key, and one read loses its only distinct position."""
    pool = _kmer_pool(CHAIN + 3, 11, 11)
    links, Ka, Kb = pool[:CHAIN + 1], pool[CHAIN + 1], pool[CHAIN + 2]
    clouds = {}
    for i in range(CHAIN):
        units = [EMPTY] * 65535
        units[0], units[65534] = {links[i]}, {links[i + 1]}
        clouds[f"c{i:03d}"] = units
    clouds["c000"][6] = {Kb}              # contig position 6
    clouds[f"c{CHAIN - 1:03d}"][518] = {Ka}  # contig position 256 * 65534 + 518 = 2^24 + 6
    clouds["A"] = [EMPTY, {Ka}]
    clouds["B"] = [EMPTY, {Kb}]
    chain = [f"c{i:03d}" for i in range(1, CHAIN)]
    _, model, lines = _run(tmp_path, clouds, ["c000"], [(chain, 1, 1, 1), (["A", "B"], 1, 1, 1)], 1)
    assert list(clouds).index("B") == list(clouds).index("A") + 1
    assert model.scores[("A", (1 << 24) + 5)] == [1, 1] and model.scores[("B", 5)] == [1, 1]
    assert lines[-2:] == [f"A {(1 << 24) + 5} 1 1", "B 5 1 1"]
    assert model.contig.max_pos == CHAIN * 65534


def _synthetic_report(path):
    """A few hundred reads of a 150-copy HOR array with 4 kb flanks (so prefix and suffix classes are non-empty), and
    the k-mers that occur once in the array."""
    from collections import Counter
    from centroflye_b200 import synth
    unit = synth.hor_unit(4, 60, 0.25, seed=21)
    genome, a0, alen = synth.simulate_genome(unit, 150, 0.03, 22, flank_len=4000)
    reads = synth.simulate_reads(genome, a0, alen, unit, 60, 0.02, 23, median_len=7000, sigma=0.4, min_len=5200,
                                 max_len=20000)
    synth.write_ncrf_report(str(path), reads, unit)
    array = synth._SYM[genome[a0:a0 + alen]].tobytes().decode("ascii")
    counts = Counter(array[i:i + 19] for i in range(len(array) - 18))
    return {kmer for kmer, c in counts.items() if c == 1}


@pytest.mark.gpu
def test_end_to_end_synthetic_report(tmp_path):
    """ReadPlacer.run() on a synthetic report in both golden variants against the restatement over py_oracle clouds;
    once, the same classes through a foreign dict of those clouds write the same file as the device clouds."""
    import argparse
    from centroflye_b200.ncrf_parser import NCRF_Report
    from centroflye_b200.read_placer import ReadPlacer
    from oracle.make_placer_golden import VARIANTS as PARAMS
    report = tmp_path / "report.ncrf"
    genomic = _synthetic_report(report)
    kfn = tmp_path / "kmers.txt"
    kfn.write_text("".join(kmer + "\n" for kmer in sorted(genomic)))
    rep = NCRF_Report(str(report))
    assert len(rep.records) >= 200
    for tag in VARIANTS:
        v = PARAMS[tag]
        params = argparse.Namespace(ncrf=str(report), genomic_kmers=str(kfn), k_cloud=19, outdir=str(tmp_path / tag), **v)
        with contextlib.redirect_stdout(io.StringIO()):
            placer = ReadPlacer(params)
            placer.run()
        got = open(os.path.join(params.outdir, "read_positions.csv")).read()
        clouds = py_oracle.filter_clouds(py_oracle.reads_kmer_clouds(rep.records, 1, 19, genomic),
                                         min_mult=v["min_kmer_mult"])
        prefix, internal, suffix = rep.classify(large_threshold=v["prefix_threshold"])
        assert prefix and internal and suffix
        model = py_oracle.place_reads(prefix, internal, suffix, clouds, v["min_cloud_kmer_freq"], v["min_unit"],
                                      v["min_inters"])
        assert _split(got.splitlines()) == _split(model.lines)
        assert placer.cloud_contig.read_positions == model.contig.read_positions
        assert dict(placer.cloud_contig.coverage) == dict(model.contig.coverage)
        assert placer.cloud_contig.max_pos == model.contig.max_pos
        assert sum(not ln.endswith(" None") for ln in model.lines) > len(prefix) + 10
        if tag == "default":
            foreign = _Clouds((r, _Cloud(u)) for r, u in clouds.items())
            pl = _placer(tmp_path, v["min_cloud_kmer_freq"])
            with contextlib.redirect_stdout(io.StringIO()):
                pl.add_prefix_reads(prefix, foreign)
                pl.add_reads(internal, foreign, v["min_unit"], v["min_inters"])
                pl.add_reads(suffix, foreign, v["min_unit"], v["min_inters"])
            assert open(pl.position_outfile).read() == got
