"""rr's keep decisions against exact infix edit distances of whole reads.

The reference is _infix_distance (tests/test_gpu_read_recruitment.py), the row-wise DP of edlib's HW mode, run on whole
reads on the host; every (unit, read) pair is computed once per module, both strands, and reused for every threshold,
path, format and chunk size.  The rule is rr.cpp's: a read is kept iff min(d_unit, d_reverse_complement) <= threshold,
or threshold < 0.  What this checks is what the reference binary's goldens never reach:

* segmentation: a read longer than SEGMENT is cut into segments that overlap by |unit| + threshold and is kept if any
  segment hits.  A hit within t edits spans at most m + t read bases, so the tight overlap is m + t - 1: a hit that
  starts one base before a segment boundary then ends on the last base of the segment.  The seeded corpus plants such
  hits (copies with exactly t interior insertions) before the first, second and fourth boundary and in the last segment,
  and reads whose length makes the segment count change.  On the host, the plan restated in numpy with overlaps m + t - 1
  and m + t reproduces every whole-read decision and m + t - 2 loses a kept read, so the corpus tells a correct overlap
  from a short one.  On the device, recruit(), recruit_file and recruit_file_units (one worker and three) must match the
  whole-read decisions at SEGMENT 8192 and, monkeypatched, at 64, 256 and 1040;
* the word classes of rr_filter_kernel<NW>: exact distances on both strands at the first and last length of every
  class;
* threshold ties on the early-exit path: cfk_rr_filter_units with one unit at thresholds d - 1, d and d + 1, and where
  the scan stops (cfk_rr_filter's out_dist without exact).
Bytes are compared as rr_filter.cu documents: a read byte the unit does not hold ('N', lowercase) matches nothing."""
import gzip

import numpy as np
import pytest

from test_gpu_read_recruitment import _infix_distance, _mutate, _rnd

gpu = pytest.mark.gpu

# (unit length m, planted insertions t, SEGMENT): t small against m, so that a planted copy needs its whole span
CASES = [(65, 5, 64), (65, 5, 256), (65, 5, 8192), (300, 20, 256), (300, 20, 8192), (1100, 30, 1040), (24, 2, 64),
         (24, 2, 8192)]
CASE_IDS = [f"m{m}-t{t}-S{s}" for m, t, s in CASES]
LONG_READ = 1 << 20  # the read of about 1 Mbase, for the shortest unit
# unit length -> words of its class in rr_filter_kernel<NW> (cfk_rr_words): the first and last length of every class
WORD_CLASS_LIMITS = {128: 4, 255: 4, 256: 4, 512: 9, 575: 9, 576: 9, 577: 17, 1087: 17, 1088: 17, 1089: 33, 2111: 33,
                     2112: 33, 2113: 52, 3327: 52, 3328: 52}

# ---- the reference ------------------------------------------------------------------------------------------------------

_DIST = {}  # (unit, read) -> (infix distance of the unit, of its reverse complement)


def _distances(unit, reads):
    """int64[R, 2]: the exact infix distances of the unit and of its reverse complement in every whole read."""
    from centroflye_b200.read_recruitment import reverse_complement
    rc = reverse_complement(unit)
    out = np.empty((len(reads), 2), dtype=np.int64)
    for i, s in enumerate(reads):
        if (unit, s) not in _DIST:
            _DIST[unit, s] = (_infix_distance(unit, s), _infix_distance(rc, s))
        out[i] = _DIST[unit, s]
    return out


def _keep(dist, threshold):
    """rr.cpp's rule on the distances of _distances."""
    return np.ones(len(dist), dtype=bool) if threshold < 0 else dist.min(axis=1) <= threshold


def _end_scores(unit, texts):
    """The last row of _infix_distance's DP for every row of texts (uint8[N, W], padded with zeros, a byte no unit
    holds): out[i, e] is the least edit distance of the unit to an infix of texts[i] that ends at e.  Its running minimum
    at e is the infix distance of texts[i, :e]; columns up to e never read the bytes behind e."""
    n, w = texts.shape
    ar = np.arange(w + 1, dtype=np.int32)
    ne = {c: (texts != c).astype(np.int32) for c in set(unit.encode())}
    prev, cur = np.zeros((n, w + 1), dtype=np.int32), np.empty((n, w + 1), dtype=np.int32)
    for i, c in enumerate(unit.encode()):
        cur[:, 0] = i + 1
        np.minimum(prev[:, :-1] + ne[c], prev[:, 1:] + 1, out=cur[:, 1:])
        cur -= ar
        np.minimum.accumulate(cur, axis=1, out=prev)
        prev += ar
    return prev


def _prefix_minima(unit, texts, width, cells=1 << 22):
    """[np.minimum.accumulate of _end_scores(unit, text[:width])] for every text, in batches of about `cells`."""
    out = []
    rows = max(1, cells // (width + 1))
    for b in range(0, len(texts), rows):
        batch = np.zeros((len(texts[b:b + rows]), width), dtype=np.uint8)
        for i, s in enumerate(texts[b:b + rows]):
            s = s[:width].encode()
            batch[i, :len(s)] = np.frombuffer(s, dtype=np.uint8)
        out.extend(np.minimum.accumulate(_end_scores(unit, batch), axis=1))
    return out


# ---- the segment plan, restated -------------------------------------------------------------------------------------------

def _n_seg(lens, overlap, segment):
    """max(1, ceil(max(len - o, 1) / S)) segments per read; segment j covers [j S, min(j S + S + o, len))."""
    return np.maximum(1, -(-np.maximum(np.asarray(lens, dtype=np.int64) - overlap, 1) // segment))


class _Segments:
    """The infix distance of every segment a plan with overlap in [o_lo, o_hi] can make, both strands: one DP per
    segment start j S of every read over its longest segment, S + o_hi bases; a shorter segment is a prefix of it."""

    def __init__(self, unit, reads, segment, o_lo, o_hi):
        from centroflye_b200.read_recruitment import reverse_complement
        self.segment, self.o_hi = segment, o_hi
        self.lens = np.array([len(s) for s in reads], dtype=np.int64)
        starts = [(r, j * segment) for r, n in enumerate(_n_seg(self.lens, o_lo, segment).tolist()) for j in range(n)]
        texts = [reads[r][a:a + segment + o_hi] for r, a in starts]
        self.at = {key: i for i, key in enumerate(starts)}
        self.minima = [_prefix_minima(u, texts, segment + o_hi) for u in (unit, reverse_complement(unit))]

    def keep(self, overlap, threshold):
        """Per read: does any segment of the plan with this overlap hold the unit within threshold edits?"""
        assert overlap <= self.o_hi
        out = np.zeros(len(self.lens), dtype=bool)
        for r, (n, n_seg) in enumerate(zip(self.lens.tolist(), _n_seg(self.lens, overlap, self.segment).tolist())):
            for j in range(n_seg):
                i, a = self.at[r, j * self.segment], j * self.segment
                end = min(self.segment + overlap, n - a)
                out[r] |= min(self.minima[0][i][end], self.minima[1][i][end]) <= threshold
        return out


# ---- the corpus ---------------------------------------------------------------------------------------------------------

def _planted(rng, core, t):
    """core with exactly t single-base insertions, all in its middle half: edit distance t, span len(core) + t."""
    m = len(core)
    pos = np.sort(rng.integers(m // 4, m - m // 4 + 1, size=t)).tolist()
    parts = [core[a:b] + "ACGT"[int(rng.integers(4))] for a, b in zip([0] + pos[:-1], pos)]
    return "".join(parts) + core[pos[-1] if pos else 0:]


class _Case:
    """The unit of (m, t) (a seeded random unit) and the reads of (m, t, S) as (name, sequence)."""

    def __init__(self, m, t, segment):
        from centroflye_b200.read_recruitment import reverse_complement
        self.m, self.t, self.segment = m, t, segment
        rng = np.random.default_rng([m, t])
        self.unit = _rnd(rng, m)
        strands = (self.unit, reverse_complement(self.unit))
        long_read = _rnd(rng, LONG_READ) if m < 32 else None
        rng = np.random.default_rng([m, t, segment])
        S, span, o = segment, m + t, m + t  # o: recruit()'s overlap at threshold t
        reads, k = [], 0

        def copy():
            nonlocal k
            k += 1
            return _planted(rng, strands[k % 2], t)

        for j in (0, 1, 3):  # the hit starts one base before the boundary after segment j
            reads.append((f"before_boundary_{j}", _rnd(rng, (j + 1) * S - 1) + copy() + _rnd(rng, int(rng.integers(0, S)))))
            reads.append((f"on_boundary_{j} x", _rnd(rng, (j + 1) * S) + copy() + _rnd(rng, int(rng.integers(0, 50)))))
        # the hit ends on the last base: in the last of three segments only, and where the segment count goes 1 -> 2
        reads.append(("last_segment", _rnd(rng, 2 * S + o + int(rng.integers(1, S)) - span) + copy()))
        for d in (-1, 0, 1):
            reads.append((f"length_S+o{d:+d}\tend", _rnd(rng, S + o + d - span) + copy()))
        reads.append(("length_S+o+1 start", copy() + _rnd(rng, S + o + 1 - span)))
        # shorter than the unit: nothing, a random stretch, the reverse complement less t bases (a tie at threshold t)
        reads += [("empty", ""), ("short_random", _rnd(rng, m // 2)), ("short_rc", strands[1][t:]),
                  ("short_prefix", strands[0][:m - 3])]
        # N and lowercase: matched by nothing the unit holds
        c = copy()
        reads.append(("with_N", _rnd(rng, 90) + c[:len(c) // 2] + "N" + c[len(c) // 2 + 1:] + "N" * 30))
        c = copy()
        h = len(c) // 3
        reads.append(("with_lowercase", _rnd(rng, S - 1) + c[:h] + c[h:h + 3].lower() + c[h + 3:] + _rnd(rng, 40).lower()))
        reads.append(("lowercase_unit", _rnd(rng, 20) + strands[0].lower() + _rnd(rng, 20)))
        reads.append(("n_flanks", "N" * (S - 1) + copy() + "N" * 17))
        reads += [(f"random_{i}", _rnd(rng, int(rng.integers(1, 2 * S)))) for i in range(3)]
        reads.append(("mutated", _rnd(rng, S - 40) + _mutate(rng, strands[1], 0.08) + _rnd(rng, 300)))
        if long_read is not None:  # planted before a boundary of every S here, and twice more at random
            at = [100 * 8192 - 1, int(rng.integers(0, LONG_READ // 2)), LONG_READ - span]
            s = long_read
            for a in at:
                s = s[:a] + copy() + s[a + span:]
            reads.append(("long", s[:LONG_READ]))
        self.reads = reads
        self.seqs = [s for _, s in reads]
        planted = [d for (name, _), d in zip(reads, _distances(self.unit, self.seqs).min(axis=1).tolist())
                   if not name.startswith(("random", "short_random", "lowercase_unit", "empty"))]
        # every planted copy's own distance and that minus one (t and t - 1 when the copy is tight)
        self.thresholds = sorted({d for d in planted if d <= t} | {d - 1 for d in planted if 1 <= d <= t})


_CASES = {}


def _case(m, t, segment):
    if (m, t, segment) not in _CASES:
        _CASES[m, t, segment] = _Case(m, t, segment)
    return _CASES[m, t, segment]


# ---- 1. the overlap bound, on the host --------------------------------------------------------------------------------

@pytest.mark.parametrize("m,t,segment", CASES, ids=CASE_IDS)
def test_overlap_bound_on_the_host(m, t, segment):
    c = _case(m, t, segment)
    assert t in c.thresholds and max(c.thresholds) == t and t < m
    dist = _distances(c.unit, c.seqs)
    segs = _Segments(c.unit, c.seqs, segment, m + min(c.thresholds) - 2, m + t)
    for threshold in c.thresholds:
        want = _keep(dist, threshold)
        for o in (m + threshold - 1, m + threshold):  # the tight bound, and what recruit() uses
            got = segs.keep(o, threshold)
            assert np.array_equal(got, want), (threshold, o, [c.reads[r][0] for r in np.flatnonzero(got != want)])
        short = segs.keep(m + threshold - 2, threshold)
        assert not (short & ~want).any()  # a segment is an infix of its read
        if threshold == t:  # the corpus tells the tight overlap from one base less
            lost = [c.reads[r][0] for r in np.flatnonzero(want & ~short)]
            assert lost, "no planted copy needs its whole span"
    n_seg = _n_seg(segs.lens, m + t, segment)
    assert n_seg.max() >= 4 and (segs.lens > segment).sum() >= 8


def test_word_class_placement():
    """cfk_rr_words: the first and last unit length of every class of rr_filter_kernel<NW>, NW words of 64 bases."""
    from centroflye_b200 import _lib
    lib = _lib.load()
    assert {m: lib.cfk_rr_words(m) for m in WORD_CLASS_LIMITS} == WORD_CLASS_LIMITS
    assert [lib.cfk_rr_words(m) for m in (0, -1, 1, 64, 65, 3329, 4000)] == [-1, -1, 4, 4, 4, -1, -1]


# ---- 2. recruit(), in memory ----------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("m,t,segment", CASES, ids=CASE_IDS)
def test_recruit_decisions_equal_whole_read_dp(m, t, segment, monkeypatch):
    from centroflye_b200 import read_recruitment as rr
    assert rr.SEGMENT == 8192
    c = _case(m, t, segment)
    dist = _distances(c.unit, c.seqs)
    for s in sorted({segment, rr.SEGMENT}):
        monkeypatch.setattr(rr, "SEGMENT", s)
        for threshold in c.thresholds + [-1]:
            got = rr.recruit(c.unit, c.seqs, threshold)
            want = _keep(dist, threshold)
            assert np.array_equal(got, want), (s, threshold, [c.reads[r][0] for r in np.flatnonzero(got != want)])


# ---- 3. exact distances at the word-class limits -------------------------------------------------------------------------

def _class_corpus(m):
    """A seeded unit of m bases and reads around it: mutated copies on both strands with a long tail (the early exit
    stops before the end), the unit itself, a read shorter than the unit, five Ns inside a copy, a copy with three
    insertions, a random read."""
    from centroflye_b200.read_recruitment import reverse_complement
    rng = np.random.default_rng(m + 7)
    unit = _rnd(rng, m)
    rc = reverse_complement(unit)
    reads = [_rnd(rng, 40) + _mutate(rng, unit, 0.03) + _rnd(rng, 300), _rnd(rng, 100) + _mutate(rng, rc, 0.08) + _rnd(rng, 200),
             unit, rc[m // 3:], unit[:m // 2] + "NNNNN" + unit[m // 2:] + _rnd(rng, 100), _rnd(rng, 30) + _planted(rng, rc, 3),
             _rnd(rng, m + 100)]
    return unit, reads


@gpu
@pytest.mark.parametrize("m", sorted(WORD_CLASS_LIMITS))
def test_exact_distances_at_word_class_limits(m):
    from centroflye_b200 import read_recruitment as rr
    unit, reads = _class_corpus(m)
    want = _distances(unit, reads)
    threshold = max(3, m // 50)
    keep, dist = rr.recruit(unit, reads, threshold, exact=True)
    assert np.array_equal(dist, want)
    assert np.array_equal(keep, _keep(want, threshold))
    assert want[2, 0] == 0 and want[3, 1] == m // 3


# ---- 4. threshold ties on the early-exit path -----------------------------------------------------------------------------

TIE_UNITS = (128, 576, 577, 1089, 2113)  # one unit of every word class


def _tie_corpus():
    """The class corpora of TIE_UNITS, and twenty reads of the 128-base unit mutated at rates from 0 to 0.38, so that
    its distances take enough values for more than one launch of its class."""
    units, reads, own = [], [], []
    for m in TIE_UNITS:
        unit, rs = _class_corpus(m)
        units.append(unit)
        own.append(list(range(len(reads), len(reads) + len(rs))))
        reads += rs
    rng = np.random.default_rng(128)
    for i in range(20):
        own[0].append(len(reads))
        reads.append(_rnd(rng, 30) + _mutate(rng, units[0], 0.02 * i) + _rnd(rng, 400))
    return units, reads, own


def _whole_reads_on_device(eng, reads):
    lens = np.array([len(s) for s in reads], dtype=np.int64)
    offs = np.zeros(len(reads), dtype=np.int64)
    np.cumsum(((lens + 15) & ~15)[:-1], out=offs[1:])
    text = np.zeros(int(offs[-1] + lens[-1]) + 32, dtype=np.uint8)
    for o, s in zip(offs.tolist(), reads):
        text[o:o + len(s)] = np.frombuffer(s.encode(), dtype=np.uint8)
    order = np.argsort(-lens, kind="stable").astype(np.int32)
    return [eng._to_dev(a) for a in (text, offs, lens, order)]


@gpu
def test_filter_units_keep_flips_at_the_distance():
    """cfk_rr_filter_units with every unit repeated at thresholds d - 1, d and d + 1 for distances d of its reads
    (every distinct one for the 128-base unit: more than 64 entries, several launches of its class)."""
    import torch
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200.engine import default_engine
    eng = default_engine()
    units, reads, own = _tie_corpus()
    dist = [_distances(u, reads).min(axis=1) for u in units]
    entries = []  # (unit index, threshold)
    for u in range(len(units)):
        ds = sorted(set(dist[u].tolist()) if u == 0 else set(dist[u][own[u]].tolist()))
        entries += [(u, th) for d in ds for th in (d - 1, d, d + 1) if th >= 0]
    assert sum(u == 0 for u, _ in entries) > 64
    masks = [rr.build_masks(u) for u in units]
    d_text, d_off, d_len, d_order = _whole_reads_on_device(eng, reads)
    d_peq = eng._to_dev(np.concatenate([masks[u][0].reshape(-1) for u, _ in entries]).view(np.int64))
    d_sym = eng._to_dev(np.concatenate([masks[u][1] for u, _ in entries]))
    unit_m = np.array([len(units[u]) for u, _ in entries], dtype=np.int32)
    unit_t = np.array([th for _, th in entries], dtype=np.int32)
    R, U, p = len(reads), len(entries), eng._p
    d_keep = eng._zeros(U * R, torch.uint8)
    _lib.call("cfk_rr_filter_units", p(d_text), p(d_off), p(d_len), p(d_order), R, U, p(d_peq), p(d_sym),
              unit_m.ctypes.data, unit_t.ctypes.data, p(d_keep), eng._stream())
    got = d_keep[:U * R].cpu().numpy().reshape(U, R).astype(bool)
    ties = 0
    for row, (u, th) in zip(got, entries):
        assert np.array_equal(row, dist[u] <= th), (len(units[u]), th, np.flatnonzero(row != (dist[u] <= th)).tolist())
        ties += int((dist[u] == th).sum())
    assert ties >= len(entries) // 3


@gpu
def test_early_exit_stops_where_the_minimum_comes_within_the_threshold():
    """cfk_rr_filter without exact, with out_dist: a strand scans its read 16 bytes (one load) at a time and stops
    after the load in which its running minimum comes within the threshold, so out_dist holds that minimum then; a
    strand that never comes within it scans the whole read and holds the exact distance."""
    import torch
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    from centroflye_b200.engine import default_engine
    eng = default_engine()
    units, reads, own = _tie_corpus()
    p, stopped_early = eng._p, 0
    for unit, mine in zip(units, own):
        rs = [reads[r] for r in mine]
        n = np.array([len(s) for s in rs])
        minima = [_prefix_minima(u, rs, int(n.max())) for u in (unit, rr.reverse_complement(unit))]
        dist = np.array([[mm[i][n[i]] for mm in minima] for i in range(len(rs))])
        assert np.array_equal(dist, _distances(unit, rs))
        peq, sym_of, _ = rr.build_masks(unit)
        d_peq, d_sym = eng._to_dev(peq.reshape(-1).view(np.int64)), eng._to_dev(sym_of)
        d_text, d_off, d_len, d_order = _whole_reads_on_device(eng, rs)
        for th in sorted({th for d in dist.min(axis=1).tolist() for th in (d - 1, d, d + 1) if th >= 0}):
            want = np.empty((len(rs), 2), dtype=np.int64)
            for i in range(len(rs)):
                for s in range(2):
                    within = np.flatnonzero(minima[s][i][1:n[i] + 1] <= th)  # column c + 1: c + 1 bases read
                    end = min(int(n[i]), (int(within[0]) + 16) // 16 * 16) if within.size else int(n[i])
                    want[i, s] = minima[s][i][end]
                    stopped_early += end < n[i]
            d_keep, d_dist = eng._zeros(len(rs), torch.uint8), eng._zeros(2 * len(rs), torch.int32)
            _lib.call("cfk_rr_filter", p(d_text), p(d_off), p(d_len), p(d_order), len(rs), p(d_peq), p(d_sym), len(unit),
                      th, 0, p(d_dist), p(d_keep), eng._stream())
            got = d_dist[:2 * len(rs)].cpu().numpy().reshape(-1, 2)
            assert np.array_equal(got, want), (len(unit), th, got.tolist(), want.tolist())
            assert np.array_equal(d_keep[:len(rs)].cpu().numpy().astype(bool), dist.min(axis=1) <= th)
    assert stopped_early >= 20


# ---- 5. end to end ---------------------------------------------------------------------------------------------------------

def _formats(tmp_path, reads):
    """FASTA with 60-column lines, FASTQ and gzip FASTQ of the reads -> {format: path}."""
    fa = "".join(f">{n}\n" + "".join(s[i:i + 60] + "\n" for i in range(0, len(s), 60)) for n, s in reads).encode()
    fq = "".join(f"@{n}\n{s}\n+\n{'I' * len(s)}\n" for n, s in reads).encode()
    paths = {f: str(tmp_path / f"reads.{f}") for f in ("fasta", "fastq", "fastq.gz")}
    open(paths["fasta"], "wb").write(fa)
    open(paths["fastq"], "wb").write(fq)
    with gzip.open(paths["fastq.gz"], "wb") as f:
        f.write(fq)
    return paths


def _expected(reads, keep):
    """>name\\nsequence\\n of every kept read in file order, the name cut at the first whitespace."""
    return "".join(f">{n.split()[0]}\n{s}\n" for (n, s), k in zip(reads, keep.tolist()) if k).encode()


@gpu
@pytest.mark.parametrize("segment", [256, 8192])
def test_output_files_equal_whole_read_dp(tmp_path, monkeypatch, segment):
    """recruit_file per job, recruit_file_units for all jobs (their largest m + t sets the overlap; one job keeps
    everything) on one worker and three: every output is the kept reads of the whole-read DP, byte for byte."""
    from centroflye_b200 import read_recruitment as rr
    monkeypatch.setattr(rr, "SEGMENT", segment)
    cases = [_case(m, t, s) for m, t, s in CASES if s == segment]
    reads = [(f"{c.m}_{name}", s) for c in cases for name, s in c.reads if len(s) < LONG_READ]
    seqs = [s for _, s in reads]
    jobs = [(c.unit, th) for c in cases for th in (c.t, c.t - 1)] + [(cases[-1].unit, -1)]
    assert len({len(u) + th for u, th in jobs if th >= 0}) == len(jobs) - 1
    want = [_expected(reads, _keep(_distances(u, seqs), th)) for u, th in jobs]
    assert all(w.count(b">") >= 8 for w in want[0:-1:2]) and want[-1].count(b">") == len(reads)
    for fmt, path in _formats(tmp_path, reads).items():
        for chunk in (1000, 1 << 24):  # 1000 bytes: less than one record for most of them
            where = f"{fmt}_{chunk}"
            for i, (unit, th) in enumerate(jobs):
                out = str(tmp_path / f"{where}_single{i}.fa")
                stats = {}
                rr.recruit_file(unit, path, out, th, chunk_bytes=chunk, stats=stats)
                assert stats["fallback"] is None and stats["records"] == len(reads)
                assert open(out, "rb").read() == want[i], (where, len(unit), th)
            for devices in (None, [0, 0, 0]):
                outs = [str(tmp_path / f"{where}_{devices is not None}_{i}.fa") for i in range(len(jobs))]
                stats = {}
                rr.recruit_file_units([(u, o, th) for (u, th), o in zip(jobs, outs)], path, chunk_bytes=chunk,
                                      stats=stats, devices=devices)
                assert stats["fallback"] is None
                for i, (o, (unit, th)) in enumerate(zip(outs, jobs)):
                    assert open(o, "rb").read() == want[i], (where, devices, len(unit), th)
