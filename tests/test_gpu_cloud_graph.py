"""Stages B-D at the limits of their layouts, against plain restatements of the reference.

* ``sparse_dist_edges`` restates distance_based_kmer_recruitment.py:111-149 with sorted int64 keys instead of dense
  n_kmers x n_kmers matrices, so the cases can be as large as the kernels' layouts need: clouds around every multiple of
  the sketch's 32-entry rows and 128-entry windows, shared-memory bank pile-ups, same-hash ids inside a unit, more hot
  ids than the level-2 set holds, passes at SK_ND_MAX distances and at exactly SK_CAP entries.
* ``restate_clouds`` restates read_kmer_cloud.py:18-31 on the packed reads for stage B: k from 1 to 31, unit offsets at
  every residue mod 16, hit counts around the warp's 512-entry list, repetitive units, the block form.

The restatements check themselves without a GPU (dense matrices, the golden points, the C oracle); everything that
runs a kernel is marked gpu.
"""
import contextlib
import itertools
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")


def _header_define(name):
    with open(os.path.join(ROOT, "include", "cfk.h")) as f:
        m = re.search(rf"^#define\s+{name}\s+(\d+)", f.read(), re.M)
    assert m, f"{name} not found in include/cfk.h"
    return int(m.group(1))


SKETCH_BITS = _header_define("CFK_SKETCH_BITS")
SKETCH_LOAD_DIV = _header_define("CFK_SKETCH_LOAD_DIV")
SKETCH_MIN_COV = _header_define("CFK_SKETCH_MIN_COV")
SKETCH_MAX_COV = _header_define("CFK_SKETCH_MAX_COV")
# layout constants of cfk.cu the cases are built around
SK_WINDOW, SK_L2_MAX, SK_Q_SLOTS = 128, 192, 256
CLW_LIST, CL_SMEM_IDS = 512, 8192


def sk_hash(ids, bits=SKETCH_BITS):
    """Counter index of an id in the stage-C sketch (cfk.cu sk_hash): (id * 0x9E3779B1 mod 2^32) >> (32 - bits)."""
    ids = np.asarray(ids, dtype=np.uint64)
    return ((ids * np.uint64(0x9E3779B1)) & np.uint64(0xFFFFFFFF)) >> np.uint64(32 - bits)


def sk_bank(h):
    """Shared-memory bank of a byte counter (4-byte words, 32 banks)."""
    return (np.asarray(h, dtype=np.uint64) >> np.uint64(2)) & np.uint64(31)


def sk_cap(bits):
    """Cloud entries one sketch pass is planned for (cfk.cu SK_CAP)."""
    return (1 << bits) // SKETCH_LOAD_DIV


# ---- stage C/D reference ----------------------------------------------------------------------------------------
def _flatten(units):
    """units: list (per read) of lists (per unit) of sorted id arrays -> (unit_ptr, ids, unit_last), int64."""
    flat = [np.asarray(u, dtype=np.int64) for rd in units for u in rd]
    sizes = np.array([u.size for u in flat], dtype=np.int64)
    ptr = np.zeros(sizes.size + 1, dtype=np.int64)
    np.cumsum(sizes, out=ptr[1:])
    ids = np.concatenate(flat) if flat else np.empty(0, np.int64)
    per_read = np.array([len(rd) for rd in units], dtype=np.int64)
    last = np.repeat(np.cumsum(per_read) - 1, per_read)
    return ptr, ids, last


def _canon(e):
    e = np.asarray(e, dtype=np.int64).reshape(-1, 4)
    return e[np.lexsort((e[:, 3], e[:, 2], e[:, 1], e[:, 0]))]


def sparse_dist_edges(units, min_d, max_d, min_cov, rel=0.8):
    """get_kmer_dist_map + filter_dist_tuples (dbkr.py:111-149) on integer ids -> (edges, n_increments).

    edges: int64[n, 4] rows (a, b, d, cnt), sorted.  For every d, the products of unit i and unit i + d of every read
    are formed at once (np.repeat over the left unit's entries, a ragged arange over the right unit's), pairs a == b are
    dropped, and (d, a, b) -- ids renumbered densely, so any universe below 2^32 fits -- is one int64 key; np.unique
    counts the keys, a second np.unique totals them over d per (a, b).  An edge is kept iff cnt >= min_cov and
    cnt / total >= rel in float64.  n_increments counts the products with a != b (the `+= 1` of dbkr.py:126)."""
    ptr, ids, last = _flatten(units)
    empty = np.empty((0, 4), dtype=np.int64)
    dmin = max(int(min_d), 1)
    if ids.size == 0:
        return empty, 0
    uniq, dense = np.unique(ids, return_inverse=True)
    dense = dense.astype(np.int64)
    n = np.int64(uniq.size)
    sizes = np.diff(ptr)
    unit_of = np.repeat(np.arange(sizes.size, dtype=np.int64), sizes)
    rem = last[unit_of] - unit_of  # units behind each entry's unit inside its read
    dtop = min(int(max_d), int(rem.max()))
    if dtop < dmin:
        return empty, 0
    assert (dtop - dmin + 1) * int(n) * int(n) < (1 << 63)
    keys, n_incr = [], 0
    for d in range(dmin, dtop + 1):
        left = np.flatnonzero(rem >= d)
        right = unit_of[left] + d
        cnt = sizes[right]
        tot = int(cnt.sum())
        if tot == 0:
            continue
        a = np.repeat(dense[left], cnt)
        b = dense[np.repeat(ptr[right] - (np.cumsum(cnt) - cnt), cnt) + np.arange(tot, dtype=np.int64)]
        keep = a != b
        n_incr += int(keep.sum())
        keys.append(((d - dmin) * n + a[keep]) * n + b[keep])
    if not keys:
        return empty, n_incr
    key, cnt = np.unique(np.concatenate(keys), return_counts=True)
    d = key // (n * n) + dmin
    pair = key % (n * n)
    _, inv = np.unique(pair, return_inverse=True)
    total = np.bincount(inv, weights=cnt)[inv]
    keep = (cnt >= min_cov) & (cnt.astype(np.float64) / total >= rel)
    edges = np.stack([uniq[pair[keep] // n], uniq[pair[keep] % n], d[keep], cnt[keep]], axis=1)
    return _canon(edges), n_incr


def _edge_set(e):
    return {tuple(int(x) for x in row) for row in np.asarray(e).reshape(-1, 4)}


def _diff(got, want):
    g, w = _edge_set(got), _edge_set(want)
    return f"missing {sorted(w - g)[:6]} ({len(w - g)} in all), extra {sorted(g - w)[:6]} ({len(g - w)} in all)"


def _unit(x):
    return np.unique(np.asarray(x, dtype=np.int64))


# ---- stage C/D cases (deterministic; the ones built around the sketch's hash take its bit width) ----------------
WINDOW_SIZES = [0, 1, 31, 32, 33, 127, 128, 129, 255, 256, 257, 383, 384, 385]


def _window_case():
    """Clouds of every size around the 32-entry rows and 128-entry windows, mixed inside reads of 1, 2, 5 and 40
    units.  Unit i of a read draws from pool (start + i) mod 8 (disjoint 400-id pools), so ids recur at fixed
    distances across reads."""
    rng = np.random.default_rng(11)
    pools = rng.permutation(5000)[:3200].reshape(8, 400)
    sizes = itertools.cycle(rng.permutation(WINDOW_SIZES * 3))
    units = []
    for n_units in [1] * 4 + [2] * 6 + [5] * 8 + [40]:
        s = int(rng.integers(0, 8))
        units.append([_unit(rng.choice(pools[(s + i) % 8], size=next(sizes), replace=False)) for i in range(n_units)])
    return units, 5000


def _bank_case(bits):
    """Windows whose counters pile into shared-memory banks: 128 entries in one bank (distinct counters while the bank
    has enough of them), windows with 5-8 entries in each of several banks, and a two-window unit whose first window
    is one bank.  The same units in 8 reads; outside the one-bank unit each entry is kept with probability 0.9."""
    rng = np.random.default_rng(21)
    n_kmers = 1 << 16
    all_ids = np.arange(n_kmers, dtype=np.int64)
    h = sk_hash(all_ids, bits).astype(np.int64)
    bank = sk_bank(h).astype(np.int64)
    used = np.zeros(n_kmers, dtype=bool)

    def take(b, n, lo=0, hi=n_kmers):
        """n unused ids of bank b inside [lo, hi), distinct counters first."""
        pool = all_ids[(bank == b) & ~used & (all_ids >= lo) & (all_ids < hi)]
        pool = pool[rng.permutation(pool.size)]
        _, first = np.unique(h[pool], return_index=True)
        rest = np.setdiff1d(np.arange(pool.size), first)
        pick = pool[np.concatenate([first, rest])[:n]]
        assert pick.size == n
        used[pick] = True
        return pick

    one_bank = np.sort(take(0, 128))
    mixed_full = np.concatenate([take(b, 8) for b in range(1, 17)])                                   # 16 banks x 8
    mixed_3rows = np.concatenate([take(b, c) for b, c in zip(range(17, 25), [8, 8, 7, 7, 6, 6, 5, 5])]
                                 + [take(b, 1) for b in range(25, 32)] + [take(0, 20)])               # 79 entries
    other_bank = take(5, 128)
    two_windows = np.concatenate([take(7, 128, hi=n_kmers // 2),
                                  np.concatenate([take(b, 4, lo=n_kmers // 2) for b in range(0, 32, 2)])])
    layout = [one_bank, mixed_full, mixed_3rows, other_bank, two_windows]
    units = [[layout[0]] + [_unit(u[rng.random(u.size) < 0.9]) for u in layout[1:]] for _ in range(8)]
    return units, n_kmers, layout


def _collision_case(bits, min_cov):
    """Same-hash pairs P < F in one unit with >= 31 other ids between them, so F (>= 32 positions later) is the one
    flagged SK_DUP.  Three groups, each with its own source A in unit 0 of its reads (unit 1 holds 40 fillers of other
    hashes from between P and F, plus):
      flagged_only  F in min_cov reads, P only in the last: F's count reaches min_cov only where F is flagged
      both          P and F in min_cov reads: both reach min_cov, F always flagged
      neither       F in min_cov - 1 reads, P in the next min_cov - 1: their shared counter passes min_cov - 1, so a
                    candidate is made, but no id reaches min_cov."""
    rng = np.random.default_rng(31 + min_cov)
    n_kmers = 1 << 16
    all_ids = np.arange(n_kmers, dtype=np.int64)
    h = sk_hash(all_ids, bits).astype(np.int64)
    c = min_cov
    units, groups = [], {}
    for gi, outcome in enumerate(("flagged_only", "both", "neither")):
        lo = gi * 20000
        while True:
            p = int(rng.integers(lo + 1, lo + 8000))
            f_cands = all_ids[(h == h[p]) & (all_ids > p + 1500) & (all_ids < p + 9000)]
            if f_cands.size and h[lo] != h[p]:
                break
        f = int(f_cands[0])
        between = all_ids[p + 1:f]
        fillers = between[h[p + 1:f] != h[p]]
        a = lo  # the source: the group's lowest id, below P
        groups[outcome] = (a, p, f)
        if outcome == "flagged_only":
            rows = [(False, True)] * (c - 1) + [(True, True)]
        elif outcome == "both":
            rows = [(True, True)] * c
        else:
            rows = [(False, True)] * (c - 1) + [(True, False)] * (c - 1)
        for with_p, with_f in rows:
            u1 = list(rng.choice(fillers, size=40, replace=False)) + [p] * with_p + [f] * with_f
            units.append([_unit([a]), _unit(u1)])
    return units, n_kmers, groups


def _level2_case():
    """Source 0: 250 ids in unit 1 of each of its 8 reads -- all hot in one pass, more than the level-2 set holds.
    Source 1: 150 ids in unit 1 of each of its 40 reads (two windows per unit) -- the hot-position queue fills and
    drains in nearly every step without the set overflowing."""
    rng = np.random.default_rng(41)
    hot250, hot150 = 2 + np.arange(250), 300 + np.arange(150)
    units = []
    for src, hot, n_reads in ((0, hot250, 8), (1, hot150, 40)):
        for _ in range(n_reads):
            units.append([_unit([src]), _unit(np.concatenate([hot, rng.choice(np.arange(1000, 5000), 20, replace=False)]))])
    return units, 5000


def _nd_case():
    """40-unit reads of 2-6 entry clouds from disjoint per-position pools: passes are planned at SK_ND_MAX distances,
    and pairs reaching the last unit of a read are counted in multi-distance passes."""
    rng = np.random.default_rng(51)
    pools = np.arange(40 * 8).reshape(40, 8)
    units = [[_unit(rng.choice(pools[j], size=int(rng.integers(2, 7)), replace=False)) for j in range(40)]
             for _ in range(12)]
    return units, 320


def _occ32_case():
    """Sources with exactly 32 (register window of sketch_source) and 33 (the general path) occurrences; an id in the
    LAST unit of each of their reads; and a source whose 36 reads end at every distance from 0 to 8."""
    rng = np.random.default_rng(61)
    a32, a33, z, a_var, z_var = 0, 1, 2, 3, 4
    pools = 10 + np.arange(4 * 120).reshape(4, 120)
    units = []
    for r in range(40):
        u0 = [x for x, n in ((a32, 32), (a33, 33)) if r < n]
        units.append([_unit(u0)] + [_unit(rng.choice(pools[j], 60, replace=False)) for j in range(3)] + [_unit([z])])
    for r in range(36):
        n_units = 1 + r % 9
        rd = [_unit([a_var])] + [_unit(rng.choice(pools[j % 4], 8, replace=False)) for j in range(n_units - 1)]
        if n_units > 1:
            rd[-1] = _unit(np.concatenate([rd[-1], [z_var]]))
        units.append(rd)
    return units, 600


def _cap_case(bits):
    """Source X: 9 occurrences with cap/8 entries at distance 1 -- one distance alone exceeds SK_CAP.  Source Y: 8
    occurrences with cap/8 entries -- distance 1 fills SK_CAP exactly, distance 2 (one entry) no longer fits."""
    per = sk_cap(bits) // 8
    sx, sy = 10 + np.arange(per), 10 + per + np.arange(per)
    units = [[_unit([0]), _unit(sx), _unit([5])] for _ in range(9)]
    units += [[_unit([1]), _unit(sy), _unit([6])] for _ in range(8)]
    return units, int(10 + 2 * per)


def _param_case():
    """60 reads of 1-12 units over 12 overlapping pools used cyclically: pairs recur at several distances, so the ratio
    test matters; clouds of 0-19 entries."""
    rng = np.random.default_rng(71)
    units = []
    for _ in range(60):
        s, n_units = int(rng.integers(0, 12)), int(rng.integers(1, 13))
        units.append([_unit(rng.choice(np.arange(((s + i) % 12) * 20, ((s + i) % 12) * 20 + 30),
                                       size=int(rng.integers(0, 20)), replace=False)) for i in range(n_units)])
    return units, 250


def _ratio_case():
    """Counts on both sides of 254 / 255 / 256 (X_k -> Y_k in 253 + k reads), and ratios at the 0.8 threshold:
    4 of 5 and 8 of 10 (both exactly 0.8 in float64: kept) and 79 of 99 (just below: dropped)."""
    xs, ys = 10 + np.arange(5), 20 + np.arange(5)
    units = [[_unit(xs[r < 253 + np.arange(5)]), _unit(ys[r < 253 + np.arange(5)])] for r in range(257)]
    for a, n1, n2 in ((40, 4, 1), (42, 8, 2), (44, 79, 20)):
        units += [[_unit([a]), _unit([a + 1])]] * n1 + [[_unit([a]), _unit([]), _unit([a + 1])]] * n2
    return units, 50



def _fanout_case():
    """300 sources in unit 0 of 3 reads, the same 42 targets in each of the 17 units behind them.  A source's pass spans
    16 distances (3 x 42 entries each), and at a ratio threshold below 1/17 each of its candidates (a, b, d0, d1) yields
    an edge per distance: far more edges than candidate records plus the edge buffer's slack of 1024."""
    sources, targets = 100 + np.arange(300), np.arange(42)
    return [[_unit(sources)] + [_unit(targets)] * 17 for _ in range(3)], 400


_CASES = {}


def _case(name, *args):
    key = (name,) + args
    if key not in _CASES:
        _CASES[key] = globals()[f"_{name}_case"](*args)
    return _CASES[key]


_REFS = {}


def _ref(case_key, units, min_d, max_d, min_cov, rel=0.8, reads=None):
    key = (case_key, min_d, max_d, min_cov, rel, reads)
    if key not in _REFS:
        sub = units if reads is None else units[reads[0]:reads[1]]
        _REFS[key] = sparse_dist_edges(sub, min_d, max_d, min_cov, rel)
    return _REFS[key]


# ---- stage B reference -------------------------------------------------------------------------------------------
def _kmers_at_every_base(batch, k):
    from centroflye_b200.encode import unpack_codes
    codes = unpack_codes(batch.packed, batch.packed.size * 16).astype(np.uint64)
    n = codes.size - k + 1
    km = np.zeros(n, dtype=np.uint64)
    for i in range(k):
        km = (km << np.uint64(2)) | codes[i:i + n]
    return km


def _unit_kmers(batch, units, k):
    """-> (k-mer of every k-mer start of every unit, its unit index)."""
    nk = np.maximum(units.unit_len.astype(np.int64) - k + 1, 0)
    starts = np.repeat(units.unit_off - (np.cumsum(nk) - nk), nk) + np.arange(int(nk.sum()), dtype=np.int64)
    return _kmers_at_every_base(batch, k)[starts], np.repeat(np.arange(units.n_units, dtype=np.int64), nk)


def restate_clouds(batch, units, k, rare_keys):
    """ReadKMerCloud.fromNCRF_record (read_kmer_cloud.py:18-31) on the packed reads -> (unit_ptr int64[U+1], ids
    uint32[E]): the cloud of a unit is the sorted unique ranks, in the sorted rare set, of the unit's k-mers."""
    rare = np.unique(np.asarray(rare_keys, dtype=np.uint64))
    km, unit_of = _unit_kmers(batch, units, k)
    r = np.searchsorted(rare, km)
    hit = r < rare.size
    hit[hit] = rare[r[hit]] == km[hit]
    key = np.unique((unit_of[hit] << 32) | r[hit].astype(np.int64))
    ptr = np.zeros(units.n_units + 1, dtype=np.int64)
    np.cumsum(np.bincount(key >> 32, minlength=units.n_units), out=ptr[1:])
    return ptr, (key & 0xFFFFFFFF).astype(np.uint32)


STAGE_B_KS = [1, 2, 5, 11, 16, 17, 31]


def _stage_b_case(k):
    """-> (batch, units, rare keys u64).  Reads 0-15: the first unit starts at residue r mod 16 of the packed stream,
    unit lengths cycle through 0, k - 1, k, k + 1, k + 31, k + 32 (random lengths in between), the last unit ends at the
    read's last base, runs of A and T hold the all-A / all-T k-mers; a read shorter than k and one of exactly k.  Then
    units whose k-mers are all rare: 511 / 512 / 513 hits (the warp's shared list holds 512), 3000 bases, a period-7
    repeat of 3000 bases and a period-13 repeat of 500 (a few ids, sorted runs across the 32-entry tiles of the warp
    unique), and a 9200-base unit (more than the block form's 8192 shared-memory k-mer starts).  The rare set holds 40 %
    of the other units' k-mers, all-A, all-T and keys >= 4^k that can never match."""
    from centroflye_b200.ingest import pack_reads, units_from_boundaries
    rng = np.random.default_rng(500 + k)
    reads, bounds = [], []
    shape_lens = [0, k - 1, k, k + 1, k + 31, k + 32]
    for r in range(16):
        n = int(rng.integers(300, 700))
        seq = rng.integers(0, 4, size=n, dtype=np.uint8)
        if r % 4 == 0:
            seq[10:10 + k + 3] = 0
            seq[60:60 + k + 3] = 3
        b, i = [r], 0
        while True:
            ln = shape_lens[(i // 2) % len(shape_lens)] if i % 2 == 0 else int(rng.integers(0, 2 * k + 40))
            if b[-1] + ln >= n:
                break
            b.append(b[-1] + ln)
            i += 1
        b.append(n)
        reads.append(seq)
        bounds.append(b)
    for n in (k - 1, k):
        reads.append(rng.integers(0, 4, size=n, dtype=np.uint8))
        bounds.append([0, n])
    n_shape = len(reads)
    lim = [511 + k - 1, 512 + k - 1, 513 + k - 1, 3000]
    seq = rng.integers(0, 4, size=int(sum(lim)) + 37, dtype=np.uint8)
    reads.append(seq)
    bounds.append([5] + list(5 + np.cumsum(lim)))
    rep = np.concatenate([np.tile(rng.integers(0, 4, size=7, dtype=np.uint8), 3000 // 7 + 1)[:3000],
                          np.tile(rng.integers(0, 4, size=13, dtype=np.uint8), 500 // 13 + 1)[:500]])
    reads.append(rep)
    bounds.append([0, 3000, 3500])
    big = rng.integers(0, 4, size=9300, dtype=np.uint8)
    big[4000:6000] = np.tile(rng.integers(0, 4, size=11, dtype=np.uint8), 2000 // 11 + 1)[:2000]
    reads.append(big)
    bounds.append([3, 9203])
    batch = pack_reads(reads, [f"r{i}" for i in range(len(reads))])
    units = units_from_boundaries(batch, bounds)
    km, unit_of = _unit_kmers(batch, units, k)
    first_lim_unit = int(units.read_unit_ptr[n_shape])
    shape_km = np.unique(km[unit_of < first_lim_unit])
    rare = np.concatenate([shape_km[rng.random(shape_km.size) < 0.4], km[unit_of >= first_lim_unit],
                           np.array([0, (1 << (2 * k)) - 1], dtype=np.uint64),
                           np.array([1 << (2 * k), (1 << (2 * k)) + 7, 1 << 62, (1 << 63) + 5, (1 << 64) - 2],
                                    dtype=np.uint64)])
    return batch, units, np.unique(rare)


_B_CASES = {}


def _b_case(k):
    if k not in _B_CASES:
        _B_CASES[k] = _stage_b_case(k)
    return _B_CASES[k]


# ==== self-checks of the restatements (no GPU) ====================================================================
def test_sketch_hash_restatement():
    assert 10 <= SKETCH_BITS <= 13 and SKETCH_LOAD_DIV >= 1 and (SKETCH_MIN_COV, SKETCH_MAX_COV) == (3, 255)
    for bits in (10, 13):
        for x in (0, 1, 2, 12345, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF):
            want = ((x * 0x9E3779B1) % (1 << 32)) >> (32 - bits)
            assert int(sk_hash([x], bits)[0]) == want and int(sk_bank([want])[0]) == (want >> 2) & 31


@pytest.mark.parametrize("seed", range(6))
def test_sparse_reference_equals_dense(seed):
    from test_gpu_kernels import _numpy_edges
    rng = np.random.default_rng(900 + seed)
    n_kmers = int(rng.integers(20, 300))
    units = [[_unit(rng.choice(n_kmers, size=int(rng.integers(0, min(n_kmers, 40))), replace=False))
              for _ in range(int(rng.integers(1, 14)))] for _ in range(int(rng.integers(1, 30)))]
    for min_d, max_d, min_cov, rel in ((1, 150, 2, 0.8), (0, 3, 1, 0.8), (2, 2, 3, 0.5), (3, 9, 0, 0.8),
                                       (1, 40, 4, 0.3)):
        want, incr = _numpy_edges(units, n_kmers, min_d, max_d, min_cov, rel)
        got, n = sparse_dist_edges(units, min_d, max_d, min_cov, rel)
        assert n == incr and _edge_set(got) == want and len(got) == len(want)


def _golden_units(arr):
    rare, kmers, ptr = arr["rare"], arr["clouds_kmers"], arr["clouds_unit_ptr"]
    ids = np.searchsorted(rare, kmers)
    assert np.array_equal(rare[ids], kmers)
    rptr = np.concatenate([[0], np.cumsum(arr["clouds_units_per_read"])])
    return [[ids[ptr[u]:ptr[u + 1]] for u in range(rptr[r], rptr[r + 1])] for r in range(rptr.size - 1)], rare


def _golden_points():
    from conftest import all_case_points
    return all_case_points()


@pytest.mark.parametrize("case,pi", _golden_points())
def test_sparse_reference_equals_golden(golden, case, pi):
    """The 13 golden points: the edges and increments the reference computed; py_oracle's dict form as well on the
    points of at most 3 million increments."""
    from oracle import py_oracle
    meta, arr = golden(case).point(pi)
    p = meta["params"]
    units, rare = _golden_units(arr)
    sub = units[p["min_nreads"]:p["max_nreads"]]
    got, incr = sparse_dist_edges(sub, p["min_distance"], p["max_distance"], p["min_coverage"])
    assert incr == meta["n_increments"] and len(got) == meta["n_edges"]
    stored = np.stack([np.searchsorted(rare, arr["edge_a"]), np.searchsorted(rare, arr["edge_b"]),
                       arr["edge_d"].astype(np.int64), arr["edge_cnt"].astype(np.int64)], axis=1)
    assert np.array_equal(got, _canon(stored))
    if meta["n_increments"] > 3 * 10 ** 6:  # pure-Python counting of the larger points takes 5-15 s each
        return
    clouds = {r: [set(u.tolist()) for u in rd] for r, rd in enumerate(units)}
    cnt = py_oracle.dist_counts(clouds, p["min_nreads"], p["max_nreads"], p["min_distance"], p["max_distance"])
    selected, edges = py_oracle.filter_edges(cnt, p["min_coverage"])
    assert sum(cnt.values()) == incr
    assert _edge_set(got) == {(a, b, d, c) for d, a, b, c in edges}
    assert set(np.unique(got[:, :2]).tolist()) == selected


@pytest.mark.parametrize("seed", range(3))
def test_sparse_reference_equals_c_oracle(seed):
    """Mid-size random graphs (a few million increments, a sparse id universe near 2^32), and read windows."""
    from oracle import c_oracle
    rng = np.random.default_rng(700 + seed)
    universe = rng.choice(np.arange((1 << 32) - 5000, (1 << 32) - 1), size=3100, replace=False)
    units = []
    for _ in range(80):
        s, n_units = int(rng.integers(0, 20)), int(rng.integers(1, 30))
        units.append([_unit(universe[rng.choice(np.arange(((s + i) % 20) * 150, ((s + i) % 20) * 150 + 200),
                                               size=int(rng.integers(0, 60)), replace=False)])
                      for i in range(n_units)])
    ptr, ids, last = _flatten(units)
    uniq = np.unique(ids)
    dense_ids = np.searchsorted(uniq, ids).astype(np.uint32)  # the C oracle indexes a table by id
    rptr = np.concatenate([[0], np.cumsum([len(rd) for rd in units])])
    for min_d, max_d, min_cov, reads in ((1, 150, 3, (0, 80)), (0, 5, 1, (0, 80)), (2, 30, 4, (7, 51))):
        got, incr = sparse_dist_edges(units[reads[0]:reads[1]], min_d, max_d, min_cov)
        c = c_oracle.dist_edges(ptr, dense_ids, last.astype(np.int32), uniq.size, min_d, max_d, min_cov,
                                unit_lo=int(rptr[reads[0]]), unit_hi=int(rptr[reads[1]]), threads=4)
        assert incr == c["n_increments"] and incr > 10 ** 5
        e = c["edges"].astype(np.int64)
        e[:, 0], e[:, 1] = uniq[e[:, 0]], uniq[e[:, 1]]
        assert np.array_equal(got, _canon(e))


@pytest.mark.parametrize("k", STAGE_B_KS)
def test_cloud_restatement_equals_c_oracle(k):
    from oracle import c_oracle
    batch, units, rare = _b_case(k)
    ptr, ids = restate_clouds(batch, units, k, rare)
    cptr, cids = c_oracle.clouds(c_oracle.unpacked_codes(batch), units, k, rare)
    assert np.array_equal(ptr, cptr) and np.array_equal(ids, cids)
    sizes = np.diff(ptr)
    n_lim = int(units.read_unit_ptr[-4])
    if k >= 16:  # random k-mers are distinct: the hit counts around the shared list are distinct ids as well
        assert sizes[n_lim:n_lim + 3].tolist() == [CLW_LIST - 1, CLW_LIST, CLW_LIST + 1]
    assert np.any(sizes[units.read_unit_ptr[-3]:units.read_unit_ptr[-2]] <= 13)  # the repeats: a few ids per unit
    assert units.unit_len[-1] - k + 1 > CL_SMEM_IDS
    assert sorted(set((units.unit_off[units.read_unit_ptr[:16]] % 16).tolist())) == list(range(16))
    assert sizes.sum() > 0 and 0 in rare.tolist()


def test_cases_are_built_as_described():
    """The sketch cases hold the layouts they are named after (at the header's CFK_SKETCH_BITS)."""
    bits = SKETCH_BITS
    units, n_kmers, layout = _bank_case(bits)
    assert len(set(sk_bank(sk_hash(layout[0], bits)).tolist())) == 1 and layout[0].size == SK_WINDOW
    assert np.bincount(sk_bank(sk_hash(layout[1], bits)).astype(np.int64)).max() == 8
    for c in (3, 4, 7):
        units, _, groups = _collision_case(bits, c)
        want = _edge_set(sparse_dist_edges(units, 1, 1, c)[0])
        for outcome, (a, p, f) in groups.items():
            assert sk_hash([p], bits)[0] == sk_hash([f], bits)[0]
            for rd in units:
                if rd[0].tolist() == [a] and p in rd[1] and f in rd[1]:
                    assert np.searchsorted(rd[1], f) - np.searchsorted(rd[1], p) >= 32
            has = {x for x in (p, f) if (a, x, 1, c) in want}
            assert has == {"flagged_only": {f}, "both": {p, f}, "neither": set()}[outcome]
    units, _ = _level2_case()
    assert units[0][1].size - 20 > SK_L2_MAX >= units[-1][1].size - 20 > SK_Q_SLOTS - SK_WINDOW
    units, _ = _cap_case(bits)
    assert sum(u[1].size for u in units[:9]) > sk_cap(bits) and sum(u[1].size for u in units[9:]) == sk_cap(bits)
    units, _ = _fanout_case()
    e = sparse_dist_edges(units, 1, 20, 3, 0.05)[0]
    assert len(e) > 8 * len(np.unique(e[:, 0] * 400 + e[:, 1]))
    units, _ = _ratio_case()
    e = _edge_set(sparse_dist_edges(units, 1, 2, 4)[0])
    assert (40, 41, 1, 4) in e and (42, 43, 1, 8) in e and not any(x[:2] == (44, 45) for x in e)


# ==== GPU ========================================================================================================
@pytest.fixture(scope="module")
def eng():
    from centroflye_b200.engine import default_engine
    return default_engine()


@pytest.fixture(scope="module")
def bits(eng):
    """The sketch width the loaded library was built with (include/cfk.h unless overridden at build time)."""
    return int(eng.lib.cfk_sketch_bits())


@contextlib.contextmanager
def _settings(eng, **kw):
    old = {k: getattr(eng, k) for k in kw}
    for k, v in kw.items():
        setattr(eng, k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            setattr(eng, k, v)


def _modes(min_cov):
    """Stage-C kernel forms serving min_cov: exact tables always; the sketch with banked and unbanked codes."""
    out = [("exact", 1)]
    if SKETCH_MIN_COV <= min_cov <= SKETCH_MAX_COV:
        out += [("sketch", 1), ("sketch", 0)]
    return out


def _upload(eng, units):
    from centroflye_b200.engine import CloudCSR
    ptr, ids, last = _flatten(units)
    csr = CloudCSR(unit_ptr=eng._to_dev(ptr), ids=eng._to_dev(ids.astype(np.uint32).view(np.int32)),
                   n_units=int(last.size), n_entries=int(ids.size))
    return csr, eng._to_dev(last.astype(np.int32))


def _run(eng, dev, n_kmers, min_d, max_d, min_cov, rel=0.8, **kw):
    csr, dlast = dev
    res = eng.dist_edges(csr, dlast, n_kmers, min_d, max_d, min_cov, rel, **kw)
    e = _canon(res.edges.cpu().numpy().view(np.uint32).astype(np.int64))
    sel = np.sort(res.selected.cpu().numpy().view(np.uint32).astype(np.int64))
    return e, sel, res


def _check(eng, units, n_kmers, min_d, max_d, min_cov, rel=0.8, want=None, dev=None, **kw):
    """Every kernel form against the reference: the edge set, n_increments, and selected = the edges' endpoints."""
    we, wincr = want if want is not None else sparse_dist_edges(units, min_d, max_d, min_cov, rel)
    wsel = np.unique(we[:, :2])
    dev = dev if dev is not None else _upload(eng, units)
    out = {}
    for mode, banked in _modes(min_cov):
        with _settings(eng, pair_mode=mode, sketch_banked=banked):
            e, sel, res = _run(eng, dev, n_kmers, min_d, max_d, min_cov, rel, **kw)
        tag = f"{mode} banked={banked}"
        assert eng.last_pair_kernel == ("pair_sketch_kernel" if mode == "sketch" else "pair_candidates_kernel")
        assert res.n_increments == wincr, tag
        assert np.array_equal(e, we), f"{tag}: {_diff(e, we)}"
        assert np.array_equal(sel, wsel), tag
        out[(mode, banked)] = res
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("min_d,max_d,min_cov", [(1, 3, 3), (0, 7, 5)])
def test_window_boundaries(eng, min_d, max_d, min_cov):
    units, n_kmers = _case("window")
    want = _ref(("window",), units, min_d, max_d, min_cov)
    assert len(want[0]) > 1000
    _check(eng, units, n_kmers, min_d, max_d, min_cov, want=want)


@pytest.mark.gpu
@pytest.mark.parametrize("min_cov", [3, 6])
def test_bank_overflow(eng, bits, min_cov):
    units, n_kmers, _ = _case("bank", bits)
    want = _ref(("bank", bits), units, 1, 4, min_cov)
    assert len(want[0]) > 1000
    _check(eng, units, n_kmers, 1, 4, min_cov, want=want)


@pytest.mark.gpu
@pytest.mark.parametrize("min_cov", [3, 4, 7])
def test_hash_collisions(eng, bits, min_cov):
    units, n_kmers, groups = _case("collision", bits, min_cov)
    want = _ref(("collision", bits, min_cov), units, 1, 1, min_cov)
    w = _edge_set(want[0])
    a, p, f = groups["flagged_only"]
    assert (a, f, 1, min_cov) in w and not any(e[:2] == (a, p) for e in w)
    a, p, f = groups["both"]
    assert (a, f, 1, min_cov) in w and (a, p, 1, min_cov) in w
    a, p, f = groups["neither"]
    assert not any(e[:2] in ((a, p), (a, f)) for e in w)
    _check(eng, units, n_kmers, 1, 1, min_cov, want=want)


@pytest.mark.gpu
@pytest.mark.parametrize("min_cov", [3, 5])
def test_level2_set_and_queue(eng, min_cov):
    units, n_kmers = _case("level2")
    want = _ref(("level2",), units, 1, 3, min_cov)
    assert {(0, x, 1, 8) for x in range(2, 252)} <= _edge_set(want[0])
    res = _check(eng, units, n_kmers, 1, 3, min_cov, want=want)
    assert res[("sketch", 1)].n_splits > 0 and res[("sketch", 0)].n_splits > 0


@pytest.mark.gpu
@pytest.mark.parametrize("max_d", [4, 20, 150])
def test_pass_planning(eng, bits, max_d):
    """Sources with 32 / 33 occurrences, reads ending inside the distance range, passes at SK_ND_MAX distances, one
    distance over SK_CAP and one filling it exactly."""
    for name, args in (("occ32", ()), ("nd", ()), ("cap", (bits,))):
        units, n_kmers = _case(name, *args)
        want = _ref((name,) + args, units, 1, max_d, 3)
        assert len(want[0]) > 0
        if name == "occ32":
            assert (1, 2, 4, 33) in _edge_set(want[0]) or max_d < 4
        _check(eng, units, n_kmers, 1, max_d, 3, want=want)


@pytest.mark.gpu
@pytest.mark.parametrize("min_d,max_d,min_cov", [
    (0, 1, 3), (1, 1, 3), (0, 3, 3), (2, 3, 3), (3, 3, 3), (7, 7, 3), (0, 150, 3), (2, 150, 3), (7, 150, 3),
    (1, 10 ** 4, 3), (7, 10 ** 4, 4), (1, 150, 1), (1, 150, 2), (1, 150, 4), (2, 7, 254)])
def test_parameters(eng, min_d, max_d, min_cov):
    units, n_kmers = _case("param")
    _check(eng, units, n_kmers, min_d, max_d, min_cov, want=_ref(("param",), units, min_d, max_d, min_cov))


@pytest.mark.gpu
@pytest.mark.parametrize("min_cov", [1, 2, 3, 4, 254, 255, 256])
def test_coverage_and_ratio_edges(eng, min_cov):
    units, n_kmers = _case("ratio")
    want = _ref(("ratio",), units, 0, 3, min_cov)
    w = _edge_set(want[0])
    assert ((40, 41, 1, 4) in w) == (min_cov <= 4) and ((42, 43, 1, 8) in w) == (min_cov <= 8)
    assert not any(e[:2] == (44, 45) for e in w)
    for i in range(5):
        assert ((10 + i, 20 + i, 1, 253 + i) in w) == (253 + i >= min_cov)
    _check(eng, units, n_kmers, 0, 3, min_cov, want=want)


@pytest.mark.gpu
@pytest.mark.parametrize("reads", [(0, 60), (0, 1), (5, 23), (53, 60), (10, 10)])
def test_read_window(eng, reads):
    """unit_lo / unit_hi on read boundaries: the reference on that read subset (dbkr.py islice(min_n, max_n))."""
    units, n_kmers = _case("param")
    rptr = np.concatenate([[0], np.cumsum([len(rd) for rd in units])])
    want = _ref(("param",), units, 1, 150, 3, reads=reads)
    _check(eng, units, n_kmers, 1, 150, 3, want=want, unit_lo=int(rptr[reads[0]]), unit_hi=int(rptr[reads[1]]))


@pytest.mark.gpu
@pytest.mark.parametrize("name,min_d,max_d,min_cov,rel", [
    ("param", 1, 150, 3, 0.8), ("level2", 1, 3, 3, 0.8), ("window", 1, 3, 3, 0.8), ("fanout", 1, 20, 3, 0.05)])
def test_buffer_growth(eng, name, min_d, max_d, min_cov, rel):
    """Candidate and edge buffers sized from hints of one entry.  The candidate buffer then always overflows and is
    grown (sketch chunks leave holes in the candidates).  The edge buffer starts at the candidate count + 1024, which
    only a case with more edges than that outgrows: "fanout" at a low ratio threshold, where the edge loop must run."""
    units, n_kmers = _case(name)[:2]
    want = _ref((name,), units, min_d, max_d, min_cov, rel)
    dev = _upload(eng, units)
    for mode, banked in _modes(min_cov):
        with _settings(eng, pair_mode=mode, sketch_banked=banked, cand_hint=1, edge_hint=1):
            e, sel, res = _run(eng, dev, n_kmers, min_d, max_d, min_cov, rel)
            n_cand = eng.last_pair_counters[0]
        tag = f"{mode} banked={banked}"
        assert n_cand > 1, tag  # the candidate loop ran
        if name == "fanout":  # the first edge buffer held n_cand + 1024 edges: the edge loop ran
            assert len(e) > n_cand + 1024, f"{tag}: {len(e)} edges, {n_cand} candidates"
        assert res.n_increments == want[1] and np.array_equal(e, want[0]), f"{tag}: {_diff(e, want[0])}"
        assert np.array_equal(sel, np.unique(want[0][:, :2]))


@pytest.mark.gpu
@pytest.mark.parametrize("prefetch", ["1", "0"])
def test_sketch_prefetch_switch(eng, bits, monkeypatch, prefetch):
    """CFK_SKETCH_PREFETCH (read on every call) forces the L2 prefetch of each pass's code blocks on / off."""
    monkeypatch.setenv("CFK_SKETCH_PREFETCH", prefetch)
    units, n_kmers = _case("param")
    _check(eng, units, n_kmers, 1, 150, 3, want=_ref(("param",), units, 1, 150, 3))
    units, n_kmers, _ = _case("bank", bits)
    _check(eng, units, n_kmers, 1, 4, 3, want=_ref(("bank", bits), units, 1, 4, 3))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["param", "occ32"])
def test_sharding_by_source(eng, name):
    """a_begin / a_end / a_stride: [0, h) in one part and [h, n) in three strided ones are disjoint, and together they
    are the whole graph and its increments."""
    units, n_kmers = _case(name)
    want = _ref((name,), units, 1, 150, 3)
    dev = _upload(eng, units)
    h = n_kmers // 3
    for mode, banked in _modes(3):
        with _settings(eng, pair_mode=mode, sketch_banked=banked):
            parts = [_run(eng, dev, n_kmers, 1, 150, 3, a_begin=0, a_end=h)]
            parts += [_run(eng, dev, n_kmers, 1, 150, 3, a_begin=h + r, a_stride=3) for r in range(3)]
        sets = [_edge_set(p[0]) for p in parts]
        assert sum(len(s) for s in sets) == len(set().union(*sets)) == len(want[0])
        assert set().union(*sets) == _edge_set(want[0]), mode
        assert sum(p[2].n_increments for p in parts) == want[1]
        assert all(min(e[0] for e in s) >= h for s in sets[1:] if s) and all(e[0] < h for e in sets[0])


# ---- stage B ----------------------------------------------------------------------------------------------------
def _gpu_clouds(eng, batch, units, k, rare):
    reads, dunits = eng.upload_reads(batch, k), eng.upload_units(units, k)
    index = eng.build_index(eng._to_dev(rare.view(np.int64)))
    csr = eng.build_clouds(reads, dunits, k, index)
    return (csr.unit_ptr.cpu().numpy()[:units.n_units + 1], csr.ids.cpu().numpy().view(np.uint32)[:csr.n_entries],
            index)


@pytest.mark.gpu
@pytest.mark.parametrize("k", STAGE_B_KS)
@pytest.mark.parametrize("cap_mult,filter_bytes", [(0, None), (1, 0), (1, 1 << 60), (0, 0)])
def test_cloud_build(eng, k, cap_mult, filter_bytes):
    """The warp form of stage B with the probe table sized by the engine or at n + 1 slots (long chains that wrap), with
    and without the bitmap pre-filter."""
    from oracle import c_oracle
    batch, units, rare = _b_case(k)
    kw = {"index_cap_mult": cap_mult}
    if filter_bytes is not None:
        kw["index_filter_bytes"] = filter_bytes
    with _settings(eng, **kw):
        ptr, ids, index = _gpu_clouds(eng, batch, units, k, rare)
    if cap_mult == 1:  # the engine's floor of 64 slots holds the rare sets of k = 1, 2
        assert index.cap == max(64, rare.size + 1) and (k < 5 or index.cap == rare.size + 1)
    assert (index.filter is not None) == (filter_bytes == 0)
    wptr, wids = restate_clouds(batch, units, k, rare)
    assert np.array_equal(ptr, wptr) and np.array_equal(ids, wids)
    cptr, cids = c_oracle.clouds(c_oracle.unpacked_codes(batch), units, k, rare)
    assert np.array_equal(ptr, cptr) and np.array_equal(ids, cids)


BLOCK_KS = [1, 5, 11, 17, 31]


def _stage_b_kernels(eng, k):
    """Names of the stage-B kernels one build_clouds call launches (torch.profiler, CUDA activity)."""
    import torch
    batch, units, rare = _b_case(k)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _gpu_clouds(eng, batch, units, k, rare)
        torch.cuda.synchronize()
    return sorted({m.group(0) for e in prof.events() for m in [re.search(r"cloud_build\w*_kernel", e.name)] if m})


def _stage_b_child(out_dir):
    """Runs in a process started with CFK_CLOUD_MODE=block (the library latches the form on its first call)."""
    import json
    from centroflye_b200.engine import Engine
    eng = Engine()
    for k in BLOCK_KS:
        batch, units, rare = _b_case(k)
        ptr, ids, _ = _gpu_clouds(eng, batch, units, k, rare)
        np.savez(os.path.join(out_dir, f"k{k}.npz"), unit_ptr=ptr, ids=ids)
    with open(os.path.join(out_dir, "kernels.json"), "w") as f:
        json.dump(_stage_b_kernels(eng, BLOCK_KS[0]), f)


@pytest.mark.gpu
def test_cloud_build_block_form(eng, tmp_path):
    """The block form, in a child process started with CFK_CLOUD_MODE=block, against the restatement.  The kernels the
    child launched are read from the profiler, so a switch that stopped working would fail here instead of testing the
    warp form twice (this process, without the switch, serves as the probe's control)."""
    import json
    assert _stage_b_kernels(eng, BLOCK_KS[0]) == ["cloud_build_warp_kernel"]
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {TESTS!r}]; import test_gpu_cloud_graph as t; "
            f"t._stage_b_child({str(tmp_path)!r})")
    flags = ["-s"] if sys.flags.no_user_site else []
    env = dict(os.environ, CFK_CLOUD_MODE="block")
    res = subprocess.run([sys.executable, *flags, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    with open(tmp_path / "kernels.json") as f:
        assert json.load(f) == ["cloud_build_kernel"]
    for k in BLOCK_KS:
        batch, units, rare = _b_case(k)
        got = np.load(tmp_path / f"k{k}.npz")
        wptr, wids = restate_clouds(batch, units, k, rare)
        assert np.array_equal(got["unit_ptr"], wptr) and np.array_equal(got["ids"], wids), f"k={k}"


@pytest.mark.gpu
def test_filter_clouds(eng):
    """filter_clouds against py_oracle.filter_clouds for every pair of bounds from {0, 2, 2.5, 3, -inf, inf}."""
    from centroflye_b200.engine import CloudCSR
    from oracle import py_oracle
    rng = np.random.default_rng(81)
    n_kmers = 120
    units = [[_unit(rng.choice(n_kmers, size=int(rng.integers(0, 12)), replace=False))
              for _ in range(int(rng.integers(1, 6)))] for _ in range(40)]
    ptr, ids, last = _flatten(units)
    csr = CloudCSR(unit_ptr=eng._to_dev(ptr), ids=eng._to_dev(ids.astype(np.int32)), n_units=int(last.size),
                   n_entries=int(ids.size))
    clouds = {r: [set(u.tolist()) for u in rd] for r, rd in enumerate(units)}
    assert len(set(np.bincount(ids).tolist())) > 5  # multiplicities on both sides of every bound
    bounds = [0, 2, 2.5, 3, -math.inf, math.inf]
    for lo, hi in itertools.product(bounds, bounds):
        out = eng.filter_clouds(csr, n_kmers, lo, hi)
        want = py_oracle.filter_clouds(clouds, lo, hi)
        wsets = [u for r in range(len(units)) for u in want[r]]
        wptr = np.concatenate([[0], np.cumsum([len(u) for u in wsets])])
        wids = np.concatenate([np.sort(np.fromiter(u, dtype=np.int64, count=len(u))) for u in wsets])
        assert np.array_equal(out.unit_ptr.cpu().numpy()[:len(wsets) + 1], wptr), (lo, hi)
        assert np.array_equal(out.ids.cpu().numpy()[:out.n_entries], wids), (lo, hi)
