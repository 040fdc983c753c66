"""Kernel-level GPU tests through the C ABI: sort, scan, select, and the stage-C corner paths
(shared-memory table splitting, 64-bit slots, long occurrence lists) against numpy restatements."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from centroflye_b200.engine import default_engine
    return default_engine()


@pytest.mark.parametrize("n", [0, 1, 2, 31, 4095, 4096, 4097, 8192, 12289, 100003, 1 << 20, (1 << 20) + 77])
def test_sort_u64(eng, n):
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    if n > 10:
        keys[: n // 3] = keys[n // 3: 2 * (n // 3)]  # duplicates
    dev = eng._to_dev(keys.view(np.int64)) if n else eng._empty(0, eng.torch.int64)[:0]
    out = eng.sort_keys(dev)
    assert np.array_equal(out.cpu().numpy().view(np.uint64)[:n], np.sort(keys))


@pytest.mark.parametrize("n", [1, 5, 2047, 2048, 2049, 70001, 3 * 2048 * 1024 + 5])
def test_exclusive_scan(eng, n):
    rng = np.random.default_rng(n)
    v = rng.integers(0, 5000, size=n, dtype=np.int32)
    out = eng.exclusive_scan(eng._to_dev(v)).cpu().numpy()
    want = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(v.astype(np.int64), out=want[1:])
    assert np.array_equal(out[: n + 1], want)


@pytest.fixture(params=["exact", "sketch"])
def pair_mode(eng, request):
    """Both stage-C kernels: exact shared-memory tables and the counter sketch (3 <= min_cov <= 255)."""
    old, eng.pair_mode = eng.pair_mode, request.param
    yield request.param
    eng.pair_mode = old


def _csr_from_units(units, n_kmers):
    """units: list (per read) of lists (per unit) of sorted id arrays."""
    flat = [u for rd in units for u in rd]
    ptr = np.zeros(len(flat) + 1, dtype=np.int64)
    np.cumsum([len(u) for u in flat], out=ptr[1:])
    ids = np.concatenate(flat).astype(np.uint32) if flat else np.empty(0, np.uint32)
    last = np.concatenate([np.full(len(rd), 0) for rd in units]).astype(np.int32)
    pos = 0
    for rd in units:
        last[pos:pos + len(rd)] = pos + len(rd) - 1
        pos += len(rd)
    return ptr, ids, last


def _numpy_edges(units, n_kmers, min_d, max_d, min_cov, thr=0.8):
    """Dense restatement of dbkr.py:111-149 on integer ids (indicator-matrix products)."""
    dmax = min(max_d, max(len(rd) for rd in units) - 1)
    cnt = {}
    for d in range(max(min_d, 1), dmax + 1):
        c = np.zeros((n_kmers, n_kmers), dtype=np.int64)
        for rd in units:
            for i in range(len(rd) - d):
                c[np.ix_(rd[i], rd[i + d])] += 1
        np.fill_diagonal(c, 0)
        cnt[d] = c
    total = sum(cnt.values()) if cnt else np.zeros((n_kmers, n_kmers), dtype=np.int64)
    edges = set()
    for d, c in cnt.items():
        a, b = np.nonzero((c >= min_cov) & (c / np.maximum(total, 1) >= thr))
        edges |= {(int(x), int(y), d, int(c[x, y])) for x, y in zip(a, b)}
    return edges, int(sum(int(c.sum()) for c in cnt.values()))


def _run_dist(eng, units, n_kmers, min_d, max_d, min_cov, **kw):
    from centroflye_b200.engine import CloudCSR
    ptr, ids, last = _csr_from_units(units, n_kmers)
    csr = CloudCSR(unit_ptr=eng._to_dev(ptr), ids=eng._to_dev(ids.view(np.int32)), n_units=len(last),
                   n_entries=int(ids.size))
    res = eng.dist_edges(csr, eng._to_dev(last), n_kmers, min_d, max_d, min_cov, **kw)
    e = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    sel = set(res.selected.cpu().numpy().view(np.uint32).tolist())
    return {tuple(int(x) for x in row) for row in e}, sel, res


def test_dist_table_splitting(eng, pair_mode):
    """Clouds far larger than one warp table force the id-range splitting path."""
    rng = np.random.default_rng(1)
    n_kmers = 6000
    units = [[np.sort(rng.choice(n_kmers, size=3500, replace=False)) for _ in range(3)] for _ in range(5)]
    want, incr = _numpy_edges(units, n_kmers, 1, 150, 3)
    got, sel, res = _run_dist(eng, units, n_kmers, 1, 150, 3)
    assert res.n_increments == incr
    assert res.n_splits >= 0
    assert got == want
    assert sel == {e[0] for e in want} | {e[1] for e in want}


def test_dist_wide_slots_and_long_lists(eng, pair_mode):
    """An id present in > 32 units of one read (multi-chunk occurrence list) in a universe too large for
    32-bit slots: exercises the 64-bit table and counts > 1 per read."""
    rng = np.random.default_rng(2)
    n_real = 400
    n_kmers = (1 << 21) + 3  # ids are only < n_real, but slot width is chosen from n_kmers
    n_units = 2200
    rd = []
    for u in range(n_units):
        extra = rng.choice(np.arange(1, n_real), size=3, replace=False)
        rd.append(np.sort(np.concatenate([[0], extra])))
    units = [rd, [np.array([0, 7, 9]), np.array([0, 9]), np.array([7])]]
    dense_units = units
    want, incr = _numpy_edges(dense_units, n_real, 2, 40, 4)
    got, sel, res = _run_dist(eng, units, n_kmers, 2, 40, 4)
    assert res.n_increments == incr
    assert got == want


_SAT_CACHE = {}


def _saturation_case(min_cov):
    if min_cov not in _SAT_CACHE:
        rng = np.random.default_rng(7)
        n_kmers = 1500
        core = np.arange(0, 500, 2)            # 250 ids present in every unit of the long read: all hot together
        rd = [np.sort(np.concatenate([core, rng.choice(np.arange(501, 1400), size=40, replace=False)]))
              for _ in range(100)]
        noise = [[np.sort(rng.choice(1400, size=rng.integers(1, 200), replace=False)) for _ in range(rng.integers(1, 6))]
                 for _ in range(30)]
        # P = 1450 then, five units later, Q = 1451 in 260 short reads and R = 1452 in 254 of them:
        # cnt[5][P][Q] = 260 and cnt[5][P][R] = 254 sit on either side of min_cov = 255
        pairs = [[np.array([1450, int(rng.integers(0, 1400))]), *[np.empty(0, np.int64)] * 4,
                  np.array([1451, 1452] if i < 254 else [1451])] for i in range(260)]
        units = [rd] + noise + pairs
        _SAT_CACHE[min_cov] = (units, n_kmers) + _numpy_edges(units, n_kmers, 1, 12, min_cov)
    return _SAT_CACHE[min_cov]


@pytest.mark.parametrize("min_cov", [3, 254, 255])
def test_dist_sketch_saturation_and_set_overflow(eng, pair_mode, min_cov):
    """Counts far above the 8-bit sketch counters (a pair co-occurring in > 255 unit pairs), min_cov at both ends of
    the sketch range, and more simultaneous hot ids than the level-2 set holds (forces the id-range split)."""
    units, n_kmers, want, incr = _saturation_case(min_cov)
    got, sel, res = _run_dist(eng, units, n_kmers, 1, 12, min_cov)
    assert res.n_increments == incr
    assert got == want
    assert sel == {e[0] for e in want} | {e[1] for e in want}
    assert (1450, 1451, 5, 260) in got and ((1450, 1452, 5, 254) in got) == (min_cov <= 254)
    if pair_mode == "sketch" and min_cov == 3:  # only at a low threshold do all 250 core ids turn hot in one pass
        assert res.n_splits > 0


@pytest.mark.parametrize("seed", range(4))
def test_dist_sketch_random_clouds(eng, pair_mode, seed):
    """Random ragged clouds (empty units, one-unit reads, ids shared between neighbouring units)."""
    rng = np.random.default_rng(100 + seed)
    n_kmers = int(rng.integers(50, 700))
    units = []
    for _ in range(int(rng.integers(1, 60))):
        n_u = int(rng.integers(1, 40))
        base = rng.choice(n_kmers, size=min(n_kmers, int(rng.integers(1, 90))), replace=False)
        rd = []
        for _ in range(n_u):
            keep = base[rng.random(base.size) < 0.7]
            extra = rng.choice(n_kmers, size=int(rng.integers(0, 30)), replace=False)
            rd.append(np.unique(np.concatenate([keep, extra])) if rng.random() > 0.1 else np.empty(0, np.int64))
        units.append(rd)
    min_cov = int(rng.integers(3, 7))
    want, incr = _numpy_edges(units, n_kmers, 1, 150, min_cov)
    got, sel, res = _run_dist(eng, units, n_kmers, 1, 150, min_cov)
    assert res.n_increments == incr
    assert got == want


def test_dist_sharded_by_source_equals_whole(eng):
    rng = np.random.default_rng(3)
    n_kmers = 900
    units = [[np.sort(rng.choice(n_kmers, size=rng.integers(0, 120), replace=False)) for _ in range(rng.integers(1, 9))]
             for _ in range(40)]
    whole, _, res = _run_dist(eng, units, n_kmers, 1, 150, 2)
    want, incr = _numpy_edges(units, n_kmers, 1, 150, 2)
    assert whole == want and res.n_increments == incr
    parts = set()
    total_incr = 0
    for r in range(3):
        got, _, res_r = _run_dist(eng, units, n_kmers, 1, 150, 2, a_begin=r, a_stride=3)
        assert not (parts & got)
        parts |= got
        total_incr += res_r.n_increments
    assert parts == whole and total_incr == incr


@pytest.mark.parametrize("world", [1, 3, 8])
def test_occurrence_slices_concatenate_to_the_whole_inversion(eng, world):
    """What ShardedRecruiter.global_occurrences all-gathers: the lists of id slice r, in rank order, are the lists of
    Engine.build_occurrences (ragged clouds; ids absent from every cloud; more ranks than some slices have ids)."""
    from centroflye_b200.engine import CloudCSR
    rng = np.random.default_rng(11 + world)
    for n_kmers in (5, 333, 4000):
        units = [[np.sort(rng.choice(n_kmers, size=rng.integers(0, min(n_kmers, 150)), replace=False))
                  for _ in range(rng.integers(1, 12))] for _ in range(30)]
        ptr, ids, last = _csr_from_units(units, n_kmers)
        csr = CloudCSR(unit_ptr=eng._to_dev(ptr), ids=eng._to_dev(ids.view(np.int32)), n_units=len(last),
                       n_entries=int(ids.size))
        dlast = eng._to_dev(last)
        occ_ptr, occ, occ_last = eng.build_occurrences(csr, n_kmers, unit_last=dlast)
        want_ptr, want_occ = occ_ptr.cpu().numpy(), occ.cpu().numpy()
        # independent restatement: unit indices holding id a, ascending
        lists = [[] for _ in range(n_kmers)]
        for u in range(len(last)):
            for a in ids[ptr[u]: ptr[u + 1]]:
                lists[int(a)].append(u)
        assert want_occ.tolist() == [u for lst in lists for u in lst]
        assert np.array_equal(np.diff(want_ptr), [len(lst) for lst in lists])
        mults, occs = [], []
        for r in range(world):
            lo, hi = n_kmers * r // world, n_kmers * (r + 1) // world
            mult, sptr = eng.occurrence_slice_count(csr, lo, hi)
            n_occ = int(sptr[hi - lo].item())
            occs.append(eng.occurrence_slice_fill(csr, lo, hi, sptr, n_occ).cpu().numpy())
            mults.append(mult.cpu().numpy())
            assert n_occ == int(want_ptr[hi] - want_ptr[lo])
        assert np.array_equal(np.concatenate(mults), np.diff(want_ptr))
        assert np.array_equal(np.concatenate(occs), want_occ)
        assert np.array_equal(eng.occurrence_last(occ, dlast).cpu().numpy(), occ_last.cpu().numpy())
        assert np.array_equal(occ_last.cpu().numpy(), last[want_occ])


def test_table_select_partitions_cover_table(eng):
    from centroflye_b200 import synth
    from centroflye_b200.ingest import batch_from_synth
    unit = synth.random_unit(150, 3)
    genome, a0, alen = synth.simulate_genome(unit, 60, 0.02, 4, flank_len=300)
    reads = synth.simulate_reads(genome, a0, alen, unit, 5, 0.04, 5, median_len=6000, sigma=0.2, min_len=5300, max_len=9000)
    batch, _ = batch_from_synth(reads, len(unit))
    dev = eng.upload_reads(batch, 17)
    table = eng.count_docfreq(dev, 17)
    allk, nr, nm = eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True)
    whole = dict(zip(allk.cpu().numpy().tolist(), zip(nr.cpu().numpy().tolist(), nm.cpu().numpy().tolist())))
    merged = {}
    for part in range(3):
        k_, r_, m_ = eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True, n_parts=3, part=part)
        for key, a, b in zip(k_.cpu().numpy().tolist(), r_.cpu().numpy().tolist(), m_.cpu().numpy().tolist()):
            assert key not in merged
            merged[key] = (a, b)
    assert merged == whole
    # owner-side merge of two half read sets equals counting everything at once
    from centroflye_b200.ingest import pack_reads
    from centroflye_b200.encode import unpack_codes
    codes = [unpack_codes(batch.packed, int(batch.read_off[-1] + batch.read_len[-1]))[o:o + n]
             for o, n in zip(batch.read_off, batch.read_len)]
    half = len(codes) // 2
    t_sum = eng.new_table(table.cap)
    for part_codes in (codes[:half], codes[half:]):
        b = pack_reads(part_codes, [f"r{i}" for i in range(len(part_codes))])
        t_part = eng.count_docfreq(eng.upload_reads(b, 17), 17)
        eng.merge_into(t_sum, *eng.table_select(t_part, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True))
    k2, r2, m2 = eng.table_select(t_sum, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True)
    assert dict(zip(k2.cpu().numpy().tolist(), zip(r2.cpu().numpy().tolist(), m2.cpu().numpy().tolist()))) == whole


def test_table_partition_matches_owner_rule(eng):
    from centroflye_b200.dist import key_owner_np
    rng = np.random.default_rng(9)
    keys = np.unique(rng.integers(0, 1 << 40, size=20000, dtype=np.uint64))
    nr = rng.integers(1, 50, size=keys.size, dtype=np.uint32)
    nm = rng.integers(0, 5, size=keys.size, dtype=np.uint32)
    table = eng.new_table(3 * keys.size + 7)
    eng.merge_into(table, eng._to_dev(keys.view(np.int64)), eng._to_dev(nr.view(np.int32)), eng._to_dev(nm.view(np.int32)))
    for parts in (1, 3, 8):
        counts = eng.part_count(table, parts)
        k_, r_, m_ = eng.part_scatter(table, parts, counts)
        counts = counts.cpu().numpy()
        owner = key_owner_np(keys, parts)
        assert np.array_equal(counts, np.bincount(owner, minlength=parts))
        got_k = k_.cpu().numpy().view(np.uint64)
        off = np.concatenate([[0], np.cumsum(counts)])
        for p in range(parts):
            seg = got_k[off[p]:off[p + 1]]
            assert (key_owner_np(seg, parts) == p).all()
        order = np.argsort(got_k)
        assert np.array_equal(got_k[order], keys)
        assert np.array_equal(r_.cpu().numpy().view(np.uint32)[order], nr)
        assert np.array_equal(m_.cpu().numpy().view(np.uint32)[order], nm)


@pytest.fixture(params=["stream", "resident", "tiled"])
def docfreq_mode(eng, request):
    """The stage-A kernels: two-phase (emit records per read, apply them per hash partition), (read, pass) items
    updating the table directly, and one block per read."""
    old, eng.docfreq_mode = eng.docfreq_mode, request.param
    yield request.param
    eng.docfreq_mode = old


def _repetitive_read(rng, length, unit_len, div):
    unit = rng.integers(0, 4, size=unit_len, dtype=np.uint8)
    out = np.tile(unit, length // unit_len + 1)[:length].copy()
    flip = rng.random(length) < div
    out[flip] = rng.integers(0, 4, size=int(flip.sum()), dtype=np.uint8)
    return out


@pytest.mark.parametrize("k", [1, 5, 19, 31])
def test_docfreq_read_shapes(eng, docfreq_mode, k):
    """Stage A on reads of every shape the kernels treat differently: shorter than k, exactly k, one set pass,
    several passes (> 29 k k-mers), too long to stay resident in shared memory (> 655 kb), all highly repetitive
    (so n_multi matters) -- against the C restatement of dbkr.py:39-63."""
    from centroflye_b200.ingest import pack_reads
    from oracle import c_oracle
    rng = np.random.default_rng(100 + k)
    lens = [0, k - 1, k, k + 1, 63, 64, 65, 1000, 8191, 8192, 8200, 29000, 31000, 70001, 131072, 300000, 700000, 5000, 5000]
    codes = [_repetitive_read(rng, max(n, 0), int(rng.integers(20, 400)), 0.02) for n in lens]
    codes[-1] = codes[-2].copy()  # the same read twice: n_reads 2, n_multi per read as before
    batch = pack_reads(codes, [f"r{i}" for i in range(len(codes))])
    table = eng.count_docfreq(eng.upload_reads(batch, k), k)
    keys, nr, nm = eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True)
    keys = keys.cpu().numpy().view(np.uint64)
    order = np.argsort(keys)
    wk, wr, wm = c_oracle.docfreq(c_oracle.unpacked_codes(batch), batch, k)
    assert np.array_equal(keys[order], wk)
    assert np.array_equal(nr.cpu().numpy().view(np.uint32)[order], wr)
    assert np.array_equal(nm.cpu().numpy().view(np.uint32)[order], wm)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_docfreq_claim_races(eng, docfreq_mode, seed):
    """The atomics-free per-read set of the two-phase kernel resolves racing claims in its verify phase.  Reads made
    to provoke them: tiny alphabets / short periods (a few distinct k-mers hit by thousands of positions at once),
    many exact copies of one segment at varying offsets, and random reads in between -- against the C restatement of
    dbkr.py:39-63 at a k where nearly every position of the periodic reads is a duplicate."""
    from centroflye_b200.ingest import pack_reads
    from oracle import c_oracle
    rng = np.random.default_rng(seed)
    k = [7, 11, 19][seed - 1]
    codes = []
    for period in (1, 2, 3, 5, 17, 64, 171):
        unit = rng.integers(0, 4, size=period, dtype=np.uint8)
        for n in (5000, 40000, 90000):
            codes.append(np.tile(unit, n // period + 1)[:n].copy())
    seg = rng.integers(0, 4, size=3000, dtype=np.uint8)
    for _ in range(40):
        parts = [seg if rng.random() < 0.7 else rng.integers(0, 4, size=int(rng.integers(10, 4000)), dtype=np.uint8)
                 for _ in range(int(rng.integers(2, 30)))]
        codes.append(np.concatenate(parts))
    for _ in range(60):
        codes.append(_repetitive_read(rng, int(rng.integers(5000, 120000)), int(rng.integers(150, 2100)), 0.06))
    batch = pack_reads(codes, [f"r{i}" for i in range(len(codes))])
    table = eng.count_docfreq(eng.upload_reads(batch, k), k)
    keys, nr, nm = eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True)
    keys = keys.cpu().numpy().view(np.uint64)
    order = np.argsort(keys)
    wk, wr, wm = c_oracle.docfreq(c_oracle.unpacked_codes(batch), batch, k)
    assert np.array_equal(keys[order], wk)
    assert np.array_equal(nr.cpu().numpy().view(np.uint32)[order], wr)
    assert np.array_equal(nm.cpu().numpy().view(np.uint32)[order], wm)


def test_stream_count_splits_oversized_partitions(eng):
    """Phase 2 of the two-phase stage A plans a partition for cfk_docfreq_part_target() k-mer occurrences but its
    block's table holds fewer distinct k-mers: reads without repeats (every k-mer new) overflow it, and the kernel must
    take the partition again by halves of its hash range -- same counts, no fall-back to the single-kernel form."""
    from centroflye_b200.ingest import pack_reads
    from oracle import c_oracle
    rng = np.random.default_rng(5)
    codes = [rng.integers(0, 4, size=int(rng.integers(20000, 60000)), dtype=np.uint8) for _ in range(60)]
    codes += [codes[3][1000:30000].copy(), codes[7].copy()]  # two reads sharing long stretches with others
    batch = pack_reads(codes, [f"r{i}" for i in range(len(codes))])
    k = 21
    assert int(eng.lib.cfk_docfreq_part_target()) > int(eng.lib.cfk_docfreq_part_distinct())
    old, eng.docfreq_mode = eng.docfreq_mode, "stream"
    old_group = eng.stream_group
    try:
        for group in (1, 8):  # grouped units that do not fit are retried partition by partition, then split
            eng.stream_group = group
            before = eng.stream_fallbacks
            table = eng.count_docfreq(eng.upload_reads(batch, k), k)
            assert table.dense and eng.stream_fallbacks == before
            keys, nr, nm = eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True)
            keys = keys.cpu().numpy().view(np.uint64)
            order = np.argsort(keys)
            wk, wr, wm = c_oracle.docfreq(c_oracle.unpacked_codes(batch), batch, k)
            assert np.array_equal(keys[order], wk)
            assert np.array_equal(nr.cpu().numpy().view(np.uint32)[order], wr)
            assert np.array_equal(nm.cpu().numpy().view(np.uint32)[order], wm)
    finally:
        eng.docfreq_mode, eng.stream_group = old, old_group


def test_stream_partition_buffers_grow(eng):
    """A k-mer present in every read adds one record per read to ONE partition: with a deliberately small first guess
    the buffers overflow, phase 1 reports the size it needed and the call repeats itself with it."""
    from centroflye_b200.ingest import pack_reads
    from oracle import c_oracle
    rng = np.random.default_rng(9)
    shared = rng.integers(0, 4, size=400, dtype=np.uint8)
    codes = [np.concatenate([rng.integers(0, 4, size=5200, dtype=np.uint8), shared,
                             rng.integers(0, 4, size=300, dtype=np.uint8)]) for _ in range(700)]
    batch = pack_reads(codes, [f"r{i}" for i in range(len(codes))])
    k = 19
    old = (eng.docfreq_mode, eng.part_slack, dict(eng.part_cap_seen))
    eng.docfreq_mode, eng.part_slack = "stream", 0.2
    eng.part_cap_seen.clear()
    plan = eng.stream_plan
    eng.stream_plan = lambda *a, **kw: (plan(*a, **kw)[0], 64)  # 64 records per partition buffer: far too few
    try:
        rare = eng.rare_kmers(eng.upload_reads(batch, k), k, 600, 700, 3)
        assert max(eng.part_cap_seen.values()) > 64  # the measured size was remembered
        wk, wr, wm = c_oracle.docfreq(c_oracle.unpacked_codes(batch), batch, k)
        want = wk[(wr >= 600) & (wr <= 700) & (wm <= 3)]
        assert want.size >= 400 - k
        assert np.array_equal(np.sort(rare.cpu().numpy().view(np.uint64)), want)
    finally:
        eng.stream_plan = plan
        eng.docfreq_mode, eng.part_slack = old[0], old[1]
        eng.part_cap_seen.clear()
        eng.part_cap_seen.update(old[2])


def test_negative_max_nonuniq_selects_nothing(eng):
    """dbkr.py:57-62: with max_nonuniq < 0 the test `non_unique_freqs[kmer] <= max_nonuniq` fails for every k-mer, so
    all_kmers ends empty and so does the rare set (ADVICE r1: the u32 conversion must not turn -1 into "everything")."""
    from centroflye_b200.ingest import pack_reads
    rng = np.random.default_rng(2)
    codes = [_repetitive_read(rng, 9000, 300, 0.03) for _ in range(12)]
    batch = pack_reads(codes, [f"r{i}" for i in range(len(codes))])
    for mode in ("stream", "resident"):
        old, eng.docfreq_mode = eng.docfreq_mode, mode
        try:
            assert eng.rare_kmers(eng.upload_reads(batch, 15), 15, 1, 100, -1).numel() == 0
            assert eng.rare_kmers(eng.upload_reads(batch, 15), 15, 5, 4, 3).numel() == 0  # empty band
            assert eng.rare_kmers(eng.upload_reads(batch, 15), 15, 1, 100, 3).numel() > 0
        finally:
            eng.docfreq_mode = old


def test_merge_sorted_runs(eng):
    """cfk_merge_sorted_runs: runs of distinct keys (sizes 0, 1, many) merged by ranking == numpy sort."""
    from centroflye_b200 import _lib
    import torch
    rng = np.random.default_rng(4)
    keys = np.unique(rng.integers(0, 1 << 62, size=200000, dtype=np.int64))
    rng.shuffle(keys)
    sizes = [0, 1, 70000, 3, keys.size - 70004]
    runs, at = [], 0
    for s in sizes:
        runs.append(np.sort(keys[at:at + s]))
        at += s
    cat = np.concatenate(runs)
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    d_cat, d_ptr = eng._to_dev(cat), eng._to_dev(ptr)
    out = eng._empty(cat.size, torch.int64)
    _lib.call("cfk_merge_sorted_runs", eng._p(d_cat), eng._p(d_ptr), len(sizes), int(cat.size), eng._p(out), eng._stream())
    assert np.array_equal(out.cpu().numpy(), np.sort(keys))


def test_cloud_build_with_index_filter(eng):
    """The bitmap pre-filter of stage B (cfk_index_filter_build; used when the rare-set index outgrows L2) must not change
    a single cloud: same CSR with the filter forced on as without it."""
    import bench
    unit, batch, units = bench.simulate("cenx", 0.03)
    k = 19
    reads, dunits = eng.upload_reads(batch, k), eng.upload_units(units, k)
    rare = eng.rare_kmers(reads, k, 6, 40, 3)
    assert rare.numel() > 1000
    old = eng.index_filter_bytes
    try:
        eng.index_filter_bytes = 1 << 60
        plain = eng.build_index(rare)
        assert plain.filter is None
        eng.index_filter_bytes = 0
        filtered = eng.build_index(rare)
        assert filtered.filter is not None and filtered.filter_bits >= 20
    finally:
        eng.index_filter_bytes = old
    a, b = eng.build_clouds(reads, dunits, k, plain), eng.build_clouds(reads, dunits, k, filtered)
    assert a.n_entries == b.n_entries > 0
    assert np.array_equal(a.unit_ptr.cpu().numpy(), b.unit_ptr.cpu().numpy())
    assert np.array_equal(a.ids.cpu().numpy(), b.ids.cpu().numpy())


def test_stream_launch_finish_equals_synchronous_call(eng):
    """docfreq_stream_launch / docfreq_stream_finish (the streaming bench enqueues batch i + 1 before reading batch i's
    counters back): same rare keys and the same table as the synchronous docfreq_stream, also when the first launch
    finds its partition buffers too small and is repeated."""
    import torch
    from centroflye_b200.ingest import pack_reads
    rng = np.random.default_rng(12)
    batches = []
    for b in range(3):
        codes = [_repetitive_read(rng, int(rng.integers(6000, 50000)), int(rng.integers(200, 2100)), 0.05) for _ in range(40)]
        batches.append(pack_reads(codes, [f"b{b}r{i}" for i in range(len(codes))]))
    k, band = 17, (3, 30, 3)
    old = (eng.docfreq_mode, dict(eng.part_cap_seen), eng.part_slack)
    eng.docfreq_mode = "stream"
    try:
        want = []
        for batch in batches:
            rare, table = eng.docfreq_stream(eng.upload_reads(batch, k), k, band=band, want_table=True)
            keys, nr, nm = eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True)
            o = np.argsort(keys.cpu().numpy().view(np.uint64))
            want.append((np.sort(rare.cpu().numpy().view(np.uint64)), keys.cpu().numpy().view(np.uint64)[o],
                         nr.cpu().numpy()[o], nm.cpu().numpy()[o]))
        eng.part_cap_seen.clear()
        eng.part_slack = 0.05  # the first launches overflow and are repeated inside finish()
        n_max = max(int(b.n_bases) for b in batches)
        bufs = [torch.empty(2 * n_max, dtype=torch.int64, device=eng.device) for _ in range(2)]
        handles, got = [], []
        for i, batch in enumerate(batches):
            handles.append(eng.docfreq_stream_launch(eng.upload_reads(batch, k), k, band=band, table_buf=bufs[i & 1]))
            if i >= 1:
                got.append(eng.docfreq_stream_finish(handles[i - 1]))
                rare, table = got[-1]
                keys, nr, nm = eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True)
                o = np.argsort(keys.cpu().numpy().view(np.uint64))
                w = want[i - 1]
                assert np.array_equal(np.sort(rare.cpu().numpy().view(np.uint64)), w[0])
                assert np.array_equal(keys.cpu().numpy().view(np.uint64)[o], w[1])
                assert np.array_equal(nr.cpu().numpy()[o], w[2]) and np.array_equal(nm.cpu().numpy()[o], w[3])
        rare, table = eng.docfreq_stream_finish(handles[-1])
        assert np.array_equal(np.sort(rare.cpu().numpy().view(np.uint64)), want[-1][0]) and table.cap == want[-1][1].size
    finally:
        eng.docfreq_mode, eng.part_slack = old[0], old[2]
        eng.part_cap_seen.clear()
        eng.part_cap_seen.update(old[1])


def test_stream_rare_output_too_small_on_both_paths(eng):
    """A rare output too small for the band: rare_kmers and a docfreq_stream_launch / docfreq_stream_finish pair both
    run phase 2 again on the records they keep (phase 1 once per call), return what a call with ample room returns and
    leave a hint large enough for the next call."""
    from centroflye_b200 import synth
    from centroflye_b200.ingest import batch_from_synth
    unit = synth.hor_unit(4, 60, 0.25, seed=5)
    genome, a0, alen = synth.simulate_genome(unit, 120, 0.02, 6, flank_len=2000)
    batch, _ = batch_from_synth(synth.simulate_reads(genome, a0, alen, unit, 20, 0.05, 7, median_len=7000, sigma=0.4,
                                                     min_len=5200, max_len=20000), len(unit))
    k, band, key = 19, (8, 24, 3), ("stream", False)
    old = (eng.docfreq_mode, dict(eng.select_hint))
    emit, emits = eng.emit_records, []

    def counted(*a, **kw):
        emits.append(1)
        return emit(*a, **kw)
    eng.docfreq_mode = "stream"
    try:
        reads = eng.upload_reads(batch, k)
        eng.select_hint[key] = 1 << 20
        want = np.sort(eng.rare_kmers(reads, k, *band).cpu().numpy().view(np.uint64))
        assert want.size > 100
        eng.emit_records = counted
        eng.select_hint[key] = 1
        got = eng.rare_kmers(reads, k, *band)
        assert len(emits) == 1 and np.array_equal(np.sort(got.cpu().numpy().view(np.uint64)), want)
        assert eng.select_hint[key] > want.size
        eng.select_hint[key] = 1
        got, table = eng.docfreq_stream_finish(eng.docfreq_stream_launch(reads, k, band=band))
        assert len(emits) == 2 and table is None and np.array_equal(np.sort(got.cpu().numpy().view(np.uint64)), want)
        assert eng.select_hint[key] > want.size
    finally:
        eng.__dict__.pop("emit_records", None)
        eng.docfreq_mode = old[0]
        eng.select_hint.clear()
        eng.select_hint.update(old[1])
