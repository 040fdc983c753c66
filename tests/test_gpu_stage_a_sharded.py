"""Two-phase stage A in the layouts of the multi-GPU exchange, and at the limits of phase 2, on ONE device.

Phase 1 (cfk_docfreq_emit) writes one record per distinct k-mer of a read into hash partitions; cfk_records_pack lays
a rank's partitions back to back; the all-to-all (dist.exchange_records) hands every rank its partition range, one
padded run per source rank; phase 2 (cfk_docfreq_count_parts) counts a partition over all sources.  Here the
all-to-all is restated in-process (exchange_local, itself checked against exchange_records under gloo), so the real
kernels see the exact buffers W ranks would give them, padding included -- and the real ShardedRecruiter runs with W
processes sharing one GPU, its collectives routed through the host.  References: the C oracle (oracle/c_oracle.py)
and numpy restatements of the record format and of phase 2.
"""
import datetime
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT  # noqa: F401  (puts the repo root on sys.path)

U32_MAX = 0xFFFFFFFF
KEY_BITS = np.uint64((1 << 62) - 1)
BIT63 = np.uint64(1 << 63)
TABLE_SLOTS = 3072  # slots of one phase-2 table: 2-key buckets, CFK_DOCFREQ_PART_DISTINCT * 2 / 3 of them


# ---- the record format (include/cfk.h: base j of the k-mer at bits 2j..2j+1; keys put the first base on top) ------
def key_to_raw(keys, k):
    """Library key (first base in the most significant bits) -> the order phase 1's records hold a k-mer in."""
    keys = np.asarray(keys, dtype=np.uint64)
    raw = np.zeros_like(keys)
    for j in range(k):  # base j of the k-mer
        raw |= ((keys >> np.uint64(2 * (k - 1 - j))) & np.uint64(3)) << np.uint64(2 * j)
    return raw


def raw_to_key(raw, k):
    """Phase 1's k-mer bits (bit 63 and the bits above 2k ignored) -> library key."""
    raw = np.asarray(raw, dtype=np.uint64)
    keys = np.zeros_like(raw)
    for j in range(k):
        keys = (keys << np.uint64(2)) | ((raw >> np.uint64(2 * j)) & np.uint64(3))
    return keys


def count_np(records, k):
    """Phase 2 restated: raw records (bit 63 = the read held the k-mer twice) -> (keys, n_reads, n_multi) by key."""
    records = np.asarray(records, dtype=np.uint64)
    keys, inv = np.unique(raw_to_key(records & KEY_BITS, k), return_inverse=True)
    nr = np.bincount(inv, minlength=keys.size).astype(np.uint32)
    nm = np.bincount(inv, weights=(records >> np.uint64(63)).astype(np.float64), minlength=keys.size).astype(np.uint32)
    return keys, nr, nm


def _scan(c):
    """exclusive_scan of Engine, restated with torch on the tensor's own device."""
    return torch.cat([torch.zeros(1, dtype=torch.int64, device=c.device), torch.cumsum(c.to(torch.int64), 0)])


# ---- the record all-to-all, in one process ----------------------------------------------------------------------
def exchange_local(sends, counts, world):
    """dist.exchange_records for all W ranks at once.  sends[s] = rank s's send buffer, laid out by
    padded_run_offsets(counts[s], world); counts[s] = int32[n_parts] records per partition.  -> per destination d:
    (recv, recv_counts, offsets), recv source-major with every source's run padded to RUN_ALIGN (the padding travels:
    it holds what the sender had there), offsets = padded_run_offsets(recv_counts) as global_rare_stream computes them."""
    from centroflye_b200.dist import padded_run_offsets
    per = counts[0].numel() // world
    starts, sizes = [], []
    for s in range(world):
        _, size = padded_run_offsets(counts[s], world, _scan)
        size = [int(x) for x in size.tolist()]
        sizes.append(size)
        starts.append(np.concatenate([[0], np.cumsum(size)]).tolist())
    out = []
    for d in range(world):
        recv_counts = torch.cat([counts[s][d * per: (d + 1) * per] for s in range(world)])
        n = sum(sizes[s][d] for s in range(world))
        recv = sends[0].new_empty(max(n, 1))
        if n:
            recv[:n] = torch.cat([sends[s][starts[s][d]: starts[s][d] + sizes[s][d]] for s in range(world)])
        offsets, _ = padded_run_offsets(recv_counts, world, _scan)
        out.append((recv, recv_counts, offsets))
    return out


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _init_gloo(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    # a rank that takes another branch than its peers raises after this long instead of hanging the test
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(minutes=3))


# ================================================================================================================
# host restatements, checked without a GPU
# ================================================================================================================
def test_key_raw_forms_are_inverse():
    rng = np.random.default_rng(1)
    for k in range(1, 32):
        x = rng.integers(0, 1 << (2 * k), size=2000, dtype=np.uint64)
        x[:2] = [0, (1 << (2 * k)) - 1]
        assert np.array_equal(raw_to_key(key_to_raw(x, k), k), x)
        assert np.array_equal(key_to_raw(raw_to_key(x, k), k), x)
        # known answer from the bases themselves: key = sum b_j 4^(k-1-j), raw = sum b_j 4^j
        bases = rng.integers(0, 4, size=k)
        key = sum(int(b) << (2 * (k - 1 - j)) for j, b in enumerate(bases))
        raw = sum(int(b) << (2 * j) for j, b in enumerate(bases))
        assert int(key_to_raw([key], k)[0]) == raw and int(raw_to_key([raw], k)[0]) == key


@pytest.mark.parametrize("k", [5, 15, 31])
def test_record_restatement_matches_oracle(k):
    """The gloo tests' restatement of phase 1 (_records_np, keys) in the device's raw form, counted by count_np,
    gives the C oracle's document frequencies: the host model the GPU tests below rely on."""
    from centroflye_b200.ingest import pack_reads
    from oracle import c_oracle
    from test_dist_gloo import _records_np
    rng = np.random.default_rng(k)
    codes = [_repetitive_read(rng, int(rng.integers(k - 1, 3000)), int(rng.integers(3, 300)), 0.05) for _ in range(12)]
    codes.append(codes[4].copy())
    batch = pack_reads(codes, [f"r{i}" for i in range(len(codes))])
    recs = _records_np(batch, k)
    raw = key_to_raw(recs & KEY_BITS, k) | (recs & BIT63)
    keys, nr, nm = count_np(raw, k)
    wk, wr, wm = c_oracle.docfreq(c_oracle.unpacked_codes(batch), batch, k)
    assert wk.size > 1000 and (wm > 0).any() and (wr > 1).any()
    assert np.array_equal(keys, wk) and np.array_equal(nr, wr) and np.array_equal(nm, wm)


def _exchange_worker(rank, world, port, out_dir):
    _init_gloo(rank, world, port)
    try:
        from centroflye_b200.dist import RUN_ALIGN, exchange_records, padded_run_offsets
        rng = np.random.default_rng(100 + world)  # every rank builds every rank's send buffer
        per = 7
        counts = [rng.integers(0, 40, size=world * per).astype(np.int32) for _ in range(world)]
        for c in counts:
            c[rng.random(c.size) < 0.3] = 0
            c[rng.integers(c.size)] = RUN_ALIGN  # a partition that ends exactly on a line
        counts[0][(world - 1) * per:] = 0  # rank 0 sends nothing to the last rank
        if world > 2:
            counts[1][:] = 0  # rank 1 sends nothing at all
        counts = [torch.from_numpy(c) for c in counts]
        sends = []
        for c in counts:
            _, sizes = padded_run_offsets(c, world, _scan)
            sends.append(torch.from_numpy(rng.integers(-(1 << 62), 1 << 62, size=max(int(sizes.sum()), 1))))
        want_recv, want_counts, want_off = exchange_local(sends, counts, world)[rank]
        recv, recv_counts, flags, n_sent = exchange_records(sends[rank], counts[rank], world, flags=torch.tensor([rank]))
        assert flags == [world - 1] and n_sent == int(counts[rank].sum())
        assert torch.equal(recv_counts, want_counts)
        off, sizes = padded_run_offsets(recv_counts, world, _scan)
        assert torch.equal(off, want_off)
        n = int(sizes.sum())
        assert recv.numel() == want_recv.numel() == max(n, 1)
        assert torch.equal(recv[:n], want_recv[:n])  # the runs and the padding between them
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_exchange_local_matches_exchange_records(tmp_path, world):
    mp.spawn(_exchange_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


# ================================================================================================================
# device helpers
# ================================================================================================================
@pytest.fixture(scope="module")
def eng():
    """An engine of this module's own: the tests here change its sizes, hints and mode and make it fall back on
    purpose (stream_fallbacks), none of which may reach the shared default_engine() other modules check."""
    from centroflye_b200.engine import Engine
    return Engine("cuda:0")


def _repetitive_read(rng, length, unit_len, div):
    unit = rng.integers(0, 4, size=unit_len, dtype=np.uint8)
    out = np.tile(unit, length // unit_len + 1)[:length].copy()
    flip = rng.random(length) < div
    out[flip] = rng.integers(0, 4, size=int(flip.sum()), dtype=np.uint8)
    return out


def _shard_codes(seed=7):
    """Repetitive reads (n_multi matters), exact copies next to their original (dealt to different shards), reads
    that share long stretches with others, and reads shorter than k."""
    rng = np.random.default_rng(seed)
    codes = [_repetitive_read(rng, int(rng.integers(3000, 20000)), int(rng.integers(40, 900)), 0.04) for _ in range(24)]
    for i in range(4):
        codes.insert(2 * i + 1, codes[2 * i].copy())
    for _ in range(6):
        src = codes[int(rng.integers(len(codes)))]
        a = int(rng.integers(0, src.size // 2))
        codes.append(np.concatenate([rng.integers(0, 4, size=700, dtype=np.uint8), src[a: a + src.size // 2],
                                     rng.integers(0, 4, size=300, dtype=np.uint8)]))
    codes += [codes[3][:10].copy(), codes[5][100:131].copy()]
    return codes


def _deal(codes, world):
    """Reads dealt round-robin over the shards; at W = 5 the middle shard gets no reads."""
    from centroflye_b200.ingest import pack_reads
    takers = [s for s in range(world) if not (world == 5 and s == 2)]
    mine = {s: [] for s in range(world)}
    for i, c in enumerate(codes):
        mine[takers[i % len(takers)]].append((i, c))
    return [pack_reads([c for _, c in mine[s]], [f"r{i}" for i, _ in mine[s]]) for s in range(world)]


_ORACLE = {}


def _oracle(codes, k):
    from centroflye_b200.ingest import pack_reads
    from oracle import c_oracle
    key = (id(codes), k)
    if key not in _ORACLE:
        batch = pack_reads(codes, [f"r{i}" for i in range(len(codes))])
        _ORACLE[key] = c_oracle.docfreq(c_oracle.unpacked_codes(batch), batch, k)
    return _ORACLE[key]


_CODES = _shard_codes()
N_PARTS = 120  # divisible by every world size below


def _emit(eng, batch, k, n_parts):
    """The real phase 1 of one shard -> (records, cursors, part_cap, k-mer occurrences)."""
    reads = eng.upload_reads(batch, k)
    n_local = batch.n_kmers(k)
    part_cap = 3 * (n_local // n_parts) + 2 * batch.n_reads + 512
    records, cursors, counters = eng.emit_records(reads, k, n_parts, part_cap)
    c = counters.cpu().tolist()
    assert c[1] == 0
    if c[0]:
        part_cap = int(cursors.max()) + 16
        records, cursors, counters = eng.emit_records(reads, k, n_parts, part_cap)
        assert counters.cpu().tolist()[:2] == [0, 0]
    return records, cursors, part_cap, n_local


def _poison(k):
    """A record whose k-mer occurs in the reads, with bit 63 set: a count that reads it comes out wrong."""
    wk, _, _ = _oracle(_CODES, k)
    return int((key_to_raw(wk[len(wk) // 2: len(wk) // 2 + 1], k) | BIT63).view(np.int64)[0])


def _fill_outside(buf, starts, lens, value):
    """buf (device int64) = value everywhere outside the runs [starts[i], starts[i] + lens[i])."""
    keep = np.zeros(buf.numel() + 1, dtype=np.int64)
    np.add.at(keep, np.asarray(starts, dtype=np.int64), 1)
    np.add.at(keep, np.asarray(starts, dtype=np.int64) + np.asarray(lens, dtype=np.int64), -1)
    hole = np.cumsum(keep)[:-1] == 0
    buf[torch.from_numpy(hole).to(buf.device)] = value
    return int(hole.sum())


def _count(eng, records, cursors, n_parts, part_cap, k, room, **kw):
    """Engine.count_records with band (1, U32_MAX, U32_MAX) and room for `room` rare keys -> sorted (keys, n_reads,
    n_multi) on the host, and the host counters."""
    eng.select_hint[("stream", True)] = room
    rare, nr, nm, counters, max_rare = eng.count_records(records, cursors, n_parts, part_cap, k,
                                                         band=(1, U32_MAX, U32_MAX), with_counts=True, **kw)
    c = counters.cpu().tolist()
    assert c[1] == 0 and c[4] <= max_rare
    keys = rare[: c[4]].cpu().numpy().view(np.uint64)
    o = np.argsort(keys)
    return keys[o], nr[: c[4]].cpu().numpy().view(np.uint32)[o], nm[: c[4]].cpu().numpy().view(np.uint32)[o], c


# ================================================================================================================
# phase 2 in the exchange layout (GPU)
# ================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("k", [11, 19, 31])
def test_count_over_exchanged_runs(eng, k, world):
    """Every shard's real phase 1 and cfk_records_pack, the all-to-all restated, then phase 2 per destination as
    global_rare_stream calls it (n_src = W, padded offsets, part_cap = 1, n_parts / W local partitions), the padding
    between runs full of poison: the union over destinations is the oracle's table, every key from one destination,
    at every grouping of partitions."""
    from centroflye_b200.dist import RUN_ALIGN, padded_run_offsets
    sends, counts = [], []
    for batch in _deal(_CODES, world):
        records, cursors, part_cap, n_local = _emit(eng, batch, k, N_PARTS)
        c = cursors.clamp(max=part_cap)
        offsets, _ = padded_run_offsets(c, world, eng.exclusive_scan)
        sends.append(eng.pack_records(records, part_cap, c, offsets, n_local + RUN_ALIGN * world))
        counts.append(c)
    assert sum(int(c.sum()) for c in counts) > 0 and (world != 5 or int(counts[2].sum()) == 0)
    poison = _poison(k)
    wk, wr, wm = _oracle(_CODES, k)
    exchanged, holes = [], 0
    for recv, recv_counts, offsets in exchange_local(sends, counts, world):
        # poison in the padding, and behind the last run: a run read at another run's offset stays in the buffer
        recv = torch.cat([recv, recv.new_empty(int(recv_counts.max()) + RUN_ALIGN)])
        holes += _fill_outside(recv, offsets.cpu().numpy(), recv_counts.cpu().numpy(), poison)
        exchanged.append((recv, recv_counts, offsets))
    assert holes > 0
    retried = 0
    for group in (1, 8, 64):
        got = []
        for recv, recv_counts, offsets in exchanged:
            keys, nr, nm, c = _count(eng, recv, recv_counts, N_PARTS // world, 1, k, wk.size + 1024, n_src=world,
                                     offsets=offsets, group=group)
            assert c[0] == 0 and c[5] == keys.size
            retried += c[6]
            got.append((keys, nr, nm))
        keys = np.concatenate([g[0] for g in got])
        assert np.unique(keys).size == keys.size  # a k-mer has one owner
        o = np.argsort(keys)
        assert np.array_equal(keys[o], wk)
        assert np.array_equal(np.concatenate([g[1] for g in got])[o], wr)
        assert np.array_equal(np.concatenate([g[2] for g in got])[o], wm)
    assert retried > 0  # some unit outgrew its table and was taken again partition by partition


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 5])
@pytest.mark.parametrize("k", [11, 31])
def test_count_over_strided_sources(eng, k, world):
    """The other multi-source layout: source s's partition p at records[s * src_stride + p * part_cap], cursors[s *
    n_parts + p] records of it.  Whatever lies beyond a cursor is poison and must not be read; a cursor beyond part_cap
    (what phase 1 leaves after an overflow) must be clamped to part_cap."""
    poison = _poison(k)
    shards = [_emit(eng, batch, k, N_PARTS) for batch in _deal(_CODES, world)]
    cur = np.concatenate([s[1].cpu().numpy()[:N_PARTS] for s in shards]).astype(np.int64)
    cap = int(cur.max())  # the fullest partition fills its buffer exactly
    stride = N_PARTS * cap
    host = np.full(world * stride + cap + 4096, poison, dtype=np.int64)  # (a tail: an unclamped read stays inside)
    for s, (records, cursors, part_cap, _) in enumerate(shards):
        r = records.cpu().numpy()
        for p in range(N_PARTS):
            n = int(cur[s * N_PARTS + p])
            host[s * stride + p * cap: s * stride + p * cap + n] = r[p * part_cap: p * part_cap + n]
    cur[cur == cap] = cap + 1000  # read unclamped, these would run into the next buffer (or the poisoned tail)
    records = eng._to_dev(host)
    cursors = eng._to_dev(cur.astype(np.int32))
    wk, wr, wm = _oracle(_CODES, k)
    for group in (1, 8):
        keys, nr, nm, c = _count(eng, records, cursors, N_PARTS, cap, k, wk.size + 1024, n_src=world,
                                 src_stride=stride, group=group)
        assert c[0] == 0
        assert np.array_equal(keys, wk) and np.array_equal(nr, wr) and np.array_equal(nm, wm)


@pytest.mark.gpu
@pytest.mark.parametrize("n_parts,world", [(7, 1), (2369, 1), (5000, 8)])
def test_records_pack_against_numpy(eng, n_parts, world):
    """cfk_records_pack: partition p's first min(cursors[p], part_cap) records to out[offsets[p]...], nothing else
    written -- over more partitions than its grid has blocks (148 * 16), with empty and exactly full partitions,
    cursors beyond part_cap (an overflowed phase 1) and the padded offsets of the exchange."""
    from centroflye_b200 import _lib
    from centroflye_b200.dist import padded_run_offsets
    rng = np.random.default_rng(n_parts)
    part_cap = 37
    cursors = rng.integers(0, part_cap + 1, size=n_parts).astype(np.int32)
    cursors[rng.random(n_parts) < 0.2] = 0
    cursors[rng.random(n_parts) < 0.2] = part_cap
    cursors[rng.random(n_parts) < 0.05] = part_cap + 9
    cursors[-1] = part_cap  # the last partition, which no first-round block of the grid reaches
    counts = np.minimum(cursors, part_cap)
    offsets, sizes = padded_run_offsets(torch.from_numpy(counts), world, _scan)
    offsets = offsets.numpy()
    records = rng.integers(-(1 << 62), 1 << 62, size=n_parts * part_cap)
    sentinel = -0x2152411021524111
    n_out = int(sizes.sum()) + 64
    out = torch.full((n_out,), sentinel, dtype=torch.int64, device=eng.device)
    d_rec, d_cur, d_off = eng._to_dev(records), eng._to_dev(cursors), eng._to_dev(offsets)  # alive across the call
    _lib.call("cfk_records_pack", eng._p(d_rec), part_cap, eng._p(d_cur), eng._p(d_off), n_parts, eng._p(out),
              eng._stream())
    want = np.full(n_out, sentinel, dtype=np.int64)
    for p in range(n_parts):
        want[offsets[p]: offsets[p] + counts[p]] = records[p * part_cap: p * part_cap + counts[p]]
    assert np.array_equal(out.cpu().numpy(), want)


# ================================================================================================================
# phase 2 at its limits, on synthetic records (GPU)
# ================================================================================================================
K_SYN = 31


def _dense_runs(runs, n_src, poison):
    """runs[s * n_parts + p] = uint64 raw records of source s, partition p -> (records, cursors, offsets) on the device
    in the receive layout of the exchange: source-major, every source's run padded to RUN_ALIGN, poison in the holes and
    behind the last run."""
    from centroflye_b200.dist import RUN_ALIGN, padded_run_offsets
    counts = torch.tensor([r.size for r in runs], dtype=torch.int32)
    offsets, sizes = padded_run_offsets(counts, n_src, _scan)
    host = np.full(int(sizes.sum()) + int(counts.max()) + RUN_ALIGN, poison, dtype=np.uint64)
    for r, o in zip(runs, offsets.tolist()):
        host[o: o + r.size] = r
    return _dev(host.view(np.int64)), _dev(counts.numpy()), _dev(offsets.numpy())


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _count_one_partition(eng, recs, n_src, room):
    """One partition's raw records counted by phase 2: one strided source (n_src = 1) or n_src dense runs."""
    recs = np.asarray(recs, dtype=np.uint64)
    poison = recs[0] | BIT63
    if n_src == 1:
        return _count(eng, _dev(recs.view(np.int64)), _dev(np.array([recs.size], dtype=np.int32)), 1,
                      max(recs.size, 1), K_SYN, room)
    records, cursors, offsets = _dense_runs(np.array_split(recs, n_src), n_src, poison)
    return _count(eng, records, cursors, 1, 1, K_SYN, room, n_src=n_src, offsets=offsets)


@pytest.mark.gpu
@pytest.mark.parametrize("n_src", [1, 3])
@pytest.mark.parametrize("multi", ["all", "some"])
def test_count_16_bit_read_counter(eng, n_src, multi):
    """A k-mer's further reads and further repeated reads share one 32-bit word in phase 2 (16 bits each): a k-mer in
    65 536 reads is exact, one in 65 537 reads must be reported (counters[0]) so the caller falls back.  Spread over
    three sources no source alone reaches the limit."""
    rng = np.random.default_rng(3 + n_src)
    key = np.uint64(int(rng.integers(0, 1 << 62)) & ((1 << (2 * K_SYN)) - 1))
    fill = np.unique(rng.integers(0, 1 << (2 * K_SYN), size=3000, dtype=np.uint64))
    fill = fill[fill != key]
    for n in (65536, 65537):
        recs = np.full(n, key, dtype=np.uint64)
        flagged = np.ones(n, bool) if multi == "all" else rng.random(n) < 0.3
        recs[flagged] |= BIT63
        both = np.concatenate([recs, fill])
        rng.shuffle(both)
        keys, nr, nm, c = _count_one_partition(eng, both, n_src, fill.size + 1024)
        if n == 65537:
            assert c[0] != 0
            continue
        assert c[0] == 0
        wk, wr, wm = count_np(both, K_SYN)
        assert np.array_equal(keys, wk) and np.array_equal(nr, wr) and np.array_equal(nm, wm)
        at = np.searchsorted(wk, raw_to_key([key], K_SYN)[0])
        assert nr[at] == 65536 and nm[at] == int(flagged.sum())


def _distinct_records(rng, d):
    """d distinct random k-mers, each in 1 to 3 records, bit 63 at random; shuffled."""
    keys = np.unique(rng.integers(0, 1 << (2 * K_SYN), size=d + d // 8 + 16, dtype=np.uint64))[:d]
    assert keys.size == d
    recs = np.repeat(keys, rng.integers(1, 4, size=d))
    recs[rng.random(recs.size) < 0.2] |= BIT63
    rng.shuffle(recs)
    return recs


@pytest.mark.gpu
@pytest.mark.parametrize("tables", [1, 2, 4, 16, 32, 64])
def test_count_split_stack(eng, tables):
    """One partition with more distinct k-mers than a table holds is counted by halves of its hash range, down to 64
    sub-ranges.  0.8 * tables * CFK_DOCFREQ_PART_DISTINCT distinct k-mers need `tables` sub-ranges and must come out
    exact (the margin: a sub-range's share depends on the hash)."""
    distinct = int(eng.lib.cfk_docfreq_part_distinct())
    assert distinct * 4 // 3 == TABLE_SLOTS
    rng = np.random.default_rng(tables)
    d = int(0.8 * tables * distinct)
    recs = _distinct_records(rng, d)
    for n_src in (1, 2):
        keys, nr, nm, c = _count_one_partition(eng, recs, n_src, d + 1024)
        assert c[0] == 0 and (c[6] > 0) == (d > TABLE_SLOTS)
        wk, wr, wm = count_np(recs, K_SYN)
        assert np.array_equal(keys, wk) and np.array_equal(nr, wr) and np.array_equal(nm, wm)


@pytest.mark.gpu
def test_count_split_stack_gives_up(eng):
    """1.3 * 64 tables' slots of distinct k-mers in one partition: even its 64 sub-ranges overflow -> counters[0]."""
    rng = np.random.default_rng(64)
    recs = _distinct_records(rng, int(1.3 * 64 * TABLE_SLOTS))
    for n_src in (1, 3):
        _, _, _, c = _count_one_partition(eng, recs, n_src, 1 << 20)
        assert c[0] != 0


@pytest.mark.gpu
def test_count_rare_output_too_small(eng):
    """Phase 2 with three dense sources and a rare output smaller than the band's k-mers: counters[4] is the true
    number, nothing is written past max_rare, and what was written is a part of the true set with its counts."""
    from centroflye_b200 import _lib
    rng = np.random.default_rng(8)
    n_parts, n_src, k = 6, 3, K_SYN
    keys = np.unique(rng.integers(0, 1 << (2 * k), size=20000, dtype=np.uint64))
    recs = np.repeat(keys, rng.integers(1, 7, size=keys.size))
    recs[rng.random(recs.size) < 0.15] |= BIT63
    rng.shuffle(recs)
    part = (recs & KEY_BITS) % np.uint64(n_parts)  # phase 2 only needs a k-mer's records in one partition
    src = rng.integers(0, n_src, size=recs.size)
    runs = [recs[(src == s) & (part == p)] for s in range(n_src) for p in range(n_parts)]
    records, cursors, d_off = _dense_runs(runs, n_src, recs[0] | BIT63)
    lo, hi, mn = 2, 4, 1
    wk, wr, wm = count_np(recs, k)
    band = (wr >= lo) & (wr <= hi) & (wm <= mn)
    n_true = int(band.sum())
    assert n_true > 1000
    for max_rare in (0, n_true // 3, n_true - 1, n_true):
        spare = 257
        out_k = torch.full((max_rare + spare,), -7, dtype=torch.int64, device=eng.device)
        out_r = torch.full((max_rare + spare,), -7, dtype=torch.int32, device=eng.device)
        out_m = torch.full((max_rare + spare,), -7, dtype=torch.int32, device=eng.device)
        counters = eng._counters()
        _lib.call("cfk_docfreq_count_parts", eng._p(records), 1, eng._p(cursors), eng._p(d_off), n_parts, n_src, 0, 1,
                  k, lo, hi, mn, eng._p(out_k), eng._p(out_r), eng._p(out_m), max_rare, None, 0, eng._p(counters),
                  eng.n_sms, eng._stream())
        c = counters.cpu().tolist()
        assert c[0] == 0 and c[4] == n_true and c[5] == wk.size
        for out in (out_k, out_r, out_m):
            assert (out[max_rare:].cpu().numpy() == -7).all()
        got = out_k[:max_rare].cpu().numpy().view(np.uint64)
        at = np.searchsorted(wk, got)
        assert np.unique(got).size == max_rare and (wk[np.minimum(at, wk.size - 1)] == got).all() and band[at].all()
        assert np.array_equal(out_r[:max_rare].cpu().numpy().view(np.uint32), wr[at])
        assert np.array_equal(out_m[:max_rare].cpu().numpy().view(np.uint32), wm[at])


# ================================================================================================================
# whole stage A on one GPU at the counter limit
# ================================================================================================================
SHORT_LEN, SHORT_K = 48, 19


def _shared_kmer_codes(n, seed=11):
    """n random reads of 48 bases that all hold one 19-mer; every fourth holds it twice (at 0 and at 29)."""
    rng = np.random.default_rng(seed)
    shared = rng.integers(0, 4, size=SHORT_K, dtype=np.uint8)
    codes = rng.integers(0, 4, size=(n, SHORT_LEN), dtype=np.uint8)
    at = rng.integers(0, SHORT_LEN - SHORT_K + 1, size=n)
    twice = np.arange(n) % 4 == 0
    at[twice] = 0
    cols = at[:, None] + np.arange(SHORT_K)
    codes[np.arange(n)[:, None], cols] = shared
    codes[twice, SHORT_LEN - SHORT_K:] = shared
    key = 0
    for b in shared:
        key = (key << 2) | int(b)
    return list(codes), np.uint64(key), int(twice.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [65536, 65537])
def test_stage_a_at_read_counter_limit(eng, n):
    """65 536 reads sharing a k-mer are counted by the two-phase path; 65 537 are not: phase 1 first overflows (the
    k-mer's records all land in one partition) and is launched again, then phase 2 reports the k-mer and the call
    falls back to the single-kernel form -- exactly once per call, with the oracle's counts either way."""
    from centroflye_b200.ingest import pack_reads
    from oracle import c_oracle
    codes, key, n_twice = _shared_kmer_codes(n)
    batch = pack_reads(codes, [f"s{i}" for i in range(n)])
    k = SHORT_K
    wk, wr, wm = c_oracle.docfreq(c_oracle.unpacked_codes(batch), batch, k)
    at = np.searchsorted(wk, key)
    assert wk[at] == key and wr[at] == n and wm[at] == n_twice
    emit, emits = eng.emit_records, []

    def counted(*a, **kw):
        emits.append(1)
        return emit(*a, **kw)
    eng.docfreq_mode = "stream"
    eng.emit_records = counted
    try:
        reads = eng.upload_reads(batch, k)
        eng.part_cap_seen.clear()
        before = eng.stream_fallbacks
        table = eng.count_docfreq(reads, k)
        assert len(emits) == 2  # the first partition buffers are too small for the shared k-mer's records
        assert eng.stream_fallbacks == before + (n > 65536) and table.dense == (n <= 65536)
        keys, nr, nm = eng.table_select(table, 0, U32_MAX, U32_MAX, with_counts=True)
        keys = keys.cpu().numpy().view(np.uint64)
        o = np.argsort(keys)
        assert np.array_equal(keys[o], wk)
        assert np.array_equal(nr.cpu().numpy().view(np.uint32)[o], wr)
        assert np.array_equal(nm.cpu().numpy().view(np.uint32)[o], wm)
        eng.part_cap_seen.clear()
        before, emits[:] = eng.stream_fallbacks, []
        rare = eng.rare_kmers(reads, k, 60000, U32_MAX, U32_MAX)
        assert len(emits) == 2 and eng.stream_fallbacks == before + (n > 65536)
        assert rare.cpu().numpy().view(np.uint64).tolist() == [int(key)]
    finally:
        eng.__dict__.pop("emit_records", None)


# ================================================================================================================
# the sharded path: W processes on one GPU (GPU)
# ================================================================================================================
def _collectives_through_host():
    """torch.distributed's all_to_all_single, all_gather_into_tensor and all_reduce, made to take CUDA tensors over
    gloo: the wrapper moves them to the host and the result back.  dist.py looks these functions up at every call."""
    a2a, gather, reduce = dist.all_to_all_single, dist.all_gather_into_tensor, dist.all_reduce

    def all_to_all_single(output, input, output_split_sizes=None, input_split_sizes=None, group=None):
        host = torch.empty(output.shape, dtype=output.dtype)
        a2a(host, input.cpu(), output_split_sizes, input_split_sizes, group=group)
        output.copy_(host)

    def all_gather_into_tensor(output, input, group=None):
        host = torch.empty(output.shape, dtype=output.dtype)
        gather(host, input.cpu(), group=group)
        output.copy_(host)

    def all_reduce(tensor, op=dist.ReduceOp.SUM, group=None):
        host = tensor.cpu()
        reduce(host, op=op, group=group)
        tensor.copy_(host)

    dist.all_to_all_single, dist.all_gather_into_tensor, dist.all_reduce = all_to_all_single, all_gather_into_tensor, all_reduce


RECRUIT = dict(k=19, max_nonuniq=3, min_d=1, max_d=150, min_cov=4)


def _recruit_reads():
    from centroflye_b200 import synth
    unit = synth.hor_unit(4, 60, 0.25, seed=5)
    genome, a0, alen = synth.simulate_genome(unit, 120, 0.02, 6, flank_len=2000)
    reads = synth.simulate_reads(genome, a0, alen, unit, 20, 0.05, 7, median_len=7000, sigma=0.4, min_len=5200,
                                 max_len=20000)
    return unit, reads


def _check_step(out, want, batch, units, k):
    """One ShardedRecruiter.step against c_oracle.recruit of the whole read set."""
    from oracle import c_oracle
    index, csr, res = out
    assert np.array_equal(index.sorted_keys.cpu().numpy().view(np.uint64), want["rare"]), "rare set"
    ptr, ids = c_oracle.clouds(c_oracle.unpacked_codes(batch), units, k, want["rare"])
    assert np.array_equal(csr.unit_ptr.cpu().numpy()[: units.n_units + 1], ptr), "this rank's cloud sizes"
    assert np.array_equal(csr.ids.cpu().numpy().view(np.uint32)[: ids.size], ids), "this rank's clouds"
    assert res.n_increments == want["n_increments"]
    got = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    canon = lambda e: e[np.lexsort((e[:, 3], e[:, 2], e[:, 1], e[:, 0]))]  # noqa: E731
    assert np.array_equal(canon(got), canon(want["edges"])), "edge set"
    assert np.array_equal(np.sort(res.selected.cpu().numpy().view(np.uint32)), want["selected"]), "unique k-mers"


def _sharded_worker(rank, world, port, out_dir, case):
    torch.cuda.set_device(0)
    _init_gloo(rank, world, port)
    try:
        _collectives_through_host()
        from centroflye_b200.dist import ShardedRecruiter
        from centroflye_b200.engine import Engine, band_to_int
        from centroflye_b200.ingest import batch_from_synth, pack_reads, units_from_boundaries
        from oracle import c_oracle
        eng = Engine("cuda:0")
        emits = []
        emit = eng.emit_records

        def counted(*a, **kw):
            emits.append(1)
            return emit(*a, **kw)
        eng.emit_records = counted
        k, mn, min_d, max_d, min_cov = (RECRUIT[x] for x in ("k", "max_nonuniq", "min_d", "max_d", "min_cov"))
        if case in ("plain", "empty_rank"):
            lo, hi = band_to_int(0.9 * 20 * 0.4, 3.0 * 20 * 0.4)
            unit, reads = _recruit_reads()
            whole_batch, whole_units = batch_from_synth(reads, len(unit))
            want = c_oracle.recruit(whole_batch, whole_units, k, lo, hi, mn, min_d, max_d, min_cov, threads=2)
            assert want["rare"].size > 100 and want["edges"].shape[0] > 20
            if case == "plain":
                mine = reads[rank::world]
            else:  # the last rank holds no reads at all
                mine = reads[rank::world - 1] if rank < world - 1 else []
            batch, units = batch_from_synth(mine, len(unit))
            rec = ShardedRecruiter(eng, batch, units, k, rank, world)
            step = lambda: rec.step(lo, hi, mn, min_d, max_d, min_cov)  # noqa: E731
            eng.docfreq_mode = "stream"
            for _ in range(2):  # the second step runs with the adapted partition grouping and output sizes
                _check_step(step(), want, batch, units, k)
            assert eng.stream_fallbacks == 0
            if case == "plain":
                # the table-based exchanges give the same rare set: all-to-all of the tables, nominate-then-sum
                eng.docfreq_mode = "resident"
                for nominate in (False, True):
                    rec.nominate = nominate
                    index = step()[0]
                    assert np.array_equal(index.sorted_keys.cpu().numpy().view(np.uint64), want["rare"])
                # phase 1 of rank 1 overflows: every rank launches it again with the size all ranks need
                eng.docfreq_mode = "stream"
                if rank == 1:
                    plan = eng.stream_plan
                    eng.stream_plan = lambda *a, **kw: (plan(*a, **kw)[0], 64)
                del emits[:]
                _check_step(step(), want, batch, units, k)
                assert len(emits) == 2 and eng.stream_fallbacks == 0
        elif case == "counter_limit":
            # 65 537 reads share one k-mer but no rank holds 65 536 of them: only the summed count crosses the limit
            codes, key, _ = _shared_kmer_codes(65537)
            mine = codes[rank::world]
            batch = pack_reads(mine, [f"s{i}" for i in range(rank, 65537, world)])
            units = units_from_boundaries(batch, [[0, SHORT_LEN]] * len(mine))
            whole = pack_reads(codes, [f"s{i}" for i in range(65537)])
            wk, wr, wm = c_oracle.docfreq(c_oracle.unpacked_codes(whole), whole, SHORT_K)
            lo, hi, mn = 2, U32_MAX, U32_MAX
            assert key in wk[wr >= 65537]
            rec = ShardedRecruiter(eng, batch, units, SHORT_K, rank, world)
            eng.docfreq_mode = "stream"
            assert rec.global_rare_stream(lo, hi, mn) is None  # on every rank
            index = rec.step(lo, hi, mn, min_d, max_d, min_cov)[0]  # falls back to the table exchange
            assert np.array_equal(index.sorted_keys.cpu().numpy().view(np.uint64), wk[wr >= lo])
        else:
            raise AssertionError(case)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def _spawn(tmp_path, world, case):
    mp.spawn(_sharded_worker, args=(world, _free_port(), str(tmp_path), case), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 4])
def test_sharded_recruiter_on_one_gpu(tmp_path, world):
    """ShardedRecruiter.step with W ranks sharing one GPU == c_oracle.recruit of the whole read set (rare set, edges,
    unique k-mers, increments, every rank's own clouds), twice; == the table-based exchanges; and again after one
    rank's phase 1 ran out of partition buffer (every rank launches phase 1 exactly twice)."""
    _spawn(tmp_path, world, "plain")


@pytest.mark.gpu
def test_sharded_recruiter_rank_without_reads(tmp_path):
    _spawn(tmp_path, 3, "empty_rank")


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_counter_limit_across_ranks(tmp_path, world):
    """A k-mer in 65 537 reads, none of the ranks holding 65 536 of them: phase 2 of its owner reports it, every rank
    leaves the record exchange together (global_rare_stream -> None) and step() takes the table exchange instead."""
    _spawn(tmp_path, world, "counter_limit")
