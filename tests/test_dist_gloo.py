"""world_size-2 and -3 tests of the multi-GPU exchange logic (centroflye_b200/dist.py) on the gloo backend, CPU tensors.

The device kernels cannot run here; what is checked is everything AROUND them: the variable-size all-to-all /
all-gather helpers, the owner rule, the additivity of (n_reads, n_multi) over read shards, the global numbering
of all-gathered cloud shards, and that dealing source k-mers round-robin partitions the edge set.  The per-shard
counting itself is done by the CPU oracle (test infrastructure), in place of libcfk.so.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT  # noqa: F401  (puts the repo root on sys.path)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dataset():
    from centroflye_b200 import synth
    from centroflye_b200.ingest import batch_from_synth
    unit = synth.hor_unit(3, 50, 0.25, seed=3)
    genome, a0, alen = synth.simulate_genome(unit, 90, 0.03, 4, flank_len=800)
    reads = synth.simulate_reads(genome, a0, alen, unit, 14, 0.04, 5, median_len=6500, sigma=0.3, min_len=5200,
                                 max_len=12000)
    return unit, reads, batch_from_synth


KEY_BITS = np.uint64((1 << 62) - 1)


def _records_np(batch, k):
    """What cfk_docfreq_emit produces, restated: one record per distinct k-mer of a read, bit 63 = seen twice in it."""
    from oracle import c_oracle
    codes = c_oracle.unpacked_codes(batch)
    recs = []
    for r in range(batch.n_reads):
        seq = codes[int(batch.read_off[r]): int(batch.read_off[r]) + int(batch.read_len[r])].astype(np.uint64)
        km = np.zeros(seq.size - k + 1, dtype=np.uint64)
        for j in range(k):
            km = (km << np.uint64(2)) | seq[j: seq.size - k + 1 + j]
        u, c = np.unique(km, return_counts=True)
        recs.append(u | ((c > 1).astype(np.uint64) << np.uint64(63)))
    return np.concatenate(recs)


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import torch.distributed as tdist_mod
        from centroflye_b200 import dist as cdist
        from oracle import c_oracle

        # --- helpers --------------------------------------------------------------------------------------
        send_counts = torch.tensor([rank + 1 + p for p in range(world)], dtype=torch.int64)
        recv_counts = cdist.exchange_counts(send_counts)
        assert recv_counts.tolist() == [p + 1 + rank for p in range(world)]
        send = torch.cat([torch.full((int(c),), 100 * rank + p, dtype=torch.int64) for p, c in enumerate(send_counts)])
        got = cdist.all_to_all_v(send, send_counts.tolist(), recv_counts.tolist())
        want = torch.cat([torch.full((int(c),), 100 * p + rank, dtype=torch.int64) for p, c in enumerate(recv_counts)])
        assert torch.equal(got, want)
        cat, counts = cdist.all_gather_v(torch.arange(3 * rank, dtype=torch.int32))  # rank 0 contributes nothing
        assert counts == [3 * r for r in range(world)]
        assert torch.equal(cat, torch.cat([torch.arange(3 * r, dtype=torch.int32) for r in range(world)]))

        # --- sharded stage A == global stage A ---------------------------------------------------------------
        unit, reads, batch_from_synth = _dataset()
        k, lo, hi, max_nonuniq = 15, 3, 12, 2
        whole_batch, whole_units = batch_from_synth(reads, len(unit))
        my_batch, my_units = batch_from_synth(reads[rank::world], len(unit))
        keys, nr, nm = c_oracle.docfreq(c_oracle.unpacked_codes(my_batch), my_batch, k)
        owner = cdist.key_owner_np(keys, world)
        order = np.argsort(owner, kind="stable")
        send_counts = np.bincount(owner, minlength=world).astype(np.int64)
        recv_counts = cdist.exchange_counts(torch.from_numpy(send_counts)).tolist()
        rk = cdist.all_to_all_v(torch.from_numpy(keys[order].view(np.int64)), send_counts.tolist(), recv_counts).numpy()
        rr = cdist.all_to_all_v(torch.from_numpy(nr[order].astype(np.int64)), send_counts.tolist(), recv_counts).numpy()
        rm = cdist.all_to_all_v(torch.from_numpy(nm[order].astype(np.int64)), send_counts.tolist(), recv_counts).numpy()
        assert (cdist.key_owner_np(rk.view(np.uint64), world) == rank).all()
        uk, inv = np.unique(rk.view(np.uint64), return_inverse=True)
        sum_r = np.bincount(inv, weights=rr, minlength=uk.size).astype(np.int64)
        sum_m = np.bincount(inv, weights=rm, minlength=uk.size).astype(np.int64)
        mine = uk[(sum_m <= max_nonuniq) & (sum_r >= lo) & (sum_r <= hi)]
        rare_all, _ = cdist.all_gather_v(torch.from_numpy(mine.view(np.int64)))
        rare = np.sort(rare_all.numpy().view(np.uint64))
        gk, gr, gm = c_oracle.docfreq(c_oracle.unpacked_codes(whole_batch), whole_batch, k)
        want_rare = gk[(gm <= max_nonuniq) & (gr >= lo) & (gr <= hi)]
        assert rare.size > 50 and np.array_equal(rare, want_rare)

        # --- the default stage-A exchange: all-to-all of per-read records by partition range -------------------------------
        # what cfk_docfreq_emit produces is restated with numpy (one record per distinct k-mer of a read, bit 63 = seen
        # twice in that read, partition = hash range); the exchange itself is the product code (cdist.exchange_records)
        n_parts = 6 * world
        recs = _records_np(my_batch, k)
        key_bits = KEY_BITS
        part = (cdist.mix64_np(recs & key_bits) % np.uint64(n_parts)).astype(np.int64)
        by_part = np.argsort(part, kind="stable")
        counts = torch.from_numpy(np.bincount(part, minlength=n_parts).astype(np.int32))
        scan = lambda c: torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(c.to(torch.int64), 0)])  # noqa: E731
        soff, ssizes = cdist.padded_run_offsets(counts, world, scan)
        per = n_parts // world
        assert all(int(soff[g * per]) % cdist.RUN_ALIGN == 0 for g in range(world))  # every rank's run starts aligned
        send = torch.full((int(ssizes.sum()),), -1, dtype=torch.int64)  # -1 = padding, must never be counted
        sorted_recs = torch.from_numpy(recs[by_part].view(np.int64))
        dense = np.concatenate([[0], np.cumsum(counts.numpy().astype(np.int64))])
        for p_ in range(n_parts):
            send[int(soff[p_]): int(soff[p_]) + int(counts[p_])] = sorted_recs[dense[p_]: dense[p_ + 1]]
        recv, recv_counts, flags, n_sent = cdist.exchange_records(send, counts, world, flags=torch.tensor([rank, 0, 7 + rank]))
        assert flags == [world - 1, 0, 7 + world - 1] and n_sent == recs.size
        roff, rsizes = cdist.padded_run_offsets(recv_counts, world, scan)
        assert recv.numel() >= int(rsizes.sum())
        # source-major layout: run (s, q) = the records of local partition q sent by rank s, all of partition rank * per + q
        runs = []
        for s_ in range(world):
            assert int(roff[s_ * per]) % cdist.RUN_ALIGN == 0
            for q in range(per):
                run = recv[int(roff[s_ * per + q]): int(roff[s_ * per + q]) + int(recv_counts[s_ * per + q])].numpy().view(np.uint64)
                assert ((cdist.mix64_np(run & key_bits) % np.uint64(n_parts)) == np.uint64(rank * per + q)).all()
                runs.append(run)
        got = np.concatenate(runs)
        keys_o, inv = np.unique(got & key_bits, return_inverse=True)
        nr_o = np.bincount(inv, minlength=keys_o.size)
        nm_o = np.bincount(inv, weights=(got >> np.uint64(63)).astype(np.float64), minlength=keys_o.size).astype(np.int64)
        mine_rare = keys_o[(nm_o <= max_nonuniq) & (nr_o >= lo) & (nr_o <= hi)]
        all_rare, _ = cdist.all_gather_v(torch.from_numpy(np.sort(mine_rare).view(np.int64)))
        assert np.array_equal(np.sort(all_rare.numpy().view(np.uint64)), want_rare)

        # --- nominate-then-sum (ShardedRecruiter.global_rare_keys): same rare set for ~1 % of the traffic --------------
        import torch.distributed as tdist
        for lo2, hi2 in ((3, 12), (4, 9), (7, 40)):
            share = -(-lo2 // world)
            if share < 2:  # the product falls back to the full exchange for such a band (global_rare_keys)
                assert world > 2
                continue
            nominated = keys[nr >= share]
            allk, _ = cdist.all_gather_v(torch.from_numpy(nominated.view(np.int64)))
            union = torch.unique(allk).numpy().view(np.uint64)
            pos = np.searchsorted(keys, union)
            pos_c = np.minimum(pos, max(keys.size - 1, 0))
            held = (pos < keys.size) & (keys[pos_c] == union)
            sums = torch.from_numpy(np.stack([np.where(held, nr[pos_c], 0), np.where(held, nm[pos_c], 0)]).astype(np.int64))
            tdist.all_reduce(sums)
            sums = sums.numpy()
            got2 = union[(sums[0] >= lo2) & (sums[0] <= hi2) & (sums[1] <= max_nonuniq)]
            assert np.array_equal(got2, gk[(gm <= max_nonuniq) & (gr >= lo2) & (gr <= hi2)])
            assert nominated.size < keys.size

        # --- all-gathered cloud shards + round-robin sources == whole graph ----------------------------------
        ptr, ids = c_oracle.clouds(c_oracle.unpacked_codes(my_batch), my_units, k, rare)
        cnt_all, last_all, ids_all, unit_counts = cdist.gather_cloud_shards(
            torch.from_numpy(np.diff(ptr).astype(np.int32)), torch.from_numpy(c_oracle.unit_last_of(my_units)),
            torch.from_numpy(ids.view(np.int32)))
        # the same three arrays gathered one by one (each call exchanging its own lengths)
        cnt_1, unit_counts_1 = cdist.all_gather_v(torch.from_numpy(np.diff(ptr).astype(np.int32)))
        last_1, _ = cdist.all_gather_v(torch.from_numpy(c_oracle.unit_last_of(my_units)))
        ids_1, _ = cdist.all_gather_v(torch.from_numpy(ids.view(np.int32)))
        assert unit_counts == unit_counts_1 and torch.equal(cnt_all, cnt_1) and torch.equal(last_all, last_1)
        assert torch.equal(ids_all, ids_1)
        unit_last, base = cdist.merge_cloud_shards(cnt_all, unit_counts, last_all)
        assert unit_counts[rank] == my_units.n_units and int(base[-1]) == sum(unit_counts)
        gptr = np.zeros(cnt_all.numel() + 1, dtype=np.int64)
        np.cumsum(cnt_all.numpy(), out=gptr[1:])
        gids = np.ascontiguousarray(ids_all.numpy().view(np.uint32))
        gl = np.ascontiguousarray(unit_last.numpy())
        assert (gl >= np.arange(gl.size)).all() and gl[-1] == gl.size - 1
        # --- occurrence lists built once over all ranks (ShardedRecruiter.global_occurrences): the orchestration is the
        # product code, the two device passes are restated with numpy behind the engine's method names -------------------
        class _SliceEngine:
            device, torch, use_occ_last = torch.device("cpu"), torch, True

            @staticmethod
            def exclusive_scan(c):
                return torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(c.to(torch.int64), 0)])

            @staticmethod
            def _zeros(n, dtype):
                return torch.zeros(max(int(n), 1), dtype=dtype)

            def _lists(self, lo, hi):
                unit_of = np.repeat(np.arange(gptr.size - 1), np.diff(gptr))
                keep = (gids >= lo) & (gids < hi)
                order = np.lexsort((unit_of[keep], gids[keep]))
                return gids[keep][order].astype(np.int64) - lo, unit_of[keep][order]

            def occurrence_slice_count(self, csr, lo, hi):
                mult = torch.from_numpy(np.bincount(self._lists(lo, hi)[0], minlength=hi - lo).astype(np.int32))
                return mult, self.exclusive_scan(mult)

            def occurrence_slice_fill(self, csr, lo, hi, ptr, n_occ):
                occ = self._lists(lo, hi)[1]
                assert occ.size == n_occ == int(ptr[hi - lo])
                return torch.from_numpy(occ.astype(np.int32))

            @staticmethod
            def occurrence_last(occ, unit_last_t):
                return unit_last_t[occ.to(torch.int64)]

        sr = object.__new__(cdist.ShardedRecruiter)
        sr.eng, sr.torch, sr.dist, sr.world, sr.rank, sr.group, sr.bytes_exchanged = _SliceEngine(), torch, tdist_mod, world, rank, None, 0
        occ_ptr, occ, occ_last = sr.global_occurrences(None, unit_last, int(rare.size))
        unit_of = np.repeat(np.arange(gptr.size - 1), np.diff(gptr))
        by_id = np.lexsort((unit_of, gids))
        assert np.array_equal(occ.numpy(), unit_of[by_id])  # every id's units, ascending: the whole inversion
        assert np.array_equal(np.diff(occ_ptr.numpy()), np.bincount(gids, minlength=rare.size))
        assert np.array_equal(occ_last.numpy(), gl[unit_of[by_id]])

        part = c_oracle.dist_edges(gptr, gids, gl, rare.size, 1, 150, 2)  # all sources, on the global numbering
        e = part["edges"]
        mine_e = e[e[:, 0] % world == rank]  # what this rank's a = rank, rank + G, ... pass would emit
        flat, _ = cdist.all_gather_v(torch.from_numpy(np.ascontiguousarray(mine_e).view(np.int32).reshape(-1)))
        got_e = flat.numpy().view(np.uint32).reshape(-1, 4)
        # reference: the unsharded read set (unit numbering differs, edges do not depend on it)
        wptr, wids = c_oracle.clouds(c_oracle.unpacked_codes(whole_batch), whole_units, k, want_rare)
        whole = c_oracle.dist_edges(wptr, wids, c_oracle.unit_last_of(whole_units), want_rare.size, 1, 150, 2)
        canon = lambda x: x[np.lexsort((x[:, 3], x[:, 2], x[:, 1], x[:, 0]))]  # noqa: E731
        assert whole["edges"].shape[0] > 20
        assert np.array_equal(canon(got_e), canon(whole["edges"]))
        assert part["n_increments"] == whole["n_increments"]
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_exchange(tmp_path, world):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def _stage_a_engine(recs, calls, unfit=False):
    """An Engine whose device steps of two-phase stage A are restated with numpy on CPU tensors; stream_plan,
    _adapt_stream_group, grow_part_cap and docfreq_stream_finish are the product's.  calls receives the part_cap of every
    phase-1 launch; unfit: phase 2 reports a partition that did not fit."""
    import types
    from centroflye_b200.dist import mix64_np
    from centroflye_b200.engine import Engine
    eng = object.__new__(Engine)
    eng.torch, eng.device, eng.events = torch, torch.device("cpu"), None
    eng.lib = types.SimpleNamespace(cfk_docfreq_part_target=lambda: 20000, cfk_docfreq_part_distinct=lambda: 6144)
    eng.part_slack, eng.stream_group, eng.part_cap_seen, eng.select_hint, eng.stream_fallbacks = 1.25, 1, {}, {}, 0

    def emit_records(reads, k, n_parts, part_cap):  # cfk_docfreq_emit: records[p * part_cap + i], i < cursors[p]
        calls.append(part_cap)
        part = (mix64_np(recs & KEY_BITS) % np.uint64(n_parts)).astype(np.int64)
        need = np.bincount(part, minlength=n_parts)
        records = np.full(n_parts * part_cap, -1, dtype=np.int64)
        for p in range(n_parts):
            mine = recs[part == p][:part_cap].view(np.int64)
            records[p * part_cap: p * part_cap + mine.size] = mine
        counters = torch.zeros(8, dtype=torch.int64)
        counters[0] = int(need.max() > part_cap)
        return torch.from_numpy(records), torch.from_numpy(need.astype(np.int32)), counters

    def pack_records(records, part_cap, counts, offsets, n_out):  # cfk_records_pack
        out = torch.full((n_out,), -1, dtype=torch.int64)
        for p, (c, o) in enumerate(zip(counts.tolist(), offsets.tolist())):
            out[o: o + c] = records[p * part_cap: p * part_cap + c]
        return out

    def count_records(records, cursors, n_parts, part_cap, k, band=None, with_counts=False, dense=None, n_src=1,
                      src_stride=0, offsets=None, group=1):  # cfk_docfreq_count_parts over the runs of every source
        got = np.concatenate([records[o: o + c].numpy() for c, o in zip(cursors.tolist(), offsets.tolist())])
        got = got.view(np.uint64)
        keys, inv = np.unique(got & KEY_BITS, return_inverse=True)
        nr = np.bincount(inv, minlength=keys.size)
        nm = np.bincount(inv, weights=(got >> np.uint64(63)).astype(np.float64), minlength=keys.size)
        lo, hi, mn = band
        rare = keys[(nm <= mn) & (nr >= lo) & (nr <= hi)].view(np.int64)
        max_rare = int(eng.select_hint.get(("stream", False), 1 << 20))
        out = torch.zeros(max(max_rare, 1), dtype=torch.int64)
        out[: min(rare.size, max_rare)] = torch.from_numpy(rare[:max_rare])
        counters = torch.tensor([int(unfit), 0, 0, 0, rare.size, keys.size, 0, 0], dtype=torch.int64)
        return out, None, None, counters, max_rare

    def readback(h, stats):  # the pinned copy and its event
        h["host"], h["done"] = stats.clone(), types.SimpleNamespace(synchronize=lambda: None)

    eng.emit_records, eng.pack_records, eng.count_records, eng._readback = emit_records, pack_records, count_records, readback
    eng.exclusive_scan = lambda c: torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(c.to(torch.int64), 0)])
    eng.sort_keys = lambda keys: torch.from_numpy(np.sort(keys.numpy().view(np.uint64)).view(np.int64))
    eng.merge_sorted_runs = lambda keys, counts: eng.sort_keys(keys)  # cfk_merge_sorted_runs: runs of distinct keys
    return eng


def _rare_stream_worker(rank, world, port, out_dir):
    """ShardedRecruiter.global_rare_stream itself, its device steps restated (_stage_a_engine): the same rare set on
    every rank, also after one rank's phase 1 overflowed; all ranks fall back together when one rank's phase 2 cannot."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import types
        from centroflye_b200 import dist as cdist
        from oracle import c_oracle
        unit, reads, batch_from_synth = _dataset()
        k, lo, hi, max_nonuniq = 15, 3, 12, 2
        whole_batch, _ = batch_from_synth(reads, len(unit))
        gk, gr, gm = c_oracle.docfreq(c_oracle.unpacked_codes(whole_batch), whole_batch, k)
        want_rare = gk[(gm <= max_nonuniq) & (gr >= lo) & (gr <= hi)]
        my_batch, _ = batch_from_synth(reads[rank::world], len(unit))
        recs = _records_np(my_batch, k)
        n_local = int(np.maximum(my_batch.read_len - k + 1, 0).sum())
        n_total = torch.tensor([n_local])
        dist.all_reduce(n_total)
        for case in ("plain", "emit_overflow", "unfit"):
            calls = []
            eng = _stage_a_engine(recs, calls, unfit=case == "unfit" and rank == world - 1)
            if case == "emit_overflow" and rank == 1:  # this rank's first partition buffers are far too small
                plan = eng.stream_plan
                eng.stream_plan = lambda *a, **kw: (plan(*a, **kw)[0], 64)
            sr = object.__new__(cdist.ShardedRecruiter)
            sr.eng, sr.torch, sr.dist, sr.world, sr.rank, sr.group, sr.k = eng, torch, dist, world, rank, None, k
            sr.reads, sr.n_kmers_local, sr.n_kmers_total = types.SimpleNamespace(n_reads=my_batch.n_reads), n_local, int(n_total)
            sr.bytes_exchanged = 0
            got = sr.global_rare_stream(lo, hi, max_nonuniq)
            n_parts = eng.stream_plan(int(n_total), my_batch.n_reads, n_ranks=world, n_kmers_local=n_local)[0]
            assert n_parts >= 2 * world
            if case == "unfit":
                assert got is None and len(calls) == 1 and eng.stream_fallbacks == int(rank == world - 1)
                continue
            assert np.array_equal(got.numpy().view(np.uint64), want_rare) and want_rare.size > 50
            assert eng.stream_fallbacks == 0
            if case == "plain":
                assert len(calls) == 1 and eng.part_cap_seen == {}
            else:  # every rank went again, with the largest partition of all ranks, and remembers it
                part = (cdist.mix64_np(recs & KEY_BITS) % np.uint64(n_parts)).astype(np.int64)
                biggest = torch.tensor([int(np.bincount(part, minlength=n_parts).max())])
                dist.all_reduce(biggest, op=dist.ReduceOp.MAX)
                assert len(calls) == 2 and calls[1] == int(int(biggest) * 1.05) + 256
                assert eng.part_cap_seen == {n_parts: int(biggest)}
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_rare_stream(tmp_path, world):
    mp.spawn(_rare_stream_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def test_owner_rule_is_a_partition():
    from centroflye_b200.dist import key_owner_np, mix64_np
    rng = np.random.default_rng(0)
    keys = rng.integers(0, 1 << 62, size=5000, dtype=np.uint64)
    for parts in (1, 2, 3, 8):
        o = key_owner_np(keys, parts)
        assert o.min() >= 0 and o.max() < parts
        if parts > 1:
            assert np.bincount(o, minlength=parts).min() > 5000 / parts * 0.8
    # murmur3 finaliser known answers (restated independently: python ints)
    def mix(x):
        m = (1 << 64) - 1
        x ^= x >> 33; x = (x * 0xff51afd7ed558ccd) & m; x ^= x >> 33; x = (x * 0xc4ceb9fe1a85ec53) & m; x ^= x >> 33
        return x
    assert [int(v) for v in mix64_np(keys[:50])] == [mix(int(v)) for v in keys[:50]]


@pytest.mark.parametrize("world", [1, 2, 5, 8])
def test_padded_run_offsets_layout(world):
    """Every rank's run starts on a RUN_ALIGN boundary, partitions inside a run are back to back, nothing overlaps
    (ragged counts, empty partitions, empty runs)."""
    from centroflye_b200.dist import RUN_ALIGN, padded_run_offsets
    scan = lambda c: torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(c.to(torch.int64), 0)])  # noqa: E731
    rng = np.random.default_rng(world)
    for per in (1, 3, 40):
        counts = rng.integers(0, 50, size=world * per).astype(np.int32)
        counts[rng.random(counts.size) < 0.3] = 0
        if world > 1:
            counts[per: 2 * per] = 0  # rank 1 gets nothing at all
        off, sizes = padded_run_offsets(torch.from_numpy(counts), world, scan)
        off, sizes = off.numpy(), sizes.numpy()
        assert (sizes % RUN_ALIGN == 0).all()
        run_start = np.concatenate([[0], np.cumsum(sizes)])
        for g in range(world):
            c = counts[g * per: (g + 1) * per].astype(np.int64)
            assert off[g * per] == run_start[g]
            assert np.array_equal(off[g * per: (g + 1) * per], run_start[g] + np.concatenate([[0], np.cumsum(c)[:-1]]))
            assert run_start[g] + c.sum() <= run_start[g + 1] < run_start[g] + c.sum() + RUN_ALIGN
