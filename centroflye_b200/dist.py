"""Recruitment sharded over the GPUs of one box: one process per GPU, torch.distributed for the plumbing.

The reference is single-process (SURVEY.md §2); this is the partitioning of SURVEY.md §8e:

  reads         sharded by record across ranks (every rank holds whole reads and their units)
  stage A       phase 1 of the two-phase kernel pair on the rank's own reads (one 8-byte record per distinct k-mer of
                a read, in n_parts hash partitions) -> all-to-all of the records, partition range g to rank g ->
                phase 2 on the owned partitions with one record run per source rank: n_reads / n_multi of the WHOLE
                read set, max_nonuniq and the rare band in the same kernel -> the rare keys are all-gathered, so
                every rank holds the same sorted set (n_reads and n_multi are sums over reads, dbkr.py:55-59, hence
                additive over read shards).  The earlier table-based exchanges are kept for docfreq_mode != stream.
  stage B       local: clouds of the rank's own units against the global rare set
  stage C/D     the cloud CSR is all-gathered (units concatenated in rank order) and the SOURCE k-mer ids are
                dealt round-robin: rank r handles a = r, r + G, ...  No counter ever crosses a rank boundary
                because all of cnt[.][a][.] lives with a's owner; edges / endpoint flags are gathered at the end.

The collectives are written against torch.distributed only (all_to_all_single, all_gather_into_tensor), so the
exchange logic below runs unchanged on gloo/CPU tensors (tests/test_dist_gloo.py) and NCCL/CUDA tensors.
"""
import os

import numpy as np

from ._lib import CfkError
from .engine import stream_counters

U32_MAX = 0xFFFFFFFF
_GOLDEN = np.uint64(0x9E3779B97F4A7C15)


# ---- host restatement of the device hash (tests, and host-side routing of small key lists) ------------------
def mix64_np(x):
    x = np.asarray(x, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint64(33)
        x *= np.uint64(0xff51afd7ed558ccd)
        x ^= x >> np.uint64(33)
        x *= np.uint64(0xc4ceb9fe1a85ec53)
        x ^= x >> np.uint64(33)
    return x


def key_owner_np(keys, n_parts):
    """owner(key) of cfk_table_select / cfk_table_part_* (csrc/cfk.cu key_owner)."""
    return (mix64_np(np.asarray(keys, dtype=np.uint64) ^ _GOLDEN) % np.uint64(n_parts)).astype(np.int64)


# ---- variable-size collectives on top of torch.distributed ---------------------------------------------------
def exchange_counts(send_counts, group=None):
    """send_counts[p] = records this rank sends to p  ->  recv_counts[p] = records p sends to this rank."""
    import torch.distributed as dist
    recv = send_counts.new_empty(send_counts.shape)
    dist.all_to_all_single(recv, send_counts, group=group)
    return recv


def all_to_all_v(send, send_counts, recv_counts, group=None):
    """Rows of `send` are grouped by destination (send_counts rows each); returns the rows received,
    grouped by source.  Counts are python ints."""
    import torch.distributed as dist
    out = send.new_empty((int(sum(recv_counts)),) + tuple(send.shape[1:]))
    dist.all_to_all_single(out, send.contiguous(), output_split_sizes=[int(c) for c in recv_counts],
                           input_split_sizes=[int(c) for c in send_counts], group=group)
    return out


def gather_counts(values, device, group=None):
    """A few per-rank integers -> int64 list[world][len(values)] on the host (one small all-gather, one host sync)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    mine = torch.tensor([int(v) for v in values], dtype=torch.int64, device=device)
    out = torch.empty(world * mine.numel(), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(out, mine, group=group)
    return out.view(world, mine.numel()).cpu().tolist()


def all_gather_v(t, group=None, counts=None):
    """Concatenation over ranks (rank order) of a 1-d tensor whose length differs per rank -> (cat, counts).
    counts: the per-rank lengths when the caller already has them (gather_counts), else they are exchanged first.
    Every rank's slot of the gather starts on a 128-byte boundary (see padded_run_offsets: NCCL moves unaligned
    chunks at less than half the speed)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    if counts is None:
        counts = [c[0] for c in gather_counts([t.numel()], t.device, group)]
    counts = [int(c) for c in counts]
    if world == 1:
        return t, counts
    per_line = max(128 // t.element_size(), 1)
    width = -(-max(max(counts), 1) // per_line) * per_line
    padded = t.new_empty(width)
    padded[: t.numel()] = t
    gathered = t.new_empty(world * width)
    dist.all_gather_into_tensor(gathered, padded, group=group)
    if all(c == width for c in counts):
        return gathered, counts
    parts = [gathered[r * width: r * width + c] for r, c in enumerate(counts)]
    return torch.cat(parts), counts


RUN_ALIGN = 16  # records: every rank's run of the exchange starts on a 128-byte boundary


def padded_run_offsets(counts, world, exclusive_scan):
    """Where partition p's records start in a buffer that holds `world` runs (partition range g = run g, or source g's
    records on the receiving side) back to back, every run starting on a multiple of RUN_ALIGN records: NCCL copies a
    run whose start is not 16-byte aligned at less than half the speed (measured: 2.6 vs 1.1 ms for 0.9 GB on two
    B200s, the splits of the all-to-all being odd numbers of 8-byte records).  counts: int32[world * per];
    exclusive_scan(int32 tensor) -> int64[n + 1].  Returns (offsets int64[world * per], run sizes with padding int64[world])."""
    import torch
    per = counts.numel() // world
    dense = exclusive_scan(counts)[: counts.numel()]
    sizes = counts.view(world, per).sum(1, dtype=torch.int64)
    padded = (sizes + (RUN_ALIGN - 1)) // RUN_ALIGN * RUN_ALIGN
    extra = padded - sizes
    shift = torch.cumsum(extra, 0) - extra
    return dense + torch.repeat_interleave(shift, per), padded


def exchange_records(send, part_counts, world, group=None, flags=None):
    """The record all-to-all of stage A.  `send` holds this rank's records laid out by padded_run_offsets(part_counts)
    (partition p: part_counts[p] records; the run of partition range g -- what rank g gets -- starts on a multiple of
    RUN_ALIGN), n_parts = world * parts_per_rank.  Returns (recv, recv_counts, flags, n_sent): recv = the records of
    this rank's partition range, source-major, laid out by padded_run_offsets(recv_counts) (source s's run of
    partitions starts aligned; recv_counts[s * parts_per_rank + q] = records of local partition q from source s) --
    the (records, cursors, offsets) cfk_docfreq_count_parts takes.  One host sync (the split sizes); `flags` (small
    int64 tensor) rides along and comes back as a python list, all-reduced with MAX; n_sent = records this rank sent."""
    import os
    import torch
    import torch.distributed as dist
    trace = os.environ.get("CFK_EXCHANGE_TRACE") and send.is_cuda
    marks = []

    def mark(name):
        if trace:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks.append((name, e))
    mark("start")
    n_parts = int(part_counts.numel())
    per = n_parts // world
    recv_counts = torch.empty_like(part_counts)
    dist.all_to_all_single(recv_counts, part_counts.contiguous(), group=group)
    mark("counts_a2a")
    pad = lambda c: (c.view(world, per).sum(1, dtype=torch.int64) + (RUN_ALIGN - 1)) // RUN_ALIGN * RUN_ALIGN  # noqa: E731
    sizes = torch.cat([pad(part_counts), pad(recv_counts), part_counts.sum(dtype=torch.int64).view(1)])
    if flags is not None:
        flags = flags.to(torch.int64).clone()
        dist.all_reduce(flags, op=dist.ReduceOp.MAX, group=group)
        sizes = torch.cat([sizes, flags])
    mark("flags_allreduce")
    host = sizes.cpu().tolist()
    mark("host_sync")
    n_send, n_recv, n_records = host[:world], host[world:2 * world], host[2 * world]
    host = host[:2 * world] + host[2 * world + 1:]
    recv = send.new_empty(max(int(sum(n_recv)), 1))
    dist.all_to_all_single(recv[: int(sum(n_recv))], send[: int(sum(n_send))].contiguous(),
                           output_split_sizes=[int(c) for c in n_recv], input_split_sizes=[int(c) for c in n_send],
                           group=group)
    mark("records_a2a")
    if trace:
        torch.cuda.synchronize()
        if dist.get_rank(group) == 0:
            print("[exchange]", {b[0]: round(a[1].elapsed_time(b[1]), 3) for a, b in zip(marks[:-1], marks[1:])},
                  "sent", int(sum(n_send)), flush=True)
    return recv, recv_counts, host[2 * world:], int(n_records)


def gather_cloud_shards(cnt, last, ids, group=None):
    """This rank's (|cloud| per unit int32[U], last unit of the read int32[U], cloud ids[E]) -> the rank-order
    concatenations (cnt_all, last_all, ids_all, unit_counts).  One host sync (both lengths in one small gather); the
    two per-unit arrays travel in one all-gather (rank r's slot = its counts, then its lasts), the ids in a second."""
    import torch
    sizes = gather_counts([cnt.numel(), ids.numel()], cnt.device, group)
    unit_counts = [int(c[0]) for c in sizes]
    both, _ = all_gather_v(torch.cat([cnt, last]), group, counts=[2 * c for c in unit_counts])
    pieces = torch.split(both, [c for u in unit_counts for c in (u, u)])
    ids_all, _ = all_gather_v(ids.contiguous(), group, counts=[c[1] for c in sizes])
    return torch.cat(pieces[0::2]), torch.cat(pieces[1::2]), ids_all, unit_counts


def merge_cloud_shards(cnt_all, unit_counts, last_all):
    """Per-rank (|cloud| per unit, index of the last unit of the read, local numbering) -> global numbering.

    cnt_all / last_all are the rank-order concatenations; unit_counts[r] = units of rank r.  Returns
    (unit_last_global, unit_base) with unit_base[r] = first global unit index of rank r."""
    import torch
    base = np.zeros(len(unit_counts) + 1, dtype=np.int64)
    np.cumsum(np.asarray(unit_counts, dtype=np.int64), out=base[1:])
    shift = torch.repeat_interleave(torch.as_tensor(base[:-1], device=last_all.device),
                                    torch.as_tensor(np.asarray(unit_counts, dtype=np.int64), device=last_all.device))
    return (last_all.to(torch.int64) + shift).to(torch.int32), base


class ShardedRecruiter:
    """Whole recruitment path over `world` GPUs; `batch` / `units` are THIS rank's reads (ingest.ReadBatch / UnitIndex)."""

    def __init__(self, engine, batch, units, k, rank, world, group=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.eng, self.k, self.rank, self.world, self.group = engine, k, rank, world, group
        self.batch, self.units = batch, units
        self.reads = engine.upload_reads(batch, k)
        self.dunits = engine.upload_units(units, k)
        self.n_kmers_local = int(np.maximum(batch.read_len - k + 1, 0).sum())
        n = torch.tensor([batch.n_bases, self.n_kmers_local], dtype=torch.int64, device=engine.device)
        dist.all_reduce(n, group=group)
        self.n_bases_total, self.n_kmers_total = int(n[0].item()), int(n[1].item())
        self.last_increments = 0
        self.bytes_exchanged = 0
        self.nominate = True  # stage A exchange: nominate-then-sum (False: all-to-all of every table record)
        self.shard_occurrences = os.environ.get("CFK_SHARD_OCC", "1") != "0"  # False: every rank inverts all clouds

    # ---- stage A exchange ---------------------------------------------------------------------------------
    def global_rare_stream(self, lo, hi, max_nonuniq):
        """Two-phase stage A over all ranks -> sorted rare keys of the WHOLE read set (identical on every rank), or
        None when phase 2 could not hold a partition (the caller falls back to the table-based exchange).
        emit (local reads) -> pack -> all-to-all of the records (partition range g to rank g) -> count with one record
        run per source rank -> all-gather of the rare keys.  Two host syncs: the split sizes, and phase 2's counters."""
        eng, t, W = self.eng, self.torch, self.world
        if lo > hi or max_nonuniq < 0:
            return eng._empty(0, t.int64)[:0]
        n_parts, part_cap = eng.stream_plan(self.n_kmers_total, self.reads.n_reads, n_ranks=W,
                                            n_kmers_local=self.n_kmers_local)
        for launches in (1, 2, 3):
            records, cursors, ecounters = eng.emit_records(self.reads, self.k, n_parts, part_cap)
            with eng._stage("exchange_pack"):
                counts = cursors.clamp(max=part_cap)
                offsets, _ = padded_run_offsets(counts, W, eng.exclusive_scan)
                send = eng.pack_records(records, part_cap, counts, offsets,
                                        self.n_kmers_local + RUN_ALIGN * W)  # records <= k-mer occurrences
            with eng._stage("exchange_docfreq"):
                recv, recv_counts, flags, n_sent = exchange_records(send, counts, W, self.group,
                                                                    flags=eng.emit_stats(cursors, ecounters))
            self.bytes_exchanged += 8 * n_sent + 4 * n_parts
            s = stream_counters(emit=flags)  # all-reduced: every rank takes the same branch
            if not s.emit_overflow:
                break
            part_cap = eng.grow_part_cap(n_parts, s.biggest_part, launches)  # some rank ran out of room: all go again
            del records, send, recv
        roff, _ = padded_run_offsets(recv_counts, W, eng.exclusive_scan)
        h = eng.docfreq_count_launch(recv, recv_counts, n_parts // W, 1, self.k, (lo, hi, max_nonuniq), n_src=W,
                                     offsets=roff)
        out = eng.docfreq_stream_finish(h)
        ok = t.tensor([0 if out is None else 1], dtype=t.int64, device=eng.device)
        self.dist.all_reduce(ok, op=self.dist.ReduceOp.MIN, group=self.group)
        if int(ok.item()) == 0:
            return None
        with eng._stage("exchange_rare"):
            # every rank sorts its own keys; the gathered runs (distinct keys: a k-mer has one owner) are merged by rank
            mine = eng.sort_keys(out[0].clone()) if out[0].numel() > 1 else out[0].contiguous()
            allk, counts = all_gather_v(mine, self.group)
            self.bytes_exchanged += 8 * int(mine.numel())
            if allk.numel() == 0:
                return allk
            return eng.merge_sorted_runs(allk, counts)

    def global_rare_keys(self, table, lo, hi, max_nonuniq):
        """Local table -> sorted rare keys of the WHOLE read set (identical on every rank).

        Nominate, then sum: n_reads is a sum over ranks, so a k-mer with lo or more reads in total has at least
        ceil(lo / G) of them on SOME rank.  Every rank nominates its k-mers with that many reads (a few 10^5 -- the
        10^8 error k-mers seen once stay home), the nominations are all-gathered and de-duplicated, every rank looks
        its own counts of the union up (cfk_table_lookup), one all-reduce sums them and every rank applies the band:
        the same sorted set everywhere, exactly the set of the full exchange below, for ~1 % of its traffic."""
        eng, t, W = self.eng, self.torch, self.world
        share = -(-int(lo) // W)  # ceil(lo / W)
        if self.nominate and share >= 2 and lo <= hi:
            mine = eng.table_select(table, share, 0xFFFFFFFF, 0xFFFFFFFF)
            allk, _ = all_gather_v(mine.contiguous(), self.group)
            self.bytes_exchanged += 8 * int(mine.numel())
            union = t.unique(allk)  # sorted; keys < 2^62, so the int64 order is the uint64 order
            nr, nm = eng.table_lookup(table, union)
            sums = t.stack([nr.to(t.int64), nm.to(t.int64)])
            self.dist.all_reduce(sums, group=self.group)
            self.bytes_exchanged += 16 * int(union.numel())
            keep = (sums[0] >= int(lo)) & (sums[0] <= int(hi)) & (sums[1] <= int(max_nonuniq))
            return union[keep].contiguous()
        counts = eng.part_count(table, W)
        send_counts = counts.cpu().tolist()
        keys, nreads, nmulti = eng.part_scatter(table, W, counts)
        recv_counts = exchange_counts(counts, self.group).cpu().tolist()
        rk = all_to_all_v(keys, send_counts, recv_counts, self.group)
        rr = all_to_all_v(nreads, send_counts, recv_counts, self.group)
        rm = all_to_all_v(nmulti, send_counts, recv_counts, self.group)
        self.bytes_exchanged += 16 * int(sum(send_counts))
        n_recv = int(rk.numel())
        owned = eng.new_table(max(1024, int(n_recv / eng.table_load) + 1))
        if n_recv:
            eng.merge_into(owned, rk, rr, rm)
        mine = eng.table_select(owned, lo, hi, max_nonuniq) if lo <= hi else eng._empty(0, t.int64)[:0]
        allk, _ = all_gather_v(mine.contiguous(), self.group)
        return eng.sort_keys(allk.clone()) if allk.numel() else allk

    # ---- stage B exchange ---------------------------------------------------------------------------------
    def global_clouds(self, csr):
        """Local CloudCSR -> (global CloudCSR, global unit_last) with units concatenated in rank order."""
        from .engine import CloudCSR
        eng, t = self.eng, self.torch
        U = csr.n_units
        cnt = (csr.unit_ptr[1:U + 1] - csr.unit_ptr[:U]).to(t.int32) if U else eng._empty(0, t.int32)[:0]
        cnt_all, last_all, ids_all, unit_counts = gather_cloud_shards(cnt, self.dunits.unit_last[:U],
                                                                      csr.ids[: csr.n_entries], self.group)
        self.bytes_exchanged += 8 * U + 4 * csr.n_entries
        unit_last, _ = merge_cloud_shards(cnt_all, unit_counts, last_all)
        n_units = int(cnt_all.numel())
        unit_ptr = eng.exclusive_scan(cnt_all) if n_units else eng._zeros(1, t.int64)
        return CloudCSR(unit_ptr=unit_ptr, ids=ids_all, n_units=n_units, n_entries=int(ids_all.numel())), unit_last

    # ---- stage C prologue ---------------------------------------------------------------------------------
    def global_occurrences(self, gcsr, unit_last, n_kmers):
        """The occurrence lists of the all-gathered clouds, built once over all ranks instead of once per rank: rank r
        inverts the ids of [n r / G, n (r + 1) / G) (two binary searches per unit bound its slice of the sorted list),
        the list lengths and the lists are all-gathered in rank order = id order.  One host sync (every rank's number of
        occurrences).  -> (occ_ptr, occ, occ_last) as Engine.build_occurrences returns them."""
        eng, t, W = self.eng, self.torch, self.world
        bounds = [n_kmers * i // W for i in range(W + 1)]
        lo, hi = bounds[self.rank], bounds[self.rank + 1]
        mult, ptr = eng.occurrence_slice_count(gcsr, lo, hi)
        totals = t.empty(W, dtype=t.int64, device=eng.device)
        self.dist.all_gather_into_tensor(totals, ptr[hi - lo: hi - lo + 1].contiguous(), group=self.group)
        totals = [int(c) for c in totals.cpu().tolist()]
        if sum(totals) >= 1 << 32:
            raise CfkError("occurrence lists: 2^32 or more cloud entries")
        occ = eng.occurrence_slice_fill(gcsr, lo, hi, ptr, totals[self.rank])
        mult_all, _ = all_gather_v(mult.contiguous(), self.group, counts=[bounds[i + 1] - bounds[i] for i in range(W)])
        occ_all, _ = all_gather_v(occ.contiguous(), self.group, counts=totals)
        self.bytes_exchanged += 4 * (hi - lo) + 4 * totals[self.rank]
        occ_ptr = eng.exclusive_scan(mult_all) if n_kmers else eng._zeros(1, t.int64)
        return occ_ptr, occ_all, eng.occurrence_last(occ_all, unit_last)

    # ---- whole path ---------------------------------------------------------------------------------------
    def step(self, lo, hi, max_nonuniq, min_d, max_d, min_cov, rel_threshold=0.8, gather=True, on_clouds=None):
        """-> (index, local CloudCSR, DistResult); with gather=True every rank ends up with all edges / endpoints.
        on_clouds(index, csr) is called as soon as the rare set and this rank's clouds are final."""
        from .engine import DistResult
        eng, t = self.eng, self.torch
        if lo > hi or max_nonuniq < 0:  # dbkr.py:57-62 deletes every k-mer when max_nonuniq < 0; an empty band holds none
            rare = eng._empty(0, t.int64)[:0]
        else:
            rare = self.global_rare_stream(lo, hi, max_nonuniq) if eng.docfreq_mode == "stream" else None
        if rare is None:
            table = eng._count_docfreq_direct(self.reads, self.k)  # hashed table: this exchange looks keys up
            with eng._stage("exchange_docfreq"):
                rare = self.global_rare_keys(table, lo, hi, max_nonuniq)
            del table
        index = eng.build_index(rare, presorted=True)
        csr = eng.build_clouds(self.reads, self.dunits, self.k, index)
        if on_clouds is not None:
            on_clouds(index, csr)
        with eng._stage("gather_clouds"):
            gcsr, unit_last = self.global_clouds(csr)
        occurrences = None
        if self.shard_occurrences and index.n and gcsr.n_entries:
            with eng._stage("occurrences"):
                occurrences = self.global_occurrences(gcsr, unit_last, index.n)
        res = eng.dist_edges(gcsr, unit_last, index.n, min_d, max_d, min_cov, rel_threshold,
                             a_begin=self.rank, a_stride=self.world, occurrences=occurrences)
        stats = t.tensor([res.n_increments, res.n_candidates, res.n_pair_candidates, res.n_splits], dtype=t.int64,
                         device=eng.device)
        self.dist.all_reduce(stats, group=self.group)
        self.last_increments = int(stats[0].item())
        with eng._stage("gather_edges"):
            # the recruited k-mers (endpoints of kept edges) are the union over ranks: every rank gets all of them;
            # the edges themselves stay sharded by source k-mer (rank r holds the sources a = r mod G) unless gather
            edges = res.edges.reshape(-1)
            if gather:
                edges, _ = all_gather_v(edges.contiguous(), self.group)
            flags = eng._zeros(index.n, t.int32)
            if res.selected.numel():
                flags[res.selected.to(t.int64)] = 1
            self.dist.all_reduce(flags, op=self.dist.ReduceOp.MAX, group=self.group)
            selected = t.nonzero(flags[: index.n]).reshape(-1).to(t.int32)
        s = stats.cpu().tolist()
        out = DistResult(edges=edges.view(-1, 4), selected=selected, n_candidates=s[1], n_increments=s[0],
                         n_splits=s[3], n_pair_candidates=s[2])
        return index, csr, out

    def e2e_step(self, lo, hi, max_nonuniq, min_d, max_d, min_cov):
        """Pinned host buffers -> host results, sharded like the work: every rank reads back its own clouds and the
        edges of its own source k-mers; rank 0 also the recruited k-mers and the rare set.  Returns this rank's
        (h2d, d2h) bytes."""
        eng = self.eng
        self.reads = eng.upload_reads(self.batch, self.k)
        self.dunits = eng.upload_units(self.units, self.k)
        early = {}

        def clouds_home(index, csr):  # the clouds (and the rare set) travel while the distance graph is computed
            want = dict(unit_ptr=csr.unit_ptr, ids=csr.ids)
            if self.rank == 0:
                want["rare_keys"] = index.sorted_keys
            early.update(eng.start_host_copy(**want))

        index, csr, res = self.step(lo, hi, max_nonuniq, min_d, max_d, min_cov, gather=False, on_clouds=clouds_home)
        want = dict(edges=res.edges)
        if self.rank == 0:
            want["selected"] = res.selected
        out = eng.to_host(**want)  # pinned result buffers; synchronises
        eng.finish_host_copies()
        out.update(early)
        d2h = sum(x.numel() * x.element_size() for x in out.values())
        return self.reads.h2d_bytes + self.dunits.h2d_bytes, d2h
