"""Device pipeline of the recruitment path: PyTorch owns memory and streams, libcfk.so does the work.

Stages (reference function each one replaces, paths under /root/reference/scripts):

  count_docfreq   get_kmer_freqs_from_ncrf_report   distance_based_kmer_recruitment.py:39-63
  select / index  get_rare_kmers band + kmer_index  distance_based_kmer_recruitment.py:74-79,103
  build_clouds    ReadKMerCloud.fromNCRF_record     read_kmer_cloud.py:18-31
  filter_clouds   filter_reads_kmer_clouds          read_kmer_cloud.py:43-54
  dist_edges      get_kmer_dist_map + filter_dist_tuples  distance_based_kmer_recruitment.py:85-149

There is no CPU fallback: constructing an Engine without CUDA or without libcfk.so raises.
"""
import contextlib
import math
import os
from collections import namedtuple
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import CfkError
from .encode import check_k

U32_MAX = 0xFFFFFFFF
SKETCH_MIN_COV, SKETCH_MAX_COV = 3, 255  # include/cfk.h CFK_SKETCH_MIN_COV / CFK_SKETCH_MAX_COV


def band_to_int(left, right):
    """Integer form of ``left <= freq <= right`` for integer freq (floats come from dbkr.py:74-75)."""
    lo = max(0, math.ceil(left))
    hi = math.floor(right)
    return lo, min(hi, U32_MAX)


@dataclass
class DeviceReads:
    packed: object      # int32[n_words]
    read_off: object    # int64[R]
    read_len: object    # int64[R]
    order: object       # int32[R]  read indices, longest first (work order of the stage-A kernel)
    n_reads: int
    n_bases: int
    h2d_bytes: int
    max_len: int = 0    # longest read (bases)


@dataclass
class DeviceUnits:
    unit_off: object    # int64[U]
    unit_len: object    # int32[U]
    unit_kbase: object  # int64[U+1]
    unit_last: object   # int32[U]  index of the last unit of the same read
    n_units: int
    n_kmer_starts: int
    h2d_bytes: int


@dataclass
class DocFreqTable:
    slots: object       # int64[2 * cap]: per slot (key as uint64 bits, -1 = empty ; n_reads | n_multi << 32)
    cap: int
    dense: bool = False  # True: every slot is occupied and in no particular order (two-phase stage A): scans only


StreamCounters = namedtuple("StreamCounters", "unfit n_rare n_distinct n_retried emit_overflow biggest_part")


def stream_counters(c=(), emit=()):
    """Host int64 values of two-phase stage A -> StreamCounters; the only code that knows where each value sits.
    c = the counters of cfk_docfreq_count_parts (include/cfk.h: a partition did not fit, internal error, -, -, rare
    k-mers found, distinct k-mers, units retried), optionally followed by Engine.emit_stats (the one readback of a
    launch); emit = emit_stats alone (the sharded path's all-reduced phase-1 flags).  Internal errors raise."""
    unfit, internal, _, _, n_rare, n_distinct, n_retried, _, *tail = [int(x) for x in c] or [0] * 8
    emit_overflow, emit_internal, biggest_part = tail or [int(x) for x in emit] or [0, 0, 0]
    if internal:
        raise CfkError("stage A: phase 2 reported an internal error")
    if emit_internal:
        raise CfkError("stage A: per-read k-mer set overflowed (internal error)")
    return StreamCounters(unfit, n_rare, n_distinct, n_retried, emit_overflow, biggest_part)


@dataclass
class KmerIndex:
    sorted_keys: object  # int64[n]   ascending as uint64; rank = id
    idx_keys: object     # int64[cap]
    idx_vals: object     # int32[cap]
    cap: int
    n: int
    filter: object = None   # int32[2^filter_bits / 32] bitmap of hash prefixes, only for an index beyond L2
    filter_bits: int = 0


@dataclass
class CloudCSR:
    unit_ptr: object    # int64[U+1]
    ids: object         # int32[E]   sorted unique ids inside every unit
    n_units: int
    n_entries: int


@dataclass
class DistResult:
    edges: object        # int32[n_edges, 4]  (a, b, d, cnt) as uint32 bit patterns, unordered
    selected: object     # int32[n_selected]  ids that are an endpoint of a kept edge, unordered
    n_candidates: int        # (a, b, d) with cnt >= min_cov (the reference's candidate dict, dbkr.py:133-138)
    n_increments: int        # executions of `+= 1` at dbkr.py:126
    n_splits: int
    n_pair_candidates: int = 0  # (a, b, distance chunk) records handed from stage C to stage D


class Engine:
    def __init__(self, device=None):
        import torch
        self.torch = torch
        if not torch.cuda.is_available():
            raise CfkError("centroflye_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.n_sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        self.cand_hint = 1 << 20
        self.edge_hint = 1 << 20
        self.select_hint = {}  # (lo > 0, with_counts) -> output capacity that held last time
        self.sketch_banked = 1    # stage C sketch: bank-aware placement of the codes (0: the ids' own order)
        self.use_occ_last = 1     # stage C/D read unit_last through a per-occurrence copy (0: chase unit_last[g])
        self.index_cap_mult = 0   # slots per key of the rare-set probe table; 0 = by size (build_index)
        self.index_filter_bytes = 96 << 20  # a probe table larger than this gets a bitmap pre-filter (cfk_index_filter_build)
        self.table_load = 0.75  # distinct k-mers <= occurrences, so the stage-A table is at most this full (measured: 0.45 / 0.6 / 0.75 -> 26.4 / 26.0 / 25.8 ms per step)
        # stage C kernel: "auto" = sketch where it applies, "exact" = always the exact tables, "sketch" = insist
        self.pair_mode = os.environ.get("CFK_PAIR_MODE", "auto")
        # stage A kernel: "stream" = two-phase (emit hash-partitioned records, apply them partition by partition),
        # "resident" = (read, pass) items updating the table directly, "tiled" = one block per read
        self.docfreq_mode = os.environ.get("CFK_DOCFREQ_MODE", "stream")
        if self.docfreq_mode not in ("stream", "resident", "tiled"):
            raise CfkError(f"CFK_DOCFREQ_MODE must be stream, resident or tiled, got {self.docfreq_mode!r}")
        self.part_slack = 1.25  # records per partition buffer / expected records per partition (stream mode)
        self.stream_group = 1   # partitions per phase-2 unit; adapted after every call (_adapt_stream_group)
        self.part_cap_seen = {}  # n_parts -> largest partition (records) phase 1 produced so far
        self.stream_fallbacks = 0  # two-phase calls that handed stage A to the single-kernel form
        self._stat_pool, self._stat_next = [], 0  # pinned result slots of docfreq_stream_launch
        self.events = None  # set to a list to collect (stage, start_event, end_event) per C-ABI call group
        self._host_pool = {}  # name -> pinned uint8 buffer for results (to_host)
        self._copy_stream = None  # side stream of start_host_copy

    # ---- plumbing ---------------------------------------------------------------------------
    def _stream(self):
        """The stream every C-ABI call of this engine is enqueued on.  The library launches on the CURRENT device, so
        an engine bound to another GPU of the same process makes its device current first (a side effect the caller
        sees; one process per GPU never pays for it)."""
        t = self.torch
        if t.cuda.current_device() != self.device.index:
            t.cuda.set_device(self.device)
        return t.cuda.current_stream(self.device).cuda_stream

    def _to_dev(self, arr, dtype=None):
        t = self.torch.from_numpy(np.ascontiguousarray(arr))
        if dtype is not None:
            t = t.to(dtype)
        return t.pin_memory().to(self.device, non_blocking=True)

    def _staged(self, owner, name, arr):
        """Pinned staging copy of a host array, made once per owner object (ReadBatch / UnitIndex are immutable
        after ingestion) and reused by every later upload: page-locking 40 MB costs more than copying it."""
        cache = owner.__dict__.setdefault("_cfk_pinned", {})
        hit = cache.get(name)
        if hit is None or hit[0] is not arr:
            src = np.ascontiguousarray(arr)
            src = src.view(np.int32) if src.dtype == np.uint32 else src
            hit = (arr, self.torch.from_numpy(src).pin_memory())
            cache[name] = hit
        return hit[1].to(self.device, non_blocking=True)

    def to_host(self, **tensors):
        """Device tensors -> host tensors through pinned result buffers kept by the engine (one stream-ordered
        copy each, one synchronize at the end).  The returned tensors alias the pool: they are valid until the
        next to_host() call with the same names."""
        t = self.torch
        out = {}
        for name, src in tensors.items():
            src = src.contiguous()
            nbytes = src.numel() * src.element_size()
            buf = self._host_pool.get(name)
            if buf is None or buf.numel() < nbytes:
                buf = t.empty(max(nbytes + nbytes // 8, 1 << 16), dtype=t.uint8, pin_memory=True)
                self._host_pool[name] = buf
            dst = buf[:nbytes].view(src.dtype).view(src.shape)
            dst.copy_(src, non_blocking=True)
            out[name] = dst
        t.cuda.current_stream(self.device).synchronize()
        return out

    def start_host_copy(self, **tensors):
        """Like to_host(), but on a side stream and without waiting: the copies start as soon as the work already
        enqueued on the current stream has produced the tensors, and overlap whatever is enqueued afterwards
        (the cloud CSR goes home while stage C runs).  finish_host_copies() waits for them."""
        t = self.torch
        if self._copy_stream is None:
            self._copy_stream = t.cuda.Stream(self.device)
        ready = t.cuda.Event()
        ready.record(t.cuda.current_stream(self.device))
        self._copy_stream.wait_event(ready)
        out = {}
        with t.cuda.stream(self._copy_stream):
            for name, src in tensors.items():
                src = src.contiguous()
                src.record_stream(self._copy_stream)
                nbytes = src.numel() * src.element_size()
                buf = self._host_pool.get(name)
                if buf is None or buf.numel() < nbytes:
                    buf = t.empty(max(nbytes + nbytes // 8, 1 << 16), dtype=t.uint8, pin_memory=True)
                    self._host_pool[name] = buf
                dst = buf[:nbytes].view(src.dtype).view(src.shape)
                dst.copy_(src, non_blocking=True)
                out[name] = dst
        return out

    def finish_host_copies(self):
        if self._copy_stream is not None:
            self._copy_stream.synchronize()

    def _empty(self, n, dtype):
        return self.torch.empty(max(int(n), 1), dtype=dtype, device=self.device)

    def _zeros(self, n, dtype):
        return self.torch.zeros(max(int(n), 1), dtype=dtype, device=self.device)

    def _counters(self):
        return self.torch.zeros(8, dtype=self.torch.int64, device=self.device)

    @staticmethod
    def _p(t):
        return None if t is None else t.data_ptr()

    @contextlib.contextmanager
    def _stage(self, name):
        """CUDA-event bracket on the launching stream (only when self.events is a list)."""
        if self.events is None:
            yield
            return
        t = self.torch
        a, b = t.cuda.Event(enable_timing=True), t.cuda.Event(enable_timing=True)
        a.record(t.cuda.current_stream(self.device))
        yield
        b.record(t.cuda.current_stream(self.device))
        self.events.append((name, a, b))

    def stage_times_ms(self):
        """Sum of elapsed ms per stage name (synchronises)."""
        self.torch.cuda.synchronize(self.device)
        out = {}
        for name, a, b in self.events or []:
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return out

    def launch_count(self):
        return int(self.lib.cfk_launch_count())

    # ---- uploads ----------------------------------------------------------------------------
    def upload_reads(self, batch, k):
        """ReadBatch -> device (pinned staging, async copies)."""
        derived = batch.__dict__.setdefault("_cfk_derived", {})  # host arrays made once per (immutable) batch
        if "order" not in derived:
            derived["order"] = np.argsort(-batch.read_len, kind="stable").astype(np.int32)
        order = derived["order"]
        packed = batch.packed.view(np.int32)
        h2d = packed.nbytes + batch.read_off.nbytes + batch.read_len.nbytes + order.nbytes
        return DeviceReads(packed=self._staged(batch, "packed", batch.packed),
                           read_off=self._staged(batch, "read_off", batch.read_off),
                           read_len=self._staged(batch, "read_len", batch.read_len),
                           order=self._staged(batch, "order", order),
                           n_reads=batch.n_reads, n_bases=batch.n_bases, h2d_bytes=h2d,
                           max_len=int(batch.read_len.max()) if batch.n_reads else 0)

    def upload_units(self, units, k):
        derived = units.__dict__.setdefault("_cfk_derived", {})  # host arrays made once per (immutable) unit index
        if ("kbase", k) not in derived:
            nk = np.maximum(units.unit_len.astype(np.int64) - k + 1, 0)
            kbase = np.zeros(units.n_units + 1, dtype=np.int64)
            np.cumsum(nk, out=kbase[1:])
            derived[("kbase", k)] = kbase
        if "last" not in derived:
            last = np.zeros(units.n_units, dtype=np.int32)
            ptr = units.read_unit_ptr
            last[:] = np.repeat(ptr[1:] - 1, np.diff(ptr))
            derived["last"] = last
        kbase, last = derived[("kbase", k)], derived["last"]
        h2d = units.unit_off.nbytes + units.unit_len.nbytes + kbase.nbytes + last.nbytes
        return DeviceUnits(unit_off=self._staged(units, "unit_off", units.unit_off),
                           unit_len=self._staged(units, "unit_len", units.unit_len),
                           unit_kbase=self._staged(units, f"kbase{k}", kbase), unit_last=self._staged(units, "last", last),
                           n_units=units.n_units, n_kmer_starts=int(kbase[-1]), h2d_bytes=h2d)

    # ---- stage A ----------------------------------------------------------------------------
    def new_table(self, cap):
        slots = self._empty(2 * int(cap), self.torch.int64)
        _lib.call("cfk_table_init", self._p(slots), int(cap), self._stream())
        return DocFreqTable(slots=slots, cap=int(cap))

    def count_docfreq(self, reads, k, n_kmers_hint=None):
        """One pass over all reads -> DocFreqTable (every distinct k-mer with n_reads and n_multi)."""
        k = check_k(k)
        if self.docfreq_mode == "stream" and reads.n_reads:
            out = self.docfreq_stream(reads, k, want_table=True)
            if out is not None:
                return out[1]
        return self._count_docfreq_direct(reads, k, n_kmers_hint)

    def rare_kmers(self, reads, k, lo, hi, max_nonuniq):
        """Stage A + the band of get_rare_kmers in one go -> unordered rare keys (int64 tensor of uint64 bits)."""
        k = check_k(k)
        if lo > hi or max_nonuniq < 0:
            return self._empty(0, self.torch.int64)[:0]
        if self.docfreq_mode == "stream" and reads.n_reads:
            out = self.docfreq_stream(reads, k, band=(lo, hi, max_nonuniq))
            if out is not None:
                return out[0]
        table = self._count_docfreq_direct(reads, k, None)
        return self.table_select(table, lo, hi, max_nonuniq)

    def _count_docfreq_direct(self, reads, k, n_kmers_hint=None):
        """The single-kernel forms of stage A (global hash table): "resident" (default of this path) or "tiled"."""
        total_k = n_kmers_hint if n_kmers_hint is not None else max(reads.n_bases - reads.n_reads * (k - 1), 0)
        cap = max(1024, int(total_k / self.table_load) + 1)
        item_ptr = None
        if self.docfreq_mode != "tiled" and reads.n_reads:
            n_pass = self._empty(reads.n_reads, self.torch.int32)
            _lib.call("cfk_docfreq_plan", self._p(reads.read_len), self._p(reads.order), reads.n_reads, k,
                      self._p(n_pass), self._stream())
            item_ptr = self.exclusive_scan(n_pass[:reads.n_reads])
        while True:
            table = self.new_table(cap)
            counters = self._counters()
            with self._stage("docfreq"):
                if item_ptr is not None:
                    _lib.call("cfk_docfreq_count_resident", self._p(reads.packed), self._p(reads.read_off),
                              self._p(reads.read_len), self._p(reads.order), self._p(item_ptr), reads.n_reads, k,
                              self._p(table.slots), cap, self._p(counters), self.n_sms, self._stream())
                else:
                    _lib.call("cfk_docfreq_count", self._p(reads.packed), self._p(reads.read_off),
                              self._p(reads.read_len), self._p(reads.order), reads.n_reads, k, self._p(table.slots),
                              cap, self._p(counters), self.n_sms, self._stream())
            c = counters.cpu()
            if int(c[1]):
                raise CfkError("stage A: per-read k-mer set overflowed (internal error)")
            if int(c[0]) == 0:
                return table
            cap *= 2

    # -- two-phase stage A: cfk_docfreq_emit (reads -> hash-partitioned records) + cfk_docfreq_count_parts
    def stream_plan(self, n_kmers, n_reads, n_ranks=1, n_kmers_local=None):
        """(n_parts, part_cap): n_parts hash partitions for n_kmers k-mer occurrences of the WHOLE job (a multiple of
        n_ranks: partition range g of the exchange belongs to rank g), each planned for cfk_docfreq_part_target()
        occurrences; part_cap = records one partition buffer of THIS rank holds.  The first guess leaves room for two
        k-mers present in every local read on top of the mean; a call whose buffers overflowed is repeated with the
        size it measured, and later calls start from the largest size seen (self.part_cap_seen)."""
        target = int(self.lib.cfk_docfreq_part_target())
        n_parts = max(1, -(-int(n_kmers) // target))
        n_parts = -(-n_parts // n_ranks) * n_ranks
        local = int(n_kmers if n_kmers_local is None else n_kmers_local)
        mean = -(-local // n_parts)
        guess = int(mean * self.part_slack) + 2 * min(int(n_reads), 16384) + 512
        seen = self.part_cap_seen.get(n_parts)
        part_cap = int(seen * 1.1) + 256 if seen else guess
        return n_parts, max(1, min(part_cap, local + 1))

    def emit_records(self, reads, k, n_parts, part_cap):
        """Phase 1 -> (records int64[n_parts * part_cap], cursors int32[n_parts], counters).  counters[0] != 0:
        some partition buffer was too small (cursors then hold the sizes that would have been needed)."""
        t = self.torch
        if reads.max_len >= (1 << 30):
            raise CfkError("stage A (two-phase): reads of 2^30 bases or more are not supported")
        n_pass = self._empty(reads.n_reads, t.int32)
        _lib.call("cfk_docfreq_emit_plan", self._p(reads.read_len), self._p(reads.order), reads.n_reads, k,
                  self._p(n_pass), self._stream())
        item_ptr = self.exclusive_scan(n_pass[:reads.n_reads])
        records = self._empty(n_parts * part_cap, t.int64)
        cursors = self._zeros(n_parts, t.int32)
        counters = self._counters()
        with self._stage("docfreq_emit"):
            _lib.call("cfk_docfreq_emit", self._p(reads.packed), self._p(reads.read_off), self._p(reads.read_len),
                      self._p(reads.order), self._p(item_ptr), reads.n_reads, k, self._p(records), part_cap, n_parts,
                      self._p(cursors), self._p(counters), self.n_sms, self._stream())
        return records, cursors, counters

    def count_records(self, records, cursors, n_parts, part_cap, k, band=None, with_counts=False, dense=None,
                      n_src=1, src_stride=0, offsets=None, group=1):
        """Phase 2 over n_parts partitions -> (rare_keys, rare_nreads, rare_nmulti, counters, max_rare); the rare
        outputs are None without a band.  `dense` (int64[2 * max_dense]) receives the whole table when given."""
        t = self.torch
        lo, hi, mn = (0, 0, 0) if band is None else band
        hint_key = ("stream", bool(with_counts))
        max_rare = int(self.select_hint.get(hint_key, 1 << 20)) if band is not None else 0
        rare = self._empty(max_rare, t.int64) if band is not None else None
        rare_nr = self._empty(max_rare, t.int32) if band is not None and with_counts else None
        rare_nm = self._empty(max_rare, t.int32) if band is not None and with_counts else None
        counters = self._counters()
        with self._stage("docfreq_count"):
            _lib.call("cfk_docfreq_count_parts", self._p(records), part_cap, self._p(cursors), self._p(offsets), n_parts,
                      n_src, src_stride, int(group), int(k), int(lo), int(min(hi, U32_MAX)), int(min(mn, U32_MAX)),
                      self._p(rare), self._p(rare_nr), self._p(rare_nm), max_rare, self._p(dense),
                      0 if dense is None else dense.numel() // 2, self._p(counters), self.n_sms, self._stream())
        return rare, rare_nr, rare_nm, counters, max_rare

    def _adapt_stream_group(self, n_distinct, n_parts, n_retried):
        """Partitions counted as one unit by the next phase 2: as many as keep a unit's distinct k-mers near 60 % of
        the block's table (any value is exact; a unit that does not fit is retried partition by partition)."""
        cap = int(self.lib.cfk_docfreq_part_distinct())
        per_part = max(1.0, n_distinct / max(1, n_parts))
        group = int(max(1, min(64, 0.6 * cap / per_part)))
        if n_retried * 20 > n_parts / max(1, self.stream_group):  # more than 5 % of the units did not fit
            group = max(1, min(group, self.stream_group // 2))
        self.stream_group = group

    def emit_stats(self, cursors, counters):
        """int64[3] device tensor: phase 1's overflow flag, its internal-error flag, its largest partition."""
        t = self.torch
        return t.stack([counters[0], counters[1], cursors.max().to(t.int64)])

    def grow_part_cap(self, n_parts, biggest, launches):
        """Phase 1 overflowed on its `launches`-th launch and needed `biggest` records in its largest partition -> the
        part_cap to launch it again with.  Later plans start from the largest size seen (stream_plan)."""
        if launches >= 3:
            raise CfkError("stage A: partition buffers overflowed three times (internal error)")
        self.part_cap_seen[n_parts] = max(self.part_cap_seen.get(n_parts, 0), biggest)
        return int(biggest * 1.05) + 256

    def docfreq_stream(self, reads, k, band=None, with_counts=False, want_table=False, table_buf=None):
        """Two-phase stage A on one GPU -> (rare, table) or None when phase 2 could not hold a partition (more than
        65536 reads sharing a k-mer, or a partition that does not fit after 64-fold splitting): the caller falls back
        to the single-kernel form.  rare = unordered keys inside band = (lo, hi, max_nonuniq) (a tuple with the two
        count tensors when with_counts); table = the dense DocFreqTable when want_table.  One host sync at the end
        (two when the table is wanted and no table_buf -- int64[2 * slots], at least one slot per k-mer occurrence --
        is given: its size then comes from phase 1)."""
        return self.docfreq_stream_finish(self._stream_launch(reads, k, band, with_counts, want_table, table_buf))

    def docfreq_stream_launch(self, reads, k, band=None, with_counts=False, table_buf=None):
        """Enqueue both phases of stage A for one batch and return a handle; nothing is read back yet, so the next
        batch can be enqueued behind it.  docfreq_stream_finish(handle) waits for THIS batch's counters only."""
        return self._stream_launch(reads, k, band, with_counts, table_buf is not None, table_buf)

    def _stream_launch(self, reads, k, band, with_counts, want_table, table_buf):
        n_parts, part_cap = self.stream_plan(max(reads.n_bases - reads.n_reads * (k - 1), 0), reads.n_reads)
        h = dict(reads=reads, k=k, band=band, with_counts=with_counts, want_table=want_table,
                 table_buf=table_buf if want_table else None, n_parts=n_parts, n_src=1, offsets=None, launches=0)
        return self._stream_emit(h, part_cap)

    def _stream_emit(self, h, part_cap):
        """Phase 1 of a handle (again after an overflow, with a larger part_cap), then its phase 2."""
        h.update(records=None, dense=None, rare=None)  # a repeat lets go of the buffers that were too small first
        records, cursors, counters = self.emit_records(h["reads"], h["k"], h["n_parts"], part_cap)
        dense = h["table_buf"]
        if h["want_table"] and dense is None:
            n_rec = int(cursors.clamp(max=part_cap).sum(dtype=self.torch.int64).item())  # distinct k-mers <= records
            dense = self._empty(2 * max(n_rec, 1), self.torch.int64)
        h.update(records=records, cursors=cursors, part_cap=part_cap, dense=dense,
                 emit=self.emit_stats(cursors, counters), launches=h["launches"] + 1)
        return self._stream_count(h)

    def docfreq_count_launch(self, records, cursors, n_parts, part_cap, k, band, n_src=1, offsets=None):
        """Phase 2 alone, on records the multi-GPU exchange delivered -> a handle for docfreq_stream_finish."""
        return self._stream_count(dict(records=records, cursors=cursors, n_parts=n_parts, part_cap=part_cap, k=k,
                                       band=band, with_counts=False, dense=None, n_src=n_src, offsets=offsets, emit=None))

    def _stream_count(self, h):
        """Phase 2 on the records the handle keeps; its counters (+ phase 1's emit_stats, if it ran) go home."""
        rare, rare_nr, rare_nm, counters, h["max_rare"] = self.count_records(
            h["records"], h["cursors"], h["n_parts"], h["part_cap"], h["k"], h["band"], h["with_counts"], h["dense"],
            n_src=h["n_src"], offsets=h["offsets"], group=self.stream_group)
        h["rare"] = (rare, rare_nr, rare_nm)
        self._readback(h, counters if h["emit"] is None else self.torch.cat([counters, h["emit"]]))
        return h

    def _readback(self, h, stats):
        """stats (<= 16 int64 on the device) -> h["host"], pinned, once h["done"] (an event) has completed."""
        t = self.torch
        if "host" not in h:  # one slot of a small pinned ring per handle (page-locking costs far more than the copy)
            self._stat_pool = self._stat_pool or [t.empty(16, dtype=t.int64, pin_memory=True) for _ in range(8)]
            h["host"] = self._stat_pool[self._stat_next % len(self._stat_pool)][: stats.numel()]
            self._stat_next += 1
        h["host"].copy_(stats, non_blocking=True)
        h["done"] = t.cuda.Event()
        h["done"].record(t.cuda.current_stream(self.device))

    def docfreq_stream_finish(self, h):
        """-> (rare, table) of a launched batch, like docfreq_stream.  Waits for this batch's counters only.  A phase 1
        that ran out of partition buffer is launched again with the size it measured (three launches in all at most);
        a rare output that was too small gets phase 2 again, on the records the handle keeps."""
        while True:
            h["done"].synchronize()
            s = stream_counters(h["host"])
            if s.emit_overflow:  # what phase 2 reported is void
                self._stream_emit(h, self.grow_part_cap(h["n_parts"], s.biggest_part, h["launches"]))
            elif s.unfit:
                self.stream_fallbacks += 1
                return None
            elif h["band"] is not None and s.n_rare > h["max_rare"]:
                self.select_hint[("stream", bool(h["with_counts"]))] = s.n_rare + 1024  # the size is now known
                self._stream_count(h)
            else:
                break
        if h["emit"] is not None:
            self.part_cap_seen[h["n_parts"]] = max(self.part_cap_seen.get(h["n_parts"], 0), s.biggest_part)
        self._adapt_stream_group(s.n_distinct, h["n_parts"], s.n_retried)
        n = s.n_distinct
        table = None if h["dense"] is None else DocFreqTable(slots=h["dense"][:2 * n], cap=n, dense=True)
        if h["band"] is None:
            return None, table
        self.select_hint[("stream", bool(h["with_counts"]))] = max(h["max_rare"], int(s.n_rare * 1.05) + 1024)
        rare = tuple(x[:s.n_rare] for x in h["rare"] if x is not None)
        return (rare if h["with_counts"] else rare[0]), table

    def pack_records(self, records, part_cap, counts, offsets, n_out):
        """Phase 1's partition buffers -> int64[n_out] holding partition p's counts[p] records from offsets[p] on
        (cfk_records_pack)."""
        out = self._empty(n_out, self.torch.int64)
        _lib.call("cfk_records_pack", self._p(records), part_cap, self._p(counts), self._p(offsets), int(counts.numel()),
                  self._p(out), self._stream())
        return out

    def count_total(self, reads, batch, k, canonical=False):
        """Total occurrences of every k-mer over all reads (no per-read de-duplication) -> DocFreqTable whose n_reads
        field holds the count (better_consensus_unit_reconstruction.py:127-135).  canonical=True merges the two strands
        of a k-mer (`jellyfish count -C`, ext/tandemQUAST/scripts/select_kmers.py:131-133)."""
        k = check_k(k)
        tile = int(self.lib.cfk_kmer_count_tile())
        nk = np.maximum(batch.read_len - k + 1, 0)
        tiles_per_read = (nk + tile - 1) // tile
        tile_read = np.repeat(np.arange(batch.n_reads, dtype=np.int32), tiles_per_read)
        first = np.cumsum(tiles_per_read) - tiles_per_read
        tile_start = (np.arange(tile_read.size, dtype=np.int64) - np.repeat(first, tiles_per_read)) * tile
        d_read, d_start = self._to_dev(tile_read), self._to_dev(tile_start)
        cap = max(1024, int(int(nk.sum()) / self.table_load) + 1)
        while True:
            table = self.new_table(cap)
            counters = self._counters()
            _lib.call("cfk_kmer_count_canonical" if canonical else "cfk_kmer_count_total", self._p(reads.packed),
                      self._p(reads.read_off), self._p(reads.read_len),
                      self._p(d_read), self._p(d_start), int(tile_read.size), k, self._p(table.slots), cap,
                      self._p(counters), self._stream())
            if int(counters.cpu()[0]) == 0:
                return table
            cap *= 2

    def table_select(self, table, lo, hi, max_nonuniq, with_counts=False, n_parts=0, part=0):
        """Compacted (keys[, n_reads, n_multi]) of slots inside the band, unordered."""
        t = self.torch
        args = (self._p(table.slots), table.cap, int(lo), int(min(hi, U32_MAX)), int(min(max_nonuniq, U32_MAX)),
                n_parts, part)
        hint_key = (int(lo) > 0, bool(with_counts))
        max_out = int(self.select_hint.get(hint_key, 1 << 20))
        while True:  # one pass over the table when the hint holds; a second one with the exact size otherwise
            counters = self._counters()
            keys = self._empty(max_out, t.int64)
            nreads = self._empty(max_out, t.int32) if with_counts else None
            nmulti = self._empty(max_out, t.int32) if with_counts else None
            with self._stage("table_select"):
                _lib.call("cfk_table_select", *args, self._p(keys), self._p(nreads), self._p(nmulti), max_out,
                          self._p(counters), self._stream())
            n = int(counters.cpu()[0])
            if n <= max_out:
                break
            max_out = n
        self.select_hint[hint_key] = max(max_out, int(n * 1.05) + 1024)
        if with_counts:
            return keys[:n], nreads[:n], nmulti[:n]
        return keys[:n]

    def table_lookup(self, table, keys):
        """(n_reads, n_multi) int32 tensors of the given keys (0 / 0 where the table does not hold the key)."""
        t = self.torch
        if table.dense:
            raise CfkError("table_lookup needs a hashed table; the two-phase stage A returns a dense one "
                           "(use count_docfreq with docfreq_mode='resident')")
        n = int(keys.numel())
        nreads, nmulti = self._empty(n, t.int32), self._empty(n, t.int32)
        _lib.call("cfk_table_lookup", self._p(table.slots), table.cap, self._p(keys.contiguous()), n, self._p(nreads),
                  self._p(nmulti), self._stream())
        return nreads[:n], nmulti[:n]

    def part_count(self, table, n_parts):
        """int64[n_parts] (device): occupied slots per hash partition (owner = mix64(key ^ golden) % n_parts)."""
        counts = self._zeros(n_parts, self.torch.int64)
        _lib.call("cfk_table_part_count", self._p(table.slots), table.cap, n_parts, self._p(counts), self._stream())
        return counts

    def part_scatter(self, table, n_parts, counts):
        """All occupied slots grouped by partition: (keys, n_reads, n_multi), partition p contiguous."""
        t = self.torch
        total = int(counts.sum().item())
        cursors = (t.cumsum(counts, 0) - counts).contiguous()
        keys, nreads, nmulti = self._empty(total, t.int64), self._empty(total, t.int32), self._empty(total, t.int32)
        _lib.call("cfk_table_part_scatter", self._p(table.slots), table.cap, n_parts, self._p(cursors), self._p(keys),
                  self._p(nreads), self._p(nmulti), self._stream())
        return keys[:total], nreads[:total], nmulti[:total]

    def merge_into(self, table, keys, nreads, nmulti):
        counters = self._counters()
        _lib.call("cfk_table_merge", self._p(keys), self._p(nreads), self._p(nmulti), int(keys.numel()),
                  self._p(table.slots), table.cap, self._p(counters), self._stream())
        if int(counters.cpu()[0]):
            raise CfkError("owner-side table full during merge")

    # ---- rare set -> sorted ids + probe table ------------------------------------------------
    def sort_keys(self, keys):
        keys = keys.contiguous()
        _lib.call("cfk_sort_u64", self._p(keys), int(keys.numel()), self._stream())
        return keys

    def merge_sorted_runs(self, keys, counts):
        """Back-to-back sorted runs of distinct keys, counts[r] keys in run r -> one sorted tensor (cfk_merge_sorted_runs)."""
        n = int(keys.numel())
        run_ptr = self._to_dev(np.concatenate([[0], np.cumsum(np.asarray(counts, dtype=np.int64))]))
        merged = self._empty(n, self.torch.int64)
        _lib.call("cfk_merge_sorted_runs", self._p(keys.contiguous()), self._p(run_ptr), len(counts), n, self._p(merged),
                  self._stream())
        return merged[:n]

    def build_index(self, keys, presorted=False):
        t = self.torch
        n = int(keys.numel())
        with self._stage("sort_rare"):
            sorted_keys = keys.contiguous() if presorted else self.sort_keys(keys.clone())
        # slots per key: stage B probes this table once per k-mer and is bound by L2 sector throughput, so every probe
        # saved counts; 8x keeps chains near 1 probe while the table (12 B per slot) still sits in the 126 MB L2
        mult = self.index_cap_mult or (8 if n <= (1 << 20) else 4 if n <= (1 << 22) else 2)
        cap = max(64, mult * n + 1)
        idx_keys = t.full((cap,), -1, dtype=t.int64, device=self.device)
        idx_vals = self._zeros(cap, t.int32)
        counters = self._counters()
        with self._stage("index_build"):
            _lib.call("cfk_index_build", self._p(sorted_keys), n, self._p(idx_keys), self._p(idx_vals), cap,
                      self._p(counters), self._stream())
        filt, bits = None, 0
        if 12 * cap > self.index_filter_bytes:  # stage B would probe DRAM: a bitmap that stays in L2 goes first
            bits = int(min(30, max(20, math.ceil(math.log2(max(16 * n, 2))))))  # >= 16 bits per key: ~6 % false positives
            filt = self._zeros((1 << bits) // 32, t.int32)
            _lib.call("cfk_index_filter_build", self._p(sorted_keys), n, bits, self._p(filt), self._stream())
        return KmerIndex(sorted_keys=sorted_keys, idx_keys=idx_keys, idx_vals=idx_vals, cap=cap, n=n, filter=filt,
                         filter_bits=bits)

    def index_from_host_keys(self, keys_u64):
        """Sorted unique uint64 numpy keys -> KmerIndex (genomic_kmers arriving as set[str])."""
        keys = np.unique(np.asarray(keys_u64, dtype=np.uint64))
        return self.build_index(self._to_dev(keys.view(np.int64)), presorted=True)

    # ---- stage B ----------------------------------------------------------------------------
    def exclusive_scan(self, counts_i32):
        t = self.torch
        n = int(counts_i32.numel())
        out = self._empty(n + 1, t.int64)
        scratch = self._empty(int(self.lib.cfk_scan_scratch_elems(n)), t.int64)
        _lib.call("cfk_exclusive_scan", self._p(counts_i32), self._p(out), n, self._p(scratch), self._stream())
        return out

    def build_clouds(self, reads, units, k, index):
        k = check_k(k)
        t = self.torch
        U = units.n_units
        if U == 0:
            return CloudCSR(unit_ptr=self._zeros(1, t.int64), ids=self._empty(0, t.int32), n_units=0, n_entries=0)
        tmp = self._empty(units.n_kmer_starts, t.int32)
        cnt = self._empty(U, t.int32)
        with self._stage("cloud_build"):
            _lib.call("cfk_cloud_build", self._p(reads.packed), self._p(units.unit_off), self._p(units.unit_len),
                      self._p(units.unit_kbase), U, k, self._p(index.idx_keys), self._p(index.idx_vals), index.cap,
                      self._p(index.filter), int(index.filter_bits), self._p(tmp), self._p(cnt), self._stream())
        unit_ptr = self.exclusive_scan(cnt[:U])
        E = int(unit_ptr[U].item())
        ids = self._empty(E, t.int32)
        _lib.call("cfk_cloud_compact", self._p(tmp), self._p(units.unit_kbase), self._p(unit_ptr), U, self._p(ids),
                  self._stream())
        return CloudCSR(unit_ptr=unit_ptr, ids=ids[:E], n_units=U, n_entries=E)

    def id_histogram(self, csr, n_kmers, unit_lo=0, unit_hi=None):
        t = self.torch
        unit_hi = csr.n_units if unit_hi is None else unit_hi
        mult = self._zeros(n_kmers, t.int32)
        _lib.call("cfk_id_histogram", self._p(csr.unit_ptr), self._p(csr.ids), unit_lo, unit_hi, self._p(mult),
                  self._stream())
        return mult

    def filter_clouds(self, csr, n_kmers, min_mult=2, max_mult=math.inf):
        t = self.torch
        U = csr.n_units
        if U == 0:
            return csr
        big = 1 << 62
        lo = -big if min_mult == -math.inf else (big if min_mult == math.inf else int(math.ceil(min_mult)))
        hi = big if max_mult == math.inf else (-big if max_mult == -math.inf else int(math.floor(max_mult)))
        mult = self.id_histogram(csr, n_kmers)
        cnt = self._empty(U, t.int32)
        _lib.call("cfk_cloud_filter_count", self._p(csr.unit_ptr), self._p(csr.ids), U, self._p(mult), lo, hi,
                  self._p(cnt), self._stream())
        new_ptr = self.exclusive_scan(cnt[:U])
        E = int(new_ptr[U].item())
        new_ids = self._empty(E, t.int32)
        _lib.call("cfk_cloud_filter_write", self._p(csr.unit_ptr), self._p(csr.ids), U, self._p(mult), lo, hi,
                  self._p(new_ptr), self._p(new_ids), self._stream())
        return CloudCSR(unit_ptr=new_ptr, ids=new_ids[:E], n_units=U, n_entries=E)

    # ---- stage C / D ------------------------------------------------------------------------
    def build_occurrences(self, csr, n_kmers, unit_lo=0, unit_hi=None, unit_last=None):
        """-> (occ_ptr, occ, occ_last): the inverted cloud CSR; occ_last (unit_last gathered per occurrence) is None
        when unit_last is not given."""
        t = self.torch
        unit_hi = csr.n_units if unit_hi is None else unit_hi
        mult = self.id_histogram(csr, n_kmers, unit_lo, unit_hi)
        occ_ptr = self.exclusive_scan(mult[:n_kmers]) if n_kmers else self._zeros(1, t.int64)
        n_occ = int(occ_ptr[n_kmers].item()) if n_kmers else 0
        if n_occ >= 1 << 32:
            raise CfkError("occurrence lists: 2^32 or more cloud entries")
        occ = self._empty(n_occ, t.int32)
        cursor = self._empty(n_kmers, t.int32)
        _lib.call("cfk_occ_fill", self._p(csr.unit_ptr), self._p(csr.ids), unit_lo, unit_hi, self._p(occ_ptr), n_kmers,
                  self._p(cursor), self._p(occ), self._stream())
        _lib.call("cfk_occ_sort", self._p(occ_ptr), self._p(occ), n_kmers, self._stream())
        return occ_ptr, occ, self.occurrence_last(occ, unit_last)

    def occurrence_slice_count(self, csr, id_lo, id_hi):
        """First half of inverting the ids of [id_lo, id_hi) only (ShardedRecruiter.global_occurrences): -> (mult
        int32[id_hi - id_lo], ptr int64[id_hi - id_lo + 1] = its exclusive scan); nothing is read back."""
        t = self.torch
        n = id_hi - id_lo
        if n == 0:
            return self._empty(0, t.int32)[:0], self._zeros(1, t.int64)
        mult = self._zeros(n, t.int32)
        _lib.call("cfk_occ_slice_histogram", self._p(csr.unit_ptr), self._p(csr.ids), csr.n_units, id_lo, id_hi,
                  self._p(mult), self._stream())
        return mult, self.exclusive_scan(mult)

    def occurrence_slice_fill(self, csr, id_lo, id_hi, ptr, n_occ):
        """Second half: the slice's occurrence lists back to back (n_occ = ptr[-1], read back by the caller), each sorted."""
        t = self.torch
        n = id_hi - id_lo
        occ = self._empty(n_occ, t.int32)
        if n == 0 or n_occ == 0:
            return occ[:n_occ]
        cursor = self._empty(n, t.int32)
        _lib.call("cfk_occ_slice_fill", self._p(csr.unit_ptr), self._p(csr.ids), csr.n_units, id_lo, id_hi, self._p(ptr),
                  self._p(cursor), self._p(occ), self._stream())
        _lib.call("cfk_occ_sort", self._p(ptr), self._p(occ), n, self._stream())
        return occ[:n_occ]

    def occurrence_last(self, occ, unit_last):
        """occ_last[i] = unit_last[occ[i]] (None when the engine is told not to keep the per-occurrence copy)."""
        if unit_last is None or not self.use_occ_last:
            return None
        n_occ = int(occ.numel())
        occ_last = self._empty(n_occ, self.torch.int32)
        _lib.call("cfk_occ_last", self._p(occ), n_occ, self._p(unit_last), self._p(occ_last), self._stream())
        return occ_last

    def dist_edges(self, csr, unit_last, n_kmers, min_d, max_d, min_cov, rel_threshold=0.8,
                   unit_lo=0, unit_hi=None, a_begin=0, a_end=None, a_stride=1, occurrences=None):
        """Fused get_kmer_dist_map + filter_dist_tuples over source ids a_begin, a_begin+stride, ... < a_end."""
        t = self.torch
        if min_d < 0:
            raise ValueError("min_d < 0: the reference loop (dbkr.py:121) is undefined for negative distances")
        a_end = n_kmers if a_end is None else a_end
        empty = DistResult(edges=t.empty((0, 4), dtype=t.int32, device=self.device),
                           selected=self._empty(0, t.int32)[:0], n_candidates=0, n_increments=0, n_splits=0)
        if n_kmers == 0 or csr.n_entries == 0 or max_d < max(min_d, 1):
            return empty
        if occurrences is not None:
            occ_ptr, occ, occ_last = occurrences
        else:
            with self._stage("occurrences"):
                occ_ptr, occ, occ_last = self.build_occurrences(csr, n_kmers, unit_lo, unit_hi, unit_last)
        min_cov_u = int(min(max(min_cov, 0), U32_MAX))
        # stage C flavour: the sketch kernel serves min_cov in [3, 255]; the exact tables serve anything
        use_sketch = self.pair_mode != "exact" and SKETCH_MIN_COV <= min_cov_u <= SKETCH_MAX_COV
        if self.pair_mode == "sketch" and not use_sketch:
            raise CfkError(f"pair_mode=sketch needs {SKETCH_MIN_COV} <= min_coverage <= {SKETCH_MAX_COV}")
        if use_sketch:
            n_codes = int(self.lib.cfk_sketch_codes_elems(csr.n_entries, csr.n_units))
            codes = self._empty(n_codes, t.int16)
            perm = self._empty(n_codes, t.int32) if self.sketch_banked and n_codes < (1 << 32) else None
            with self._stage("sketch_codes"):
                _lib.call("cfk_sketch_codes", self._p(csr.unit_ptr), self._p(csr.ids), csr.n_units, self._p(codes),
                          self._p(perm), self._stream())
        else:
            usplit = self._empty(7 * csr.n_units, t.int32)
            _lib.call("cfk_unit_splits", self._p(csr.unit_ptr), self._p(csr.ids), csr.n_units, csr.n_entries, n_kmers,
                      self._p(usplit), self._stream())
        max_cand = int(self.cand_hint)
        while True:
            cand = self._empty(max_cand * 4, t.int32)
            counters = self._counters()
            with self._stage("pair_candidates"):
                if use_sketch:
                    _lib.call("cfk_pair_sketch", self._p(csr.unit_ptr), self._p(csr.ids), self._p(codes), self._p(perm),
                              self._p(unit_last), self._p(occ_ptr), self._p(occ), self._p(occ_last), csr.n_entries, n_kmers,
                              a_begin, a_end, a_stride, int(min_d), int(max_d), min_cov_u, self._p(cand), max_cand,
                              self._p(counters), self.n_sms, self._stream())
                else:
                    _lib.call("cfk_pair_candidates", self._p(csr.unit_ptr), self._p(csr.ids), self._p(unit_last),
                              self._p(occ_ptr), self._p(occ), self._p(usplit), csr.n_entries, n_kmers, a_begin, a_end,
                              a_stride, int(min_d), int(max_d), min_cov_u, self._p(cand), max_cand, self._p(counters),
                              self.n_sms, self._stream())
            c = counters.cpu()
            self.last_pair_counters = [int(x) for x in c.tolist()]
            self.last_pair_kernel = "pair_sketch_kernel" if use_sketch else "pair_candidates_kernel"
            n_cand = int(c[0])
            if n_cand <= max_cand:
                break
            # the size is now known: one more pass (the sketch kernel hands out the array in per-warp chunks of 256, so
            # the total moves by a few chunks from run to run: leave room for one chunk per warp)
            max_cand = n_cand + (self.n_sms * 32 * 256 if use_sketch else 0)
            del cand
        self.cand_hint = max(self.cand_hint, int(n_cand * 1.05) + 1024)
        selected = self._zeros(n_kmers, t.uint8)
        max_edges = max(int(self.edge_hint), n_cand + 1024)
        while True:
            edges = self._empty(max_edges * 4, t.int32)
            counters2 = self._counters()
            with self._stage("pair_join"):
                _lib.call("cfk_pair_join", self._p(cand), n_cand, self._p(occ_ptr), self._p(occ), self._p(occ_last),
                          self._p(unit_last),
                          int(min_d), int(max_d), min_cov_u, float(rel_threshold), self._p(edges), max_edges,
                          self._p(selected), self._p(counters2), self._stream())
            c2 = counters2.cpu()
            n_edges = int(c2[0])
            if n_edges <= max_edges:
                break
            max_edges = n_edges
            del edges
        self.edge_hint = max(self.edge_hint, int(n_edges * 1.05) + 1024)
        sel_idx = self._empty(n_kmers, t.int32)
        counters3 = self._counters()
        _lib.call("cfk_flag_indices", self._p(selected), n_kmers, self._p(sel_idx), self._p(counters3),
                  self._stream())
        n_sel = int(counters3.cpu()[0])
        return DistResult(edges=edges[: n_edges * 4].view(n_edges, 4), selected=sel_idx[:n_sel],
                          n_candidates=int(c2[2]), n_pair_candidates=int(c[4]) if use_sketch else n_cand,
                          n_increments=int(c[2]),
                          n_splits=int(c[3]))

    # ---- whole path -------------------------------------------------------------------------
    def recruit(self, reads, units, k, lo, hi, max_nonuniq, min_d, max_d, min_cov, rel_threshold=0.8,
                unit_lo=0, unit_hi=None, on_clouds=None):
        """main() of the reference script on device-resident inputs; returns device-resident results.
        on_clouds(index, csr) is called as soon as the rare set and the clouds are final (before the distance graph):
        the place to start their trip to the host (start_host_copy)."""
        rare = self.rare_kmers(reads, k, lo, hi, max_nonuniq)
        index = self.build_index(rare)
        csr = self.build_clouds(reads, units, k, index)
        if on_clouds is not None:
            on_clouds(index, csr)
        dist = self.dist_edges(csr, units.unit_last, index.n, min_d, max_d, min_cov, rel_threshold,
                               unit_lo=unit_lo, unit_hi=unit_hi)
        return index, csr, dist


_default_engine = None


def default_engine():
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine()
    return _default_engine


def to_host_u64(t):
    return t.cpu().numpy().view(np.uint64)


def to_host_u32(t, pinned=False):
    """Device tensor -> numpy uint32 view.  pinned: through a page-locked buffer of its own (the array keeps it alive;
    torch caches the allocation), 129 MB of edges in ~3 ms instead of ~60 ms through pageable memory."""
    if pinned and t.is_cuda and t.numel():
        import torch
        dst = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        with torch.cuda.device(t.device):
            dst.copy_(t, non_blocking=True)
            torch.cuda.current_stream(t.device).synchronize()
        return dst.numpy().view(np.uint32)
    return t.cpu().numpy().view(np.uint32)
