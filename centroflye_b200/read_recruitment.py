"""The read recruitment pre-filter of the reference (``scripts/read_recruitment/rr.cpp``, SURVEY.md §8f rank 4) on the
device: same command line (``rr unit.fasta reads.fasta[.gz] output.fasta edit_distance_threshold``), same output file.

rr.cpp:73-90 aligns the unit and its reverse complement against every read with edlib in HW mode (the whole unit
against any infix of the read, k = threshold) and copies the read to the output when either alignment exists.  Here the
two alignments of every read are bit-parallel scans on the GPU (csrc/rr_filter.cu): cfk_rr_filter, one thread per read
and strand, for units of up to 3328 bases, and cfk_rr_filter_long, one warp per read and strand, for units of up to
32768 bases.

The command line streams (recruit_file): the read file goes through in chunks of a fixed size -- a reader thread reads
or inflates it, a native scanner (csrc/seq_scan.cpp, cfk_seq_scan) finds the records of a chunk, the device gathers
the sequences, filters them and assembles ``>name\\nsequence\\n`` of the kept reads in input order, and a writer thread
appends that to the output.  Host and device memory follow the chunk size, not the input size.  recruit_file_units is
the same pipeline for several (unit, output, threshold) jobs: the file is read and scanned once, one filter launch per
word class covers every unit, and each output gets the bytes recruit_file writes for that job alone (recruit_file is
its one-job case; main_units / scripts/rr_multi.py is its command line); with devices= it deals every chunk's records
out to several GPUs in contiguous ranges, and the outputs are the same bytes.  read_sequences() and
recruit() are the in-memory form of the same computation, and the specification the streaming form is tested against.

The read file may be FASTA / FASTQ, plain, gzip or bgzip, or unaligned BAM; nothing but its bytes tells them apart.  A
file whose first gzip member is a BGZF block (bgzip, BAM) is inflated on the run's first device (_DeviceInflater:
cfk_bgzf_blocks finds the blocks on the host, csrc/bgzf.cu inflates a chunk's worth at once); other gzip files are
inflated by zlib on the reader thread.  A stream that starts with "BAM\\1" is scanned by cfk_bam_scan instead of
cfk_seq_scan and gathered by cfk_rr_bam_gather; it yields the reads ``samtools fastq -n -F 0x900`` writes (_read_bam).
"""
import gzip
import os
import queue
import sys
import threading
import time

import numpy as np

from . import _lib
from ._lib import CfkError

_COMPLEMENT = {"A": "T", "T": "A", "G": "C", "C": "G"}
SEGMENT = 8192  # read bases per device work item (a multiple of 16: segments start on 16-byte boundaries)


def reverse_complement(unit):
    """rr.cpp:11-39,58-63; a unit symbol outside ACGT trips the reference's assert."""
    try:
        return "".join(_COMPLEMENT[c] for c in reversed(unit))
    except KeyError as e:
        raise AssertionError(f"complement(): unexpected symbol {e.args[0]!r} in the unit") from None


def read_sequences(path):
    """(name, sequence) of every FASTA / FASTQ record, plain or gzip -- what kseq_read yields: the name is the header up
    to the first whitespace, sequence lines are joined until a line starting with '>', '@' or '+'; after '+' as many
    quality characters as the sequence has bases are skipped.  A file whose (inflated) bytes start with "BAM\\1" is
    unaligned BAM, read by _read_bam."""
    with open(path, "rb") as f:
        magic = f.read(2)
    opener = gzip.open if magic == b"\x1f\x8b" else open
    with opener(path, "rb") as f:
        bam = f.read(4) == BAM_MAGIC
    if bam:
        yield from _read_bam(path, opener)
        return
    with opener(path, "rt") as f:
        line = f.readline()
        while line:
            if line[:1] not in (">", "@"):
                line = f.readline()
                continue
            name = (line[1:].split() or [""])[0]
            chunks = []
            line = f.readline()
            while line and line[:1] not in (">", "@", "+"):
                chunks.append(line.strip())
                line = f.readline()
            seq = "".join(chunks)
            if line[:1] == "+":
                left = len(seq)
                line = f.readline()
                while line and left > 0:
                    left -= len(line.rstrip("\r\n"))
                    line = f.readline()
            yield name, seq


BAM_MAGIC = b"BAM\1"
_BAM_PAIRS = [a + b for a in "=ACMGRSVTWYHKDBN" for b in "=ACMGRSVTWYHKDBN"]  # one SEQ byte -> its two bases
_BAM_COMPLEMENT = str.maketrans("=ACMGRSVTWYHKDBN", "=TGKCYSBAWRDMHVN")


def _bam_bases(packed, l_seq, reverse):
    """The bases of a BAM SEQ field (4-bit codes, two per byte), reverse-complemented when `reverse`."""
    seq = "".join(map(_BAM_PAIRS.__getitem__, packed))[:l_seq]
    return seq[::-1].translate(_BAM_COMPLEMENT) if reverse else seq


def _read_bam(path, opener):
    """(name, sequence) of every record of an unaligned BAM file (SAM spec §4.2), read with `opener` and struct: the FASTQ
    records ``samtools fastq -n -F 0x900`` writes -- secondary and supplementary alignments (flag & 0x900) yield
    nothing, the name is QNAME (no /1 or /2), the sequence is SEQ over "=ACMGRSVTWYHKDBN", reverse-complemented (A-T, C-G,
    M-K, R-Y, H-D, B-V; W, S, N and = are their own complements) when flag & 0x10 is set.  Quality, CIGAR and tags are
    ignored.  That this is samtools' output is the intent; it has not been checked against samtools itself."""
    import struct
    with opener(path, "rb") as f:
        def exact(n):
            b = f.read(n)
            if len(b) != n:
                raise EOFError("the BAM file ends inside a record or its header")
            return b
        exact(4)
        exact(struct.unpack("<i", exact(4))[0])  # header text
        for _ in range(struct.unpack("<i", exact(4))[0]):  # references: name, length
            exact(struct.unpack("<i", exact(4))[0] + 4)
        while True:
            head = f.read(4)
            if not head:
                return
            block_size = struct.unpack("<i", head if len(head) == 4 else exact(4))[0]
            if block_size < 32:
                raise ValueError(f"BAM record with block_size {block_size}")
            rec = exact(block_size)
            l_read_name = rec[8]
            n_cigar_op, flag, l_seq = struct.unpack_from("<HHi", rec, 12)
            at = 32 + l_read_name + 4 * n_cigar_op
            if l_read_name == 0 or l_seq < 0 or at + (l_seq + 1) // 2 + l_seq > block_size:
                raise ValueError("BAM record with fields past its block_size")
            if not flag & 0x900:
                yield rec[32:32 + l_read_name - 1].decode("ascii"), _bam_bases(rec[at:at + (l_seq + 1) // 2], l_seq,
                                                                                flag & 0x10)


MAX_SHORT_UNIT = 3328  # the longest unit of cfk_rr_filter / cfk_rr_filter_units (rr_filter_kernel<52>)


def is_long(unit):
    """Does the unit take cfk_rr_filter_long (the warp-per-segment kernel) rather than cfk_rr_filter?"""
    return len(unit) > MAX_SHORT_UNIT


def build_masks(unit):
    """-> (peq uint64[2, S, NW], sym_of uint8[256], NW) for cfk_rr_filter: units of 1..3328 bases (build_long_masks
    for longer ones)."""
    m = len(unit)
    nw = int(_lib.load().cfk_rr_words(m))
    if nw < 0:
        raise CfkError(f"read recruitment: the unit has {m} bases; 1..3328 are supported")
    return _masks(unit, nw)


def build_long_masks(unit):
    """-> (peq uint64[2, S, W, 32], sym_of uint8[256], W) for cfk_rr_filter_long: units of 1..32768 bases.  The masks of
    build_masks padded with zero words to 32 W, lane-minor: peq[strand, s, k, L] is word L * W + k."""
    m = len(unit)
    w = int(_lib.load().cfk_rr_long_words(m))
    if w < 0:
        raise CfkError(f"read recruitment: the unit has {m} bases; 1..32768 are supported")
    peq, sym_of, _ = _masks(unit, 32 * w)
    return np.ascontiguousarray(peq.reshape(2, -1, 32, w).transpose(0, 1, 3, 2)), sym_of, w


def _job_masks(unit, long_units):
    """The masks of a unit the streaming form filters: build_long_masks for a unit of more than 3328 bases when
    long_units is set, build_masks otherwise (which refuses such a unit, as the streaming form always has)."""
    if not is_long(unit):
        return build_masks(unit)
    if not long_units:
        raise CfkError(f"read recruitment: the unit has {len(unit)} bases; 1..3328 are supported "
                       "(long_units=True, which the rr and rr_multi command lines pass, takes up to 32768)")
    return build_long_masks(unit)


def _masks(unit, nw):
    """The match masks and symbol table of build_masks with nw words per strand."""
    lib = _lib.load()
    m = len(unit)
    n_sym = int(lib.cfk_rr_max_symbols())
    symbols = sorted(set((unit + reverse_complement(unit)).encode("latin-1")))  # both strands share one symbol table
    if len(symbols) > n_sym - 1:
        raise CfkError(f"read recruitment: the unit uses {len(symbols)} distinct symbols; at most {n_sym - 1} are supported")
    sym_of = np.zeros(256, dtype=np.uint8)
    for slot, b in enumerate(symbols, start=1):
        sym_of[b] = slot
    peq = np.zeros((2, n_sym, nw), dtype=np.uint64)
    for strand, seq in enumerate((unit, reverse_complement(unit))):
        codes = sym_of[np.frombuffer(seq.encode("latin-1"), dtype=np.uint8)]
        pos = np.arange(m)
        for slot in range(1, len(symbols) + 1):
            hit = pos[codes == slot]
            np.bitwise_or.at(peq[strand, slot], hit >> 6, np.uint64(1) << (hit & 63).astype(np.uint64))
    return peq, sym_of, nw


def _segment_plan(lens, overlap, long_unit):
    """The device work items of reads of lengths lens (int64): read r is cut into n_seg[r] = max(1, ceil(max(lens[r] -
    overlap, 1) / step)) segments, segment j covering bases [j step, min(j step + step + overlap, lens[r])).  step is
    SEGMENT, or with long_unit (a unit of more than 3328 bases in the plan) at least the overlap rounded up to 16, so a
    unit of 32 kb does not scan every base about five times.  Either way step is a multiple of 16, so a segment starts
    on a 16-byte boundary when its read does: the kernels read the text 16 bytes at a time.
    -> (n_seg, seg_read, start, seg_len), the last three per segment: its read, first base and length."""
    step = max(SEGMENT, (overlap + 15) // 16 * 16) if long_unit else SEGMENT
    n_seg = np.maximum(1, -(-np.maximum(lens - overlap, 1) // step))
    seg_read = np.repeat(np.arange(len(lens), dtype=np.int64), n_seg)
    start = (np.arange(seg_read.size, dtype=np.int64) - np.repeat(np.cumsum(n_seg) - n_seg, n_seg)) * step
    return n_seg, seg_read, start, np.minimum(step + overlap, lens[seg_read] - start)


def recruit(unit, seqs, threshold, exact=False, engine=None):
    """keep[r] (bool) for every sequence, and with exact=True the infix edit distances int32[R, 2] (unit, reverse
    complement) of cfk_rr_filter, or of cfk_rr_filter_long for a unit of more than 3328 bases (up to 32768)."""
    from .engine import default_engine
    eng = engine or default_engine()
    t = eng.torch
    long_unit = is_long(unit)
    peq, sym_of, _ = build_long_masks(unit) if long_unit else build_masks(unit)
    R = len(seqs)
    keep = np.zeros(R, dtype=bool)
    dist = np.zeros((R, 2), dtype=np.int32) if exact else None
    d_peq, d_sym = eng._to_dev(peq.reshape(-1).view(np.int64)), eng._to_dev(sym_of)
    start, budget = 0, 1 << 30  # device batches of about 1 GiB of read bytes
    while start < R:
        end, total = start, 0
        while end < R and (end == start or total + len(seqs[end]) <= budget):
            total += (len(seqs[end]) + 15) & ~15
            end += 1
        lens = np.array([len(s) for s in seqs[start:end]], dtype=np.int64)
        offs = np.zeros(end - start, dtype=np.int64)
        np.cumsum(((lens + 15) & ~15)[:-1], out=offs[1:])
        text = np.zeros(int(offs[-1] + ((lens[-1] + 15) & ~15)) + 16, dtype=np.uint8)
        for o, s in zip(offs.tolist(), seqs[start:end]):
            text[o:o + len(s)] = np.frombuffer(s.encode("latin-1"), dtype=np.uint8)
        # One thread walks one segment.  A hit within `threshold` edits spans at most |unit| + threshold read bases, so a
        # long read is cut into segments of SEGMENT bases that overlap by that much: the decision per read (any segment
        # hits) is unchanged, the longest read no longer sets the kernel's duration.  Exact distances need whole reads.
        seg_read = np.arange(end - start, dtype=np.int64)
        seg_off, seg_len = offs, lens
        if not exact and threshold >= 0:
            _, seg_read, seg_start, seg_len = _segment_plan(lens, len(unit) + int(threshold), long_unit)
            seg_off = offs[seg_read] + seg_start
        order = np.argsort(-seg_len, kind="stable").astype(np.int32)
        n = int(seg_read.size)
        d_keep = eng._zeros(n, t.uint8)
        d_dist = eng._empty(2 * n, t.int32) if exact else None
        d_text, d_offs, d_lens, d_order = eng._to_dev(text), eng._to_dev(seg_off), eng._to_dev(seg_len), eng._to_dev(order)
        p = eng._p
        with eng._stage("rr_filter"):
            if long_unit:
                m_t = np.array([len(unit), int(threshold)], dtype=np.int32)
                _lib.call("cfk_rr_filter_long", p(d_text), p(d_offs), p(d_lens), p(d_order), n, 1, p(d_peq), p(d_sym),
                          m_t.ctypes.data, m_t[1:].ctypes.data, int(bool(exact)), p(d_dist), p(d_keep), eng._stream())
            else:
                _lib.call("cfk_rr_filter", p(d_text), p(d_offs), p(d_lens), p(d_order), n, p(d_peq), p(d_sym), len(unit),
                          int(threshold), int(bool(exact)), p(d_dist), p(d_keep), eng._stream())
        hit = np.zeros(end - start, dtype=bool)
        np.logical_or.at(hit, seg_read, d_keep[:n].cpu().numpy().astype(bool))
        keep[start:end] = hit
        if exact:
            dist[start:end] = d_dist[: 2 * n].cpu().numpy().reshape(n, 2)
        start = end
    return (keep, dist) if exact else keep


CHUNK_BYTES = 64 << 20  # read-file bytes per streaming step (recruit_file); main() uses this
_BLOCK_BYTES = 8 << 20   # the reader thread's unit of readinto / inflate; four blocks are read ahead
# scanner table sizes: a record slot (32 bytes) per 128 chunk bytes, a piece slot (24 bytes) per 64; a chunk whose
# records need more is processed in parts
_REC_BYTES_PER_SLOT, _PIECE_BYTES_PER_SLOT = 128, 64


def _open_binary(path, inflate=None):
    """The read file as bytes, inflated when it starts with the gzip magic (like read_sequences).  inflate: None, or
    (device, chunk_bytes, stats) -- a file whose first member is a BGZF block is then inflated on that device
    (_DeviceInflater; device is a callable returning a torch.device)."""
    with open(path, "rb") as f:
        head = f.read(_BGZF_MAX_MEMBER)
    if head[:2] != b"\x1f\x8b":
        return open(path, "rb")
    if inflate is not None and _bgzf_blocks(np.frombuffer(head, dtype=np.uint8), 1)[0] == 1:
        return _DeviceInflater(path, *inflate)
    return gzip.open(path, "rb")


_BGZF_MAX_MEMBER = 1 << 16  # BSIZE is 16 bits: no BGZF member is larger
_BGZF_INCOMPLETE, _BGZF_NOT_BGZF = 1, 2  # cfk_bgzf_blocks flags (include/cfk.h)
_BGZF_STATUS = {1: "not a valid DEFLATE stream", 2: "inflated length differs from ISIZE", 3: "CRC32 mismatch"}


def _bgzf_blocks(buf, max_blocks, rows=None):
    """cfk_bgzf_blocks on buf (uint8 array) -> (n_blocks, consumed, inflated bytes, flags); rows: int64[max_blocks, 5]."""
    out = np.zeros(4, dtype=np.int64)
    if rows is None:
        rows = np.zeros((max_blocks, 5), dtype=np.int64)
    _lib.call("cfk_bgzf_blocks", buf.ctypes.data, buf.size, rows.ctypes.data, max_blocks, out.ctypes.data)
    return tuple(out.tolist())


class _DeviceInflater:
    """A BGZF file's inflated bytes, read with readinto() like a gzip.GzipFile: cfk_bgzf_blocks finds the blocks of the
    compressed bytes, enough of them to fill a chunk go to the device in one copy, cfk_bgzf_inflate inflates them on a
    stream of its own, and the inflated bytes come back into a pinned buffer.  From a member that is not BGZF on
    (or a last member cut short) the rest of the file goes to gzip.GzipFile on the host, so every file reads to the
    bytes -- or the error -- gzip.open gives.  A block the device rejects raises gzip.BadGzipFile with its file offset.
    stats["inflate_s"] gets the device seconds of the kernel, stats["bgzf_blocks"] the number of blocks."""

    def __init__(self, path, device, chunk_bytes, stats):
        import torch
        self.torch, self.device, self.stats = torch, device(), stats
        self.f = open(path, "rb")
        self.max_blocks = max(1, chunk_bytes // _BGZF_MAX_MEMBER)
        self.cap = self.max_blocks * _BGZF_MAX_MEMBER  # compressed bytes that always hold max_blocks blocks
        self.buf = self.have = self.file_off = None  # compressed bytes buf[:have], from file offset file_off
        self.out, self.at, self.n = None, 0, 0  # inflated bytes out[at:n] not yet read
        self.tail, self.file_eof = None, False
        self.stream = self.dev = None
        stats.setdefault("inflate_s", 0.0)
        stats.setdefault("bgzf_blocks", 0)

    def readinto(self, view):
        view = np.frombuffer(view, dtype=np.uint8)
        k = 0
        while k < view.size:
            if self.at < self.n:
                take = min(view.size - k, self.n - self.at)
                view[k:k + take] = self.out[self.at:self.at + take]
                k, self.at = k + take, self.at + take
            elif self.tail is not None:
                got = self.tail.readinto(view[k:])
                if not got:
                    break
                k += got
            elif not self._fill():
                break
        return k

    def _setup(self):
        torch = self.torch
        torch.cuda.set_device(self.device)  # the reader thread launches on the run's first device
        self.stream = torch.cuda.Stream(self.device)
        pinned = lambda n: torch.empty(n, dtype=torch.uint8, pin_memory=True)  # noqa: E731
        dev = lambda n: torch.empty(n, dtype=torch.uint8, device=self.device)  # noqa: E731
        B = self.max_blocks
        self.h_comp, self.h_rows = pinned(self.cap), pinned(40 * B)
        self.h_out, self.h_status = pinned(B * _BGZF_MAX_MEMBER), pinned(4 * B)
        self.dev = {"comp": dev(self.cap), "rows": dev(40 * B), "out": dev(B * _BGZF_MAX_MEMBER), "status": dev(4 * B)}
        self.buf, self.have, self.file_off = self.h_comp.numpy(), 0, 0
        self.rows = self.h_rows.numpy().view(np.int64).reshape(B, 5)
        self.out = self.h_out.numpy()

    def _fill(self):
        """Inflates the next blocks into self.out; False at the end of the file."""
        torch = self.torch
        if self.dev is None:
            self._setup()
        while True:
            while not self.file_eof and self.have < self.cap:  # enough compressed bytes for max_blocks blocks
                got = self.f.readinto(memoryview(self.buf)[self.have:])
                self.file_eof = not got
                self.have += got
            n, consumed, total, flags = _bgzf_blocks(self.buf[:self.have], self.max_blocks, self.rows)
            if n or flags or consumed < self.have:
                break
            self.have, self.file_off = 0, self.file_off + consumed  # nothing but zero padding: skipped, read on
            if self.file_eof:
                return False
        if n == 0:
            # a member that is not BGZF, or a last member cut short: the rest of the file, from there, on the host
            self.f.seek(self.file_off + consumed)
            self.tail = gzip.GzipFile(fileobj=self.f, mode="rb")
            return True
        d = self.dev
        status = self.h_status.numpy()[:4 * n].view(np.int32)
        with torch.cuda.stream(self.stream):
            d["comp"][:consumed].copy_(self.h_comp[:consumed], non_blocking=True)
            d["rows"][:40 * n].copy_(self.h_rows[:40 * n], non_blocking=True)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _lib.call("cfk_bgzf_inflate", d["comp"].data_ptr(), d["rows"].data_ptr(), n, d["out"].data_ptr(),
                      d["status"].data_ptr(), self.stream.cuda_stream)
            b.record()
            self.h_out[:total].copy_(d["out"][:total], non_blocking=True)
            self.h_status[:4 * n].copy_(d["status"][:4 * n], non_blocking=True)
        self.stream.synchronize()
        self.stats["inflate_s"] += a.elapsed_time(b) / 1e3
        self.stats["bgzf_blocks"] += n
        bad = np.flatnonzero(status)
        if bad.size:
            i = int(bad[0])
            start = 0 if i == 0 else int(self.rows[i - 1, 0] + self.rows[i - 1, 1] + 8)
            while self.buf[start] == 0:  # zero padding before the member
                start += 1
            raise gzip.BadGzipFile(f"BGZF block at file offset {self.file_off + start}: "
                                   f"{_BGZF_STATUS.get(int(status[i]), 'bad status')}")
        self.at, self.n = 0, total
        self.buf[:self.have - consumed] = self.buf[consumed:self.have]
        self.have -= consumed
        self.file_off += consumed
        return True

    def close(self):
        if self.tail is not None:
            self.tail.close()
        self.f.close()


class _Fallback(Exception):
    """The chunk is outside what the streaming form reproduces byte for byte (a byte >= 0x80, which str semantics
    treat differently, or a record too large for the int32 output sizes): recruit_file runs the in-memory path."""


class _BlockReader:
    """Reads (or inflates) the file block by block on a thread of its own; readinto and zlib release the GIL."""

    def __init__(self, path, block, depth=4, inflate=None):
        self.f = _open_binary(path, inflate)
        self.block, self.seconds = block, 0.0
        self.free, self.full = queue.Queue(), queue.Queue()
        for _ in range(depth):
            self.free.put(np.empty(block, dtype=np.uint8))
        self.thread = threading.Thread(target=self._run, name="rr-reader", daemon=True)
        self.thread.start()

    def _run(self):
        try:
            while True:
                buf = self.free.get()
                if buf is None:
                    return
                t0, n, view = time.perf_counter(), 0, memoryview(buf)
                while n < buf.size:
                    k = self.f.readinto(view[n:])
                    if not k:
                        break
                    n += k
                self.seconds += time.perf_counter() - t0
                self.full.put((buf, n))
                if n < buf.size:
                    return
        except BaseException as e:  # noqa: BLE001 -- handed to the consumer, which raises it
            self.full.put(e)

    def get(self):
        item = self.full.get()
        if isinstance(item, BaseException):
            raise item
        return item

    def close(self):
        self.free.put(None)
        self.thread.join()
        self.f.close()


def _grown(store, key, nbytes, make):
    """store[key], replaced by make(size) when it holds fewer than nbytes bytes (sizes are multiples of 16, and exact
    otherwise: the pinned host allocator rounds up to a power of two, and chunk sizes usually are one)."""
    buf = store.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = store[key] = make(max(int(nbytes) + 15 & ~15, 1 << 12))
    return buf


def _scan_chunks(read_fn, chunk_bytes, host, stats, inflate_device=None):
    """Chunks of the read file cut at record boundaries by cfk_seq_scan, or by cfk_bam_scan when the (inflated) file
    starts with the BAM magic: yields (slot, raw, records, pieces, text_bytes, bam) where raw (uint8 tensor) holds the
    chunk's bytes, records int64[n, 4] and pieces are the scanner's tables (numpy views of tensors in `host`, made by
    host["alloc"]): int64[m, 3] from cfk_seq_scan, or cfk_bam_scan's bam_seq int64[n, 2] when bam is set.  Two slots
    alternate: what is yielded stays valid until the next-but-one chunk is asked for.  A chunk without a complete
    record is doubled until it has one, so an ultra-long read (or a BAM header) fits any chunk size; bytes before the
    first complete record that hold none (lines outside records, the BAM header, secondary alignments) are dropped
    instead.  inflate_device: None inflates gzip input on the host; a callable returning a torch.device inflates a
    BGZF file on that device (_DeviceInflater)."""
    alloc = lambda key, nbytes: _grown(host, key, nbytes, host["alloc"])  # noqa: E731
    inflate = None if inflate_device is None else (inflate_device, chunk_bytes, stats)
    reader = _BlockReader(read_fn, max(1 << 16, min(chunk_bytes, _BLOCK_BYTES)), inflate=inflate)
    out = np.zeros(5, dtype=np.int64)
    carry, eof, slot, table_scale = np.zeros(0, dtype=np.uint8), False, 0, 1
    blk, at, k = None, 0, 0  # the reader's block being taken apart: blk[at:k] is not in a chunk yet
    bam, stream_off, rec_index = None, 0, 0  # BAM: raw[0]'s offset in the inflated stream, alignments before it
    try:
        while True:
            n, target = carry.size, max(chunk_bytes, carry.size)
            raw = alloc((slot, "raw"), target)
            raw.numpy()[:n] = carry
            while True:
                t0 = time.perf_counter()
                while n < target and not (eof and blk is None):
                    if blk is None:
                        blk, k = reader.get()
                        at, eof = 0, k < blk.size
                    if raw.numel() < target:
                        old = raw
                        raw = alloc((slot, "raw"), target)
                        raw[:n] = old[:n]
                    take = min(k - at, target - n)
                    raw.numpy()[n:n + take] = blk[at:at + take]
                    n, at = n + take, at + take
                    if at == k:
                        reader.free.put(blk)
                        blk = None
                end = eof and blk is None
                t1 = time.perf_counter()
                max_rec = table_scale * max(64, n // _REC_BYTES_PER_SLOT)
                max_piece = table_scale * max(64, n // _PIECE_BYTES_PER_SLOT)
                rec = alloc((slot, "rec"), 32 * max_rec).numpy().view(np.int64)
                buf = raw.numpy()
                if bam is None:
                    bam = bytes(buf[:4]) == BAM_MAGIC
                if bam:
                    piece = alloc((slot, "piece"), 16 * max_rec).numpy().view(np.int64)
                    _lib.call("cfk_bam_scan", buf.ctypes.data, n, int(end), int(stream_off == 0), rec_index, stream_off,
                              rec.ctypes.data, max_rec, piece.ctypes.data, out.ctypes.data)
                else:
                    piece = alloc((slot, "piece"), 24 * max_piece).numpy().view(np.int64)
                    _lib.call("cfk_seq_scan", buf.ctypes.data, n, int(end), rec.ctypes.data, max_rec, piece.ctypes.data,
                              max_piece, out.ctypes.data)
                stats["assemble_s"] += t1 - t0
                stats["scan_s"] += time.perf_counter() - t1
                n_rec, n_piece, consumed, text_bytes, flags = out.tolist()  # BAM: n_piece = alignments consumed
                if flags & _SCAN_NOT_ASCII:
                    raise _Fallback("a byte >= 0x80 in the read file")
                if n_rec:
                    break
                if flags & _SCAN_FULL:
                    table_scale *= 2
                elif end:
                    return
                elif consumed:  # nothing to yield in buf[:consumed]: keep only the rest
                    buf[:n - consumed] = buf[consumed:n]
                    n -= consumed
                    stream_off += consumed
                    rec_index += n_piece if bam else 0
                else:
                    target = 2 * n
            table = piece[:2 * n_rec].reshape(-1, 2) if bam else piece[:3 * n_piece].reshape(-1, 3)
            yield slot, raw[:n], rec[:4 * n_rec].reshape(-1, 4), table, text_bytes, bam
            if end and consumed == n:
                return
            carry, slot = buf[consumed:n], slot ^ 1
            stream_off += consumed
            rec_index += n_piece if bam else 0
    finally:
        stats["read_s"] += reader.seconds
        reader.close()


_SCAN_NOT_ASCII, _SCAN_FULL = 1, 2  # cfk_seq_scan flags (include/cfk.h)


def scan_sequences(path, chunk_bytes=CHUNK_BYTES):
    """(name, sequence) of every record, as read_sequences(path) yields them, through the native scanner and the
    chunking of recruit_file, on the host alone.  Raises _Fallback where recruit_file hands over to read_sequences."""
    import torch
    host = {"alloc": lambda n: torch.empty(n, dtype=torch.uint8)}
    stats = {"assemble_s": 0.0, "scan_s": 0.0, "read_s": 0.0}
    for _, raw, rec, piece, _, bam in _scan_chunks(path, chunk_bytes, host, stats):
        buf, p = raw.numpy(), 0
        if bam:
            for (name_off, name_len, seq_len, _), (src, rev) in zip(rec.tolist(), piece.tolist()):
                yield (buf[name_off:name_off + name_len].tobytes().decode(),
                       _bam_bases(buf[src:src + (seq_len + 1) // 2].tobytes(), seq_len, rev))
            continue
        for name_off, name_len, seq_len, seq_dst in rec.tolist():
            parts = []
            while p < len(piece) and piece[p, 2] < seq_dst + seq_len:
                parts.append(buf[piece[p, 0]:piece[p, 0] + piece[p, 1]].tobytes())
                p += 1
            yield buf[name_off:name_off + name_len].tobytes().decode(), b"".join(parts).decode()


def _write_in_memory(unit, read_fn, path, threshold):
    """The whole read set as Python strings, one recruit() call, one write: the form every input can take."""
    _write_in_memory_jobs(read_fn, [(unit, path, threshold)])


def _write_in_memory_jobs(read_fn, jobs, long_units=False):
    """_write_in_memory for every (unit, path, threshold) of jobs, reading the file once.  Every unit is checked before
    the first output is written (long_units: as in recruit_file_units)."""
    records = list(read_sequences(read_fn))
    if records:
        for unit, _, _ in jobs:
            _job_masks(unit, long_units)
    seqs = [seq for _, seq in records]
    for unit, path, threshold in jobs:
        keep = recruit(unit, seqs, threshold) if records else np.zeros(0, dtype=bool)
        with open(path, "w") as f:
            f.write("".join(f">{name}\n{seq}\n" for (name, seq), k in zip(records, keep.tolist()) if k))


def recruit_file(unit, read_fn, output_fn, threshold, chunk_bytes=CHUNK_BYTES, engine=None, stats=None,
                 long_units=False):
    """rr's whole run, from the read file to the output file: ``>name\\nsequence\\n`` of every read of read_fn (FASTA /
    FASTQ, plain, gzip or bgzip, or unaligned BAM) that holds the unit or its reverse complement within `threshold`
    edits (threshold < 0: every read), in input order -- the bytes the in-memory path (read_sequences + recruit) writes, streamed in chunks of
    about chunk_bytes.  The output appears under output_fn only when the run has finished (it is written to a temporary
    file beside it, then renamed).  An input without records gives an empty file and touches neither the device nor the
    unit, except that a BGZF file (bgzip, BAM) is inflated on the device whether it holds records or not; otherwise an invalid unit raises before any output exists.  A chunk with a byte >= 0x80 hands the whole run to
    the in-memory path.  stats: None, or a dict that receives seconds per host stage, device seconds per stage
    (CUDA events, "device_s") and counts.  long_units: as in recruit_file_units."""
    return recruit_file_units([(unit, output_fn, threshold)], read_fn, chunk_bytes, engine, stats, long_units=long_units)


def _part_file(output_fn):
    """A new temporary file beside output_fn -> (path, binary file object)."""
    out_dir, base = os.path.split(os.path.abspath(output_fn))
    i = 0
    while True:
        tmp = os.path.join(out_dir, f".{base}.{os.getpid()}.{i}.part")
        try:
            return tmp, open(tmp, "xb")
        except FileExistsError:
            i += 1


def recruit_file_units(jobs, read_fn, chunk_bytes=CHUNK_BYTES, engine=None, stats=None, devices=None, long_units=False):
    """recruit_file for every job (unit, output_fn, threshold) of `jobs` in one pass over read_fn: the file is read,
    inflated and scanned once, the device filters every chunk for all units in one launch per unit word class, and
    each output file gets the bytes recruit_file writes for that job alone.  All outputs appear together when the run
    has finished; on an error none is created or modified.  An input without records gives empty files and checks no
    unit (a BGZF input is still inflated on the device: the first of `devices`, or the engine's); otherwise every unit is checked, with recruit_file's errors, before any output exists.  A byte >= 0x80 hands
    the whole run to the in-memory path (the file is read once, then recruit() per job).  Raises ValueError for no jobs,
    or for two jobs with the same output file.  Host and device memory follow chunk_bytes times the number of jobs.

    devices: None runs on one device (`engine`, or the default engine).  A list of devices (indices or torch.device;
    repeats allowed) runs one worker per entry, each with an Engine, buffers and a thread of its own: every chunk's
    records are dealt out in contiguous ranges of about equal bases (_split_records), each worker runs the device
    work of its range, and every output is the workers' parts of each chunk in list order -- the same bytes.
    stats: as in recruit_file, plus "job_out_bytes" (output bytes per job), "devices" (the number of workers) and
    "device_s_per_device" (device seconds per stage of each worker; "device_s" is their sum).

    long_units: also take units of 3329..32768 bases (cfk_rr_filter_long, one warp per segment and strand; the plan's
    segment step grows to the overlap rounded up to 16 when that exceeds SEGMENT).  Without it such a unit raises
    CfkError, the 3328-base limit this function has always had; the rr and rr_multi command lines pass it."""
    jobs = [(unit, output_fn, int(threshold)) for unit, output_fn, threshold in jobs]
    if not jobs:
        raise ValueError("recruit_file_units: no jobs")
    real = [os.path.realpath(output_fn) for _, output_fn, _ in jobs]
    if len(set(real)) != len(real):
        raise ValueError("recruit_file_units: two jobs write the same output file")
    if devices is None:
        def engines():
            from .engine import default_engine
            return [engine or default_engine()]

        def inflate_device():
            return engines()[0].device
        n_dev = 1
    else:
        devices = list(devices)
        if not devices or engine is not None:
            raise ValueError("recruit_file_units: devices must be a non-empty list, and excludes engine")

        def engines():
            from .engine import Engine
            return [Engine(d) for d in devices]

        def inflate_device():
            import torch
            return torch.device(devices[0])  # as Engine(devices[0]) takes it
        n_dev = len(devices)
    st = {key: 0.0 for key in ("read_s", "assemble_s", "scan_s", "plan_s", "wait_s", "write_s")}
    st.update(inflate_s=0.0, bgzf_blocks=0, chunks=0, records=0, bases=0, out_bytes=0, job_out_bytes=[0] * len(jobs), fallback=None,
              devices=n_dev, device_s=None if stats is None else {},
              device_s_per_device=None if stats is None else [{} for _ in range(n_dev)])
    tmps, files = [], []
    try:
        for _, output_fn, _ in jobs:
            tmp, f = _part_file(output_fn)
            tmps.append(tmp)
            files.append(f)
        try:
            try:
                _stream([(unit, threshold) for unit, _, threshold in jobs], read_fn, files, chunk_bytes, engines, st,
                        long_units, inflate_device)
            finally:
                for f in files:
                    f.close()
        except _Fallback as e:
            st["fallback"] = str(e)
            _write_in_memory_jobs(read_fn, [(unit, tmp, threshold) for (unit, _, threshold), tmp in zip(jobs, tmps)],
                                  long_units)
        for tmp, (_, output_fn, _) in zip(tmps, jobs):
            os.replace(tmp, output_fn)
    except BaseException:
        for f in files:
            f.close()
        for tmp in tmps:
            if os.path.exists(tmp):
                os.remove(tmp)
        raise
    if stats is not None:
        stats.update(st)
    return 0


def _split_records(seq_len, n):
    """The records of one chunk dealt to n devices: bounds int64[n + 1], device g takes records bounds[g] ..
    bounds[g + 1] - 1.  The ranges are contiguous and cover every record once; none is empty unless there are fewer
    records than devices; each holds total / n bases give or take the longest record.  A record goes to the range its
    middle base falls in, so a range gains or loses at most half a record at either end.  A range can only be left
    empty by a record longer than total / n; such ranges then take one record each from their neighbours, which only
    shrinks the others."""
    R = len(seq_len)
    if R < n:
        return np.minimum(np.arange(n + 1, dtype=np.int64), R)
    ends = np.cumsum(seq_len, dtype=np.int64)
    twice_mid = 2 * ends - seq_len
    b = np.searchsorted(n * twice_mid, 2 * int(ends[-1]) * np.arange(n + 1, dtype=np.int64), side="left")
    b[0], b[n] = 0, R
    for k in range(1, n):
        b[k] = min(max(b[k], b[k - 1] + 1), R - n + k)
    return b.astype(np.int64)


class _Worker:
    """One device of recruit_file_units' pipeline: a thread (named rr-device-<index>) that runs step() on its record
    range of every chunk handed to it through `inbox` and puts step()'s result, or the exception that ended it, on
    `outbox`.  Its engine, device buffers, pinned host buffers and output buffers are its own and follow the size of
    its ranges.  Every device call of a step is on the engine's stream, so one set of device buffers serves all
    chunks.  `run` holds what every worker shares: the filter plan of the jobs and the run's error state."""

    def __init__(self, index, eng, run, peq, sym_of):
        import torch
        self.torch, self.index, self.eng, self.run = torch, index, eng, run
        self.host, self.dev, self.events, self.plan_s = {}, {}, [], 0.0
        self.free_out = [queue.Queue() for _ in run.jobs]  # two output buffers per job, handed back by the writer
        for q in self.free_out:
            q.put(0)
            q.put(1)
        self.d_peq = self.d_sym = None
        if run.filtered:
            self.d_peq, self.d_sym = eng._to_dev(peq), eng._to_dev(sym_of)
        self.inbox, self.outbox = queue.Queue(), queue.Queue()
        self.thread = threading.Thread(target=self._loop, name=f"rr-device-{index}", daemon=True)
        self.thread.start()

    def _loop(self):
        try:
            self.eng._stream()  # makes the engine's device current for this thread
            while True:
                item = self.inbox.get()
                if item is None:
                    return
                if not self.run.abort.is_set():
                    self.outbox.put(self.step(*item))
        except BaseException as e:  # noqa: BLE001 -- raised by the main thread when it collects this chunk
            self.outbox.put(e)

    def _mark(self):
        if not self.run.timed:
            return None
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def _hbuf(self, key, nbytes):
        return _grown(self.host, key, nbytes, lambda n: self.torch.empty(n, dtype=self.torch.uint8, pin_memory=True))

    def _dbuf(self, key, nbytes, dtype=None):
        t = self.torch
        buf = _grown(self.dev, key, nbytes, lambda n: t.empty(n, dtype=t.uint8, device=self.eng.device))
        return buf.view(dtype or t.uint8)

    def step(self, raw, rec, piece, text_bytes, bam, r0, r1):
        """The device work of records r0 .. r1 - 1 of a chunk as _scan_chunks yields it: their bytes of raw and their
        rows of rec and piece (bam: the bam_seq rows), rebased on the host, go to the device, which gathers their
        sequences, filters them for every unit and emits every job's output; the outputs come home into this worker's
        output buffers.  Returns the parts for the writer, [(copy-done event, job, host buffer, bytes, free queue, key)],
        in job order."""
        if r0 == r1:
            return []
        torch, run, p = self.torch, self.run, self.eng._p
        t0 = time.perf_counter()
        # the range's text is rec[r0, 3] .. the next record's (16-byte aligned, like every record's), its pieces are
        # the ones placed there, and its raw bytes run from its first name to its last name or piece (BAM: to its
        # last SEQ, which follows the name)
        t_lo = int(rec[r0, 3])
        t_hi = int(rec[r1, 3]) if r1 < rec.shape[0] else text_bytes
        lo, hi = int(rec[r0, 0]), int(rec[r1 - 1, 0] + rec[r1 - 1, 1])
        if bam:
            table, shift = piece[r0:r1], [lo, 0]
            hi = max(hi, int(piece[r1 - 1, 0] + (rec[r1 - 1, 2] + 1) // 2))
        else:
            p0, p1 = (int(x) for x in np.searchsorted(piece[:, 2], (t_lo, t_hi)))
            table, shift = piece[p0:p1], [lo, 0, t_lo]
            if p1 > p0:
                hi = max(hi, int(piece[p1 - 1, 0] + piece[p1 - 1, 1]))
        R, P, n, text_bytes = r1 - r0, table.shape[0], hi - lo, t_hi - t_lo
        h_rec = self._hbuf("rec", 32 * R)
        rec = np.subtract(rec[r0:r1], np.array([lo, 0, 0, t_lo], dtype=np.int64),
                          out=h_rec.numpy()[:32 * R].view(np.int64).reshape(R, 4))
        pb = table.nbytes
        h_piece = self._hbuf("piece", pb)
        np.subtract(table, np.array(shift, dtype=np.int64), out=h_piece.numpy()[:pb].view(np.int64).reshape(table.shape))
        seq_len = rec[:, 2]
        upper = int((rec[:, 1] + seq_len).sum()) + 3 * R
        # segments as recruit() plans them (with run.overlap); when no job has threshold >= 0 no filter runs.
        # Host layout, int64: seg_off[S] | seg_len[S] | seg_ptr[R + 1] (first segment of each record) | order[S] (int32
        # in the first half)
        S, F = 0, len(run.filtered)
        if F:
            n_seg, seg_read, seg_start, seg_len = _segment_plan(seq_len, run.overlap, run.n_short < F)
            S = int(n_seg.sum())
            nb = 8 * (3 * S + R + 1)
            hs = self._hbuf("seg", nb)
            seg = hs.numpy()[:nb].view(np.int64)
            seg_lens = seg[S:2 * S]
            seg[:S] = rec[seg_read, 3] + seg_start
            seg_lens[:] = seg_len
            seg[2 * S] = 0
            np.cumsum(n_seg, out=seg[2 * S + 1:2 * S + R + 1])
            seg[2 * S + R + 1:].view(np.int32)[:S] = np.argsort(-seg_lens, kind="stable")
        self.plan_s += time.perf_counter() - t0
        a = self._mark()
        d_raw = self._dbuf("raw", n + 16)
        d_raw[:n].copy_(raw[lo:hi], non_blocking=True)
        d_rec = self._dbuf("rec", 32 * R)
        d_rec[:32 * R].copy_(h_rec[:32 * R], non_blocking=True)
        d_piece = self._dbuf("piece", pb + 8)
        if P:
            d_piece[:pb].copy_(h_piece[:pb], non_blocking=True)
        if S:
            d_seg = self._dbuf("seg", nb)
            d_seg[:nb].copy_(hs[:nb], non_blocking=True)
        b = self._mark()
        stream = self.eng._stream()
        d_text = self._dbuf("text", text_bytes + 16)
        if bam:
            _lib.call("cfk_rr_bam_gather", p(d_raw), p(d_piece), p(d_rec), R, p(d_text), text_bytes, stream)
        else:
            _lib.call("cfk_rr_gather", p(d_raw), p(d_piece), P, p(d_text), text_bytes, stream)
        c = self._mark()
        d_keep = seg_ptr = None
        if S:
            d_keep = self._dbuf("keep", F * S)  # [unit][segment]: the short units' rows, then the long units'
            d_keep[:F * S].zero_()
            base = d_seg.data_ptr()
            seg_ptr = base + 16 * S
            args = (p(d_text), base, base + 8 * S, base + 8 * (2 * S + R + 1), S)
            k = run.n_short
            if k:
                _lib.call("cfk_rr_filter_units", *args, k, p(self.d_peq), p(self.d_sym), run.unit_m.ctypes.data,
                          run.unit_threshold.ctypes.data, p(d_keep), stream)
            if k < F:
                _lib.call("cfk_rr_filter_long", *args, F - k, p(self.d_peq) + 8 * run.short_words,
                          p(self.d_sym) + 256 * k, run.unit_m[k:].ctypes.data, run.unit_threshold[k:].ctypes.data, 0,
                          None, p(d_keep) + k * S, stream)
        d = self._mark()
        d_sizes = self._dbuf("sizes", 4 * R, torch.int32)
        d_off = self._dbuf("off", 8 * (R + 1), torch.int64)
        d_scratch = self._dbuf("scratch", 8 * int(self.eng.lib.cfk_scan_scratch_elems(R)))
        d_totals = self._dbuf("totals", 8 * len(run.jobs), torch.int64)
        d_outs = []
        for j in range(len(run.jobs)):  # sizes, offsets and scan scratch are reused: the job's emit has read them by then
            d_out = self._dbuf(("out", j), upper + 16)
            seg_keep = None if j not in run.row else p(d_keep) + run.row[j] * S
            _lib.call("cfk_rr_keep_sizes", seg_keep, None if seg_keep is None else seg_ptr, p(d_rec), R, p(d_sizes),
                      stream)
            _lib.call("cfk_exclusive_scan", p(d_sizes), p(d_off), R, p(d_scratch), stream)
            _lib.call("cfk_rr_emit", p(d_raw), p(d_text), p(d_rec), p(d_off), R, upper, p(d_out), stream)
            d_totals[j:j + 1].copy_(d_off[R:R + 1])
            d_outs.append(d_out)
        if run.timed:
            self.events.extend((("h2d", a, b), ("gather", b, c), ("filter", c, d), ("emit", d, self._mark())))
        # the range's one size read-back: into pinned memory and an event wait, not a synchronous copy to pageable
        # memory, which blocks the CUDA calls of other threads (the BGZF reader's) until the filter has finished
        J = len(run.jobs)
        h_totals = self._hbuf("totals", 8 * J)
        h_totals[:8 * J].copy_(d_totals.view(torch.uint8)[:8 * J], non_blocking=True)
        sized = torch.cuda.Event()
        sized.record()
        sized.synchronize()
        totals = h_totals.numpy()[:8 * J].view(np.int64).tolist()
        parts = []
        for j, (total, d_out) in enumerate(zip(totals, d_outs)):
            key = self.free_out[j].get()
            if run.writer_err:
                raise run.writer_err[0]
            h = self._hbuf(("out", j, key), total)
            a = self._mark()
            if total:
                h[:total].copy_(d_out[:total], non_blocking=True)
            done = torch.cuda.Event()
            done.record()
            if run.timed:
                self.events.append(("d2h", a, self._mark()))
            parts.append((done, j, h, total, self.free_out[j], key))
        return parts


def _stream(jobs, read_fn, files, chunk_bytes, engines, st, long_units=False, inflate_device=None):
    """recruit_file_units' pipeline: jobs = [(unit, threshold)], files[j] receives job j's output, engines() -> one
    engine per worker (called once the first record is seen).  While the workers' devices work on chunk i, the reader
    thread reads ahead, this thread scans chunk i + 1 and deals its records out, and the writer thread writes chunk
    i - 1, every job's parts in worker order.  Host chunk buffers come in two slots (see _scan_chunks): a slot is
    scanned into again only after every worker has finished with it."""
    import types

    import torch
    host = {"alloc": lambda n: torch.empty(n, dtype=torch.uint8)}  # pageable until the first record is seen
    # the jobs that run the filter (threshold >= 0; the others keep every read), and their units' rows in d_peq / d_sym
    # and d_keep: the units of cfk_rr_filter_units first, then the longer ones of cfk_rr_filter_long
    filtered = [j for j, (_, threshold) in enumerate(jobs) if threshold >= 0]
    filtered.sort(key=lambda j: is_long(jobs[j][0]))  # stable: job order within each group
    # One segment plan serves every unit.  A hit within t edits spans at most |unit| + t read bases, so it lies wholly
    # inside some segment whenever the segments overlap by at least that much; and a segment is an infix of its read,
    # so a hit inside a segment is a hit in the read.  Overlapping by the largest |unit| + t of all jobs therefore
    # decides every read as recruit()'s plan for each job alone does.  Segments never span records, so dealing the
    # records of a chunk out to several devices changes no decision either.
    run = types.SimpleNamespace(
        jobs=jobs, filtered=filtered, row={j: i for i, j in enumerate(filtered)},
        unit_m=np.array([len(jobs[j][0]) for j in filtered], dtype=np.int32),
        unit_threshold=np.array([jobs[j][1] for j in filtered], dtype=np.int32),
        overlap=max((len(jobs[j][0]) + jobs[j][1] for j in filtered), default=0),
        n_short=sum(not is_long(jobs[j][0]) for j in filtered), short_words=0,
        timed=st["device_s"] is not None, abort=threading.Event(), writer_err=[])
    workers, writer, writer_q = [], None, queue.Queue()

    def write_loop():
        while True:
            item = writer_q.get()
            if item is None:
                return
            done, j, h, nbytes, free, key = item
            try:
                done.synchronize()
                t0 = time.perf_counter()
                files[j].write(memoryview(h.numpy()[:nbytes]))
                st["write_s"] += time.perf_counter() - t0
            except BaseException as e:  # noqa: BLE001 -- raised by a worker at its next hand-over
                run.writer_err.append(e)
            free.put(key)

    def start():
        nonlocal writer
        masks = [_job_masks(unit, long_units) for unit, _ in jobs]  # raises on an invalid unit, before any output
        peq = sym_of = None
        if filtered:
            peq = np.concatenate([masks[j][0].reshape(-1) for j in filtered]).view(np.int64)
            sym_of = np.concatenate([masks[j][1] for j in filtered])
            run.short_words = sum(masks[j][0].size for j in filtered[:run.n_short])
        for g, eng in enumerate(engines()):
            workers.append(_Worker(g, eng, run, peq, sym_of))
        host["alloc"] = lambda n: torch.empty(n, dtype=torch.uint8, pin_memory=True)
        writer = threading.Thread(target=write_loop, name="rr-writer", daemon=True)
        writer.start()

    def collect():
        """Waits for every worker's result of the oldest chunk in flight and queues its parts for the writer."""
        for w in workers:
            t0 = time.perf_counter()
            parts = w.outbox.get()
            st["wait_s"] += time.perf_counter() - t0
            if isinstance(parts, BaseException):
                raise parts
            for part in parts:
                _, j, _, nbytes, _, _ = part
                st["out_bytes"] += nbytes
                st["job_out_bytes"][j] += nbytes
                writer_q.put(part)

    chunks = _scan_chunks(read_fn, chunk_bytes, host, st, inflate_device)
    in_flight = False
    try:
        for slot, raw, rec, piece, text_bytes, bam in chunks:  # scanning chunk i + 1 overlaps the devices' work on chunk i
            first = not workers
            if first:
                start()
            t0 = time.perf_counter()
            seq_len = rec[:, 2]
            if int((rec[:, 1] + seq_len).max()) + 3 >= 1 << 31:
                raise _Fallback("a record of 2 GiB or more")
            st["records"] += rec.shape[0]
            st["bases"] += int(seq_len.sum())
            bounds = _split_records(seq_len, len(workers)).tolist()
            for w, r0, r1 in zip(workers, bounds[:-1], bounds[1:]):
                w.inbox.put((raw, rec, piece, text_bytes, bam, r0, r1))
            st["chunks"] += 1
            st["plan_s"] += time.perf_counter() - t0
            if in_flight:
                collect()
            in_flight = True
            if first:  # chunk 0 was scanned into pageable memory: the slot's later chunks use pinned buffers
                for name in ("raw", "rec", "piece"):
                    host.pop((slot, name))
        if in_flight:
            collect()
    finally:
        chunks.close()
        run.abort.set()  # after an error, workers skip what is queued
        for w in workers:
            w.inbox.put(None)
        if writer is not None:
            writer_q.put(None)
        for w in workers:
            w.thread.join()
        if writer is not None:
            writer.join()
    if run.writer_err:
        raise run.writer_err[0]
    st["plan_s"] += sum(w.plan_s for w in workers)
    if run.timed:
        for w in workers:
            torch.cuda.synchronize(w.eng.device)
            mine = st["device_s_per_device"][w.index]
            for name, a, b in w.events:
                s = a.elapsed_time(b) / 1e3
                mine[name] = mine.get(name, 0.0) + s
                st["device_s"][name] = st["device_s"].get(name, 0.0) + s


def main(argv=None):
    argv = sys.argv[1:] if argv is None else list(argv)
    if len(argv) != 4 or argv[0] == "-h":
        print("Usage: ./rr unit.fasta reads.fasta.gz output.fasta edit_distance_threshold", end="")  # rr.cpp's text
        print(RR_READS_NOTE, file=sys.stderr)
        return 0
    unit_fn, read_fn, output_fn = argv[:3]
    try:
        threshold = int(argv[3])
    except ValueError:
        threshold = 0  # std::atoi
    unit = next(read_sequences(unit_fn))[1]  # 1..32768 bases (edlib's rr takes any length)
    recruit_file(unit, read_fn, output_fn, threshold, long_units=True)
    return 0


RR_READS_NOTE = "\nreads: FASTA or FASTQ, plain, gzip or bgzip, or unaligned BAM (told apart by their bytes)"
UNITS_USAGE = ("Usage: rr_multi.py reads.{fasta,fastq}[.gz]|reads.bam unit1.fasta output1.fasta threshold1 [unit2.fasta output2.fasta threshold2 ...]\n"
               "       --gpus N (first): deal every chunk's records over cuda:0..N-1")


def main_units(argv=None):
    """``rr_multi.py [--gpus N] reads unit1 output1 threshold1 [unit2 output2 threshold2 ...]``: what one rr run per
    triple writes, from one pass over the read file (recruit_file_units; FASTA / FASTQ, plain, gzip or bgzip, or BAM).  Each unit is the first record of its file,
    of 1..32768 bases;
    thresholds are read as main() reads them.  --gpus N runs on cuda:0 .. N-1 (devices=); without it, on one device.
    A wrong argument count, or an N that is not an integer from 1 to the number of visible devices: the usage on
    stderr, status 2."""
    argv = sys.argv[1:] if argv is None else list(argv)
    devices = None
    if argv[:1] == ["--gpus"]:
        import torch
        try:
            n = int(argv[1])
        except (IndexError, ValueError):
            n = 0
        if not 1 <= n <= torch.cuda.device_count():
            print(UNITS_USAGE, file=sys.stderr)
            return 2
        devices, argv = list(range(n)), argv[2:]
    if len(argv) < 4 or (len(argv) - 1) % 3:
        print(UNITS_USAGE, file=sys.stderr)
        return 2
    jobs = []
    for unit_fn, output_fn, text in zip(argv[1::3], argv[2::3], argv[3::3]):
        try:
            threshold = int(text)
        except ValueError:
            threshold = 0  # std::atoi, as in main()
        jobs.append((next(read_sequences(unit_fn))[1], output_fn, threshold))
    recruit_file_units(jobs, argv[0], devices=devices, long_units=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
