"""Deterministic synthetic inputs for the recruitment path (SURVEY.md §8d).

The reference ships a genome simulator only (scripts/simulate_tandem_repeat.py:15-34:
unit x multiplicity with binomial substitutions, 200 kb random flanks); the
reads behind its published numbers came from SimLoRD + the external NCRF
aligner, neither of which is available.  This module owns the rest:

* ``simulate_genome``   same model as the reference simulator (i.i.d. substitutions
  at ``div_rate`` over the array, random flanks), re-stated on ``numpy.random.default_rng``
  so it runs on the GPU box where /root/reference does not exist;
* ``simulate_reads``    long reads (log-normal lengths, both strands, i.i.d.
  sub/ins/del errors 1:1:1) and, for the array-overlapping part of every read,
  the TRUTH alignment against the motif in NCRF's two-row form;
* ``write_ncrf_report`` the text format scripts/ncrf_parser.py:74-77 parses
  ('-' strand records are written reverse-complemented so the parser's RC path,
  :96-100, is exercised; motif name = motif sequence, the post-``sed`` form of
  scripts/run_ncrf_parallel.py:72);
* ``SynthRead.direct_units`` the gap-free read bases + unit boundaries the device
  consumes, produced without going through text (bench inputs at 10^8 bases).
  tests/test_synth.py checks both routes agree.
"""
from dataclasses import dataclass

import os

import numpy as np

from .encode import ascii_to_codes, codes_to_ascii

GAP = 4
_SYM = np.frombuffer(b"ACGT-", dtype=np.uint8)
_COMP = np.array([3, 2, 1, 0, 4], dtype=np.uint8)


def read_fasta_first(path):
    seq = []
    with open(path) as f:
        for line in f:
            if line.startswith(">"):
                if seq:
                    break
                continue
            seq.append(line.strip())
    return "".join(seq).upper()


def random_unit(length, seed):
    return codes_to_ascii(np.random.default_rng(seed).integers(0, 4, size=length, dtype=np.uint8))


def hor_unit(n_monomers=12, monomer_len=171, divergence=0.25, seed=0):
    """A higher-order-repeat unit shaped like DXZ1 (12 diverged ~171 bp monomers, 2052 bp): every
    monomer is an independently mutated copy of one random ancestor."""
    rng = np.random.default_rng(seed)
    ancestor = rng.integers(0, 4, size=monomer_len, dtype=np.uint8)
    parts = []
    for _ in range(n_monomers):
        m = ancestor.copy()
        mut = rng.random(monomer_len) < divergence
        m[mut] = (m[mut] + rng.integers(1, 4, size=int(mut.sum()), dtype=np.uint8)) & 3
        parts.append(m)
    return codes_to_ascii(np.concatenate(parts))


def simulate_genome(unit, multiplicity, div_rate, seed, flank_len=200000):
    """-> (flanked genome codes, array start, array length)."""
    rng = np.random.default_rng(seed)
    u = ascii_to_codes(unit)
    arr = np.tile(u, multiplicity)
    mut = rng.random(arr.size) < div_rate
    arr[mut] = (arr[mut] + rng.integers(1, 4, size=int(mut.sum()), dtype=np.uint8)) & 3
    left = rng.integers(0, 4, size=flank_len, dtype=np.uint8)
    right = rng.integers(0, 4, size=flank_len, dtype=np.uint8)
    return np.concatenate([left, arr, right]), flank_len, arr.size


GENOME_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "genomes")


def load_genome(name):
    """A genome made by the reference's own simulate_tandem_repeat.py (oracle/make_genomes.py wrote it 2-bit packed
    under tests/golden/genomes/) -> (flanked genome codes, array start, array length, unit string)."""
    d = np.load(os.path.join(GENOME_DIR, name + ".npz"))
    packed, n = d["packed"], int(d["n"])
    codes = np.empty(packed.size * 4, dtype=np.uint8)
    for j in range(4):
        codes[j::4] = (packed >> (2 * j)) & 3
    return codes[:n], int(d["array_start"]), int(d["array_len"]), str(d["unit"])


@dataclass
class SynthRead:
    r_id: str
    r_len: int
    r_st: int          # forward-strand read coordinates of the aligned part
    r_en: int
    strand: str
    r_row: np.ndarray  # alignment rows on the motif's forward strand, codes 0..3, 4 = gap
    m_row: np.ndarray
    unit_cols: np.ndarray  # first column of every full motif copy + end column of the last (may be empty)

    @property
    def r_al_len(self):
        return int((self.r_row != GAP).sum())

    @property
    def m_al_len(self):
        return int((self.m_row != GAP).sum())

    def direct_units(self, motif_len):
        """(gap-free read codes, unit boundaries in gap-free read offsets).

        Applies the 20 % partial prefix / suffix rule of scripts/ncrf_parser.py:49-52
        to the truth columns; an empty boundary array means "no full motif copy".
        """
        keep = self.r_row != GAP
        bases = self.r_row[keep]
        if self.unit_cols.size == 0:
            return bases, np.empty(0, dtype=np.int64)
        coords = [int(c) for c in self.unit_cols]
        n_cols = self.r_row.size
        if coords[0] > motif_len * 0.2:
            coords.insert(0, 0)
        if coords[-1] < n_cols - motif_len * 0.2:
            coords.append(n_cols)
        before = np.concatenate([[0], np.cumsum(keep)])  # read bases before column c
        return bases, before[np.asarray(coords, dtype=np.int64)].astype(np.int64)


def _draw_lengths(rng, n, median, sigma, lo, hi):
    return np.clip(np.exp(rng.normal(np.log(median), sigma, size=n)), lo, hi).astype(np.int64)


def simulate_reads(genome, array_start, array_len, motif, coverage, error_rate, seed,
                   median_len=35000, sigma=0.5, min_len=5000, max_len=300000,
                   min_aligned=1, id_prefix="read", shard=None):
    """Reads overlapping the array, with their truth alignment to the motif.

    Coverage is over the flanked genome; reads whose overlap with the array is
    shorter than ``min_aligned`` genome bases carry no alignment and are skipped
    (NCRF would not report them).  ``shard=(r, n)`` materialises only reads i with i % n == r of the
    SAME read set (lengths, positions and per-read seeds are drawn for all reads first).
    """
    rng = np.random.default_rng(seed)
    motif_codes = ascii_to_codes(motif)
    L = motif_codes.size
    G = genome.size
    n_reads = int(np.ceil(coverage * G / (median_len * np.exp(sigma * sigma / 2))))
    lengths = _draw_lengths(rng, n_reads, median_len, sigma, min_len, max_len)
    starts = rng.integers(0, G, size=n_reads)
    strands = rng.random(n_reads) < 0.5
    seeds = rng.integers(0, 2**63 - 1, size=n_reads)
    a_lo, a_hi = array_start, array_start + array_len
    e3 = error_rate / 3.0
    reads = []
    for i in range(n_reads):
        if shard is not None and i % shard[1] != shard[0]:
            continue
        s = int(starts[i])
        e = min(G, s + int(lengths[i]))
        a0, a1 = max(s, a_lo), min(e, a_hi)
        n = a1 - a0
        if n < max(min_aligned, 1):
            continue
        r = np.random.default_rng(int(seeds[i]))
        u = r.random(n)
        ins = r.random(n) < e3
        ins[-1] = False
        g = genome[a0:a1]
        r_base = g.copy()
        sub = u < e3
        r_base[sub] = (g[sub] + r.integers(1, 4, size=int(sub.sum()), dtype=np.uint8)) & 3
        r_base[(u >= e3) & (u < 2 * e3)] = GAP
        n_ins = int(ins.sum())
        col = np.arange(n, dtype=np.int64)
        col[1:] += np.cumsum(ins[:-1])
        n_cols = n + n_ins
        r_row = np.empty(n_cols, dtype=np.uint8)
        m_row = np.empty(n_cols, dtype=np.uint8)
        phase = (np.arange(a0, a1, dtype=np.int64) - a_lo) % L
        r_row[col] = r_base
        m_row[col] = motif_codes[phase]
        ins_col = col[ins] + 1
        r_row[ins_col] = r.integers(0, 4, size=n_ins, dtype=np.uint8)
        m_row[ins_col] = GAP
        # full motif copies inside [a0, a1)
        first = a0 + ((-(a0 - a_lo)) % L)
        n_full = (a1 - first) // L if first <= a1 else 0
        if n_full > 0:
            pos = first + L * np.arange(n_full + 1, dtype=np.int64)
            unit_cols = np.where(pos < a1, col[np.minimum(pos, a1 - 1) - a0], n_cols)
        else:
            unit_cols = np.empty(0, dtype=np.int64)
        left_flank = a0 - s
        al_len = int((r_row != GAP).sum())
        r_len = left_flank + al_len + (e - a1)
        reads.append(SynthRead(r_id=f"{id_prefix}_{i}", r_len=r_len, r_st=left_flank, r_en=left_flank + al_len,
                               strand="-" if strands[i] else "+", r_row=r_row, m_row=m_row,
                               unit_cols=unit_cols.astype(np.int64)))
    return reads


def _row_text(row, rc):
    if rc:
        row = _COMP[row][::-1]
    return _SYM[row].tobytes().decode("ascii")


def ncrf_record_lines(read, motif):
    """The two text lines of one record, as NCRF would print them."""
    minus = read.strand == "-"
    if minus:  # the file holds read-strand coordinates and reverse-complemented rows
        st, en = read.r_len - read.r_en, read.r_len - read.r_st
    else:
        st, en = read.r_st, read.r_en
    score = int((read.r_row == read.m_row).sum())
    l1 = f"{read.r_id} {read.r_len} {read.r_al_len}bp {st}-{en} {_row_text(read.r_row, minus)}"
    l2 = f"{motif}{read.strand} {read.m_al_len}bp score={score} {_row_text(read.m_row, minus)}"
    return l1, l2


def write_ncrf_report(path, reads, motif, header=True):
    with open(path, "w") as f:
        if header:
            f.write("# synthetic NCRF report (centroflye_b200.synth)\n\n")
        for rd in reads:
            l1, l2 = ncrf_record_lines(rd, motif)
            f.write(l1 + "\n" + l2 + "\n\n")


def make_dataset(unit, multiplicity, div_rate, genome_seed, coverage, error_rate, read_seed,
                 flank_len=200000, **read_kw):
    genome, a0, alen = simulate_genome(unit, multiplicity, div_rate, genome_seed, flank_len=flank_len)
    return simulate_reads(genome, a0, alen, unit, coverage, error_rate, read_seed, **read_kw)


# ---- compressed read files: BGZF (SAM spec §4.1) and unaligned BAM (§4.2) ---------------------------------------------

BGZF_BLOCK = 65280  # input bytes per block, as bgzip and htslib write them
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
BAM_CODES = "=ACMGRSVTWYHKDBN"


def bgzf_member(data, level=6, strategy=None, flush_at=()):
    """One BGZF block holding `data` (at most 65536 bytes): zlib raw deflate at `level` / `strategy`, with a Z_FULL_FLUSH
    after each offset of flush_at (several DEFLATE blocks in one member), a gzip header with the BC subfield, CRC32 and
    ISIZE."""
    import struct
    import zlib
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY if strategy is None else strategy)
    parts, at = [], 0
    for cut in list(flush_at) + [len(data)]:
        parts.append(c.compress(bytes(data[at:cut])))
        if cut < len(data):
            parts.append(c.flush(zlib.Z_FULL_FLUSH))
        at = cut
    parts.append(c.flush())
    payload = b"".join(parts)
    bsize = 18 + len(payload) + 8 - 1
    if bsize > 0xffff:
        raise ValueError("bgzf_member: the block does not compress into 64 KiB")
    head = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize)
    return head + payload + struct.pack("<II", zlib.crc32(data) & 0xffffffff, len(data))


def bgzf_compress(data, level=6, strategy=None, block=BGZF_BLOCK, eof=True):
    """`data` as BGZF: one member per `block` bytes, then the 28-byte end-of-file block."""
    data = memoryview(bytes(data))
    out = [bgzf_member(data[i:i + block], level, strategy) for i in range(0, len(data), block)]
    return b"".join(out) + (BGZF_EOF if eof else b"")


def write_bgzf(path, data, **kw):
    with open(path, "wb") as f:
        f.write(bgzf_compress(data, **kw))


def bam_record(name, seq, flag=0, cigar=(), qual=None, tags=b"", ref_id=-1, pos=-1):
    """One BAM alignment record (block_size included).  seq is text over BAM_CODES (other bytes are written as N); it is
    stored as given, reverse-complemented or not; cigar = [(length, op index 0..8)]; qual None writes 0xff bytes."""
    import struct
    name_b = name.encode() + b"\0"
    l_seq = len(seq)
    lut = np.full(256, 15, dtype=np.uint8)
    lut[np.frombuffer(BAM_CODES.encode(), dtype=np.uint8)] = np.arange(16, dtype=np.uint8)
    nib = np.append(lut[np.frombuffer(seq.encode("latin-1"), dtype=np.uint8)], np.uint8(0))
    packed = ((nib[0:l_seq:2] << 4) | nib[1:l_seq + 1:2][:(l_seq + 1) // 2]).tobytes()
    q = b"\xff" * l_seq if qual is None else bytes(qual)
    body = struct.pack("<iiBBHHHiiii", ref_id, pos, len(name_b), 255, 4680, len(cigar), flag, l_seq, -1, -1, 0)
    body += name_b + b"".join(struct.pack("<I", (n << 4) | op) for n, op in cigar) + packed + q + bytes(tags)
    return struct.pack("<i", len(body)) + body


def bam_bytes(records, refs=(("chr1", 248956422),), text="@HD\tVN:1.6\tSO:unknown\n"):
    """The inflated stream of a BAM file: magic, header text, references, then the records (bam_record keyword
    dicts, or already encoded bytes)."""
    import struct
    out = [b"BAM\1", struct.pack("<i", len(text)), text.encode(), struct.pack("<i", len(refs))]
    for name, length in refs:
        out += [struct.pack("<i", len(name) + 1), name.encode() + b"\0", struct.pack("<i", length)]
    out += [r if isinstance(r, (bytes, bytearray)) else bam_record(**r) for r in records]
    return b"".join(out)


def write_bam(path, records, level=6, **kw):
    """A BAM file (bam_bytes, BGZF-compressed)."""
    write_bgzf(path, bam_bytes(records, **kw), level=level)
