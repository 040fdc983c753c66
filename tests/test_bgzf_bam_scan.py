"""The host scanners of compressed read files (csrc/bam_scan.cpp): cfk_bgzf_blocks on the output of synth's BGZF writer,
and cfk_bam_scan -- through scan_sequences and directly -- against read_sequences(), the in-memory specification, which
reads BAM with gzip and struct alone."""
import gzip
import struct
import zlib

import numpy as np
import pytest

from centroflye_b200 import _lib, synth
from centroflye_b200 import read_recruitment as rr


def _blocks(data, max_blocks=1000):
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    rows = np.zeros((max_blocks, 5), dtype=np.int64)
    n, consumed, total, flags = rr._bgzf_blocks(buf, max_blocks, rows)
    return rows[:n], consumed, total, flags


# ---- cfk_bgzf_blocks ---------------------------------------------------------------------------------------------------

def test_bgzf_blocks_on_writer_output():
    data = bytes(range(256)) * 1000
    comp = synth.bgzf_compress(data, block=50000)
    rows, consumed, total, flags = _blocks(comp)
    assert flags == 0 and consumed == len(comp) and total == len(data)
    assert rows[:, 2].tolist() == [50000, 50000, 50000, 50000, 50000, 6000, 0]  # the EOF block is an empty block
    assert rows[:, 4].tolist() == np.concatenate([[0], np.cumsum(rows[:-1, 2])]).tolist()
    out = b""
    for off, length, isize, crc, dst in rows.tolist():
        block = zlib.decompress(comp[off:off + length], -15)
        assert len(block) == isize and zlib.crc32(block) == crc and dst == len(out)
        out += block
    assert out == data
    assert comp[-28:] == synth.BGZF_EOF
    assert _blocks(comp, max_blocks=2)[0].shape[0] == 2


def test_bgzf_blocks_zero_padding_and_plain_gzip_member():
    data = b"ACGT" * 30000
    comp = synth.bgzf_compress(data)
    rows, consumed, _, flags = _blocks(comp + b"\0" * 777)
    assert flags == 0 and consumed == len(comp) + 777 and rows.shape[0] == 3
    rows, consumed, _, flags = _blocks(comp[:-28] + b"\0" * 5 + synth.BGZF_EOF)
    assert flags == 0 and rows.shape[0] == 3
    plain = gzip.compress(b"tail")
    rows, consumed, _, flags = _blocks(comp + plain)
    assert flags == rr._BGZF_NOT_BGZF and consumed == len(comp) and rows.shape[0] == 3
    rows, consumed, _, flags = _blocks(comp + b"\0\0garbage")
    assert flags == rr._BGZF_NOT_BGZF and consumed == len(comp) + 2


def test_bgzf_blocks_cut_at_every_byte_of_a_member():
    a, b = synth.bgzf_member(b"first" * 100), synth.bgzf_member(b"second" * 200)
    for cut in range(len(b)):
        rows, consumed, total, flags = _blocks(a + b[:cut])
        assert rows.shape[0] == 1 and total == 500, cut
        assert consumed == len(a), cut
        assert flags == (rr._BGZF_INCOMPLETE if cut else 0), cut
    rows, consumed, total, flags = _blocks(a + b)
    assert rows.shape[0] == 2 and flags == 0 and total == 1700


def test_bgzf_blocks_general_header_and_not_bgzf():
    m = bytearray(synth.bgzf_member(b"x" * 1000))
    # FNAME and FCOMMENT after the extra field, and a second subfield before BC: still BGZF
    extra = b"ZZ\x03\x00abc" + bytes(m[12:18])
    body = m[18:]
    head = bytes([0x1f, 0x8b, 8, 4 | 8 | 16]) + bytes(m[4:10]) + struct.pack("<H", len(extra)) + extra
    head += b"name\0comment\0"
    bsize = len(head) + len(body) - 1
    i = head.index(b"BC")
    head = head[:i + 4] + struct.pack("<H", bsize) + head[i + 6:]
    rows, consumed, total, flags = _blocks(head + body)
    assert flags == 0 and rows.shape[0] == 1 and total == 1000
    assert zlib.decompress((head + body)[rows[0, 0]:rows[0, 0] + rows[0, 1]], -15) == b"x" * 1000
    big = bytearray(m)
    big[-4:] = struct.pack("<I", 65537)  # ISIZE above 65536
    assert _blocks(bytes(m) + bytes(big))[1:] == (len(m), 1000, rr._BGZF_NOT_BGZF)
    no_bc = bytearray(m)
    no_bc[12:14] = b"XC"
    assert _blocks(bytes(no_bc))[3] == rr._BGZF_NOT_BGZF
    assert _blocks(gzip.compress(b"plain"))[3] == rr._BGZF_NOT_BGZF


def test_bgzf_blocks_arguments():
    with pytest.raises(_lib.CfkError, match="bad arguments"):
        _lib.call("cfk_bgzf_blocks", None, -1, None, 0, np.zeros(4, dtype=np.int64).ctypes.data)


# ---- cfk_bam_scan ------------------------------------------------------------------------------------------------------

def _bam_records(rng, n=120):
    recs = []
    for i in range(n):
        L = int(rng.choice([0, 1, 2, 3, 15, 16, 17, 101, 2000]))
        seq = "".join(rng.choice(list(synth.BAM_CODES), size=L))
        flag = int(rng.choice([0, 4, 0x10, 0x14, 0x100, 0x800, 0x900, 0x110]))
        name = f"r{i}_" + "q" * int(rng.choice([0, 7, 254 - len(f"r{i}_")]))
        cigar = [(int(rng.integers(1, 1000)), int(rng.integers(0, 9)))] * int(rng.integers(0, 4))
        tags = b"XXZ" + b"t" * int(rng.choice([0, 9, 70000])) + b"\0"
        recs.append(dict(name=name, seq=seq, flag=flag, cigar=cigar, tags=tags,
                         qual=None if i % 2 else bytes(rng.integers(0, 60, size=L).astype(np.uint8))))
    recs.append(dict(name="all_codes", seq=synth.BAM_CODES))
    recs.append(dict(name="all_codes_rc", seq=synth.BAM_CODES * 3 + "A", flag=0x10))
    return recs


def _expected(recs):
    comp = dict(zip(synth.BAM_CODES, "=TGKCYSBAWRDMHVN"))
    out = []
    for r in recs:
        flag, seq = r.get("flag", 0), r["seq"]
        if flag & 0x900:
            continue
        out.append((r["name"], "".join(comp[c] for c in reversed(seq)) if flag & 0x10 else seq))
    return out


def test_read_sequences_reads_bam(tmp_path):
    recs = _bam_records(np.random.default_rng(1))
    path = str(tmp_path / "a.bam")
    synth.write_bam(path, recs)
    assert list(rr.read_sequences(path)) == _expected(recs)
    assert list(rr.scan_sequences(path)) == _expected(recs)


def test_bam_scan_across_chunks_and_a_large_header(tmp_path):
    recs = _bam_records(np.random.default_rng(2))
    path = str(tmp_path / "a.bam")
    synth.write_bam(path, recs, text="@CO\t" + "h" * 300000 + "\n", refs=[(f"chr{i}", 1000 + i) for i in range(500)])
    want = list(rr.read_sequences(path))
    assert want == _expected(recs)
    for chunk in (1 << 16, 100003, 1 << 20):
        assert list(rr.scan_sequences(path, chunk_bytes=chunk)) == want, chunk


def _scan(buf, at_eof, header, first_index=0, stream_offset=0, max_records=10000):
    buf = np.frombuffer(bytes(buf), dtype=np.uint8)
    rec = np.zeros((max_records, 4), dtype=np.int64)
    seq = np.zeros((max_records, 2), dtype=np.int64)
    out = np.zeros(5, dtype=np.int64)
    _lib.call("cfk_bam_scan", buf.ctypes.data, buf.size, int(at_eof), int(header), first_index, stream_offset,
              rec.ctypes.data, max_records, seq.ctypes.data, out.ctypes.data)
    n = int(out[0])
    return rec[:n], seq[:n], out.tolist()


def _decode(buf, rec, seq):
    return [(bytes(buf[a:a + b]).decode(), rr._bam_bases(bytes(buf[s:s + (L + 1) // 2]), L, rev))
            for (a, b, L, _), (s, rev) in zip(rec.tolist(), seq.tolist())]


def test_bam_scan_every_cut_of_a_small_stream():
    recs = [dict(name="a", seq="ACGTN"), dict(name="sec", seq="AC", flag=0x100), dict(name="b", seq="", flag=4),
            dict(name="c", seq="ACGTTTG", flag=0x10, cigar=[(7, 0)], tags=b"NMi\x01\0\0\0"),
            dict(name="sup", seq="G", flag=0x800), dict(name="d", seq="=ACMGRSVTWYHKDBN")]
    stream = synth.bam_bytes(recs, refs=[("c1", 10), ("c2", 20)])
    want = _expected(recs)
    for cut in range(len(stream) + 1):
        got, rest, off, index, header = [], stream, 0, 0, True
        for part, eof in ((stream[:cut], False), (None, True)):
            buf = part if part is not None else rest
            rec, seq, (n, n_aln, consumed, text, flags) = _scan(buf, eof, header, index, off)
            assert flags == 0
            assert text == sum((L + 15) & ~15 for L in rec[:, 2].tolist())
            got += _decode(buf, rec, seq)
            if header and consumed:
                header = False
            index, off, rest = index + n_aln, off + consumed, (rest if part is None else stream[consumed:])
            if part is None:
                assert consumed == len(buf)
        assert got == want, cut


def test_bam_scan_stops_when_the_tables_are_full():
    stream = synth.bam_bytes([dict(name=f"r{i}", seq="ACGT" * i) for i in range(10)])
    rec, seq, (n, n_aln, consumed, text, flags) = _scan(stream, True, True, max_records=4)
    assert n == 4 and n_aln == 4 and flags == 2
    rest = stream[consumed:]
    rec, seq, out = _scan(rest, True, False, max_records=100)
    assert out[0] == 6 and _decode(rest, rec, seq)[0] == ("r4", "ACGT" * 4)


def _record_with(**kw):
    r = bytearray(synth.bam_record("okname", "ACGTA", cigar=[(5, 0)]))
    for field, value in kw.items():
        at, fmt = {"block_size": (0, "<i"), "l_read_name": (12, "<B"), "n_cigar_op": (16, "<H"), "l_seq": (20, "<i")}[field]
        struct.pack_into(fmt, r, at, value)
    return r


@pytest.mark.parametrize("bad, match", [
    (_record_with(block_size=31), "block_size 31 is below the 32 fixed bytes"),
    (_record_with(block_size=-5), "block_size -5 is below"),
    (_record_with(l_read_name=0), "l_read_name is 0"),
    (_record_with(l_read_name=60), "the read_name field runs past block_size"),
    (_record_with(n_cigar_op=9), "the cigar field runs past block_size"),
    (_record_with(l_seq=12), "the seq field runs past block_size|the qual field runs past block_size"),
    (_record_with(l_seq=-1), "l_seq is negative"),
    (_record_with(l_read_name=6), "read_name is not NUL-terminated"),
])
def test_bam_scan_validation(bad, match):
    good = synth.bam_record("first", "AC")
    stream = synth.bam_bytes([good, bytes(bad)])
    offset = len(synth.bam_bytes([good]))
    with pytest.raises(_lib.CfkError, match=f"record 8 at offset {offset + 1000} of the inflated stream: ({match})"):
        _scan(stream, True, True, first_index=7, stream_offset=1000)


def test_bam_scan_name_bytes_and_truncation():
    for byte in (0x20, 0x7f, 0x80, 0x09):
        r = bytearray(synth.bam_record("abcdef", "A"))
        r[36 + 2] = byte
        with pytest.raises(_lib.CfkError, match=f"record 0 at offset 0 .*read_name byte 0x{byte:02x} is outside"):
            _scan(bytes(r), True, False)
    r = synth.bam_record("x" * 254, "A")  # the longest name l_read_name (a uint8) allows
    assert _decode(r, *_scan(r, True, False)[:2]) == [("x" * 254, "A")]
    stream = synth.bam_bytes([dict(name="a", seq="ACGT")])
    with pytest.raises(_lib.CfkError, match="record 0 .*ends inside the record"):
        _scan(stream[:-3], True, True)
    assert _scan(stream[:-3], False, True)[2][:3] == [0, 0, len(stream) - len(synth.bam_record("a", "ACGT"))]
    with pytest.raises(_lib.CfkError, match="ends inside its header"):
        _scan(stream[:10], True, True)
    with pytest.raises(_lib.CfkError, match="header is malformed"):
        _scan(b"BAM\2" + stream[4:], True, True)


def test_scan_sequences_names_the_bad_record(tmp_path):
    good = synth.bam_record("first", "AC")
    path = str(tmp_path / "bad.bam")
    synth.write_bgzf(path, synth.bam_bytes([good] * 3 + [bytes(_record_with(l_read_name=0))]))
    offset = len(synth.bam_bytes([good] * 3))
    with pytest.raises(_lib.CfkError, match=f"record 3 at offset {offset} of the inflated stream: l_read_name is 0"):
        list(rr.scan_sequences(path, chunk_bytes=1 << 16))


def test_bgzip_text_reads_as_before(tmp_path):
    fq = "".join(f"@q{i} d\n{'ACGT' * i}\n+\n{'I' * 4 * i}\n" for i in range(3000)).encode()
    bg, gz = str(tmp_path / "a.fq.bgz"), str(tmp_path / "a.fq.gz")
    synth.write_bgzf(bg, fq, level=1)
    with gzip.open(gz, "wb") as f:
        f.write(fq)
    want = list(rr.read_sequences(gz))
    assert list(rr.read_sequences(bg)) == want
    assert list(rr.scan_sequences(bg, chunk_bytes=1 << 16)) == want
