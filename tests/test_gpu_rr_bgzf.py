"""Compressed read files on the device: cfk_bgzf_inflate against zlib, its error statuses, and rr / rr_multi on BAM and
bgzip'd FASTA / FASTQ (read_recruitment._DeviceInflater) against the same reads as plain text."""
import gzip
import os
import struct
import zlib

import numpy as np
import pytest

from centroflye_b200 import _lib, synth
from centroflye_b200 import read_recruitment as rr
from test_gpu_read_recruitment import _rnd
from test_gpu_rr_stream import _fuzz_reads

gpu = pytest.mark.gpu


def _inflate(members, slot=None):
    """cfk_bgzf_inflate on the BGZF members given -> (status per block, inflated bytes of each block).  With slot, block
    i is written to [i * slot, i * slot + ISIZE) of an output prefilled with 0xAB, and every byte between the blocks is
    checked to be untouched."""
    import torch
    comp = b"".join(members)
    buf = np.frombuffer(comp, dtype=np.uint8)
    rows = np.zeros((len(members), 5), dtype=np.int64)
    n, consumed, total, flags = rr._bgzf_blocks(buf, len(members), rows)
    assert n == len(members) and flags == 0
    if slot is not None:
        rows[:, 4] = slot * np.arange(n)
        total = slot * n
    d_comp = torch.from_numpy(buf.copy()).cuda()
    d_rows = torch.from_numpy(rows).cuda()
    d_out = torch.full((total + 16,), 0xAB, dtype=torch.uint8, device="cuda")
    d_status = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    _lib.call("cfk_bgzf_inflate", d_comp.data_ptr(), d_rows.data_ptr(), n, d_out.data_ptr(), d_status.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    out = d_out.cpu().numpy().tobytes()
    assert out[total:] == b"\xab" * 16  # nothing written past the last block
    if slot is not None:
        for o, i in zip(rows[:, 4].tolist(), rows[:, 2].tolist()):
            assert out[o + i:o + slot] == b"\xab" * (slot - i)  # nothing written outside [out_off, out_off + ISIZE)
    return d_status.cpu().tolist(), [out[o:o + i] for o, i in zip(rows[:, 4].tolist(), rows[:, 2].tolist())]


def _payloads():
    rng = np.random.default_rng(5)
    fq = "".join(f"@read_{i} len={n}\n{_rnd(rng, n)}\n+\n{'I5#' * n}\n"[:4 * n + 40]
                 for i, n in enumerate(rng.integers(20, 600, size=400))).encode()
    return {"random": rng.integers(0, 256, size=60000).astype(np.uint8).tobytes(), "fastq": fq[:65536],
            "one byte repeated": b"A" * 65536, "empty": b"", "one": b"x", "fastq 65536": (fq * 2)[:65536]}


@gpu
def test_inflate_equals_zlib():
    strategies = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]
    members, want = [], []
    for data in _payloads().values():
        for level in (0, 1, 6, 9):
            for strategy in strategies:
                try:
                    members.append(synth.bgzf_member(data, level, strategy))
                except ValueError:  # random bytes at level 0 need more than 64 KiB of stored blocks
                    continue
                want.append(data)
        members.append(synth.bgzf_member(data, 6, flush_at=[len(data) // 5, len(data) // 2, len(data) // 2 + 1]))
        want.append(data)
    members.append(synth.BGZF_EOF)
    want.append(b"")
    for m, data in zip(members, want):  # the payloads are what zlib itself inflates
        assert zlib.decompress(m[18:-8], -15) == data
    status, got = _inflate(members)
    assert status == [0] * len(members)
    assert got == want
    assert any(len(w) == 65536 for w in want)


@gpu
def test_inflate_statuses():
    data = _payloads()["fastq"][:20000]
    crc = bytearray(synth.bgzf_member(data, 0))
    crc[18 + 5 + 100] ^= 0x20  # one byte of the stored block's data
    length = bytearray(synth.bgzf_member(data, 6))
    length[-4:] = struct.pack("<I", len(data) - 1)
    dyn = bytearray(synth.bgzf_member(data, 6))
    assert dyn[18] & 7 == 5  # BFINAL, BTYPE = dynamic
    dyn[18] |= 0xf8  # HLIT = 288: more literal/length codes than exist
    good = synth.bgzf_member(data, 6)
    status, got = _inflate([good, bytes(crc), bytes(length), bytes(dyn), good])
    assert status == [0, 3, 2, 1, 0]
    assert got[0] == got[4] == data


@gpu
def test_inflate_rejects_corrupt_streams_inside_their_blocks():
    """Every byte of a dynamic-Huffman payload replaced in turn: each block ends in a status, and writes nothing
    outside its own [out_off, out_off + ISIZE) (each block has a slot of its own, the bytes between them are checked)."""
    data = _payloads()["fastq"][:3000]
    good = synth.bgzf_member(data, 9)
    rng = np.random.default_rng(11)
    members = [good]
    for i in range(18, len(good) - 8):
        m = bytearray(good)
        m[i] = int(rng.integers(0, 256)) if m[i] else 0xff
        members.append(bytes(m))
    members.append(good)
    status, got = _inflate(members, slot=len(data) + 4096)
    assert status[0] == status[-1] == 0 and got[0] == got[-1] == data
    for m, st, out in zip(members[1:-1], status[1:-1], got[1:-1]):
        assert st in (0, 1, 2, 3)
        if st == 0:
            assert out == zlib.decompress(m[18:-8], -15)


# ---- rr and rr_multi on compressed files ------------------------------------------------------------------------------

def _reads(seed, unit, copies=2):
    rng = np.random.default_rng(seed)
    reads = []
    for c in range(copies):
        reads += [(f"c{c}_{n.split()[0]}", s) for n, s in _fuzz_reads(rng, unit)]
    return reads


def _write_fasta(path, records):
    with open(path, "w") as f:
        f.write("".join(f">{n}\n{s}\n" for n, s in records))


def _bam_of(path, reads, rng):
    """A BAM of `reads` whose read_sequences() yields them in order, among secondary / supplementary records, with half
    the reads stored reverse-complemented (flag 0x10) and odd characters, CIGAR, qualities and tags around them."""
    comp = dict(zip(synth.BAM_CODES, "=TGKCYSBAWRDMHVN"))
    recs = []
    for i, (name, seq) in enumerate(reads):
        flag = int(rng.choice([0, 4, 0x10, 0x14]))
        stored = "".join(comp[c] for c in reversed(seq)) if flag & 0x10 else seq
        recs.append(dict(name=name, seq=stored, flag=flag, cigar=[(len(seq), 0)] if seq else [],
                         qual=bytes([30]) * len(seq), tags=b"RGZgroup1\0" + b"MMZ" + b"C+m" * (i % 50) + b"\0"))
        if i % 7 == 0:
            recs.append(dict(name=name, seq=stored[:50], flag=0x100 if i % 2 else 0x800))
    synth.write_bam(path, recs, level=int(rng.choice([1, 6])), text="@HD\tVN:1.6\n@CO\t" + "x" * 100000 + "\n")


def _run(jobs, read_fn, chunk, devices=None, stats=None):
    rr.recruit_file_units(jobs, read_fn, chunk_bytes=chunk, devices=devices, long_units=True, stats=stats)
    return [open(out, "rb").read() for _, out, _ in jobs]


@gpu
def test_rr_on_bam_equals_rr_on_its_fasta(tmp_path):
    rng = np.random.default_rng(21)
    unit = _rnd(rng, 171 * 4)
    long_unit = _rnd(rng, 3400)
    reads = _reads(22, unit) + [(f"long_{i}", s) for i, (_, s) in enumerate(_reads(23, long_unit, copies=1))]
    bam, fasta = str(tmp_path / "reads.bam"), str(tmp_path / "reads.fasta")
    _bam_of(bam, reads, rng)
    _write_fasta(fasta, rr.read_sequences(bam))
    assert list(rr.read_sequences(fasta)) == reads
    jobs = [(unit, str(tmp_path / f"o{t}.fa"), t) for t in (0, 350, -1)] + [(long_unit, str(tmp_path / "long.fa"), 350)]
    ref_jobs = [(u, o + ".ref", t) for u, o, t in jobs]
    want = _run(ref_jobs, fasta, 1 << 20)
    assert want[0] and want[1] and want[3]  # something kept at every threshold
    for chunk in (1 << 20, 200003, 1 << 16):
        for devices in (None, [0, 0, 0]):
            stats = {}
            assert _run(jobs, bam, chunk, devices, stats) == want, (chunk, devices)
            assert stats["bgzf_blocks"] > 0 and stats["inflate_s"] > 0 and stats["fallback"] is None
    for t, (_, out, _) in zip((0, 350), jobs):  # rr.py's command line
        assert rr.main([_unit_file(tmp_path, unit), bam, out + ".cli", str(t)]) == 0
        assert open(out + ".cli", "rb").read() == open(out, "rb").read()


def _unit_file(tmp_path, unit):
    path = str(tmp_path / "unit.fa")
    _write_fasta(path, [("unit", unit)])
    return path


@gpu
def test_bgzip_text_equals_plain_and_gzip(tmp_path):
    rng = np.random.default_rng(31)
    unit = _rnd(rng, 171 * 3)
    reads = _reads(32, unit)
    fq = "".join(f"@{n}\n{s}\n+\n{'#' * len(s)}\n" for n, s in reads).encode()
    fa = "".join(f">{n} x\n" + "\n".join(s[i:i + 80] for i in range(0, len(s), 80)) + "\n" for n, s in reads).encode()
    jobs = [(unit, str(tmp_path / f"o{t}.fa"), t) for t in (0, 350, -1)]
    for name, text in (("fq", fq), ("fa", fa)):
        plain, gz, bgz = (str(tmp_path / f"r.{name}{ext}") for ext in ("", ".gz", ".bgz"))
        open(plain, "wb").write(text)
        with gzip.open(gz, "wb") as f:
            f.write(text)
        synth.write_bgzf(bgz, text, block=40000)
        want = _run(jobs, plain, 1 << 20)
        assert _run(jobs, gz, 1 << 20) == want
        for chunk in (1 << 20, 1 << 16):
            for devices in (None, [0, 0, 0]):
                stats = {}
                assert _run(jobs, bgz, chunk, devices, stats) == want, (name, chunk, devices)
                assert stats["bgzf_blocks"] >= len(text) // 40000


@gpu
def test_device_reader_edges_follow_gzip_open(tmp_path):
    """Zero padding (some of it longer than the reader's compressed buffer), a plain gzip member after BGZF ones,
    trailing garbage and a cut-off last member: the device reader gives the bytes, or raises the error, that gzip.open
    does."""
    text = b"".join(b">r%d\n%s\n" % (i, b"ACGT" * (i % 300)) for i in range(4000))
    body = synth.bgzf_compress(text[:300000], eof=False)
    files = {
        "padding": body + synth.bgzf_compress(text[300000:]) + b"\0" * 5000,
        "long padding": body + b"\0" * 300000 + synth.bgzf_compress(text[300000:]) + b"\0" * 200000,
        "only padding after the end": synth.bgzf_compress(text) + b"\0" * (3 << 16),
        "plain member": body + gzip.compress(text[300000:]),
        "garbage": synth.bgzf_compress(text) + b"garbage",
        "cut": synth.bgzf_compress(text, eof=False)[:-100],
    }
    stats = {}
    for (name, data), chunk in ((item, chunk) for item in files.items() for chunk in (1 << 20, 1 << 16)):
        path = str(tmp_path / name.replace(" ", "_"))
        open(path, "wb").write(data)
        try:
            want = gzip.open(path, "rb").read()
            err = None
        except (EOFError, gzip.BadGzipFile) as e:
            want, err = None, type(e)
        f = rr._open_binary(path, (lambda: __import__("torch").device("cuda", 0), chunk, stats))
        assert isinstance(f, rr._DeviceInflater), name
        got = bytearray()
        buf = bytearray(100000)
        try:
            while True:
                k = f.readinto(memoryview(buf))
                if not k:
                    break
                got += buf[:k]
        except (EOFError, gzip.BadGzipFile) as e:
            assert err is type(e), (name, chunk)
        else:
            assert err is None and bytes(got) == want, (name, chunk)
        finally:
            f.close()


@gpu
@pytest.mark.parametrize("kind, message", [("crc", "CRC32 mismatch"), ("length", "inflated length differs from ISIZE"),
                                           ("stream", "not a valid DEFLATE stream")])
def test_block_error_names_its_offset_and_leaves_no_output(tmp_path, kind, message):
    rng = np.random.default_rng(41)
    unit = _rnd(rng, 300)
    text = "".join(f">r{i}\n{_rnd(rng, 500)}\n" for i in range(3000)).encode()
    pieces = [text[i:i + 65280] for i in range(0, len(text), 65280)]
    members = [synth.bgzf_member(p, 6) for p in pieces]
    if kind == "crc":  # one flipped byte in a stored block
        bad = bytearray(synth.bgzf_member(pieces[3], 0))
        bad[100] ^= 1
    elif kind == "length":
        bad = bytearray(members[3])
        bad[-4:] = struct.pack("<I", len(pieces[3]) - 1)
    else:  # a dynamic header with HLIT = 288
        bad = bytearray(members[3])
        assert bad[18] & 7 == 5
        bad[18] |= 0xf8
    offset = sum(len(m) for m in members[:3])
    path = str(tmp_path / "bad.fa.gz")
    open(path, "wb").write(b"".join(members[:3]) + bytes(bad) + b"".join(members[4:]) + synth.BGZF_EOF)
    out = tmp_path / "out"
    out.mkdir()
    for devices in (None, [0, 0]):
        with pytest.raises(gzip.BadGzipFile, match=f"BGZF block at file offset {offset}: {message}"):
            rr.recruit_file_units([(unit, str(out / "a.fa"), 3), (unit, str(out / "b.fa"), -1)], path,
                                  chunk_bytes=1 << 18, devices=devices)
        assert os.listdir(out) == []
