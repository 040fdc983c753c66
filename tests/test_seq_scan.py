"""The native FASTA / FASTQ record scanner of the streaming rr filter (csrc/seq_scan.cpp, cfk_seq_scan) and the chunking
around it (read_recruitment._scan_chunks) against read_sequences(), the restatement of rr.cpp's kseq loop that the
goldens pin: the same records, names and sequences for every chunk size, on the golden inputs and on a seeded corpus of
the corner cases of universal newlines, str whitespace and FASTQ quality blocks."""
import gzip
import os

import numpy as np
import pytest

from test_gpu_read_recruitment import FORMATS, write_inputs

WS = " \t\x0b\x0c\x1c\x1d\x1e\x1f"  # str.isspace on ASCII, without the line breaks


def _scan(path, chunk_bytes):
    from centroflye_b200 import read_recruitment as rr
    return list(rr.scan_sequences(path, chunk_bytes=chunk_bytes))


def _want(path):
    from centroflye_b200 import read_recruitment as rr
    return list(rr.read_sequences(path))


def _write(tmp_path, name, data, gz=False):
    path = str(tmp_path / name)
    if gz:
        with gzip.open(path, "wb") as f:
            f.write(data)
    else:
        with open(path, "wb") as f:
            f.write(data)
    return path


def _fuzz_text(rng, n_records):
    """A FASTA / FASTQ mix with every corner the scanner must reproduce."""
    nl = lambda: ["\n", "\r\n", "\r"][int(rng.integers(3))]  # noqa: E731
    ws = lambda: "".join(rng.choice(list(WS), size=int(rng.integers(0, 3))))  # noqa: E731
    seq = lambda n: "".join(rng.choice(list("ACGTN"), size=n))  # noqa: E731
    out = []
    if rng.random() < 0.5:
        out.append("junk line" + nl() + nl() + "  more junk" + nl())
    for _ in range(n_records):
        kind = rng.random()
        head = rng.choice([">", "@"])
        name = rng.choice(["", " ", "r" + str(int(rng.integers(1000))), " lead\tname rest", "x\x1cy", "a\x0bb c"])
        out.append(head + name + ws() + nl())
        if kind < 0.45:  # FASTQ
            s = seq(int(rng.integers(0, 40)))
            cut = int(rng.integers(0, len(s) + 1))
            lines = [s] if rng.random() < 0.6 else [s[:cut], s[cut:]]
            for line in lines:
                out.append(ws() + line + ws() + nl())
            out.append("+" + ("comment" if rng.random() < 0.3 else "") + nl())
            q = "".join(rng.choice(list("@+>I#!"), size=max(0, len(s) + int(rng.integers(-3, 4)))))
            if rng.random() < 0.4 and len(q) > 1:  # multi-line quality
                c = int(rng.integers(1, len(q)))
                out.append(q[:c] + nl() + q[c:] + nl())
            else:
                out.append(q + nl())
        else:  # FASTA, with blank lines and whitespace inside and around lines
            for _ in range(int(rng.integers(0, 4))):
                s = seq(int(rng.integers(0, 20)))
                if rng.random() < 0.2:
                    s = s[:len(s) // 2] + " \t" + s[len(s) // 2:]
                out.append(ws() + s + ws() + nl())
                if rng.random() < 0.15:
                    out.append(nl())
    text = "".join(out)
    if rng.random() < 0.3:
        text = text.rstrip("\r\n")  # no final line break (possibly inside a quality block)
    return text


@pytest.mark.parametrize("fmt", FORMATS)
def test_golden_inputs(tmp_path, fmt):
    _, read_fn, _, _ = write_inputs(str(tmp_path), fmt)
    want = _want(read_fn)
    size = os.path.getsize(read_fn)
    for chunk in (1, 100, 4096, 30000, 1 << 16, 1 << 26):
        assert _scan(read_fn, chunk) == want, chunk
    assert size > 0


@pytest.mark.parametrize("seed", range(12))
def test_fuzz_corpus(tmp_path, seed):
    rng = np.random.default_rng(seed)
    text = _fuzz_text(rng, int(rng.integers(1, 40)))
    path = _write(tmp_path, "reads.txt", text.encode(), gz=seed % 3 == 0)
    want = _want(path)
    for chunk in sorted({1, 2, 3, 7, 16, 61, 256, len(text) // 2 + 1, len(text) + 1}):
        assert _scan(path, chunk) == want, (seed, chunk)


def test_every_split_of_an_adversarial_file(tmp_path):
    """Every chunk size from 1 byte to the whole file on a short file that packs the corners into few bytes; the
    first chunk boundary therefore falls on every byte."""
    text = ("junk\r\r\n>\t\r@ a b\r\nAC G \x0c\r\n\r\nT\n+\n@+\r>\n@q\nAC\n+x\n+@\n>e\r+\n@f\nA\r\n+\r\n"
            "\x1f\r\n>tail  x\rAAA\r\nCC\r")
    path = _write(tmp_path, "adv.txt", text.encode())
    want = _want(path)
    assert [n for n, _ in want] == ["", "a", "e", "f", "tail"]  # "@q" and "AC" are quality lines of "a"
    for chunk in range(1, len(text) + 2):
        assert _scan(path, chunk) == want, chunk


def test_records_longer_than_the_chunk(tmp_path):
    """A read many times the chunk size, single-line and in 7-column lines: the chunk grows until the record fits."""
    rng = np.random.default_rng(5)
    s = "".join(rng.choice(list("ACGT"), size=300000))
    fq = f"@short\nAC\n+\nII\n@long x\n{s}\n+\n{'I' * len(s)}\n@end\nG\n+\nI\n"
    fa = ">long\n" + "\n".join(s[i:i + 7] for i in range(0, len(s), 7)) + "\n>end\nT\n"
    for name, text in (("fq", fq), ("fa", fa)):
        path = _write(tmp_path, name, text.encode())
        want = _want(path)
        assert len(want[1 if name == "fq" else 0][1]) == len(s)
        for chunk in (1, 1000, 1 << 16):
            assert _scan(path, chunk) == want, (name, chunk)


def test_non_ascii_is_reported(tmp_path):
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    path = _write(tmp_path, "utf8.fa", ">réad\nACGT\n".encode())
    with pytest.raises(rr._Fallback):
        _scan(path, 1 << 20)
    lib = _lib.load()
    buf = np.frombuffer(b">a\nAC\n>b\xff\nGT\n", dtype=np.uint8)
    rec, piece, out = np.zeros(64, np.int64), np.zeros(64, np.int64), np.zeros(5, np.int64)
    _lib.call("cfk_seq_scan", buf.ctypes.data, buf.size, 1, rec.ctypes.data, 16, piece.ctypes.data, 16, out.ctypes.data)
    assert out[4] == rr._SCAN_NOT_ASCII and out[0] == 0


def test_scanner_tables(tmp_path):
    """The raw tables: 16-byte aligned sequence offsets, pieces placed at them, `consumed` at the first incomplete
    record, a trailing '\\r' incomplete before the end of the input, and a stop when the tables are full."""
    from centroflye_b200 import _lib
    from centroflye_b200 import read_recruitment as rr
    data = b">a x\nACG\nT\n@b\nGG\n+\nII\n>c\rAAAA\r"
    buf = np.frombuffer(data, dtype=np.uint8)
    rec, piece, out = np.zeros(64, np.int64), np.zeros(64, np.int64), np.zeros(5, np.int64)

    def scan(n, eof, max_rec=16, max_piece=16):
        _lib.call("cfk_seq_scan", buf.ctypes.data, n, int(eof), rec.ctypes.data, max_rec, piece.ctypes.data, max_piece,
                  out.ctypes.data)
        return out.tolist()

    assert scan(len(data), True) == [3, 4, len(data), 48, 0]
    assert rec[:12].reshape(3, 4).tolist() == [[1, 1, 4, 0], [12, 1, 2, 16], [23, 1, 4, 32]]
    assert piece[:12].reshape(4, 3).tolist() == [[5, 3, 0], [9, 1, 3], [14, 2, 16], [25, 4, 32]]
    assert scan(len(data), False) == [2, 3, 22, 32, 0]        # "AAAA\r" may be the first half of "\r\n"
    assert scan(len(data) - 1, False) == [2, 3, 22, 32, 0]    # ">c" may go on
    assert scan(13, False) == [1, 2, 11, 16, 0]               # the record ends where "@b" begins
    assert scan(len(data), True, max_rec=1) == [1, 2, 11, 16, rr._SCAN_FULL]
    assert scan(len(data), True, max_piece=0) == [0, 0, 0, 0, rr._SCAN_FULL]
    with pytest.raises(_lib.CfkError, match="cfk_seq_scan"):
        scan(-1, True)
