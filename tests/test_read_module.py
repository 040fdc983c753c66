"""scripts/read.py (SURVEY.md §8 a10) and the never-called get_all_kmers of scripts/read_kmer_cloud.py:57-63: the
drop-in modules against known answers worked out from the reference's source, and against what the reference classes
and module answered (tests/golden/reference_modules.json)."""
import json
import os

import pytest

from conftest import GOLDEN

SIMLORD_ID = "Read_17_length=8742bp_startpos=104652_chromosome=chrX_strand=+_numberOfErrors=1205_totalErrorProb=0.1378_passes=3.0_passesLeft=3_passesRight=2_cutPosition=4027_mult=1.5"


def _ours():
    from centroflye_b200.read import Read
    return Read


def _reference():
    with open(os.path.join(GOLDEN, "reference_modules.json")) as f:
        return json.load(f)


def test_read_plain():
    Read = _ours()
    r = Read("r1", "ACGTACGT")
    assert (r.id, r.seq, len(r), r[2], r[1:4]) == ("r1", "ACGTACGT", 8, "G", "CGT")
    assert not hasattr(r, "numb")
    with pytest.raises(TypeError):
        len(Read("no_seq"))  # seq=None, like the reference


def test_read_simlord_fields():
    r = _ours()(SIMLORD_ID, "ACGT", simulated=True)
    f = SIMLORD_ID.split("_")
    assert r.numb == 17 and r.length == 8742 and r.start_pos == 104652
    assert r.n_errors == int(f[6].split("=")[1]) == 1205
    assert r.error_rate == float(f[9].split("=")[1]) == 3.0  # field 9, whatever SimLoRD put there (read.py:15)
    assert r.mult == 1.5
    with pytest.raises((IndexError, ValueError)):
        _ours()("short_id", "ACGT", simulated=True)


def test_read_from_biopy():
    class Rec:
        id, seq = "x", bytearray(b"ACG")
    r = _ours().FromBiopyRead(Rec)
    assert r.id == "x" and r.seq == str(Rec.seq)


def test_read_equals_reference_class():
    cases = _reference()["read"]
    assert [tuple(c["args"]) for c in cases] == [("r1", "ACGTACGT", False), (SIMLORD_ID, "ACGT", True), ("r2", None, False)]
    for c in cases:
        a = _ours()(*c["args"])
        assert vars(a) == c["vars"]
        if c["args"][1] is not None:
            assert len(a) == c["len"] and a[1:3] == c["seq_1_3"]


def test_get_all_kmers_behaves_like_the_reference():
    from scripts_shim_check import load_names
    ours = load_names()
    ref = _reference()["read_kmer_cloud"]
    assert "get_all_kmers" in ours
    assert ours["get_all_kmers"]({}) == ref["get_all_kmers"]["{}"] == []
    assert ref["get_all_kmers"]["{'r': object()}"] == "AttributeError"
    with pytest.raises(AttributeError):
        ours["get_all_kmers"]({"r": object()})
    missing = {n for n in ref["public"] if n not in ours["__public__"]}
    assert not missing, f"names the reference module binds and the drop-in does not: {missing}"
