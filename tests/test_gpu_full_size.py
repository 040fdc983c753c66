"""BASELINE.json configs[1] at FULL size (1.53e8 read bases, 1.18e10 pair increments): the CUDA path against the C
oracle on every host thread, bit for bit -- rare set, clouds, increment count, all 8.8e6 edges, recruited k-mers --
plus the size-independent properties of the result and the agreement of the alternative kernels with the default
ones.  (The oracle's stage C/D needs ~9 s on 16 threads; the unmodified Python reference would need hours and ~1 TB.)"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def full():
    import bench
    from centroflye_b200.engine import default_engine
    eng = default_engine()
    unit, batch, units = bench.make_inputs(1.0)
    P = bench.PARAMS
    lo, hi = bench.band()
    reads, dunits = eng.upload_reads(batch, P["k"]), eng.upload_units(units, P["k"])
    index, csr, res = eng.recruit(reads, dunits, P["k"], lo, hi, P["max_nonuniq"], P["min_d"], P["max_d"], P["min_coverage"])
    return dict(eng=eng, batch=batch, units=units, P=P, lo=lo, hi=hi, reads=reads, dunits=dunits, index=index, csr=csr,
                res=res)


def _canon(e):
    return e[np.lexsort((e[:, 1], e[:, 0], e[:, 2]))]


def test_full_size_matches_oracle(full):
    from oracle import c_oracle
    P = full["P"]
    want = c_oracle.recruit(full["batch"], full["units"], P["k"], full["lo"], full["hi"], P["max_nonuniq"], P["min_d"],
                            P["max_d"], P["min_coverage"], threads=os.cpu_count() or 1)
    keys = full["index"].sorted_keys.cpu().numpy().view(np.uint64)
    assert np.array_equal(keys, want["rare"])
    U = full["units"].n_units
    assert np.array_equal(full["csr"].unit_ptr.cpu().numpy()[: U + 1], want["unit_ptr"])
    assert np.array_equal(full["csr"].ids.cpu().numpy().view(np.uint32), want["ids"])
    res = full["res"]
    assert res.n_increments == want["n_increments"]
    got = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    assert got.shape[0] > 8_000_000
    assert np.array_equal(_canon(got), _canon(want["edges"]))
    assert np.array_equal(np.sort(res.selected.cpu().numpy().view(np.uint32)), want["selected"])


def test_full_size_properties(full):
    P, res, csr = full["P"], full["res"], full["csr"]
    keys = full["index"].sorted_keys.cpu().numpy().view(np.uint64)
    assert (keys[1:] > keys[:-1]).all()                                   # sorted, distinct: rank = id
    ptr = csr.unit_ptr.cpu().numpy()[: full["units"].n_units + 1]
    ids = csr.ids.cpu().numpy().view(np.uint32)
    assert ptr[0] == 0 and ptr[-1] == ids.size and (np.diff(ptr) >= 0).all()
    inner = np.ones(ids.size, dtype=bool)
    inner[ptr[:-1][np.diff(ptr) > 0]] = False                             # first entry of every non-empty unit
    assert (ids[1:][inner[1:]] > ids[:-1][inner[1:]]).all()               # clouds are sets: sorted, distinct
    assert ids.max() < keys.size
    e = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    a, b, d, cnt = e[:, 0], e[:, 1], e[:, 2], e[:, 3]
    assert (a != b).all() and (d >= max(P["min_d"], 1)).all() and (d <= P["max_d"]).all() and (cnt >= P["min_coverage"]).all()
    trip = _canon(e)[:, :3]
    assert (np.abs(np.diff(trip.astype(np.int64), axis=0)).sum(axis=1) > 0).all()   # every (d, a, b) once
    sel = np.sort(res.selected.cpu().numpy().view(np.uint32))
    assert np.array_equal(sel, np.union1d(a, b))                          # recruited k-mers = endpoints of kept edges
    mult = np.bincount(ids, minlength=keys.size)
    assert (cnt <= np.minimum(mult[a], mult[b])).all()                    # a pair cannot co-occur more often than either id occurs


def test_full_size_alternative_kernels_agree(full):
    """Exact shared-memory tables vs the sketch (stage C), tiled vs resident (stage A): independent implementations,
    same results at full size."""
    eng, P = full["eng"], full["P"]
    old = (eng.pair_mode, eng.docfreq_mode)
    try:
        eng.pair_mode, eng.docfreq_mode = "exact", "tiled"
        index, csr, res = eng.recruit(full["reads"], full["dunits"], P["k"], full["lo"], full["hi"], P["max_nonuniq"],
                                      P["min_d"], P["max_d"], P["min_coverage"])
    finally:
        eng.pair_mode, eng.docfreq_mode = old
    assert np.array_equal(index.sorted_keys.cpu().numpy(), full["index"].sorted_keys.cpu().numpy())
    assert np.array_equal(csr.ids.cpu().numpy(), full["csr"].ids.cpu().numpy())
    assert res.n_increments == full["res"].n_increments and res.n_candidates == full["res"].n_candidates
    got = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    ref = full["res"].edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    assert np.array_equal(_canon(got), _canon(ref))


def test_cen6_noisy_reads_match_oracle():
    """BASELINE.json configs[2] (D6Z1 unit of 3222 bp from the reference simulator, 12 % read errors,
    --kmer-survival-rate 0.09 --coverage 50) on one GPU at 0.3 of the array (300 copies, 5e7 read bases): far more
    one-off k-mers per read than configs[1] and a different band.  The sharded form of the same instance is
    tests/test_gpu_parity.py::test_sharded_recruitment_two_gpus / bench.py --config cen6 --gpus N (parity leg)."""
    import bench
    from centroflye_b200.engine import default_engine
    from oracle import c_oracle
    eng = default_engine()
    unit, batch, units = bench.simulate("cen6", 0.3)
    P = bench.CONFIGS["cen6"]["params"]
    lo, hi = bench.band(P)
    k = P["k"]
    index, csr, res = eng.recruit(eng.upload_reads(batch, k), eng.upload_units(units, k), k, lo, hi, P["max_nonuniq"],
                                  P["min_d"], P["max_d"], P["min_coverage"])
    assert eng.stream_fallbacks == 0
    want = c_oracle.recruit(batch, units, k, lo, hi, P["max_nonuniq"], P["min_d"], P["max_d"], P["min_coverage"],
                            threads=os.cpu_count() or 1)
    assert np.array_equal(index.sorted_keys.cpu().numpy().view(np.uint64), want["rare"])
    assert np.array_equal(csr.unit_ptr.cpu().numpy()[: units.n_units + 1], want["unit_ptr"])
    assert np.array_equal(csr.ids.cpu().numpy().view(np.uint32), want["ids"])
    assert res.n_increments == want["n_increments"]
    got = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    assert np.array_equal(_canon(got), _canon(want["edges"]))
    assert np.array_equal(np.sort(res.selected.cpu().numpy().view(np.uint32)), want["selected"])
