"""BASELINE.json configs[3]: the k-size / coverage-threshold sweep ON THE cenX-SCALE SET (configs[1]'s reads, 1.53e8
bases), bit-exactness at every point against the C oracle on every host thread.

The flags are those of the reference's command line (dbkr.py:25-33): -k, --min-coverage, --bottom / --top,
--max-nonuniq.  One oracle run per (k, band, max_nonuniq) at the SMALLEST threshold of that context serves all its
thresholds: the oracle counts every (distance, a, b) exactly and the kept-edge rule `cnt >= min_coverage and
cnt / sum >= 0.8` (dbkr.py:133-147) is per edge, so the edges at a higher threshold are the rows of the result with
cnt >= threshold.  On the device the thresholds take different kernels: 2 the exact shared-memory tables
(pair_candidates_kernel), 4 and 8 the sketch (pair_sketch_kernel).

The sweep is one factor at a time around the defaults (every k at the default band; every band / max-nonuniq
combination at k = 19): 9 contexts, thresholds {2, 4, 8} at the default one and {4, 8} elsewhere = 19 points (the
72-point product would only repeat rare sets; --min-coverage 2 yields ~5e7 edges per context and is kept to one).
Edge sets of 10^7 rows are compared through two order-independent 64-bit checksums of their rows.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DEFAULT = dict(bottom=0.9, top=3.0, max_nonuniq=3)
CONTEXTS = [dict(DEFAULT, k=k) for k in (11, 15, 19, 23, 27, 31)] + \
           [dict(k=19, bottom=0.5, top=2.0, max_nonuniq=3), dict(k=19, bottom=0.9, top=3.0, max_nonuniq=0),
            dict(k=19, bottom=0.5, top=2.0, max_nonuniq=0)]


def _ctx_id(c):
    return f"k{c['k']}-b{c['bottom']}-t{c['top']}-nu{c['max_nonuniq']}"


@pytest.fixture(scope="module")
def data():
    import bench
    from centroflye_b200.engine import default_engine
    eng = default_engine()
    unit, batch, units = bench.make_inputs(1.0)
    return dict(eng=eng, batch=batch, units=units, uploads={})


@pytest.fixture(scope="module", params=CONTEXTS, ids=_ctx_id)
def ctx(request, data):
    import bench
    from centroflye_b200.engine import band_to_int
    from oracle import c_oracle
    c, P = request.param, bench.PARAMS
    lo, hi = band_to_int(c["bottom"] * P["coverage"] * P["kmer_survival_rate"], c["top"] * P["coverage"] * P["kmer_survival_rate"])
    base = 2 if c == CONTEXTS[2] else 4
    want = c_oracle.recruit(data["batch"], data["units"], c["k"], lo, hi, c["max_nonuniq"], P["min_d"], P["max_d"], base,
                            threads=os.cpu_count() or 1)
    return dict(c=c, lo=lo, hi=hi, want=want, base=base)


def _mix(x):
    x = x.copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint64(33)
        x *= np.uint64(0xff51afd7ed558ccd)
        x ^= x >> np.uint64(33)
        x *= np.uint64(0xc4ceb9fe1a85ec53)
        x ^= x >> np.uint64(33)
    return x


def _row_checksums(e):
    """Order-independent: (rows, sum and xor of one row hash, sum of a second one)."""
    e = e.astype(np.uint64)
    ab, dc = e[:, 0] | (e[:, 1] << np.uint64(32)), e[:, 2] | (e[:, 3] << np.uint64(32))
    with np.errstate(over="ignore"):
        h1 = _mix(ab ^ _mix(dc))
        h2 = _mix(dc + np.uint64(0x9E3779B97F4A7C15) * ab)
        return e.shape[0], int(h1.sum(dtype=np.uint64)), int(np.bitwise_xor.reduce(h1)) if h1.size else 0, int(h2.sum(dtype=np.uint64))


@pytest.mark.parametrize("min_cov", [2, 4, 8])
def test_sweep_point_matches_oracle(data, ctx, min_cov):
    import bench
    if min_cov < ctx["base"]:
        pytest.skip("--min-coverage 2 is swept at the default context only")
    eng, P, c, want = data["eng"], bench.PARAMS, ctx["c"], ctx["want"]
    k = c["k"]
    if k not in data["uploads"]:
        data["uploads"] = {k: (eng.upload_reads(data["batch"], k), eng.upload_units(data["units"], k))}
    reads, dunits = data["uploads"][k]
    index, csr, res = eng.recruit(reads, dunits, k, ctx["lo"], ctx["hi"], c["max_nonuniq"], P["min_d"], P["max_d"], min_cov)
    assert eng.stream_fallbacks == 0
    assert eng.last_pair_kernel == ("pair_candidates_kernel" if min_cov == 2 else "pair_sketch_kernel")
    keys = index.sorted_keys.cpu().numpy().view(np.uint64)
    assert np.array_equal(keys, want["rare"])
    U = data["units"].n_units
    assert np.array_equal(csr.unit_ptr.cpu().numpy()[: U + 1], want["unit_ptr"])
    assert np.array_equal(csr.ids.cpu().numpy().view(np.uint32), want["ids"])
    assert res.n_increments == want["n_increments"]
    keep = want["edges"][want["edges"][:, 3] >= min_cov]
    got = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
    assert got.shape == keep.shape
    assert _row_checksums(got) == _row_checksums(keep)
    want_sel = np.zeros(keys.size, dtype=bool)
    want_sel[keep[:, 0]] = True
    want_sel[keep[:, 1]] = True
    assert np.array_equal(np.sort(res.selected.cpu().numpy().view(np.uint32)), np.flatnonzero(want_sel).astype(np.uint32))
