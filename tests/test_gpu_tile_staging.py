"""D = 32 tile staging of the tensor-core label kernel (gauss_label_tc2_kernel) and the fused sub-label +
statistics kernel (niw_substats_tc_kernel): their gather threads load the rows of a tile into registers,
centre them there and store them once.  Rows past the end of a cluster are exact zeros and are not centred.
These cases put that boundary everywhere it can be: clusters that end mid-tile with the next cluster in the
same CTA's range, n not a multiple of 128, clusters of 1 and 129 points, K = 1 and K = 200, and means far
from the origin, where centring by the wrong mean or centring a padding row would show.  Each runs a full
sweep against the oracle from warm labels, so that both kernels decide the draws."""
import os

import numpy as np
import pytest

import dpmm_pkg
from oracle import dpmm_oracle as O
from tests.util import compare_sweeps, make_niw_case, set_params

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


def sized_case(sizes, seed, spread, offset):
    """make_niw_case at D = 32 with exactly sizes[k] points drawn from cluster k's own distribution (mu[k, 0],
    inv_sigma[k, 0]), in shuffled order, everything shifted by a vector of norm `offset`."""
    K, n = len(sizes), int(sum(sizes))
    case = make_niw_case(32, K, n, seed=seed, spread=spread)
    rng = np.random.default_rng(seed + 1)
    cols = []
    for k, m in enumerate(sizes):
        Lc = np.linalg.cholesky(np.linalg.inv(case["inv_sigma"][k, 0].astype(np.float64)))
        cols.append(case["mu"][k, 0].astype(np.float64)[:, None] + Lc @ rng.standard_normal((32, m)))
    x = np.concatenate(cols, axis=1)[:, rng.permutation(n)]
    shift = rng.standard_normal(32)
    shift *= offset / np.linalg.norm(shift)
    case["x"] = (x + shift[:, None]).astype(np.float32)
    case["mu"] = (case["mu"] + shift.astype(np.float32)).astype(np.float32)
    w = np.asarray(sizes, np.float64) / n
    case["weights"] = w.astype(np.float32)
    return case


def random_case(K, n, seed, spread, offset):
    sizes = np.bincount(np.random.default_rng(seed).integers(0, K, n), minlength=K)
    return sized_case(list(sizes), seed, spread, offset)


CASES = {   # name: case builder
    # ~470 tiles over 148 CTAs: clusters end mid-tile and the next cluster starts in the same CTA's range
    "ragged_ranges": lambda: random_case(5, 60001, 11, 10.0, 0.0),
    "ragged_ranges_far": lambda: random_case(5, 60001, 12, 10.0, 80.0),
    "n_not_multiple_of_tile": lambda: random_case(7, 20000 + 77, 13, 10.0, 0.0),
    "clusters_of_1_and_129": lambda: sized_case([1, 129, 1000, 129, 1, 2000], 14, 10.0, 0.0),
    "clusters_of_1_and_129_far": lambda: sized_case([129, 1, 2000, 1, 129, 777], 15, 10.0, 80.0),
    "k1": lambda: sized_case([5003], 16, 10.0, 0.0),
    "k1_far": lambda: sized_case([20000 + 5], 17, 10.0, 80.0),
    "k200": lambda: random_case(200, 60000, 18, 10.0, 0.0),
    "k200_far": lambda: random_case(200, 60000, 19, 10.0, 80.0),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_tile_staging_against_the_oracle(pkg, name):
    case = CASES[name]()
    n, K = case["n"], case["K"]
    for final in (False, True):
        g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
        o = O.OracleSweep(case["x"], O.NIW, seed=7)
        rep = compare_sweeps(g, o, case, np.random.default_rng(K + n), final=final, warm=True)
        fused, served, redone = g.fused_stats()
        g.close()
        assert fused >= 1, "the fused sub-label + statistics kernel did not run"
    # both kernels really ran, on the cluster sizes the case was built with
    os.environ["DPMM_TC_STATS"] = "1"
    try:
        g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
        set_params(g, case)
        g.sample_labels(True)
        counts = np.bincount(g.get_labels(), minlength=K + 1)[1:]
        g.sample_labels(False)
        npts, ncand, novf = g.tc_stats(overflow=True)
        g.close()
    finally:
        os.environ.pop("DPMM_TC_STATS")
    assert npts == n, "the tensor-core label path did not run"
    if "clusters_of_1" in name or name.startswith("k1"):
        np.testing.assert_array_equal(counts, np.round(case["weights"].astype(np.float64) * n).astype(np.int64))
    print(f"{name}: K={K} n={n}: {rep}; fused {fused}, served {served}, recomputed {redone}; overflow points {novf}")
