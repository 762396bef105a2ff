"""-m gpu: K1x, the FP64 Gibbs sampler that decides leaf-level labels from certified FP32 prefix sums
(csrc/gibbs_exact_kernel.cuh).  Its outputs must be those of the all-FP64 kernel K1 (KDEB200_GIBBS_EXACT=0) bit for
bit: torch.equal-strict comparison of points and labels, on Philox and on injected streams."""
import os

import numpy as np
import pytest

import kde_b200 as K
from oracle import oracle as O
from tests.util import mixture, silverman

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def thread_per_chain_kernel():
    """K1x replaces the thread-per-chain kernel; small calls would otherwise go to the warp-per-chain kernel."""
    saved = {k: os.environ.get(k) for k in ("KDEB200_GIBBS_WARP_MAX", "KDEB200_GIBBS_EXACT", "KDEB200_GIBBS_EXACT_INFLATE")}
    os.environ["KDEB200_GIBBS_WARP_MAX"] = "0"
    os.environ.pop("KDEB200_GIBBS_EXACT", None)
    os.environ.pop("KDEB200_GIBBS_EXACT_INFLATE", None)
    K.set_gibbs_precision(K.F64)
    K.gibbs_exact_redone()
    yield
    for k, v in saved.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


def run(route, trees, **kw):
    os.environ["KDEB200_GIBBS_EXACT"] = route
    try:
        return K.prodAppxMSGibbsS(None, trees, None, None, **kw)
    finally:
        os.environ.pop("KDEB200_GIBBS_EXACT", None)


def assert_same(trees, **kw):
    ref = run("0", trees, **kw)
    K.gibbs_exact_redone()
    new = run("1", trees, **kw)
    redone = K.gibbs_exact_redone()
    for a, b in zip(ref, new):
        assert a.dtype == b.dtype and a.shape == b.shape
        assert np.array_equal(a, b), "K1x differs from K1 in %d entries" % int(np.sum(a != b))
    return redone


def make_trees(seed, d, M, N, shift=0.25, weights=False):
    rng = np.random.default_rng(seed)
    trees = []
    for j in range(M):
        p = mixture(rng, d, N, shift * j)
        w = rng.uniform(0.2, 1.0, N) if weights else None
        trees.append(K.kde(p, silverman(p) if N > 2 else np.full(d, 0.7), weights=w))
    return trees


def test_c4_shape_identical_and_mostly_decided():
    trees = make_trees(11, 3, 8, 4096)
    Np, T = 1_000_000, 5
    lanes, warps = assert_same(trees, Niter=T, Np=Np, seed=123)
    leaf_draws = Np * 2 * (T + 1) * 8  # two leaf levels at N = 4096
    assert lanes < 0.01 * leaf_draws, (lanes, warps)


@pytest.mark.parametrize("d,M,N,Np,T", [
    (1, 2, 300, 3000, 5), (2, 2, 100, 2000, 5), (3, 6, 100, 1500, 5), (4, 3, 500, 1000, 3),
    (5, 3, 200, 600, 2), (6, 2, 300, 500, 2), (7, 2, 128, 400, 1), (8, 2, 150, 400, 2),
    (3, 3, 1, 300, 3), (3, 16, 20, 200, 1), (3, 2, 5001, 300, 1), (3, 3, 2, 300, 5), (3, 2, 3, 500, 2),
    (3, 2, 100_000, 200, 1),   # multi-tile leaf levels, chunks spanning several tiles
])
def test_identical_to_fp64_per_shape(d, M, N, Np, T):
    """d != 3 routes to K1 on both sides (K1x is enabled where it is measured to win) and checks the routing"""
    assert_same(make_trees(100 * d + M + N, d, M, N), Niter=T, Np=Np, seed=7 + d)


def test_weights_and_no_entropy():
    trees = make_trees(5, 3, 3, 700, weights=True)
    assert_same(trees, Niter=3, Np=2000, seed=3, addEntropy=False)


def test_lcv_bandwidths():
    rng = np.random.default_rng(6)
    trees = [K.kde(mixture(rng, 3, 400, 0.3 * j)) for j in range(3)]  # LOOCV-chosen bandwidths
    assert_same(trees, Niter=3, Np=2000, seed=4)


def test_shifted_data_and_far_apart_densities():
    rng = np.random.default_rng(8)
    a = mixture(rng, 3, 500, 0.0) + 1e3
    b = mixture(rng, 3, 500, 0.0) + 1e3 + 40.0  # the product's mass sits in the far tails of both
    trees = [K.kde(a, silverman(a)), K.kde(b, silverman(b))]
    assert_same(trees, Niter=2, Np=2000, seed=9)


def test_shard_slices():
    trees = make_trees(21, 3, 3, 1000)
    full = run("0", trees, Niter=3, Np=3000, seed=5)
    for s0, s1 in [(0, 1000), (1000, 2345), (2345, 3000)]:
        part = run("1", trees, Niter=3, Np=3000, seed=5, s0=s0, s1=s1)
        for a, b in zip(full, part):
            assert np.array_equal(a[:, s0:s1], b)


def test_injected_streams_match_oracle():
    rng = np.random.default_rng(31)
    d, M, N, Np, T = 3, 3, 150, 600, 3
    pts = [mixture(rng, d, N, 0.3 * j) for j in range(M)]
    trees = [K.kde(p, silverman(p)) for p in pts]
    otrees = [O.OKDE.kde_bw(p, silverman(p), None) for p in pts]
    nU, nN = O.prod_sizes(otrees, Np, T)
    U, G = rng.random(nU), rng.standard_normal(nN)
    assert_same(trees, Niter=T, Np=Np, randU=U, randN=G)
    p, ind = run("1", trees, Niter=T, Np=Np, randU=U, randN=G)
    op, oind = O.gibbs(otrees, Np, T, U, G)
    assert np.array_equal(ind, oind)
    scale = np.maximum(np.abs(op), 1e-3 * np.max(np.abs(op)) + 1e-300)
    assert float(np.max(np.abs(p - op) / scale)) < 1e-10


def test_inflated_bound_redoes_everything_and_still_matches():
    os.environ["KDEB200_GIBBS_EXACT_INFLATE"] = "1e6"
    try:
        lanes, warps = assert_same(make_trees(41, 3, 3, 600), Niter=2, Np=3000, seed=2)
    finally:
        os.environ.pop("KDEB200_GIBBS_EXACT_INFLATE", None)
    assert lanes > 0 and warps > 0


# ---- the certificate itself: per node and per prefix sum, K1's FP64 value lies inside the interval K1x claims ------
def check_bound(trees, mu, cadd, T=2, j=0):
    from kde_b200 import api as KA
    L = K.gibbs_sizes(trees, T)[0]
    hdr, nodes = KA._gibbs_exact_bound_probe(trees, T, j, L, mu, cadd)
    worst, nok = 0.0, 0
    for h, t in zip(hdr, nodes):
        A, B, aabs, ok, lw2max = h[:5]
        if not ok:  # K1x redoes such a draw in FP64 without looking at the bound
            continue
        nok += 1
        W = 2.0 ** lw2max
        p32, acc, p64, S64, lo, hi, lo_ck, hi_ck = t.T
        p64s, S64s = p64 / W, S64 / W  # the division's own rounding: 2^-53 relative, allowed below
        bound = p32 * (A + B * acc) + aabs
        err = np.abs(p32 - p64s)
        assert np.all(err <= bound + 2.3e-16 * p64s), float(np.max(err / bound))
        worst = max(worst, float(np.max(err / bound)))
        assert np.all(lo <= S64s * (1 + 2.3e-16)) and np.all(S64s * (1 - 2.3e-16) <= hi)
        ck = ~np.isnan(lo_ck)
        assert ck.any() and ck[-1]
        assert np.all(lo_ck[ck] <= S64s[ck] * (1 + 2.3e-16)) and np.all(S64s[ck] * (1 - 2.3e-16) <= hi_ck[ck])
    return nok, worst


def probe_queries(rng, pts, hvar, nq, offset_sd=0.0):
    """conditionals a chain meets: X near a data point (sampleIndices!) or a product mean with a Calmost (sampleIndex)"""
    d = pts.shape[0]
    mu = pts[:, rng.integers(0, pts.shape[1], nq)].T + rng.standard_normal((nq, d)) * np.sqrt(hvar)
    mu += offset_sd * np.sqrt(hvar)
    cadd = np.zeros((nq, d))
    cadd[nq // 2:] = rng.uniform(0.05, 3.0, (nq - nq // 2, d)) * hvar
    return mu, cadd


@pytest.mark.parametrize("shift", [0.0, 1e3])
def test_bound_holds_per_node_c4_shape(shift):
    rng = np.random.default_rng(71)
    pts = [mixture(rng, 3, 4096, 0.25 * j) + shift for j in range(2)]
    trees = [K.kde(p, silverman(p)) for p in pts]
    mu, cadd = probe_queries(rng, pts[0], silverman(pts[0]) ** 2, 64)
    nok, worst = check_bound(trees, mu, cadd)
    assert nok == 64
    assert worst > 1e-3  # the probe sees real FP32 errors, so a bound that is too tight would fail here


@pytest.mark.parametrize("squeeze", [0.3, 0.1, 0.03])
def test_bound_holds_with_anisotropic_bandwidths(squeeze):
    """one dimension's bandwidth far below the others: large tile radii in kernel widths, up to the range guard"""
    rng = np.random.default_rng(72)
    pts = [mixture(rng, 3, 2048, 0.25 * j) for j in range(2)]
    bws = [silverman(p) * np.array([squeeze, 1.0, 3.0]) for p in pts]
    trees = [K.kde(p, bw) for p, bw in zip(pts, bws)]
    mu, cadd = probe_queries(rng, pts[0], bws[0] ** 2, 48)
    nok, worst = check_bound(trees, mu, cadd)
    if squeeze >= 0.3:
        assert nok > 0


@pytest.mark.parametrize("offset_sd", [15.0, 21.0, 30.0, 45.0])
def test_bound_holds_for_far_conditionals(offset_sd):
    """conditionals many bandwidths from the data: totals towards 1e-99, FP32 flush-to-zero and K1's -700 clamp"""
    rng = np.random.default_rng(73)
    pts = [mixture(rng, 3, 1024, 0.25 * j) for j in range(2)]
    trees = [K.kde(p, silverman(p)) for p in pts]
    mu, cadd = probe_queries(rng, pts[0], silverman(pts[0]) ** 2, 32, offset_sd=offset_sd)
    check_bound(trees, mu, cadd)
