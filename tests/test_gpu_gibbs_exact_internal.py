"""-m gpu: K1x on internal levels -- the sampleIndex draws (variant C) of internal levels of at least 256 nodes are
decided from certified FP32 prefix sums too (csrc/gibbs_exact_kernel.cuh).  Outputs must stay those of the all-FP64
kernel K1 (KDEB200_GIBBS_EXACT=0) bit for bit, and the bound must hold node by node."""
import os

import numpy as np
import pytest

import kde_b200 as K
from kde_b200 import api as KA
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
    K.gibbs_exact_redone_internal()
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
    """K1 against K1x; returns the redo counters of the K1x call: (leaf lanes, leaf warps), (internal lanes, warps)"""
    ref = run("0", trees, **kw)
    K.gibbs_exact_redone()
    K.gibbs_exact_redone_internal()
    new = run("1", trees, **kw)
    leaf, internal = K.gibbs_exact_redone(), K.gibbs_exact_redone_internal()
    assert len(ref) == len(new)
    for a, b in zip(ref, new):
        assert a.dtype == b.dtype and a.shape == b.shape
        assert np.array_equal(a, b), "K1x differs from K1 in %d entries" % int(np.sum(a != b))
    return leaf, internal


def make_trees(seed, M, N, shift=0.25):
    rng = np.random.default_rng(seed)
    return [K.kde(p, silverman(p)) for p in (mixture(rng, 3, N, shift * j) for j in range(M))]


def test_c4_shape_identical_and_internal_mostly_decided():
    Np, T = 100_000, 5
    _, (lanes, warps) = assert_same(make_trees(11, 8, 4096), Niter=T, Np=Np, seed=321)
    certified = Np * T * 8 * 4  # sampleIndex draws on the levels of 256, 512, 1024 and 2048 nodes
    assert 0 < lanes < 0.02 * certified, (lanes, warps)


def test_multi_tile_internal_levels():
    """N = 100 000: internal levels of up to 65 536 nodes, many tiles and chunks per certified draw"""
    assert_same(make_trees(12, 2, 100_000), Niter=1, Np=300, seed=5)


def test_level_labels_identical():
    assert_same(make_trees(13, 3, 1500), Niter=3, Np=3000, seed=8, recordLabels=True)


def test_inflated_bound_redoes_internal_draws_and_still_matches():
    os.environ["KDEB200_GIBBS_EXACT_INFLATE"] = "1e6"
    try:
        (leaf, _), (lanes, warps) = assert_same(make_trees(41, 3, 1200), Niter=2, Np=3000, seed=2, recordLabels=True)
    finally:
        os.environ.pop("KDEB200_GIBBS_EXACT_INFLATE", None)
    assert leaf > 0 and lanes > 0 and warps > 0


# ---- the certificate on internal levels: per node and per prefix sum, K1's FP64 value lies inside K1x's interval ----
def check_bound(trees, level, mu, cadd, T=2, j=0, n_expect=None):
    hdr, nodes = KA._gibbs_exact_bound_probe(trees, T, j, level, mu, cadd)
    if n_expect is not None:
        assert int(hdr[0][5]) == n_expect
    worst, nok = 0.0, 0
    for h, t in zip(hdr, nodes):
        A, B, aabs, ok = h[:4]
        W = h[7]
        assert W == 2.0 ** h[4]
        if not ok:  # K1x redoes such a draw in FP64 without looking at the bound
            continue
        nok += 1
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


def internal_queries(rng, pts, hvar, nq, offset_sd=0.0, cadd_scale=(0.05, 3.0)):
    """sampleIndex conditionals: a product mean near the data and a Calmost of the other densities' kernels"""
    d = pts.shape[0]
    mu = pts[:, rng.integers(0, pts.shape[1], nq)].T + rng.standard_normal((nq, d)) * np.sqrt(hvar)
    mu += offset_sd * np.sqrt(hvar)
    cadd = rng.uniform(*cadd_scale, (nq, d)) * hvar
    return mu, cadd


@pytest.mark.parametrize("shift", [0.0, 1e3])
@pytest.mark.parametrize("n", [2048, 1024, 256])
def test_bound_holds_per_node_c4_shape(shift, n):
    rng = np.random.default_rng(81)
    pts = [mixture(rng, 3, 4096, 0.25 * j) + shift for j in range(2)]
    trees = [K.kde(p, silverman(p)) for p in pts]
    mu, cadd = internal_queries(rng, pts[0], silverman(pts[0]) ** 2, 48)
    nok, worst = check_bound(trees, int(np.log2(n)), mu, cadd, n_expect=n)
    assert nok == 48
    assert worst > 1e-3  # the probe sees real FP32 errors, so a bound that is too tight would fail here


@pytest.mark.parametrize("squeeze", [0.3, 0.1, 0.03])
def test_bound_holds_with_anisotropic_bandwidths(squeeze):
    """one dimension's bandwidth far below the others: large tile radii in kernel widths.  Below 0.3 the range guard
    (130 a1 + a0 <= 1e-3) may send every query to the FP64 redo, as on the leaf levels; where it certifies, the bound
    must hold."""
    rng = np.random.default_rng(82)
    pts = [mixture(rng, 3, 4096, 0.25 * j) for j in range(2)]
    bws = [silverman(p) * np.array([squeeze, 1.0, 3.0]) for p in pts]
    trees = [K.kde(p, bw) for p, bw in zip(pts, bws)]
    mu, cadd = internal_queries(rng, pts[0], bws[0] ** 2, 32)
    for n in (2048, 256):
        nok, _ = check_bound(trees, int(np.log2(n)), mu, cadd, n_expect=n)
        print("squeeze %g, %d nodes: %d of 32 queries certified" % (squeeze, n, nok))
        if squeeze >= 0.3:
            assert nok > 0


@pytest.mark.parametrize("offset_sd", [15.0, 21.0, 30.0, 45.0])
def test_bound_holds_for_far_conditionals(offset_sd):
    """conditionals many bandwidths from the data: totals towards 1e-99, FP32 flush-to-zero and K1's -700 clamp"""
    rng = np.random.default_rng(83)
    pts = [mixture(rng, 3, 4096, 0.25 * j) for j in range(2)]
    trees = [K.kde(p, silverman(p)) for p in pts]
    mu, cadd = internal_queries(rng, pts[0], silverman(pts[0]) ** 2, 32, offset_sd=offset_sd)
    for n in (1024, 256):
        check_bound(trees, int(np.log2(n)), mu, cadd, n_expect=n)


@pytest.mark.parametrize("cadd_scale", [(1e-4, 1e-3), (1e2, 1e4)])
def test_bound_holds_for_extreme_calmost(cadd_scale):
    """Calmost far below the node variances (c_k ~ b_k) and far above them (c_k ~ Calmost_k, flat terms)"""
    rng = np.random.default_rng(84)
    pts = [mixture(rng, 3, 4096, 0.25 * j) for j in range(2)]
    trees = [K.kde(p, silverman(p)) for p in pts]
    mu, cadd = internal_queries(rng, pts[0], silverman(pts[0]) ** 2, 32, cadd_scale=cadd_scale)
    for n in (2048, 256):
        nok, _ = check_bound(trees, int(np.log2(n)), mu, cadd, n_expect=n)
        assert nok == 32
