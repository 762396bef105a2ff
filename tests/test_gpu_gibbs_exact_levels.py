"""-m gpu: K1x decides every label from certified FP32 sums -- the sampleIndices! draws (variant B) of every internal
level, and the sampleIndex draws (variant C) of internal levels of any size, next to the leaf levels
(csrc/gibbs_exact_kernel.cuh).  Outputs must stay those of the all-FP64 kernel K1 (KDEB200_GIBBS_EXACT=0) bit for bit,
and the bound must hold node by node on the levels the earlier tests do not reach."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import kde_b200 as K
from kde_b200 import _lib
from kde_b200 import api as KA
from tests.util import mixture, silverman

pytestmark = pytest.mark.gpu

COUNTERS = (K.gibbs_exact_redone, K.gibbs_exact_redone_b, K.gibbs_exact_redone_internal)


@pytest.fixture(autouse=True)
def thread_per_chain_kernel():
    """K1x replaces the thread-per-chain kernel; small calls would otherwise go to the warp-per-chain kernel."""
    saved = {k: os.environ.get(k) for k in ("KDEB200_GIBBS_WARP_MAX", "KDEB200_GIBBS_EXACT", "KDEB200_GIBBS_EXACT_INFLATE")}
    os.environ["KDEB200_GIBBS_WARP_MAX"] = "0"
    os.environ.pop("KDEB200_GIBBS_EXACT", None)
    os.environ.pop("KDEB200_GIBBS_EXACT_INFLATE", None)
    K.set_gibbs_precision(K.F64)
    for f in COUNTERS:
        f()
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
    """K1 against K1x; returns the redo counters (lanes, warps) of the K1x call: leaf, variant B, variant C"""
    ref = run("0", trees, **kw)
    for f in COUNTERS:
        f()
    new = run("1", trees, **kw)
    counts = [f() for f in COUNTERS]
    assert len(ref) == len(new)
    for a, b in zip(ref, new):
        assert a.dtype == b.dtype and a.shape == b.shape
        assert np.array_equal(a, b), "K1x differs from K1 in %d entries" % int(np.sum(a != b))
    return counts


def make_trees(seed, M, N, shift=0.25):
    rng = np.random.default_rng(seed)
    return [K.kde(p, silverman(p)) for p in (mixture(rng, 3, N, shift * j) for j in range(M))]


def test_c4_shape_identical_with_level_labels():
    Np, T = 100_000, 5
    _, (b_lanes, _), (c_lanes, _) = assert_same(make_trees(11, 8, 4096), Niter=T, Np=Np, seed=77, recordLabels=True)
    internal_levels = 11  # 2 .. 2048 nodes
    assert b_lanes < 0.02 * Np * 8 * internal_levels, b_lanes
    assert c_lanes < 0.02 * Np * 8 * T * internal_levels, c_lanes


def test_inflated_bound_redoes_variant_b_draws_and_still_matches():
    os.environ["KDEB200_GIBBS_EXACT_INFLATE"] = "1e6"
    try:
        _, (lanes, warps), _ = assert_same(make_trees(42, 3, 1200), Niter=2, Np=3000, seed=3, recordLabels=True)
    finally:
        os.environ.pop("KDEB200_GIBBS_EXACT_INFLATE", None)
    assert lanes > 0 and warps > 0


@pytest.mark.parametrize("Np", [1, 129, 640])
def test_fewer_batches_than_resident_ctas(Np):
    """the grid is sized from the occupancy query and capped at the batch count"""
    assert_same(make_trees(43, 4, 3000), Niter=3, Np=Np, seed=9, recordLabels=True)


def test_caller_stream():
    """kdeb200_gibbs_device on a stream of the caller's: the outputs, written in stream order after a fill on that
    stream, are K1's"""
    trees = make_trees(44, 4, 2000)
    Np, T, seed = 5000, 3, 21
    ref_pts, ref_idx = run("0", trees, Niter=T, Np=Np, seed=seed)
    st = torch.cuda.Stream()
    os.environ["KDEB200_GIBBS_EXACT"] = "1"
    try:
        with torch.cuda.stream(st):
            pts = torch.full((Np, 3), float("nan"), dtype=torch.float64, device="cuda")
            idx = torch.full((Np, len(trees)), -1, dtype=torch.int64, device="cuda")
            _lib.check(_lib.lib().kdeb200_gibbs_device(KA._handles(trees), len(trees), Np, T, 1, None, None, 0, None, 0,
                                                       seed, 0, Np, pts.data_ptr(), idx.data_ptr(), None,
                                                       C.c_void_p(st.cuda_stream)))
        st.synchronize()
    finally:
        os.environ.pop("KDEB200_GIBBS_EXACT", None)
    assert np.array_equal(pts.cpu().numpy(), ref_pts.T)
    assert np.array_equal(idx.cpu().numpy(), ref_idx.T)


# ---- the certificate: per node and per prefix sum, K1's FP64 value lies inside K1x's interval ----
def check_bound(trees, level, mu, cadd, pass0, T=2, j=0, n_expect=None):
    hdr, nodes = KA._gibbs_exact_bound_probe(trees, T, j, level, mu, cadd, pass0=pass0)
    if n_expect is not None:
        assert int(hdr[0][5]) == n_expect
    worst, nok = 0.0, 0
    for h, t in zip(hdr, nodes):
        A, B, aabs, ok = h[:4]
        W = 2.0 ** h[4]  # the probe's W is the device's exp2, within 2 ulp of it
        assert abs(h[7] - W) <= 1e-15 * W
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


def queries(rng, pts, hvar, nq, offset_sd=0.0):
    """level points X (sampleIndices!) or product means (sampleIndex) near the data, and a Calmost of the other
    densities' kernels (variant C only)"""
    d = pts.shape[0]
    mu = pts[:, rng.integers(0, pts.shape[1], nq)].T + rng.standard_normal((nq, d)) * np.sqrt(hvar)
    mu += offset_sd * np.sqrt(hvar)
    cadd = rng.uniform(0.05, 3.0, (nq, d)) * hvar
    return mu, cadd


def c4_pair(rng, shift=0.0, squeeze=1.0):
    pts = [mixture(rng, 3, 4096, 0.25 * j) + shift for j in range(2)]
    bws = [silverman(p) * np.array([squeeze, 1.0, 1.0]) for p in pts]
    return pts, bws, [K.kde(p, bw) for p, bw in zip(pts, bws)]


@pytest.mark.parametrize("shift", [0.0, 1e3])
@pytest.mark.parametrize("n", [2048, 256, 32, 2])
def test_variant_b_bound_holds_per_node(shift, n):
    rng = np.random.default_rng(91)
    pts, bws, trees = c4_pair(rng, shift)
    mu, cadd = queries(rng, pts[0], bws[0] ** 2, 48)
    nok, worst = check_bound(trees, int(np.log2(n)), mu, cadd, True, n_expect=n)
    assert nok == 48
    if n >= 256:
        assert worst > 1e-3  # the probe sees real FP32 errors, so a bound that is too tight would fail here


def test_variant_b_bound_with_a_squeezed_bandwidth():
    """one bandwidth at 0.1 of the others: large radii in the level's narrowest kernel widths; where the range guard
    certifies, the bound must hold"""
    rng = np.random.default_rng(92)
    pts, bws, trees = c4_pair(rng, squeeze=0.1)
    mu, cadd = queries(rng, pts[0], bws[0] ** 2, 32)
    noks = []
    for n in (2048, 256, 8):
        nok, _ = check_bound(trees, int(np.log2(n)), mu, cadd, True, n_expect=n)
        print("squeeze 0.1, %d nodes: %d of 32 queries certified" % (n, nok))
        noks.append(nok)
    assert max(noks) > 0  # some level still certifies, so the bound is checked somewhere


def test_variant_b_variances_below_the_range_guard():
    """data and bandwidths scaled by 1e-6: node variances far below 2^-30, where the FP32 scale would be clamped.  Such
    draws are not decided (the FP64 redo serves them), and the results stay K1's"""
    rng = np.random.default_rng(95)
    pts = [1e-6 * mixture(rng, 3, 4096, 0.25 * j) for j in range(2)]
    bws = [silverman(p) for p in pts]
    trees = [K.kde(p, bw) for p, bw in zip(pts, bws)]
    mu, cadd = queries(rng, pts[0], bws[0] ** 2, 16)
    for n in (2048, 256, 2):
        nok, _ = check_bound(trees, int(np.log2(n)), mu, cadd, True, n_expect=n)
        assert nok == 0
    _, (lanes, _), _ = assert_same(trees, Niter=2, Np=2000, seed=4)
    assert lanes > 0


@pytest.mark.parametrize("offset_sd", [15.0, 30.0, 45.0])
def test_variant_b_bound_for_far_points(offset_sd):
    """level points many bandwidths from the data: totals towards 1e-99, FP32 flush-to-zero and K1's -700 clamp"""
    rng = np.random.default_rng(93)
    pts, bws, trees = c4_pair(rng)
    mu, cadd = queries(rng, pts[0], bws[0] ** 2, 32, offset_sd=offset_sd)
    for n in (1024, 64):
        check_bound(trees, int(np.log2(n)), mu, cadd, True, n_expect=n)


@pytest.mark.parametrize("n", [128, 16, 2])
def test_variant_c_bound_holds_on_small_levels(n):
    rng = np.random.default_rng(94)
    pts, bws, trees = c4_pair(rng)
    mu, cadd = queries(rng, pts[0], bws[0] ** 2, 48)
    nok, _ = check_bound(trees, int(np.log2(n)), mu, cadd, False, n_expect=n)
    assert nok == 48
