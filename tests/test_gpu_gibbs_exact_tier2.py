"""-m gpu: the FP64 tiers of K1x (csrc/gibbs_exact_kernel.cuh).  A draw the certified FP32 sums cannot decide is first
decided from warp-parallel FP64 sums of K1's node values with their own bound (xa_tier2, "tier 2"); only what that
cannot prove goes to the serial node-order sweep (xa_redo, "tier 3").  Outputs must stay those of the all-FP64 kernel
K1 (KDEB200_GIBBS_EXACT=0) bit for bit on every path.

KDEB200_GIBBS_EXACT_INFLATE multiplies both bounds.  Tier 2's relative half-width is delta = 1.001 (n + nb + 15) 2^-53
(n nodes, nb = ceil(n / 256) blocks), at least 1.001 * 18 * 2^-53 = 2.0e-15 on the smallest level (n = 2).  At inflate
1e15 delta * inflate > 2 everywhere, so the lower end of every total interval is negative, tier 2 can never prove that
K1's 1e-99 rule does not fire, and every undecided draw with a non-zero total reaches tier 3."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import kde_b200 as K
from kde_b200 import _lib
from kde_b200 import api as KA
from oracle import oracle as O
from tests.util import mixture, silverman

pytestmark = pytest.mark.gpu

COUNTERS = (K.gibbs_exact_redone, K.gibbs_exact_redone_b, K.gibbs_exact_redone_internal, K.gibbs_exact_tier3)
FORCE_TIER3 = "1e15"


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


def run(route, trees, inflate=None, **kw):
    os.environ["KDEB200_GIBBS_EXACT"] = route
    if inflate is not None:
        os.environ["KDEB200_GIBBS_EXACT_INFLATE"] = inflate
    try:
        return K.prodAppxMSGibbsS(None, trees, None, None, **kw)
    finally:
        os.environ.pop("KDEB200_GIBBS_EXACT", None)
        os.environ.pop("KDEB200_GIBBS_EXACT_INFLATE", None)


def assert_same(trees, inflate=None, **kw):
    """K1 against K1x; returns the K1x call's counters (lanes, warps): redone leaf, variant B, variant C, tier 3"""
    ref = run("0", trees, **kw)
    for f in COUNTERS:
        f()
    new = run("1", trees, inflate, **kw)
    counts = [f() for f in COUNTERS]
    assert len(ref) == len(new)
    for a, b in zip(ref, new):
        assert a.dtype == b.dtype and a.shape == b.shape
        assert np.array_equal(a, b), "K1x differs from K1 in %d entries" % int(np.sum(a != b))
    return counts


def make_trees(seed, M, N, shift=0.25, d=3):
    rng = np.random.default_rng(seed)
    return [K.kde(p, silverman(p)) for p in (mixture(rng, d, N, shift * j) for j in range(M))]


def test_c4_shape_through_tier2():
    """an FP32 bound 100 times too wide leaves most leaf warp-draws undecided; tier 2's, 100 times its own width (about
    5e-11 relative), still decides all of them"""
    Np, T = 20_000, 5
    (a_l, a_w), (b_l, _), (c_l, _), t3 = assert_same(make_trees(11, 8, 4096), "100", Niter=T, Np=Np, seed=77,
                                                      recordLabels=True)
    leaf_warp_draws = Np // 32 * 8 * (T + 1)  # one leaf level of 4096 nodes
    assert a_w > 0.5 * leaf_warp_draws, (a_w, leaf_warp_draws)
    assert b_l > 0 and c_l > 0
    assert t3 == (0, 0)


def test_huge_inflate_runs_tier3():
    (a_l, a_w), (b_l, b_w), (c_l, c_w), (t3_l, t3_w) = assert_same(make_trees(41, 3, 600), FORCE_TIER3, Niter=2,
                                                                    Np=3000, seed=2, recordLabels=True)
    assert t3_l == a_l + b_l + c_l > 0
    assert t3_w == a_w + b_w + c_w


@pytest.mark.parametrize("case", ["tiny_variances", "squeezed_bandwidth", "far_apart"])
def test_levels_outside_the_fp32_guard_go_through_tier2(case):
    """every lane of a draw the FP32 tier does not certify at all (variances below 2^-30, a bandwidth squeezed far below
    the others, product mass in the far tails) is decided by tier 2"""
    rng = np.random.default_rng(95)
    if case == "tiny_variances":
        pts = [1e-6 * mixture(rng, 3, 4096, 0.25 * j) for j in range(2)]
        bws = [silverman(p) for p in pts]
    elif case == "squeezed_bandwidth":
        pts = [mixture(rng, 3, 4096, 0.25 * j) for j in range(2)]
        bws = [silverman(p) * np.array([0.03, 1.0, 3.0]) for p in pts]
    else:
        pts = [mixture(rng, 3, 2000, 0.0) + 1e3 + 40.0 * j for j in range(2)]
        bws = [silverman(p) for p in pts]
    trees = [K.kde(p, bw) for p, bw in zip(pts, bws)]
    (a_l, _), (b_l, _), (c_l, _), t3 = assert_same(trees, Niter=2, Np=4000, seed=4, recordLabels=True)
    assert a_l + b_l + c_l > 0
    assert t3 == (0, 0)


@pytest.mark.parametrize("sep", [20.0, 40.0, 60.0])
def test_far_tails_and_cdf_edges(sep):
    """densities `sep` data spreads apart push the totals towards K1's 1e-99 rule and below; injected uniforms of 0 and
    of the largest double below 1 put targets on the first node and at the total (the n - 1 fallback).  All undecided
    draws go through tier 2 (inflate 1e3)."""
    rng = np.random.default_rng(96)
    d, M, N, Np, T = 3, 2, 300, 640, 3
    pts = [mixture(rng, d, N, 0.0) + sep * j for j in range(M)]
    trees = [K.kde(p, silverman(p)) for p in pts]
    otrees = [O.OKDE.kde_bw(p, silverman(p), None) for p in pts]
    nU, nN = O.prod_sizes(otrees, Np, T)
    U, G = rng.random(nU), rng.standard_normal(nN)
    U[rng.random(nU) < 0.2] = 0.0
    U[rng.random(nU) < 0.2] = np.nextafter(1.0, 0.0)
    (a_l, _), _, _, _ = assert_same(trees, "1e3", Niter=T, Np=Np, randU=U, randN=G, recordLabels=True)
    assert a_l > 0


def test_caller_stream():
    """kdeb200_gibbs_device on a stream of the caller's, with most draws through tier 2: the outputs, written in stream
    order after a fill on that stream, are K1's"""
    trees = make_trees(44, 4, 2000)
    Np, T, seed = 5000, 3, 21
    ref_pts, ref_idx = run("0", trees, Niter=T, Np=Np, seed=seed)
    st = torch.cuda.Stream()
    os.environ["KDEB200_GIBBS_EXACT"] = "1"
    os.environ["KDEB200_GIBBS_EXACT_INFLATE"] = "100"
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
        os.environ.pop("KDEB200_GIBBS_EXACT_INFLATE", None)
    assert np.array_equal(pts.cpu().numpy(), ref_pts.T)
    assert np.array_equal(idx.cpu().numpy(), ref_idx.T)
    lanes, _ = K.gibbs_exact_redone()
    assert lanes > 0
