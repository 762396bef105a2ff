"""-m gpu: K1m, single Gibbs calls of more than KDEB200_MAX_DENS = 16 densities (up to KDEB200_MAX_DENS_LARGE = 64).

The reference's prodAppxMSGibbsS / `*` take any number of densities; a variable's belief in belief propagation is the
product of all its incoming messages.  These products run one thread-per-chain FP64 kernel at every Np and precision,
and hold the contract of tests/test_gpu_gibbs.py: under injected streams, labels identical to the oracle and points
within 1e-10."""
import ctypes as C

import numpy as np
import pytest

import kde_b200 as K
from kde_b200 import _lib
from oracle import oracle as O
from tests import gibbs_pseudocode as PS
from tests import test_oracle_stats as STATS
from tests.util import mixture, silverman

pytestmark = pytest.mark.gpu
PT_TOL = 1e-10
NS = [1, 3, 17, 100, 40, 2000, 2, 257, 64, 9, 130, 5]  # ragged tree sizes, cycled over the densities


def make(rng, d, N, shift=0.0, weights=False, bw=None):
    pts = mixture(rng, d, N, shift)
    if bw is None:
        bw = silverman(pts) if N > 2 else np.full(d, 0.7)
    w = rng.random(N) + 0.05 if weights else None
    return K.kde(pts, bw, w), O.OKDE.kde_bw(pts, bw, w)


def family(rng, d, M, sizes=NS, weights=True):
    pairs = [make(rng, d, sizes[j % len(sizes)], 0.1 * j, weights and j % 2 == 1) for j in range(M)]
    return [p[0] for p in pairs], [p[1] for p in pairs]


def streams(otrees, Np, T, rng):
    nU, nN = O.prod_sizes(otrees, Np, T)
    return rng.random(nU), rng.standard_normal(nN)


def close(a, b):
    scale = np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b)) + 1e-300)
    return float(np.max(np.abs(a - b) / scale)) < PT_TOL


def compare(kt, ot, Np, T, rng, add_entropy=True, mask=None):
    U, G = streams(ot, Np, T, rng)
    if mask is None and add_entropy:
        ep, ei = O.gibbs(ot, Np, T, U, G, nthreads=O.max_threads())
    else:
        ep, ei = O.gibbs(ot, Np, T, U, G, add_entropy=add_entropy, mask=mask)
    gp, gi = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, randU=U, randN=G, addEntropy=add_entropy,
                                partialDimMask=mask)
    assert gi.shape == ei.shape and gp.shape == ep.shape
    nbad = int(np.sum(np.any(gi != ei, axis=0)))
    assert nbad == 0, "label mismatches in %d of %d samples" % (nbad, Np)
    assert close(gp, ep)
    return gp, gi


@pytest.mark.parametrize("M", [17, 18, 24, 32, 33, 48, 64])
@pytest.mark.parametrize("d", [1, 2, 3, 5, 8])
def test_injected_streams_match_oracle(d, M):
    rng = np.random.default_rng(100 * M + d)
    kt, ot = family(rng, d, M)
    compare(kt, ot, 150, (M + d) % 6, rng)


def test_statistical_precision_mode_runs_fp64():
    """kdeb200_set_gibbs_precision(F32) leaves these products on the FP64 kernel: labels stay exact."""
    rng = np.random.default_rng(20)
    kt, ot = family(rng, 3, 20, sizes=[300, 100, 50])
    K.set_gibbs_precision(K.F32)
    try:
        compare(kt, ot, 2000, 3, rng)
    finally:
        K.set_gibbs_precision(K.F64)


def test_partial_dim_mask_poisoned():
    """test/testPartialProd.jl at 21 densities: blind coordinates poisoned with 9999999 must not leak."""
    rng = np.random.default_rng(12)
    kt, ot, mask = [], [], []
    for j in range(21):
        kind = j % 3
        p = rng.random((2, 100)) + (10.0, 0.0, -10.0)[kind]
        if kind == 0:
            p[1, :] = 9999999.0
        if kind == 2:
            p[0, :] = 9999999.0
        kt.append(K.kde(p, [0.1, 0.1]))
        ot.append(O.OKDE.kde_bw(p, [0.1, 0.1]))
        mask.append([kind != 2, kind != 0])
    pts, _ = compare(kt, ot, 100, 3, rng, mask=mask)
    assert np.sum((0 < pts[0]) & (pts[0] < 10)) > 80 and np.sum((-10 < pts[1]) & (pts[1] < 0)) > 80
    # a dimension no density sees, and densities blind in every dimension
    kt, ot = family(rng, 3, 17, sizes=[40, 7, 100])
    mask = rng.random((17, 3)) < 0.7
    mask[:, 1] = False
    mask[4, :] = False
    pts, _ = compare(kt, ot, 130, 2, rng, mask=mask)
    assert np.all(pts[1] == 0.0)


def test_add_entropy_false_is_precision_weighted_mean():
    rng = np.random.default_rng(11)
    kt, ot = family(rng, 2, 20, sizes=[50, 30], weights=False)
    pts, ind = compare(kt, ot, 64, 5, rng, add_entropy=False)
    lam = np.stack([1.0 / (K.getBW(t)[:, 0] ** 2) for t in kt])
    for s in range(64):
        mus = np.stack([K.getPoints(t)[:, ind[j, s] - 2] for j, t in enumerate(kt)])  # label = index + 1
        assert np.allclose(pts[:, s], (lam * mus).sum(0) / lam.sum(0), rtol=1e-12, atol=1e-14)


def test_label_recording_matches_oracle():
    rng = np.random.default_rng(31)
    kt, ot = family(rng, 2, 18, sizes=[37, 5, 90, 1])
    Np, T = 150, 4
    U, G = streams(ot, Np, T, rng)
    ep, ei, er = O.gibbs(ot, Np, T, U, G, record=True)
    gp, gi, gr = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, randU=U, randN=G, recordLabels=True)
    assert gr.shape == er.shape == (Np, 18, O.gibbs_nlevels(ot))
    assert np.array_equal(gr, er) and np.array_equal(gi, ei) and close(gp, ep)
    assert np.array_equal(gr[:, :, -1] + 1, gi.T)
    _, _, g0 = K.prodAppxMSGibbsS(None, kt, None, None, Niter=0, Np=8, seed=1, recordLabels=True)
    assert (g0 == -1).all()


@pytest.mark.parametrize("M,N", [(20, 100), (40, 700)])
def test_prod_equals_gibbs_then_lcv_fit(M, N):
    """prod / `*` (kdeb200_product_kde: Gibbs and the LOOCV refit on the device; fused for <= 512 samples) equals
    Gibbs with the same Philox seed followed by kde!(points), bit for bit."""
    rng = np.random.default_rng(M)
    trees = [K.kde(mixture(rng, 2, N, 0.05 * j)) for j in range(M)]
    q = K.prod(trees, seed=77)
    pts, _ = K.prodAppxMSGibbsS(None, trees, None, None, Niter=5, Np=N, seed=77)
    ref = K.kde(pts)
    assert np.array_equal(K.getPoints(q), K.getPoints(ref))
    assert np.array_equal(K.getBW(q), K.getBW(ref))


def test_philox_mode_is_reproduced_by_injection_and_by_oracle():
    rng = np.random.default_rng(21)
    kt, ot = family(rng, 3, 24, sizes=[200, 60, 13])
    Np, T, seed = 300, 5, 20261022
    L, perU, perN, _ = K.gibbs_sizes(kt, T)
    assert L == O.gibbs_nlevels(ot) and perU == 24 * (1 + L * (1 + T)) and perN == 3 * (L + 1)
    p0, i0 = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, seed=seed)
    U, G = K.philox_streams(seed, Np, perU, perN)
    p1, i1 = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, randU=U, randN=G)
    assert np.array_equal(i0, i1) and np.array_equal(p0, p1)
    ep, ei = O.gibbs(ot, Np, T, U, G, nthreads=O.max_threads())
    assert np.array_equal(i0, ei) and close(p0, ep)


def test_sharding_slices_and_multi_context():
    rng = np.random.default_rng(9)
    kt, _ = family(rng, 3, 33, sizes=[500, 120, 31])
    Np, T = 5000 + 37, 3
    pm, im, rm = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, seed=11, recordLabels=True)
    a, ai = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, seed=11, s0=0, s1=77)
    b, bi = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, seed=11, s0=77, s1=Np)
    assert np.array_equal(np.hstack([a, b]), pm) and np.array_equal(np.hstack([ai, bi]), im)
    L, perU, perN, _ = K.gibbs_sizes(kt, T)
    U, G = K.philox_streams(11, Np, perU, perN)
    c, ci, cr = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, randU=U, randN=G, s0=130, s1=4000,
                                   recordLabels=True)
    assert np.array_equal(c, pm[:, 130:4000]) and np.array_equal(ci, im[:, 130:4000]) and np.array_equal(cr, rm[130:4000])
    K.init(0)
    try:
        assert K.init_multi(devices=[0, 0]) == 2
        p2, i2, r2 = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, seed=11, recordLabels=True)
        pj, ij = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, randU=U, randN=G)
    finally:
        assert K.init_multi(1) == 1
    assert np.array_equal(p2, pm) and np.array_equal(i2, im) and np.array_equal(r2, rm)
    assert np.array_equal(pj, pm) and np.array_equal(ij, im)


def test_pseudocode_restatement():
    """tests/gibbs_pseudocode.py, the independent transcription of the reference's chain, at 17 densities."""
    rng = np.random.default_rng(17)
    Ns = [5, 1, 9, 3, 12, 2, 7, 4, 1, 10, 6, 8, 3, 2, 11, 5, 4]
    d, Np, T = 2, 10, 2
    pts = [rng.standard_normal((d, n)) + 0.3 * j for j, n in enumerate(Ns)]
    bws = [0.3 + rng.random(d) for _ in Ns]
    wts = [rng.random(n) + 0.1 for n in Ns]
    ot = [O.OKDE.kde_bw(p, b, w) for p, b, w in zip(pts, bws, wts)]
    kt = [K.kde(p, b, w) for p, b, w in zip(pts, bws, wts)]
    U, G = streams(ot, Np, T, rng)
    pp, pi = PS.gibbs([t.arrays() for t in ot], Np, T, U, G)
    gp, gi = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, randU=U, randN=G)
    assert np.array_equal(gi, pi) and close(gp, pp)


@pytest.mark.parametrize("M", [17, 24, 64])
@pytest.mark.parametrize("vf,ic", [(2, 4), (4, 4), (8, 4)])
def test_simd_sum_edge(M, vf, ic):
    """From 16 densities on, Julia's sum(lambdas) is an @simd loop whose order depends on the host ISA
    (src/MSGibbs01.jl:141, oracle julia_sum); the kernel sums sequentially like the default oracle.  Against the
    emulated vector shapes, labels differ on at most 1 % of samples and points agree to 1e-10 elsewhere."""
    rng = np.random.default_rng(1000 * M + 10 * vf + ic)
    pairs = [make(rng, 2, 24, 0.1 * j, bw=np.array([0.4 + 0.031 * (j % 16), 0.5 + 0.017 * (j % 16)])) for j in range(M)]
    kt, ot = [p[0] for p in pairs], [p[1] for p in pairs]
    Np, T = 500, 2
    U, G = streams(ot, Np, T, rng)
    gp, gi = K.prodAppxMSGibbsS(None, kt, None, None, Niter=T, Np=Np, randU=U, randN=G)
    try:
        O.set_sum_simd(vf, ic)
        ep, ei = O.gibbs(ot, Np, T, U, G)
    finally:
        O.set_sum_simd(0, 0)
    bad = np.any(gi != ei, axis=0)
    assert bad.mean() <= 0.01
    assert np.max(np.abs(gp[:, ~bad] - ep[:, ~bad])) < 1e-10 * np.max(np.abs(ep))


def _gpu_prod(P, n, MCMC, rng):
    return K.prodAppxMSGibbsS(None, P, None, None, Niter=MCMC, Np=n, seed=int(rng.integers(1, 2 ** 62)))[0]


@pytest.mark.parametrize("D,M", [(2, 20), (2, 32), (2, 64)])
def test_reference_range_criterion(D, M):
    """rangeUnitTests' criterion (test/runtests.jl:167-201) at M beyond 16: |mean| < sqrt(1/M) and every std within
    (0.66, 1.33) sqrt(1/M), at least 5 of 10 repetitions (tests/test_oracle_many_stats.py runs the oracle)."""
    rng = np.random.default_rng(4321 + 17 * D + M)
    v = [STATS.test_prods(_gpu_prod, K.kde, rng, D=D, M=M) for _ in range(10)]
    assert sum(v) >= 5, v


def _handles(trees, gibbs=True):
    return (_lib.tree_t * len(trees))(*[t._dev(gibbs=gibbs) for t in trees])


def _c_gibbs(handles, M, Np, T=2, seed=3):
    pts = np.full(3 * max(Np, 1), 7.25)
    ind = np.full(M * max(Np, 1), -5, dtype=np.int64)
    rc = _lib.lib().kdeb200_gibbs(handles, M, Np, T, 1, None, None, 0, None, 0, seed, 0, Np, _lib.fptr(pts),
                                  _lib.iptr(ind), None)
    return rc, pts, ind


def test_refusals_and_error_codes():
    rng = np.random.default_rng(65)
    trees = [K.kde(mixture(rng, 3, 30, 0.1 * j), [0.4, 0.4, 0.4]) for j in range(65)]
    lib = _lib.lib()
    # 65 densities: code 3, nothing written
    rc, pts, ind = _c_gibbs(_handles(trees), 65, 40)
    assert rc == 3 and b"outside 1..64" in lib.kdeb200_last_error()
    assert (pts == 7.25).all() and (ind == -5).all()
    L = C.c_int(0)
    assert lib.kdeb200_gibbs_sizes(_handles(trees), 65, 2, C.byref(L), None, None, None) == 3
    bw = np.full(3, 9.5)
    assert lib.kdeb200_product_kde(_handles(trees), 65, 40, 5, 1, None, 1, _lib.fptr(pts), None, _lib.fptr(bw), None) == 3
    assert (pts == 7.25).all() and (bw == 9.5).all()
    with pytest.raises(K.KDEError):
        K.prodAppxMSGibbsS(None, trees, None, None, Np=40, seed=1)
    # 64 densities run
    rc, pts, ind = _c_gibbs(_handles(trees[:64]), 64, 40)
    assert rc == 0 and np.isfinite(pts[:120]).all() and (ind >= 2).all()
    # mixed dimensions: code 6
    mixed = trees[:16] + [K.kde(mixture(rng, 2, 30), [0.4, 0.4])] + trees[16:20]
    rc, pts, ind = _c_gibbs(_handles(mixed), 21, 40)
    assert rc == 6 and (pts == 7.25).all() and (ind == -5).all()
    # a handle made for evaluation only (kdeb200_tree_create_eval): code 7
    ev = K.kde(mixture(rng, 3, 30), [0.4, 0.4, 0.4])
    h = _handles(trees[:20])
    h[7] = ev._dev()
    rc, pts, ind = _c_gibbs(h, 20, 40)
    assert rc == 7 and b"tree_create_eval" in lib.kdeb200_last_error() and (pts == 7.25).all()
    # degenerate bandwidths (zero here) are refused with code 5 and the reason; M <= 16 still runs them verbatim
    zero = K.kde(mixture(rng, 3, 30), [0.0, 0.4, 0.4])
    deg = trees[:19] + [zero]
    rc, pts, ind = _c_gibbs(_handles(deg), 20, 40)
    assert rc == 5 and b"bandwidth" in lib.kdeb200_last_error() and (pts == 7.25).all() and (ind == -5).all()
    with pytest.raises(K.KDEError):
        K.prod(deg, seed=1)
    with np.errstate(all="ignore"):
        K.prodAppxMSGibbsS(None, trees[:15] + [zero], None, None, Np=40, seed=1)
    # the batch calls keep their limit of 16 densities per problem
    pb = np.zeros(3 * 40)
    ib = np.zeros(17 * 40, dtype=np.int64)
    nd = (C.c_int * 1)(17)
    npb = np.array([40], dtype=np.int64)
    seeds = (C.c_uint64 * 1)(1)
    rc = lib.kdeb200_gibbs_batch(1, nd, _handles(trees[:17]), _lib.iptr(npb), 2, 1, None, None, None, None, None,
                                 seeds, _lib.fptr(pb), _lib.iptr(ib))
    assert rc == 3
