"""-m gpu: K2b, many independent brute-force evaluations in one call (kdeb200_eval_batch), and batched kde!(points)
bandwidths (kdeb200_kde_lcv_batch).

Every problem of a batch must equal the single call on its own: evaluateDualTree (kdeb200_eval, FP64) bit for bit under
pruning modes 0 and 1 (within 1e-13 under mode 2), and kde(points) / lcv_bandwidths in bandwidths, nLOO_LL call counts
and every tree array."""
import ctypes as C

import numpy as np
import pytest

import kde_b200 as K
from kde_b200 import _lib
from oracle import oracle as O
from tests.util import mixture, relerr, silverman

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def one_gpu_default_pruning():
    K.init(0)
    K.set_pruning(1)
    yield
    K.set_pruning(1)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def density(rng, d, N, weights=False, lcv=False, shift=0.0):
    pts = mixture(rng, d, N, shift)
    if lcv:
        return K.kde(pts), pts
    bw = silverman(pts) if N > 2 else np.full(d, 0.5)
    return K.kde(pts, bw, rng.random(N) + 0.1 if weights else None), pts


def far_queries(bd, M):
    """queries 30 to 45 bandwidths and 1e4 away from every component: their fast-path sums are tiny, exactly zero or
    subnormal, and the kernels recompute them with exact_row"""
    d = K.Ndim(bd)
    pts = K.getPoints(bd)
    hi = pts.max(axis=1)
    bw = K.getBW(bd)[:, 0]
    q = np.repeat(hi[:, None], M, axis=1)
    q[0] += bw[0] * np.linspace(30.0, 45.0, M)
    q[:, -1] = hi + 1e4
    return q


def heterogeneous(rng):
    """(density, positions, lvFlag) problems: d = 1..8, N 1..5000 across tile and split boundaries, M 0..3000,
    weights, LCV bandwidths, LOO, far tails, a shared handle, Gibbs-upgraded handles"""
    P = []
    shared, spts = density(rng, 2, 700)
    for d, N, M, kw in [(1, 1, 17, {}), (1, 2, 0, {}), (1, 511, 300, {}), (1, 512, 768, {}), (1, 513, 769, {}),
                        (2, 255, 129, {}), (2, 256, 3000, {}), (2, 257, 100, {"weights": True}), (2, 5000, 100, {}),
                        (3, 100, 150, {"lcv": True}), (3, 1000, 2000, {"weights": True}), (4, 127, 256, {}),
                        (4, 129, 257, {}), (5, 300, 0, {}), (5, 2000, 1000, {"weights": True}), (6, 128, 100, {}),
                        (6, 4096, 200, {}), (7, 64, 1, {}), (7, 200, 200, {"lcv": True}), (8, 63, 64, {}),
                        (8, 65, 130, {"weights": True}), (8, 5000, 3000, {})]:
        bd, _ = density(rng, d, N, **kw)
        P.append((bd, mixture(rng, d, M) if M else np.zeros((d, 0)), False))
        if N <= 1000:
            P.append((bd, bd, True))                          # leave-one-out of the same density
    for d, N in [(1, 300), (3, 257), (8, 200)]:
        bd, _ = density(rng, d, N, weights=True)
        P.append((bd, far_queries(bd, 64), False))
    P.append((shared, mixture(rng, 2, 333), False))           # one handle, several problems
    P.append((shared, shared, True))
    P.append((shared, spts[:, :50], False))
    for d, N, M in [(2, 300, 120), (3, 2000, 900)]:
        bd, _ = density(rng, d, N)
        bd._dev(gibbs=True)                                   # handle already upgraded for the sampler
        P.append((bd, mixture(rng, d, M), False))
        P.append((bd, None, True))
    P.append((shared, density(rng, 2, 40)[0], False))         # pos given as another density
    P.append((K.kde(mixture(rng, 1, 90), [0.3]), rng.standard_normal(50), False))   # vector of 1-D points
    return P


def run_batch(P):
    return K.evaluateDualTree_batch([p[0] for p in P], [p[0] if p[1] is None else p[1] for p in P],
                                    [p[2] for p in P])


def single(p):
    bd, pos, lv = p
    return K.evaluateDualTree(bd, bd if pos is None else pos, lv)


def test_heterogeneous_batch_equals_single_calls_bit_for_bit():
    rng = np.random.default_rng(1)
    P = heterogeneous(rng)
    out = run_batch(P)
    assert len(out) == len(P)
    assert K.last_kernel_ms()[1] >= 2   # one launch per (d, loo) class, plus the finalize launch
    tails = 0
    for i, p in enumerate(P):
        ref = single(p)
        assert out[i].shape == ref.shape, i
        assert np.array_equal(bits(out[i]), bits(ref)), i
        tails += int(np.sum((ref == 0.0) | ((ref > 0.0) & (ref < 2.3e-308))))
    assert tails > 0   # exact zeros and subnormals from the exact_row path were compared too


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_pruning_modes(mode):
    rng = np.random.default_rng(2)
    P = heterogeneous(rng)
    K.set_pruning(mode)
    out = run_batch(P)
    for i, p in enumerate(P):
        ref = single(p)
        same = np.array_equal(bits(out[i]), bits(ref))   # also where both are NaN (one-point leave-one-out: 0/0)
        assert same or (mode == 2 and relerr(out[i], ref) <= 1e-13), i


def test_batch_against_oracle():
    rng = np.random.default_rng(3)
    P, ref = [], []
    for d, N, M, w in [(1, 200, 150, False), (2, 600, 300, True), (3, 257, 100, False), (5, 100, 80, True)]:
        pts = mixture(rng, d, N)
        bw = silverman(pts)
        ww = rng.random(N) + 0.1 if w else None
        bd, o = K.kde(pts, bw, ww), O.OKDE.kde_bw(pts, bw, ww)
        pos = mixture(rng, d, M)
        P.append((bd, pos, False))
        ref.append(o.evaluate(pos))
        P.append((bd, bd, True))
        ref.append(o.evaluate())
    out = run_batch(P)
    for i in range(len(P)):
        assert relerr(out[i], ref[i]) < 1e-12, i


def test_composition_invariance_1024_problems():
    rng = np.random.default_rng(4)
    pool = []
    for b in range(64):
        d = 1 + b % 3
        bd, _ = density(rng, d, int(rng.integers(100, 201)), weights=bool(b % 2))
        pool.append(bd)
    P = []
    for i in range(1024):
        bd = pool[int(rng.integers(0, len(pool)))]
        if i % 5 == 0:
            P.append((bd, bd, True))
        else:
            P.append((bd, mixture(rng, K.Ndim(bd), int(rng.integers(0, 201))), False))
    full = run_batch(P)
    order = rng.permutation(len(P))
    shuffled = run_batch([P[k] for k in order])
    for j, k in enumerate(order):
        assert np.array_equal(bits(shuffled[j]), bits(full[k])), k
    for k in (0, 1, 517, 1023):   # alone, and between other neighbours
        assert np.array_equal(bits(run_batch([P[k]])[0]), bits(full[k])), k
        assert np.array_equal(bits(run_batch([P[3], P[k], P[900]])[1]), bits(full[k])), k
        assert np.array_equal(bits(single(P[k])), bits(full[k])), k


def test_kde_batch_equals_kde_loop():
    rng = np.random.default_rng(5)
    sets = []
    for d in range(1, 9):
        for N in (2, 512, 513):
            sets.append(mixture(rng, d, N))
    sets.append(mixture(rng, 2, 100))
    cb, cl = [], []
    bws = K.lcv_bandwidths_batch(sets, _count=cb)
    for p, bw in zip(sets, bws):
        c = []
        ref = K.lcv_bandwidths(p, _count=c)
        cl.append(c)
        assert np.array_equal(bits(bw), bits(ref))
    assert cb == cl
    dens = K.kde_batch(sets)
    for p, a in zip(sets, dens):
        b = K.kde(p)
        for k in ("centers", "ranges", "weights", "left_child", "right_child", "lowest_leaf", "highest_leaf", "permutation"):
            assert np.array_equal(getattr(a.bt, k), getattr(b.bt, k)), k
        for k in ("means", "bandwidth", "bandwidthMin", "bandwidthMax"):
            assert np.array_equal(bits(getattr(a, k)), bits(getattr(b, k))), k
    assert K.kde_batch([]) == [] and K.evaluateDualTree_batch([], []) == []


def _raw_eval_batch(trees, M, loo, pos, precision, out):
    n = len(trees)
    h = (_lib.tree_t * max(n, 1))(*[t._dev() for t in trees])
    Ma = np.array(M, dtype=np.int64)
    la = np.array(loo, dtype=np.int32)
    return _lib.lib().kdeb200_eval_batch(n, h, _lib.iptr(Ma), la.ctypes.data_as(C.POINTER(C.c_int)), _lib.fptr(pos),
                                         precision, _lib.fptr(out))


def _err():
    return _lib.lib().kdeb200_last_error().decode()


def test_errors_name_the_problem_and_run_nothing():
    rng = np.random.default_rng(6)
    good = [density(rng, 2, 100)[0] for _ in range(3)]
    pos = mixture(rng, 2, 10)
    q = np.concatenate([np.ascontiguousarray(pos.T).ravel()] * 3)
    sentinel = -7.25
    out = np.full(30, sentinel)
    # unknown precision, and the FP32 / bounded precisions the batch does not offer: code 3
    for prec in (7, -1, K.F32, K.F64_BOUNDED, K.F32_BOUNDED):
        assert _raw_eval_batch(good, [10] * 3, [0] * 3, q, prec, out) == 3
    # NULL arguments: code 2
    h = (_lib.tree_t * 3)(*[t._dev() for t in good])
    Ma = np.full(3, 10, dtype=np.int64)
    assert _lib.lib().kdeb200_eval_batch(3, None, _lib.iptr(Ma), None, _lib.fptr(q), K.F64, _lib.fptr(out)) == 2
    assert _lib.lib().kdeb200_eval_batch(3, h, _lib.iptr(Ma), None, None, K.F64, _lib.fptr(out)) == 2
    assert "problem 0" in _err()
    h[1] = None
    assert _lib.lib().kdeb200_eval_batch(3, h, _lib.iptr(Ma), None, _lib.fptr(q), K.F64, _lib.fptr(out)) == 2
    assert "problem 1" in _err()
    # a bad bandwidth (zero variance) in problem 2: code 5, as the single call
    bad = K.kde(mixture(rng, 2, 50), [0.0, 0.3])
    with pytest.raises(K.KDEError):
        K.evaluateDualTree(bad, pos)
    assert _raw_eval_batch(good[:2] + [bad], [10] * 3, [0] * 3, q, K.F64, out) == 5
    assert "problem 2" in _err()
    assert np.all(out == sentinel)
    # a d mismatch between a density and its query block
    with pytest.raises(K.KDEError, match="problem 1"):
        K.evaluateDualTree_batch(good[:2], [pos, mixture(rng, 3, 10)])
    # fits: N < 2, NULL arguments
    d = np.array([2, 1, 2], dtype=np.int32)
    N = np.array([10, 1, 10], dtype=np.int64)
    pts = np.zeros(41)
    bw = np.full(5, sentinel)
    lcv = _lib.lib().kdeb200_kde_lcv_batch
    ip = C.POINTER(C.c_int)
    assert lcv(3, d.ctypes.data_as(ip), _lib.iptr(N), _lib.fptr(pts), _lib.fptr(bw), None) == 3
    assert "problem 1" in _err()
    assert lcv(3, d.ctypes.data_as(ip), _lib.iptr(N), None, _lib.fptr(bw), None) == 2
    assert lcv(3, None, _lib.iptr(N), _lib.fptr(pts), _lib.fptr(bw), None) == 2
    assert np.all(bw == sentinel)
    with pytest.raises(K.KDEError, match="problem 1"):
        K.kde_batch([mixture(rng, 2, 10), np.zeros((2, 1))])
    # and the batch still works afterwards
    assert _raw_eval_batch(good, [10] * 3, [0] * 3, q, K.F64, out) == 0
    assert np.array_equal(bits(out[10:20]), bits(K.evaluateDualTree(good[1], pos)))


def test_under_init_multi_runs_on_the_primary():
    rng = np.random.default_rng(7)
    P = heterogeneous(rng)[:30]
    sets = [mixture(rng, 2, 100), mixture(rng, 3, 600)]
    ref, ref_bw = run_batch(P), K.lcv_bandwidths_batch(sets)
    try:
        assert K.init_multi(devices=[0, 0]) == 2
        out, bw = run_batch(P), K.lcv_bandwidths_batch(sets)
    finally:
        assert K.init_multi(1) == 1
    for a, b in zip(out, ref):
        assert np.array_equal(bits(a), bits(b))
    for a, b in zip(bw, ref_bw):
        assert relerr(a, b) < 1e-9   # the large set's bandwidth loop shares its rows over the set, as kde_lcv does
