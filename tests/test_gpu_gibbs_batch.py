"""-m gpu: K1b, many independent Gibbs products in one call (kdeb200_gibbs_batch / kdeb200_product_kde_batch).

Every problem of a batch must equal the single call with the same arguments:
  - forced onto the thread-per-chain kernel K1 (KDEB200_GIBBS_WARP_MAX=0, KDEB200_GIBBS_EXACT=0): labels and points bit
    for bit (degenerate-bandwidth problems run the single call's verbatim warp kernel on both sides, so they are
    compared bit for bit, NaN pattern included, against the default routing);
  - under the default routing (K1w for small calls, K1x or K1 for large ones): labels identical, points within 1e-10,
    the contract test_gpu_gibbs.py holds the two single-call kernels to."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest

import kde_b200 as K
from kde_b200 import _lib
from oracle import oracle as O
from tests.util import mixture, silverman

pytestmark = pytest.mark.gpu
PT_TOL = 1e-10
ROUTE_ENV = ("KDEB200_GIBBS_WARP_MAX", "KDEB200_GIBBS_EXACT")


@contextlib.contextmanager
def route(name):
    saved = {k: os.environ.get(k) for k in ROUTE_ENV}
    try:
        for k in ROUTE_ENV:
            os.environ.pop(k, None)
        if name == "k1":
            os.environ["KDEB200_GIBBS_WARP_MAX"] = "0"
            os.environ["KDEB200_GIBBS_EXACT"] = "0"
        yield
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(autouse=True)
def default_environment():
    with route("default"):
        yield


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def close(a, b):
    scale = np.maximum(np.abs(b), 1e-3 * (np.max(np.abs(b)) if b.size else 0.0) + 1e-300)
    return b.size == 0 or float(np.max(np.abs(a - b) / scale)) < PT_TOL


class Prob:
    def __init__(self, rng, d, M, N, Np, weights=False, lcv=False, bw=None, mask=None, oracle=False):
        self.d, self.Np, self.mask = d, Np, mask
        self.trees, self.otrees = [], []
        for j in range(M):
            pts = mixture(rng, d, N, 0.25 * j)
            w = rng.random(N) + 0.1 if weights else None
            if lcv:
                self.trees.append(K.kde(pts))
            else:
                b = bw[j] if bw is not None else (silverman(pts) if N > 2 else np.full(d, 0.7))
                self.trees.append(K.kde(pts, b, w))
                if oracle:
                    self.otrees.append(O.OKDE.kde_bw(pts, b, w))

    def streams(self, rng, T):
        _, pu, pn, _ = K.gibbs_sizes(self.trees, T)
        return rng.random(self.Np * pu), rng.standard_normal(self.Np * pn)

    def single(self, T, ae, U=None, G=None, seed=None):
        return K.prodAppxMSGibbsS(None, self.trees, None, None, Niter=T, Np=self.Np, addEntropy=ae, randU=U, randN=G,
                                  partialDimMask=self.mask, seed=seed)


def heterogeneous(rng):
    P = [
        Prob(rng, 2, 2, 100, 100, oracle=True),                     # C1
        Prob(rng, 3, 6, 100, 100),                                  # testProds
        Prob(rng, 1, 3, 64, 33, oracle=True),
        Prob(rng, 4, 2, 300, 129, weights=True),
        Prob(rng, 5, 3, 50, 0),
        Prob(rng, 6, 2, 200, 1),
        Prob(rng, 7, 3, 40, 33),
        Prob(rng, 8, 2, 40, 100),
        Prob(rng, 2, 16, 20, 129),
        Prob(rng, 3, 1, 50, 100),                                   # a lone density (mask logic)
        Prob(rng, 2, 3, 2000, 3000),
        Prob(rng, 3, 2, 1, 33),                                     # one-component densities
        Prob(rng, 3, 3, 100, 100, oracle=True, mask=np.array([[1, 0, 1], [1, 1, 1], [0, 1, 1]], bool)),
        Prob(rng, 2, 2, 150, 129, lcv=True),
        Prob(rng, 2, 3, 60, 100, bw=[[0.0, 0.3], [0.3, 0.3], [0.2, 0.4]]),  # degenerate bandwidth
        Prob(rng, 4, 4, 100, 100, weights=True),
        Prob(rng, 1, 2, 500, 3000, weights=True),
    ]
    return P


def run_batch(P, T, ae, streams=None, seeds=None):
    U = G = None
    if streams is not None:
        U, G = [s[0] for s in streams], [s[1] for s in streams]
    masks = [p.mask for p in P] if any(p.mask is not None for p in P) else None
    return K.prodAppxMSGibbsS_batch([p.trees for p in P], [p.Np for p in P], Niter=T, addEntropy=ae,
                                    partialDimMasks=masks, randU=U, randN=G, seeds=seeds)


def check_against_single(P, out, T, ae, streams=None, seeds=None, degenerate=()):
    for i, p in enumerate(P):
        U, G = streams[i] if streams is not None else (None, None)
        s = None if seeds is None else seeds[i]
        bp, bi = out[i]
        assert bp.shape == (p.d, p.Np) and bi.shape == (len(p.trees), p.Np)
        if i in degenerate:
            with np.errstate(all="ignore"):
                dp, di = p.single(T, ae, U, G, s)
            assert np.array_equal(bi, di), i
            assert np.array_equal(bits(bp), bits(dp)), i
            continue
        with route("k1"):
            kp, ki = p.single(T, ae, U, G, s)
        assert np.array_equal(bi, ki), "problem %d: labels differ from K1" % i
        assert np.array_equal(bits(bp), bits(kp)), "problem %d: points differ from K1" % i
        dp, di = p.single(T, ae, U, G, s)
        assert np.array_equal(bi, di), "problem %d: labels differ from the default routing" % i
        assert close(bp, dp), "problem %d: points differ from the default routing" % i


@pytest.mark.parametrize("T,ae", [(5, True), (0, False)])
def test_heterogeneous_batch_with_injected_streams(T, ae):
    rng = np.random.default_rng(11 + T)
    P = heterogeneous(rng)
    streams = [p.streams(rng, T) for p in P]
    with np.errstate(all="ignore"):
        out = run_batch(P, T, ae, streams)
    check_against_single(P, out, T, ae, streams, degenerate=(14,))
    for i, p in enumerate(P):
        if p.otrees:
            U, G = streams[i]
            epts, eind = O.gibbs(p.otrees, p.Np, T, U, G, add_entropy=ae,
                                 mask=None if p.mask is None else p.mask)
            assert np.array_equal(out[i][1], eind), i
            assert close(out[i][0], epts), i


def test_philox_batch_with_distinct_seeds():
    rng = np.random.default_rng(5)
    P = [Prob(rng, 2, 2, 100, 100), Prob(rng, 3, 4, 80, 129), Prob(rng, 1, 2, 300, 257), Prob(rng, 5, 2, 60, 40),
         Prob(rng, 2, 2, 60, 100, bw=[[0.0, 0.3], [0.3, 0.3]])]
    seeds = [1, 2, 3, 2**63 + 5, 7]
    with np.errstate(all="ignore"):
        out = run_batch(P, 5, True, seeds=seeds)
    check_against_single(P, out, 5, True, seeds=seeds, degenerate=(4,))


def test_composition_invariance():
    rng = np.random.default_rng(8)
    P = [Prob(rng, 2, 2, 100, 100), Prob(rng, 3, 3, 70, 129), Prob(rng, 1, 2, 90, 33)]
    seeds = [10, 11, 12]
    full = run_batch(P, 3, True, seeds=seeds)
    # a batch of one equals the single call
    one = run_batch(P[:1], 3, True, seeds=seeds[:1])
    check_against_single(P[:1], one, 3, True, seeds=seeds[:1])
    # a reversed batch gives reversed blocks
    rev = run_batch(P[::-1], 3, True, seeds=seeds[::-1])
    for a, b in zip(full, rev[::-1]):
        assert np.array_equal(bits(a[0]), bits(b[0])) and np.array_equal(a[1], b[1])
    # the same problem twice gives identical blocks; one handle shared by several problems
    twice = run_batch([P[1], P[1]], 3, True, seeds=[11, 11])
    assert np.array_equal(bits(twice[0][0]), bits(twice[1][0])) and np.array_equal(twice[0][1], twice[1][1])
    assert np.array_equal(bits(twice[0][0]), bits(full[1][0]))
    t = P[0].trees[0]
    shared = [Prob.__new__(Prob) for _ in range(3)]
    for k, s in enumerate(shared):
        s.d, s.Np, s.mask, s.otrees = 2, 50 + k, None, []
        s.trees = [t, P[0].trees[1]] if k != 1 else [t, t, P[0].trees[1]]
    outs = run_batch(shared, 3, True, seeds=[1, 2, 3])
    check_against_single(shared, outs, 3, True, seeds=[1, 2, 3])
    # a mix of injected and Philox problems
    streams = [P[0].streams(rng, 3), (None, None), P[2].streams(rng, 3)]
    mix = K.prodAppxMSGibbsS_batch([p.trees for p in P], [p.Np for p in P], Niter=3, randU=[s[0] for s in streams],
                                   randN=[s[1] for s in streams], seeds=seeds)
    for i, p in enumerate(P):
        U, G = streams[i]
        with route("k1"):
            kp, ki = p.single(3, True, U, G, seeds[i])
        assert np.array_equal(mix[i][1], ki) and np.array_equal(bits(mix[i][0]), bits(kp)), i
    # the FP32 statistical mode does not apply to batches
    K.set_gibbs_precision(K.F32)
    try:
        f32 = run_batch(P, 3, True, seeds=seeds)
    finally:
        K.set_gibbs_precision(K.F64)
    for a, b in zip(full, f32):
        assert np.array_equal(bits(a[0]), bits(b[0])) and np.array_equal(a[1], b[1])


def test_many_c1_problems_ragged_blocks():
    rng = np.random.default_rng(1024)
    base = [Prob(rng, 2, 2, 100, 101) for _ in range(64)]
    P = [base[i % 64] for i in range(1024)]
    seeds = list(range(1000, 2024))
    out = run_batch(P, 5, True, seeds=seeds)
    assert all(np.isfinite(o[0]).all() and (o[1] >= 1).all() for o in out)
    for i in range(0, 1024, 32):
        with route("k1"):
            kp, ki = P[i].single(5, True, seed=seeds[i])
        assert np.array_equal(out[i][1], ki) and np.array_equal(bits(out[i][0]), bits(kp)), i
    # same trees, different seeds => different samples
    assert not np.array_equal(out[0][0], out[64][0])


def product_single(p, seed):
    d, M = p.d, len(p.trees)
    pts, ind, bw, nl = np.zeros(d * p.Np), np.zeros(M * p.Np, dtype=np.int64), np.zeros(d), (C.c_int * d)()
    _lib.check(_lib.lib().kdeb200_product_kde(K.api._handles(p.trees), M, p.Np, 5, 1, None, seed, _lib.fptr(pts),
                                              _lib.iptr(ind), _lib.fptr(bw), nl))
    return pts, ind, bw, np.array(nl[:])


def product_batch(P, seeds):
    n = len(P)
    ndens = np.array([len(p.trees) for p in P], dtype=np.int32)
    Np = np.array([p.Np for p in P], dtype=np.int64)
    sd = np.array(seeds, dtype=np.uint64)
    nd = sum(p.d for p in P)
    pts = np.zeros(sum(p.d * p.Np for p in P))
    ind = np.zeros(sum(len(p.trees) * p.Np for p in P), dtype=np.int64)
    bw, nl = np.zeros(nd), (C.c_int * nd)()
    _lib.check(_lib.lib().kdeb200_product_kde_batch(
        n, ndens.ctypes.data_as(C.POINTER(C.c_int)), K.api._handles([t for p in P for t in p.trees]), _lib.iptr(Np), 5, 1,
        None, sd.ctypes.data_as(C.POINTER(C.c_uint64)), _lib.fptr(pts), _lib.iptr(ind), _lib.fptr(bw), nl))
    out, p0, i0, b0 = [], 0, 0, 0
    for p in P:
        M = len(p.trees)
        out.append((pts[p0:p0 + p.d * p.Np], ind[i0:i0 + M * p.Np], bw[b0:b0 + p.d], np.array(nl[b0:b0 + p.d])))
        p0, i0, b0 = p0 + p.d * p.Np, i0 + M * p.Np, b0 + p.d
    return out


def test_product_batch_equals_product_kde():
    rng = np.random.default_rng(3)
    P = [Prob(rng, 2, 2, 100, 100), Prob(rng, 3, 6, 100, 100), Prob(rng, 1, 3, 50, 2), Prob(rng, 2, 2, 300, 512),
         Prob(rng, 4, 2, 100, 700), Prob(rng, 3, 2, 80, 129, mask=None), Prob(rng, 2, 2, 60, 64, bw=[[0.0, 0.3], [0.3, 0.3]])]
    seeds = [21, 22, 23, 24, 25, 26, 27]
    with np.errstate(all="ignore"):
        out = product_batch(P, seeds)
    for i, p in enumerate(P):
        with route("k1"), np.errstate(all="ignore"):
            ref = product_single(p, seeds[i])
        for a, b in zip(out[i], ref):
            assert np.array_equal(np.asarray(a).view(np.int64) if a.dtype == np.float64 else a,
                                  np.asarray(b).view(np.int64) if b.dtype == np.float64 else b), i
        with np.errstate(all="ignore"):
            dp, di, _, _ = product_single(p, seeds[i])
        assert np.array_equal(out[i][1], di), i
        if i == 6:  # degenerate bandwidths: the verbatim route on both sides, NaN pattern included
            assert np.array_equal(bits(out[i][0]), bits(dp))
        else:
            assert close(out[i][0], dp), i
    # the Python layer: prod_batch against a prod loop, host branches included
    lists = [p.trees for p in P[:5]] + [[P[0].trees[0]]]
    got = K.prod_batch(lists, seeds=seeds[:6])
    for i, ts in enumerate(lists):
        exp = K.prod(ts, seed=seeds[i])
        assert np.array_equal(K.getPoints(got[i]).shape, K.getPoints(exp).shape)
        assert close(K.getPoints(got[i]), K.getPoints(exp)), i
    lone = K.prod_batch([[P[0].trees[0]], P[0].trees], addEntropy=False, seeds=[1, 2])
    assert np.array_equal(K.getPoints(lone[0]), K.getPoints(K.prod([P[0].trees[0]], addEntropy=False)))
    assert close(K.getPoints(lone[1]), K.getPoints(K.prod(P[0].trees, addEntropy=False, seed=2)))


def raw_batch(trees, ndens, Np, T=2, U=None, nU=None, G=None, nN=None, seeds=None, pts=None, ind=None):
    nd = np.array(ndens, dtype=np.int32)
    npa = np.array(Np, dtype=np.int64)
    arr = (_lib.tree_t * max(len(trees), 1))(*trees)
    sd = np.arange(len(ndens), dtype=np.uint64) if seeds is None else seeds
    rc = _lib.lib().kdeb200_gibbs_batch(len(ndens), nd.ctypes.data_as(C.POINTER(C.c_int)), arr, _lib.iptr(npa), T, 1, None,
                                        _lib.fptr(U), _lib.iptr(nU), _lib.fptr(G), _lib.iptr(nN),
                                        None if sd is False else sd.ctypes.data_as(C.POINTER(C.c_uint64)),
                                        None if pts is False else _lib.fptr(pts if pts is not None else np.full(1000, -7.0)),
                                        None if ind is False else _lib.iptr(ind if ind is not None else np.zeros(1000, np.int64)))
    return rc, _lib.lib().kdeb200_last_error().decode()


def test_errors_name_the_problem_and_launch_nothing():
    rng = np.random.default_rng(4)
    a2, b2 = K.kde(mixture(rng, 2, 30), [0.3]), K.kde(mixture(rng, 2, 30), [0.3])
    c3 = K.kde(mixture(rng, 3, 30), [0.3])
    h = lambda t: t._dev(gibbs=True)
    pts = np.full(1000, -7.0)
    rc, msg = raw_batch([h(a2), h(b2), h(a2), h(b2), h(a2), c3._dev(gibbs=True)], [2, 2, 2], [5, 5, 5], pts=pts)
    assert rc == 6 and "problem 2" in msg, msg
    assert (pts == -7.0).all()  # nothing ran
    rc, msg = raw_batch([h(a2), h(b2)], [2, 0], [5, 5])
    assert rc == 3 and "problem 1" in msg, msg
    rc, msg = raw_batch([h(a2)] * 18, [1, 17], [5, 5])
    assert rc == 3 and "problem 1" in msg, msg
    ev = K.kde(mixture(rng, 2, 30), [0.3])
    rc, msg = raw_batch([h(a2), h(b2), ev._dev(gibbs=False)], [2, 1], [5, 5])
    assert rc == 7 and "problem 1" in msg, msg
    _, pu, pn, _ = K.gibbs_sizes([a2, b2], 2)
    U, G = rng.random(2 * 10 * pu), rng.standard_normal(2 * 10 * pn)
    rc, msg = raw_batch([h(a2), h(b2)] * 2, [2, 2], [10, 10], U=U, nU=np.array([10 * pu, 10 * pu - 2], np.int64), G=G,
                        nN=np.array([10 * pn, 10 * pn], np.int64), pts=pts)
    assert rc == 7 and "problem 1" in msg and "randU" in msg, msg
    assert (pts == -7.0).all()
    rc, msg = raw_batch([h(a2), h(b2)], [2], [5], U=U, nU=None, G=G, nN=None)
    assert rc == 2, msg
    rc, msg = raw_batch([h(a2), h(b2)], [2], [5], pts=False)
    assert rc == 2, msg
    rc, msg = raw_batch([h(a2), h(b2)], [2], [5], seeds=False)
    assert rc == 2, msg
    rc = _lib.lib().kdeb200_gibbs_batch(1, None, None, None, 2, 1, None, None, None, None, None, None, None, None)
    assert rc == 2
    rc = _lib.lib().kdeb200_product_kde_batch(1, (C.c_int * 1)(2), (_lib.tree_t * 2)(h(a2), h(b2)),
                                              _lib.iptr(np.array([1], np.int64)), 5, 1, None,
                                              np.zeros(1, np.uint64).ctypes.data_as(C.POINTER(C.c_uint64)),
                                              _lib.fptr(np.zeros(10)), None, _lib.fptr(np.zeros(2)), None)
    assert rc == 3 and "problem 0" in _lib.lib().kdeb200_last_error().decode()
    with pytest.raises(K.KDEError):
        K.prodAppxMSGibbsS_batch([[a2, c3]], [5])


def test_destroyed_trees_then_new_batch():
    rng = np.random.default_rng(6)
    P = [Prob(rng, 2, 2, 100, 100), Prob(rng, 3, 3, 80, 50)]
    run_batch(P, 3, True, seeds=[1, 2])
    for p in P:
        for t in p.trees:
            t._invalidate()
    del P
    Q = [Prob(rng, 2, 2, 120, 100), Prob(rng, 3, 3, 90, 50)]
    out = run_batch(Q, 3, True, seeds=[1, 2])
    check_against_single(Q, out, 3, True, seeds=[1, 2])
