"""-m gpu: many independent sample / rand / resample problems in one call (kdeb200_sample_batch, kdeb200_resample_batch).

Every problem of a batch must equal the single call on its own: points (as bits) and 1-based indices of kdeb200_sample
with the same handle, seed and injected streams, and for resampling the bandwidths, nLOO_LL counts and every tree array
of resample(p, Np, seed=s)."""
import ctypes as C

import numpy as np
import pytest

import kde_b200 as K
from kde_b200 import _lib
from tests.util import mixture, silverman

pytestmark = pytest.mark.gpu

SB_MAX = 2048  # problems up to this size run in the one-CTA-per-problem launch (sample_batch.cu)


@pytest.fixture(autouse=True)
def one_gpu():
    K.init(0)
    yield


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def density(rng, d, N, zeros=False):
    pts = mixture(rng, d, N)
    bw = silverman(pts) if N > 2 else np.full(d, 0.5)
    w = None
    if zeros:
        w = rng.random(N) + 0.01
        w[rng.random(N) < 0.2] = 0.0
        w[-1] = 0.5  # never all zero
    return K.kde(pts, bw, w)


def single(p, n, seed, U=None, G=None):
    """kdeb200_sample alone; U (n uniforms) and G (d x n normals) injected independently"""
    d = K.Ndim(p)
    pts = np.zeros(max(d * n, 1))
    idx = np.zeros(max(n, 1), dtype=np.int64)
    g = None if G is None else np.ascontiguousarray(np.asarray(G, dtype=np.float64).T).ravel()
    u = None if U is None else np.ascontiguousarray(U, dtype=np.float64)
    _lib.check(_lib.lib().kdeb200_sample(p._dev(), n, int(seed) & 0xFFFFFFFFFFFFFFFF, _lib.fptr(u), _lib.fptr(g),
                                         _lib.fptr(pts), _lib.iptr(idx)))
    return pts[:d * n].reshape(n, d).T, idx[:n]


def same(a, b):
    return np.array_equal(bits(a[0]), bits(b[0])) and np.array_equal(a[1], b[1])


def heterogeneous(rng):
    """(density, Np, seed): d = 1..8, N 1..5000 with zero weights, Np on both sides of SB_MAX and ~100k, a shared handle
    with two seeds, Gibbs-upgraded handles, handles whose table an earlier single call built"""
    P = []
    Nps = [0, 1, 2, SB_MAX - 1, SB_MAX, SB_MAX + 1, 100003]
    for j, (d, N) in enumerate([(1, 1), (1, 5000), (2, 2), (2, 700), (3, 129), (3, 4096), (4, 1000), (5, 33), (6, 2500),
                                (7, 64), (8, 5000), (8, 300)]):
        p = density(rng, d, N, zeros=N > 2)
        if j % 3 == 1:
            p._dev(gibbs=True)        # handle upgraded for the sampler
        if j % 4 == 2:
            K.sample(p, 5, seed=9)    # table built by a single call before the batch
        P.append((p, Nps[j % len(Nps)], int(rng.integers(0, 2 ** 63))))
        P.append((p, int(rng.integers(1, 400)), int(rng.integers(0, 2 ** 63))))
    shared = density(rng, 3, 800, zeros=True)
    P += [(shared, 500, 1), (shared, 500, 2), (shared, 3000, 3)]
    return P


def test_heterogeneous_batch_equals_single_calls_bit_for_bit():
    rng = np.random.default_rng(1)
    P = heterogeneous(rng)
    out = K.sample_batch([p for p, _, _ in P], [n for _, n, _ in P], seeds=[s for _, _, s in P])
    assert len(out) == len(P)
    for (p, n, s), got in zip(P, out):
        assert got[0].shape == (K.Ndim(p), n) and got[1].shape == (n,)
        assert same(got, single(p, n, s)), (K.Ndim(p), K.Npts(p), n)
        if n:
            assert same(got, K.sample(p, n, seed=s))
    a, b = out[-3], out[-2]  # one handle, two seeds: different draws
    assert not np.array_equal(a[1], b[1])
    ms, launches = K.last_kernel_ms()
    assert ms > 0 and launches >= 1


def test_injected_streams_equal_single_calls_and_reference_scan():
    rng = np.random.default_rng(2)
    P, U, G, ref = [], [], [], []
    shapes = [(1, 40, 17, "UN"), (2, 300, 300, "U"), (3, 500, 2048, "N"), (3, 500, 4000, ""), (4, 100, 1, "UN"),
              (5, 1000, 777, "U"), (8, 64, 2049, "N"), (2, 3, 50, "UN"), (3, 500, 3000, "U"), (2, 200, 2500, "UN"),
              (6, 90, 120, "")]
    for j, (d, N, n, mode) in enumerate(shapes):
        p = density(rng, d, N, zeros=N > 3)
        u = rng.random(n)
        if j == 7:  # ties and signed zeros: both sorts are stable with the same key order
            u[:10] = 0.0
            u[10:20] = -0.0
            u[20:30] = 0.5
        g = rng.standard_normal((d, n))
        uu = u if "U" in mode else None
        gg = g if "N" in mode else None
        s = int(rng.integers(0, 2 ** 63))
        P.append((p, n, s))
        U.append(uu)
        G.append(gg)
        ref.append(single(p, n, s, uu, gg))
    out = K.sample_batch([p for p, _, _ in P], [n for _, n, _ in P], seeds=[s for _, _, s in P], randU=U, randN=G)
    for a, b in zip(out, ref):
        assert same(a, b)
    # problem 0 (both injected) is the reference's scan (src/KDE01.jl:164-183) restated in numpy
    p, n, _ = P[0]
    got, idx = out[0]
    cw = np.cumsum(K.getWeights(p))
    cw = cw / cw[-1]
    t = np.concatenate([np.sort(U[0]), [10.0]])
    ref_pts, ref_idx, ii = np.zeros((K.Ndim(p), n)), np.zeros(n, dtype=np.int64), 0
    X, B = K.getPoints(p), K.getBW(p)
    for i in range(K.Npts(p)):
        while cw[i] > t[ii]:
            ref_pts[:, ii] = X[:, i] + B[:, i] * G[0][:, ii]
            ref_idx[ii] = i + 1
            ii += 1
    assert ii == n and np.array_equal(idx, ref_idx) and np.max(np.abs(got - ref_pts)) < 1e-14
    # a fully injected problem does not read its seed
    out2 = K.sample_batch([P[0][0]], [P[0][1]], randU=[U[0]], randN=[G[0]])
    assert same(out2[0], out[0])


def test_composition_invariance_1024_problems():
    rng = np.random.default_rng(3)
    pool = [density(rng, 1 + b % 4, int(rng.integers(50, 400)), zeros=b % 2 == 0) for b in range(64)]
    dens = [pool[i % 64] for i in range(1024)]
    Np = [int(x) for x in rng.integers(0, 300, size=1024)]
    seeds = [int(x) for x in rng.integers(0, 2 ** 63, size=1024)]
    base = K.sample_batch(dens, Np, seeds=seeds)
    for rep in range(2):
        perm = rng.permutation(1024)
        sh = K.sample_batch([dens[i] for i in perm], [Np[i] for i in perm], seeds=[seeds[i] for i in perm])
        for k, i in enumerate(perm):
            assert same(sh[k], base[i])
    for i in range(0, 1024, 7):
        assert same(K.sample_batch([dens[i]], [Np[i]], seeds=[seeds[i]])[0], base[i])


def _raw_resample(dens, Np, seeds):
    n = len(dens)
    h = (_lib.tree_t * max(n, 1))(*[p._dev() for p in dens])
    Na = np.array(Np, dtype=np.int64)
    sd = np.array(seeds, dtype=np.uint64)
    nd = sum(K.Ndim(p) for p in dens)
    pts = np.zeros(int(sum(K.Ndim(p) * m for p, m in zip(dens, Np))) + 1)
    idx = np.zeros(int(Na.sum()) + 1, dtype=np.int64)
    bw = np.zeros(nd + 1)
    calls = np.zeros(nd + 1, dtype=np.int32)
    _lib.check(_lib.lib().kdeb200_resample_batch(n, h, _lib.iptr(Na), sd.ctypes.data_as(C.POINTER(C.c_uint64)), None,
                                                 None, None, None, _lib.fptr(pts), _lib.iptr(idx), _lib.fptr(bw),
                                                 calls.ctypes.data_as(C.POINTER(C.c_int))))
    res, p0, i0, b0 = [], 0, 0, 0
    for p, m in zip(dens, Np):
        d = K.Ndim(p)
        res.append((pts[p0:p0 + d * m].reshape(m, d).T, idx[i0:i0 + m], bw[b0:b0 + d], [int(c) for c in calls[b0:b0 + d]]))
        p0, i0, b0 = p0 + d * m, i0 + m, b0 + d
    return res


def test_resample_batch_equals_resample_loop():
    rng = np.random.default_rng(4)
    dens, Np, seeds = [], [], []
    for d in range(1, 9):
        for n in (2, 3, 511, 512, 513, 2000):
            dens.append(density(rng, d, int(rng.integers(100, 300)), zeros=d % 2 == 0))
            Np.append(n)
            seeds.append(int(rng.integers(0, 2 ** 63)))
    raw = _raw_resample(dens, Np, seeds)
    for p, n, s, (pts, idx, bw, calls) in zip(dens, Np, seeds, raw):
        rp, ri = single(p, n, s)
        assert np.array_equal(bits(pts), bits(rp)) and np.array_equal(idx, ri)
        c = []
        ref_bw = K.lcv_bandwidths(rp, _count=c)
        assert np.array_equal(bits(bw), bits(ref_bw)) and calls == c, (K.Ndim(p), n)
    out = K.resample_batch(dens, Np, seeds=seeds)
    for p, n, s, a in zip(dens, Np, seeds, out):
        b = K.resample(p, n, seed=s)
        for k in ("centers", "ranges", "weights", "left_child", "right_child", "lowest_leaf", "highest_leaf", "permutation"):
            assert np.array_equal(getattr(a.bt, k), getattr(b.bt, k)), k
        for k in ("means", "bandwidth", "bandwidthMin", "bandwidthMax"):
            assert np.array_equal(bits(getattr(a, k)), bits(getattr(b, k))), k
    # Np = None: every density's own Npts
    small = dens[:4]
    for a, p, s in zip(K.resample_batch(small, seeds=seeds[:4]), small, seeds[:4]):
        assert np.array_equal(bits(a.bandwidth), bits(K.resample(p, seed=s).bandwidth))
    with pytest.raises(K.KDEError):
        K.resample_batch(small, ksType=":discrete")
    assert K.resample_batch([]) == [] and K.sample_batch([], []) == []


def _err():
    return _lib.lib().kdeb200_last_error().decode()


def test_errors_name_the_problem_and_run_nothing():
    rng = np.random.default_rng(5)
    good = [density(rng, 2, 100) for _ in range(3)]
    fresh = density(rng, 2, 120)  # a valid neighbour whose table the failing calls must not build
    L = _lib.lib()
    sentinel = -7.25

    def call(dens, Np, nU=None, nN=None, U=None, G=None, seeds=True, resample=False, null_out=False):
        n = len(dens)
        h = (_lib.tree_t * max(n, 1))(*[None if p is None else p._dev() for p in dens])
        Na = np.array(Np, dtype=np.int64)
        sd = np.arange(1, n + 1, dtype=np.uint64)
        sp = sd.ctypes.data_as(C.POINTER(C.c_uint64)) if seeds else None
        nUa = None if nU is None else np.array(nU, dtype=np.int64)
        nNa = None if nN is None else np.array(nN, dtype=np.int64)
        pts = np.full(4096, sentinel)
        idx = np.full(2048, -3, dtype=np.int64)
        bw = np.full(64, sentinel)
        po = None if null_out else _lib.fptr(pts)
        if resample:
            rc = L.kdeb200_resample_batch(n, h, _lib.iptr(Na), sp, _lib.fptr(U), _lib.iptr(nUa), _lib.fptr(G),
                                          _lib.iptr(nNa), po, _lib.iptr(idx), _lib.fptr(bw), None)
        else:
            rc = L.kdeb200_sample_batch(n, h, _lib.iptr(Na), sp, _lib.fptr(U), _lib.iptr(nUa), _lib.fptr(G),
                                        _lib.iptr(nNa), po, _lib.iptr(idx))
        assert np.all(pts == sentinel) and np.all(idx == -3) and np.all(bw == sentinel)
        return rc

    K.sample(good[0], 10, seed=1)
    before = K.last_kernel_ms()
    # NULL handle / output: code 2
    assert call([good[0], fresh, None], [10, 10, 10]) == 2 and "problem 2" in _err()
    assert call([good[0], fresh], [10, 10], null_out=True) == 2
    # Np out of range: code 3
    assert call([fresh, good[1]], [10, -1]) == 3 and "problem 1" in _err()
    assert call([fresh, good[1]], [10, 2 ** 31]) == 3 and "problem 1" in _err()
    # negative / NaN bandwidth variance: code 5, as the single call
    bad = K.kde(mixture(rng, 2, 50), [np.nan, 0.3])
    with pytest.raises(K.KDEError):
        K.sample(bad, 10, seed=1)
    assert call([fresh, good[0], bad], [10, 10, 10]) == 5 and "problem 2" in _err()
    # stream lengths neither 0 nor the full length: code 7
    U = np.zeros(64)
    assert call([fresh, good[0]], [10, 10], nU=[10, 9], nN=[0, 0], U=U, G=U) == 7 and "problem 1" in _err()
    assert call([fresh, good[0]], [10, 10], nU=[0, 0], nN=[20, 10], U=U, G=U) == 7 and "problem 1" in _err()
    # Philox problems need seeds
    assert call([fresh, good[0]], [10, 10], seeds=False) == 2
    # resample: fewer than two samples, code 3 (what kde! of fewer than two samples gives)
    assert call([fresh, good[1]], [10, 1], resample=True) == 3 and "problem 1" in _err()
    assert call([fresh, good[1]], [10, 0], resample=True) == 3 and "problem 1" in _err()
    assert K.last_kernel_ms() == before  # nothing ran
    # Python rejects length mismatches before the call
    with pytest.raises(K.KDEError):
        K.sample_batch(good, [10, 10])
    with pytest.raises(K.KDEError):
        K.sample_batch(good, [10] * 3, seeds=[1, 2])
    with pytest.raises(K.KDEError):
        K.sample_batch(good, [10] * 3, randU=[None, None])
    # and the batch still works afterwards, equal to the single calls
    out = K.sample_batch(good + [fresh], [10, 20, 30, 40], seeds=[1, 2, 3, 4])
    for p, n, s, o in zip(good + [fresh], [10, 20, 30, 40], [1, 2, 3, 4], out):
        assert same(o, single(p, n, s))


def test_lifetime_and_init_multi():
    rng = np.random.default_rng(6)
    dens = [density(rng, 1 + i % 3, 150, zeros=True) for i in range(8)]
    Np, seeds = [100, 3000, 150, 2, 512, 600, 1, 0], list(range(8))
    K.sample_batch(dens, Np, seeds=seeds)
    for p in dens:
        p._invalidate()  # destroys the handles (and their tables)
    dens2 = [density(rng, 1 + i % 3, 150, zeros=True) for i in range(8)]
    ref = [single(p, n, s) for p, n, s in zip(dens2, Np, seeds)]
    assert all(same(a, b) for a, b in zip(K.sample_batch(dens2, Np, seeds=seeds), ref))
    rNp = [100, 300, 512, 2, 50, 7, 3, 400]
    ref_r = _raw_resample(dens2, rNp, seeds)
    try:
        assert K.init_multi(devices=[0, 0]) == 2
        out = K.sample_batch(dens2, Np, seeds=seeds)
        out_r = _raw_resample(dens2, rNp, seeds)
    finally:
        assert K.init_multi(1) == 1
    assert all(same(a, b) for a, b in zip(out, ref))
    for a, b in zip(out_r, ref_r):
        assert np.array_equal(bits(a[0]), bits(b[0])) and np.array_equal(a[1], b[1])
        assert np.array_equal(bits(a[2]), bits(b[2])) and a[3] == b[3]
