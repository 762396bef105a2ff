"""Host-side mirror of KernelDensityEstimate.jl's public API for the accelerated path.

The reference's host language is Julia, which is not installed in this image (INTEGRATION.md
carries the Julia `ccall` binding).  This module is the same thin host layer in Python: same
names, argument meaning and error behaviour as the reference functions it cites, every
data-parallel step delegated to libkdeb200.so through the C-ABI (include/kdeb200.h).  Scalar
control that the reference keeps on the host (golden-section search, argument defaults) stays on
the host here too.  Nothing in this file computes a kernel sum or runs a Gibbs chain on the CPU.

Reference map (paths relative to the reference repo):
  kde / kde_bang            src/KDE01.jl:3-84          getPoints/getBW/getWeights  src/KDE01.jl:91-136
  marginal                  src/KDE01.jl:143-153       sample / rand               src/KDE01.jl:164-198
  resample                  src/BallTreeDensity01.jl:312-334
  evaluateDualTree, bd(pos) src/DualTree01.jl:370-446  evalAvgLogL / entropy       src/DualTree01.jl:450-508
  kld / minkld              src/DualTree01.jl:477-510
  nLOO_LL / golden / ksize / neighborMinMax / updateBandwidth   src/CrossValidation.jl:5-120
  prodAppxMSGibbsS / *      src/MSGibbs01.jl:645-736
"""
import ctypes as C
import math
import os

import numpy as np

from . import _lib
from ._lib import KDEError, check, fptr, iptr, lib

__all__ = [
    "KDEError", "BallTree", "BallTreeDensity", "kde", "kde_bang", "getPoints", "getBW", "getWeights", "marginal",
    "sample", "rand", "resample", "sample_batch", "rand_batch", "resample_batch", "evaluateDualTree", "evaluateDualTree_batch", "kde_batch", "lcv_bandwidths_batch", "evalAvgLogL", "entropy", "kld", "minkld", "nLOO_LL", "golden",
    "ksize", "neighborMinMax", "lcv_bandwidths", "updateBandwidth", "prodAppxMSGibbsS", "prodAppxMSGibbsS_batch", "prod_batch", "gibbs_batch_split", "Ndim", "Npts", "init", "init_multi", "multi_count", "gibbs_sizes",
    "philox_streams", "pipe_peak", "last_kernel_ms", "F64", "F32", "F64_BOUNDED", "F32_BOUNDED", "setForceEvalDirect", "set_pruning", "set_gibbs_precision", "gibbs_f32_slow_draws", "gibbs_exact_redone", "gibbs_exact_redone_internal", "gibbs_exact_redone_b", "gibbs_exact_tier3", "pruned_stats", "prod", "getKDERange", "getKDERangeLinspace",
    "getKDEMax", "getKDEMean", "getKDEfit", "intersIntgAppxIS", "eval_marginals", "to_string", "from_string",
]

F64, F32, F64_BOUNDED, F32_BOUNDED = 0, 1, 2, 3
_EUCLID = ("+", "-")


def init(device=0):
    """Bind this process to one GPU (one process per GPU)."""
    check(lib().kdeb200_init(int(device)))


def init_multi(ngpus=0, devices=None):
    """In-process multi-GPU (kdeb200_init_multi): afterwards prodAppxMSGibbsS, evaluateDualTree, entropy and
    kde(points) shard their samples / query points / leaf rows over `ngpus` devices of this process (0 = all visible).
    devices = explicit list (devices[0] = primary; repeats allowed, see include/kdeb200.h).  Returns the set's size."""
    if devices is not None:
        arr = (C.c_int * len(devices))(*[int(x) for x in devices])
        check(lib().kdeb200_init_multi_devices(arr, len(devices)))
    else:
        check(lib().kdeb200_init_multi(int(ngpus)))
    return multi_count()


def multi_count():
    n = C.c_int(0)
    check(lib().kdeb200_multi_count(C.byref(n)))
    return n.value


def setForceEvalDirect(flag):
    """setForceEvalDirect!(flag) (src/DualTree01.jl:3-9).  True (the reference's default): evaluateDualTree is the
    brute-force sum.  False: the reference switches to its dual-tree recursion (errTol = 1e-3); here the
    error-bounded tile-pruned kernel (kdeb200_set_pruning(2): every value within 1e-13 of brute force)."""
    check(lib().kdeb200_set_pruning(1 if flag else 2))


def set_pruning(mode):
    """kdeb200_set_pruning: 0 brute force everywhere, 1 (default) pruned LOO likelihood only, 2 pruned evaluations too."""
    check(lib().kdeb200_set_pruning(int(mode)))


def set_gibbs_precision(precision):
    """kdeb200_set_gibbs_precision: F64 (default, parity mode: labels exact under injected variates) or F32 (statistical
    mode only: label probabilities in packed FP32 on calls large enough for the thread-per-chain kernel)."""
    check(lib().kdeb200_set_gibbs_precision(int(precision)))


def gibbs_f32_slow_draws():
    """label draws the FP32 sampler redid in FP64 (its FP32 total under/overflowed) since the last call"""
    n = C.c_ulonglong(0)
    check(lib().kdeb200_gibbs_f32_slow_draws(C.byref(n)))
    return int(n.value)


def gibbs_exact_redone():
    """(lane-draws, warp-draws) of the FP64 sampler whose leaf-level label the certified FP32 bound could not decide and
    that were redone in FP64, since the last call"""
    n, w = C.c_ulonglong(0), C.c_ulonglong(0)
    check(lib().kdeb200_gibbs_exact_redone(C.byref(n), C.byref(w)))
    return int(n.value), int(w.value)


def gibbs_exact_redone_internal():
    """(lane-draws, warp-draws) of the FP64 sampler whose sampleIndex label on an internal level (any size) the certified
    FP32 bound could not decide and that were redone in FP64, since the last call"""
    n, w = C.c_ulonglong(0), C.c_ulonglong(0)
    check(lib().kdeb200_gibbs_exact_redone_internal(C.byref(n), C.byref(w)))
    return int(n.value), int(w.value)


def gibbs_exact_redone_b():
    """(lane-draws, warp-draws) of the FP64 sampler whose sampleIndices! label on an internal level the certified FP32
    bound could not decide and that were redone in FP64, since the last call"""
    n, w = C.c_ulonglong(0), C.c_ulonglong(0)
    check(lib().kdeb200_gibbs_exact_redone_b(C.byref(n), C.byref(w)))
    return int(n.value), int(w.value)


def gibbs_exact_tier3():
    """(lane-draws, warp-draws) of the FP64 sampler, any class, that were redone in FP64 and that the warp-parallel FP64
    sums could not decide either, so that they were summed serially in node order, since the last call"""
    n, w = C.c_ulonglong(0), C.c_ulonglong(0)
    check(lib().kdeb200_gibbs_exact_tier3(C.byref(n), C.byref(w)))
    return int(n.value), int(w.value)


def _gibbs_exact_bound_probe(trees, Niter, density, level, mu, cadd, pass0=False):
    """tests: per query conditional (rows of mu, cadd) the header and per-node table of kdeb200_gibbs_exact_bound_probe,
    as (headers [nq, 8], nodes [nq, n, 8]); pass0 probes an internal level's sampleIndices! draw (cadd unused)"""
    mu = np.ascontiguousarray(mu, dtype=np.float64)
    cadd = np.ascontiguousarray(cadd, dtype=np.float64)
    nq = mu.shape[0]
    n = max(Npts(t) for t in trees)
    out = np.zeros(nq * (8 + 8 * n))
    check(lib().kdeb200_gibbs_exact_bound_probe(_handles(trees), len(trees), int(Niter), int(density), int(level),
                                                int(bool(pass0)), fptr(mu), fptr(cadd), nq, fptr(out), out.size))
    n = int(out[5])
    per = 8 + 8 * n
    out = out[:nq * per].reshape(nq, per)
    return out[:, :8], out[:, 8:].reshape(nq, n, 8)


def pruned_stats():
    """(fraction of (query block, component tile) pairs the last pruned call kept, rows it recomputed exactly)"""
    f, r = C.c_double(0), C.c_int64(0)
    check(lib().kdeb200_pruned_stats(C.byref(f), C.byref(r)))
    return f.value, r.value


def _require_euclidean(**ops):
    # the reference threads per-dimension addop/diffop/getMu/getLambda closures through every call;
    # closures cannot cross a C-ABI and the north star forbids a CPU fallback => explicit error.
    for name, v in ops.items():
        if v is not None:
            raise KDEError("%s: only the default Euclidean (+,-) manifold is supported on the B200 path" % name)


class BallTree:
    """Field-for-field mirror of `mutable struct BallTree` (src/BallTree01.jl:10-28), 1-based ids."""

    def __init__(self, dims, num_points):
        n2 = 2 * num_points
        self.dims = int(dims)
        self.num_points = int(num_points)
        self.centers = np.zeros(n2 * dims)
        self.ranges = np.zeros(n2 * dims)
        self.weights = np.zeros(n2)
        self.left_child = np.ones(n2, dtype=np.int64)
        self.right_child = np.ones(n2, dtype=np.int64)
        self.lowest_leaf = np.ones(n2, dtype=np.int64)
        self.highest_leaf = np.ones(n2, dtype=np.int64)
        self.permutation = np.zeros(n2, dtype=np.int64)


class BallTreeDensity:
    """Mirror of `mutable struct BallTreeDensity` (src/BallTreeDensity01.jl:11-24) plus a lazily
    created device handle (kdeb200_tree_create)."""

    def __init__(self, bt, means, bandwidth):
        N, d = bt.num_points, bt.dims
        self.bt = bt
        self.multibandwidth = 0
        self.means = means
        self.bandwidth = bandwidth
        self.bandwidthMin = bandwidth[N * d:].copy()
        self.bandwidthMax = bandwidth[N * d:].copy()
        self._handle = None
        self._handle_gibbs = False
        self._bw_dirty = False  # host bandwidth changed since the device records were built

    # -- device residency --------------------------------------------------------------
    def _dev(self, gibbs=False, stale_bw_ok=False):
        """Device handle; evaluation / LOOCV callers get the leaf-only hand-over
        (kdeb200_tree_create_eval), the first Gibbs use upgrades it to the full level records.
        A handle whose bandwidth records predate an updateBandwidth! is rebuilt, unless the caller
        passes the current variances with the call itself (stale_bw_ok: entropy / nLOO_LL)."""
        if self._handle is not None and gibbs and not self._handle_gibbs:
            self._invalidate()
        if self._handle is not None and self._bw_dirty and not stale_bw_ok:
            self._invalidate()
        if self._handle is None:
            h = _lib.tree_t()
            bt = self.bt
            if gibbs:
                check(lib().kdeb200_tree_create(bt.dims, bt.num_points, fptr(self.means), fptr(self.bandwidth),
                                                fptr(bt.weights), iptr(bt.left_child), iptr(bt.right_child),
                                                iptr(bt.permutation), C.byref(h)))
            else:
                check(lib().kdeb200_tree_create_eval(bt.dims, bt.num_points, fptr(self.means),
                                                     fptr(self.bandwidth), fptr(bt.weights),
                                                     iptr(bt.permutation), C.byref(h)))
            self._handle = h
            self._handle_gibbs = gibbs
            self._bw_dirty = False
        return self._handle

    def _invalidate(self):
        if self._handle is not None:
            try:
                lib().kdeb200_tree_destroy(self._handle)
            except Exception:
                pass
            self._handle = None

    def __del__(self):
        self._invalidate()

    # -- functor: bd(pos) (src/DualTree01.jl:431-446) ----------------------------------------
    def __call__(self, pos, lvFlag=False, errTol=1e-3, addop=None, diffop=None):
        pos = np.asarray(pos, dtype=np.float64)
        if pos.ndim == 1:  # one d-dimensional point, reshape(pos, :, 1)
            pos = pos.reshape(-1, 1)
        return evaluateDualTree(self, pos, lvFlag, errTol, addop, diffop)

    def __mul__(self, other):
        return prod([self, other])

    def __repr__(self):  # Base.show (src/KDE01.jl:202-210)
        return "BallTreeDensity:\n  dims: %d\n  Npts: %d\n  bws:  %s\n" % (
            Ndim(self), Npts(self), np.round(getBW(self)[:, 0], 6).tolist())


def Ndim(bd):
    return bd.bt.dims


def Npts(bd):
    return bd.bt.num_points


# ------------------------------------------------------------------------- construction ----
def _as_matrix(points):
    p = np.asarray(points, dtype=np.float64)
    if p.ndim == 1:
        p = p.reshape(1, -1)
    if p.ndim != 2:
        raise KDEError("points must be a d x N matrix or a vector")
    return p


def _make_ball_tree_density(points, weights, bwvar):
    """makeBallTreeDensity (src/BallTreeDensity01.jl:192-231) via the library's host builder."""
    d, N = points.shape
    pts = np.ascontiguousarray(points.T).ravel()  # column-major d x N
    bt = BallTree(d, N)
    means = np.zeros(2 * N * d)
    bandwidth = np.zeros(2 * N * d)
    w = np.ascontiguousarray(weights, dtype=np.float64)
    bv = np.ascontiguousarray(bwvar, dtype=np.float64)
    check(lib().kdeb200_tree_build_host(d, N, fptr(pts), fptr(w), fptr(bv), fptr(bt.centers), fptr(bt.ranges),
                                        fptr(bt.weights), fptr(means), fptr(bandwidth), iptr(bt.left_child),
                                        iptr(bt.right_child), iptr(bt.lowest_leaf), iptr(bt.highest_leaf),
                                        iptr(bt.permutation)))
    return BallTreeDensity(bt, means, bandwidth)


def lcv_bandwidths(points, _count=None):
    """The bandwidth loop of kde!(points) (src/KDE01.jl:13-23) behind ONE library call
    (kdeb200_kde_lcv): per dimension marginal -> ksize -> golden over nLOO_LL, entirely native;
    N <= 512 runs all golden-section searches in a single kernel launch.  Returns the d standard
    deviations.  Bit-identical to the step-by-step mirror `kde(points, native_lcv=False)`."""
    pts = _as_matrix(points)
    d, N = pts.shape
    flat = np.ascontiguousarray(pts.T).ravel()
    bw = np.zeros(d)
    calls = (C.c_int * d)()
    check(lib().kdeb200_kde_lcv(d, N, fptr(flat), fptr(bw), calls))
    if _count is not None:
        _count.extend(int(c) for c in calls)
    return bw


def lcv_bandwidths_batch(point_sets, _count=None):
    """[lcv_bandwidths(p) for p in point_sets] in one library call (kdeb200_kde_lcv_batch): every set of at most 512
    points in one kernel launch, larger sets by the bandwidth loop one after the other.  Returns a list of arrays of d_i
    standard deviations, bit for bit those of lcv_bandwidths; _count, if given, receives one list of nLOO_LL call counts
    per set."""
    sets = [_as_matrix(p) for p in point_sets]
    n = len(sets)
    d = np.array([p.shape[0] for p in sets], dtype=np.int32)
    N = np.array([p.shape[1] for p in sets], dtype=np.int64)
    flat = np.concatenate([np.ascontiguousarray(p.T).ravel() for p in sets] + [np.zeros(1)])
    nb = int(d.sum())
    bw = np.zeros(nb + 1)
    calls = np.zeros(nb + 1, dtype=np.int32)
    check(lib().kdeb200_kde_lcv_batch(n, d.ctypes.data_as(C.POINTER(C.c_int)), iptr(N), fptr(flat), fptr(bw),
                                      calls.ctypes.data_as(C.POINTER(C.c_int))))
    res, b0 = [], 0
    for k in d:
        res.append(bw[b0:b0 + int(k)].copy())
        if _count is not None:
            _count.append([int(c) for c in calls[b0:b0 + int(k)]])
        b0 += int(k)
    return res


def kde_batch(point_sets):
    """[kde(p) for p in point_sets]: the leave-one-out bandwidths of all sets from one library call
    (lcv_bandwidths_batch), then each density built on the host as kde(p) builds it.  Equal bandwidths and identical
    tree arrays."""
    sets = [_as_matrix(p) for p in point_sets]
    return [kde(p, bw) for p, bw in zip(sets, lcv_bandwidths_batch(sets))]


def kde(points, ks=None, weights=None, addop=None, diffop=None, native_lcv=True):
    """kde!(points) / kde!(points, ks) / kde!(points, ks, weights)  (src/KDE01.jl:3-84).

    ks = None selects every dimension's bandwidth by leave-one-out likelihood cross validation
    (the per-dimension `ksize(marginal(p,[i]))` loop of src/KDE01.jl:17-23): in one native call
    (lcv_bandwidths) or, with native_lcv=False, step by step through the mirrors of marginal /
    ksize / golden / nLOO_LL (one kdeb200_loo_entropy call per golden-section step)."""
    _require_euclidean(addop=addop, diffop=diffop)
    pts = _as_matrix(points)
    d, N = pts.shape
    if ks is None:
        if native_lcv:
            return kde(pts, lcv_bandwidths(pts))
        p = kde(pts, [1.0])
        bwds = np.zeros(d)
        for i in range(d):
            pp = ksize(marginal(p, [i + 1]))
            bwds[i] = getBW(pp)[0, 0]
        return kde(pts, bwds)
    ks = np.atleast_1d(np.asarray(ks, dtype=np.float64)).ravel()
    if ks.size == 1:
        ks = np.repeat(ks, d)
    if ks.size != d:
        raise KDEError("kde!: bandwidth vector must have 1 or %d entries" % d)
    w = np.ones(N) if weights is None else np.asarray(weights, dtype=np.float64).ravel()
    if w.size != N:
        raise KDEError("kde!: need one weight per point")
    ssum = float(np.cumsum(w)[-1])  # sequential sum(weights)
    return _make_ball_tree_density(pts, w / ssum, ks ** 2)


kde_bang = kde  # `kde!`


def getPoints(bd, idx=None):
    """src/KDE01.jl:91-101"""
    N, d = bd.bt.num_points, bd.bt.dims
    perm = bd.bt.permutation[N:] - 1
    res = bd.bt.centers[d * N:].reshape(N, d).T
    pts = np.zeros((d, N))
    pts[:, perm] = res
    return pts if idx is None else pts[:, np.asarray(idx) - 1]


def getBW(bd, ind=None):
    """src/KDE01.jl:109-120 (standard deviations)"""
    N, d = bd.bt.num_points, bd.bt.dims
    perm = bd.bt.permutation[N:] - 1
    s = np.zeros((d, N))
    s[:, perm] = bd.bandwidth[d * N:].reshape(N, d).T
    if ind is not None and len(ind) > 0:
        s = s[:, np.asarray(ind) - 1]
    return np.sqrt(s)


def getWeights(bd, ind=None):
    """src/KDE01.jl:127-136"""
    N = bd.bt.num_points
    perm = bd.bt.permutation[N:] - 1
    wts = np.zeros(N)
    wts[perm] = bd.bt.weights[N:]
    if ind is not None and len(ind) > 0:
        wts = wts[np.asarray(ind) - 1]
    return wts


def marginal(bd, ind):
    """src/KDE01.jl:143-153 (ind is 1-based like the reference)"""
    ind = np.asarray(ind, dtype=np.int64)
    pts = getPoints(bd)
    sig = getBW(bd, [1])
    wts = getWeights(bd)
    return kde(pts[ind - 1, :], sig[ind - 1, 0], wts)


def sample(npd, Npts_, ind=None, rng=None, seed=None):
    """sample(npd, Npts[, ind]) (src/KDE01.jl:164-189) on the device (kdeb200_sample): inverse-CDF component draw from
    sorted uniforms over the cumulative weights in original point order + the kernel perturbation.  Julia's global RNG
    is not reproducible outside Julia: pass a numpy Generator `rng` (its uniforms / normals are injected) or a `seed`
    for the library's Philox streams.  Returns (points d x Npts, ind 1-based)."""
    d = npd.bt.dims
    if ind is not None:  # explicit components: no search, just the perturbation (src/KDE01.jl:185-189)
        rng = np.random.default_rng(seed) if rng is None else rng
        ind = np.asarray(ind, dtype=np.int64)
        return getPoints(npd)[:, ind - 1] + getBW(npd)[:, ind - 1] * rng.standard_normal((d, len(ind))), ind
    Npts_ = int(Npts_)
    pts = np.zeros((Npts_, d))
    idx = np.zeros(Npts_, dtype=np.int64)
    U = G = None
    if rng is not None:
        G = np.ascontiguousarray(rng.standard_normal((d, Npts_)).T).ravel()   # randn(d, Npts), column-major
        U = np.ascontiguousarray(rng.random(Npts_))
    if seed is None:
        seed = int.from_bytes(os.urandom(8), "little")
    check(lib().kdeb200_sample(npd._dev(), Npts_, int(seed) & 0xFFFFFFFFFFFFFFFF, fptr(U), fptr(G), fptr(pts), iptr(idx)))
    return pts.T, idx


def rand(p, N=1, rng=None, seed=None):
    """src/KDE01.jl:196-198"""
    return sample(p, N, rng=rng, seed=seed)[0]


def resample(p, Np=-1, ksType="lcv", rng=None, seed=None):
    """src/BallTreeDensity01.jl:312-334.  The reference's default Np=-1 and :discrete branches call
    undefined getNpts/getDim and throw; here Np=-1 means Npts(p) and :discrete is rejected."""
    if Np == -1:
        Np = Npts(p)
    if ksType in ("discrete", ":discrete"):
        raise KDEError("resample: ksType=:discrete is broken in the reference (undefined getDim) and not provided")
    samplePts, _ = sample(p, Np, rng=rng, seed=seed)
    return kde(samplePts)


def _sample_batch_args(fn, densities, Np, seeds, randU, randN):
    """handles, Np, seeds and the concatenated injected streams (or None) of a sample_batch / resample_batch call"""
    dens = list(densities)
    n = len(dens)
    Np = np.array([int(x) for x in Np], dtype=np.int64)
    if Np.size != n:
        raise KDEError("%s: need one Np per density" % fn)
    sd = _seeds(seeds, n)
    streams = []
    for name, arg, per in (("randU", randU, [1] * n), ("randN", randN, [Ndim(p) for p in dens])):
        if arg is None:
            streams += [None, None]
            continue
        if len(arg) != n:
            raise KDEError("%s: need one %s entry (or None) per density" % (fn, name))
        parts = []
        for i, a in enumerate(arg):
            if a is None:
                parts.append(np.zeros(0))
            elif name == "randU":
                parts.append(np.ascontiguousarray(a, dtype=np.float64).ravel())
            else:  # d x Np, column-major as sample takes it: point ii at [ii*d, ii*d + d)
                g = np.asarray(a, dtype=np.float64)
                if g.ndim != 2 or g.shape[0] != per[i]:
                    raise KDEError("%s: problem %d: randN must be d x Np" % (fn, i))
                parts.append(np.ascontiguousarray(g.T).ravel())
        streams += [np.concatenate(parts + [np.zeros(1)]), np.array([q.size for q in parts], dtype=np.int64)]
    handles = (_lib.tree_t * max(n, 1))()
    for i, p in enumerate(dens):
        handles[i] = p._dev()
    return dens, n, Np, sd, handles, streams


def sample_batch(densities, Np, seeds=None, randU=None, randN=None):
    """[sample(p, n, seed=s) for p, n, s in zip(densities, Np, seeds)] in one library call (kdeb200_sample_batch: one
    launch for every problem of at most 2048 samples, larger ones by the single call's route after it).  randU / randN are
    None or one entry per density, and an entry may be None (Philox(seeds[i])); randU[i] holds Np[i] uniforms, randN[i]
    is d x Np[i].  Returns a list of (points d x Np, ind), each bit for bit what sample returns for that problem alone
    with the same seed or injected streams."""
    dens, n, Np, sd, handles, (U, nU, G, nN) = _sample_batch_args("sample_batch", densities, Np, seeds, randU, randN)
    dims = [Ndim(p) for p in dens]
    pts = np.zeros(int(sum(dims[i] * Np[i] for i in range(n))) + 1)
    idx = np.zeros(int(Np.sum()) + 1, dtype=np.int64)
    check(lib().kdeb200_sample_batch(n, handles, iptr(Np), sd.ctypes.data_as(C.POINTER(C.c_uint64)), fptr(U), iptr(nU),
                                     fptr(G), iptr(nN), fptr(pts), iptr(idx)))
    out, p0, i0 = [], 0, 0
    for d, m in zip(dims, Np):
        m = int(m)
        out.append((pts[p0:p0 + d * m].reshape(m, d).T.copy(), idx[i0:i0 + m].copy()))
        p0 += d * m
        i0 += m
    return out


def rand_batch(densities, N=1, seeds=None):
    """[rand(p, N, seed=s) for p, s in zip(densities, seeds)]; N may be one count or one per density."""
    dens = list(densities)
    Ns = [int(N)] * len(dens) if np.isscalar(N) else list(N)
    return [pts for pts, _ in sample_batch(dens, Ns, seeds=seeds)]


def resample_batch(densities, Np=None, ksType="lcv", seeds=None):
    """[resample(p, n, seed=s) for p, n, s in zip(densities, Np, seeds)] in one library call (kdeb200_resample_batch):
    the samples as sample_batch draws them, then the kde! bandwidths of every sample set -- sets of at most 512 samples
    without leaving the device, in one launch.  Np = None means each density's Npts; :discrete is refused as resample
    refuses it.  Returns the densities built on the host as kde(points, bw), like kde_batch."""
    if ksType in ("discrete", ":discrete"):
        raise KDEError("resample: ksType=:discrete is broken in the reference (undefined getDim) and not provided")
    dens = list(densities)
    Ns = [Npts(p) for p in dens] if Np is None else Np
    dens, n, Nps, sd, handles, _ = _sample_batch_args("resample_batch", dens, Ns, seeds, None, None)
    dims = [Ndim(p) for p in dens]
    pts = np.zeros(int(sum(dims[i] * Nps[i] for i in range(n))) + 1)
    bw = np.zeros(int(sum(dims)) + 1)
    check(lib().kdeb200_resample_batch(n, handles, iptr(Nps), sd.ctypes.data_as(C.POINTER(C.c_uint64)), None, None, None,
                                       None, fptr(pts), None, fptr(bw), None))
    out, p0, b0 = [], 0, 0
    for d, m in zip(dims, Nps):
        m = int(m)
        out.append(kde(pts[p0:p0 + d * m].reshape(m, d).T, bw[b0:b0 + d].copy()))
        p0 += d * m
        b0 += d
    return out


# ------------------------------------------------------------------------- evaluation -------
def _eval_points(bd, pos, precision=F64):
    pos = np.asarray(pos, dtype=np.float64)
    if bd.bt.dims != pos.shape[0]:
        raise KDEError("bd and pos must have the same dimension")
    M = pos.shape[1]
    q = np.ascontiguousarray(pos.T).ravel()
    out = np.zeros(M)
    check(lib().kdeb200_eval(bd._dev(), fptr(q), M, 0, precision, fptr(out)))
    return out


def _eval_loo(bd, precision=F64):
    out = np.zeros(bd.bt.num_points)
    check(lib().kdeb200_eval(bd._dev(), None, bd.bt.num_points, 1, precision, fptr(out)))
    return out


def evaluateDualTree(bd, pos, lvFlag=False, errTol=1e-3, addop=None, diffop=None, precision=F64):
    """evaluateDualTree(bd, pos, lvFlag, errTol) (src/DualTree01.jl:370-421).

    Always the exact brute-force sum (the reference's default FORCE_EVAL_DIRECT = true); with
    setForceEvalDirect!(false) the reference's dual-tree result is only within errTol of it.
    pos may be a d x M matrix, a vector (M 1-D points, as the reference's deprecated method) or
    another BallTreeDensity.  lvFlag, or pos being bd itself, selects leave-one-out."""
    _require_euclidean(addop=addop, diffop=diffop)
    if isinstance(pos, BallTreeDensity):
        if bd.bt.dims != pos.bt.dims:
            raise KDEError("bd and pos must have the same dimension")
        if lvFlag or pos is bd:
            return _eval_loo(bd, precision)
        return _eval_points(bd, getPoints(pos), precision)
    pos = np.asarray(pos, dtype=np.float64)
    if pos.ndim == 1:
        pos = pos.reshape(1, -1)
    if bd.bt.dims != pos.shape[0]:
        raise KDEError("bd and pos must have the same dimension")
    if lvFlag:
        return _eval_loo(bd, precision)
    return _eval_points(bd, pos, precision)


def _eval_problem(i, bd, pos, lvFlag):
    """(loo, d x M query matrix or None) of one evaluateDualTree_batch problem, read as evaluateDualTree reads it"""
    if isinstance(pos, BallTreeDensity):
        if bd.bt.dims != pos.bt.dims:
            raise KDEError("evaluateDualTree_batch: problem %d: bd and pos must have the same dimension" % i)
        if lvFlag or pos is bd:
            return True, None
        return False, getPoints(pos)
    pos = np.asarray(pos, dtype=np.float64)
    if pos.ndim == 1:
        pos = pos.reshape(1, -1)
    if pos.ndim != 2 or bd.bt.dims != pos.shape[0]:
        raise KDEError("evaluateDualTree_batch: problem %d: bd and pos must have the same dimension" % i)
    if lvFlag:
        return True, None
    return False, pos


def evaluateDualTree_batch(densities, positions, lvFlags=None, precision=F64):
    """[evaluateDualTree(b, p, lv) for b, p, lv in zip(densities, positions, lvFlags)] in one library call
    (kdeb200_eval_batch: one brute-force launch per dimension and leave-one-out flag).  Each entry of positions takes
    what evaluateDualTree's pos takes (a d x M matrix, a vector of 1-D points, another BallTreeDensity; lvFlag or pos is
    the density itself selects leave-one-out).  Every result is bit for bit what evaluateDualTree returns for that
    problem alone with pruning modes 0 and 1 (within 1e-13 under mode 2).  FP64 only."""
    dens = list(densities)
    poss = list(positions)
    n = len(dens)
    if len(poss) != n:
        raise KDEError("evaluateDualTree_batch: need one position set per density")
    lvs = [False] * n if lvFlags is None else [bool(x) for x in lvFlags]
    if len(lvs) != n:
        raise KDEError("evaluateDualTree_batch: need one lvFlag per density")
    M = np.zeros(n, dtype=np.int64)
    loo = np.zeros(n, dtype=np.int32)
    blocks = []
    for i, (bd, pos, lv) in enumerate(zip(dens, poss, lvs)):
        is_loo, q = _eval_problem(i, bd, pos, lv)
        loo[i] = 1 if is_loo else 0
        if is_loo:
            M[i] = bd.bt.num_points
        else:
            M[i] = q.shape[1]
            blocks.append(np.ascontiguousarray(q.T).ravel())
    handles = (_lib.tree_t * max(n, 1))()
    for i, bd in enumerate(dens):
        handles[i] = bd._dev()
    q = np.concatenate(blocks + [np.zeros(1)])
    out = np.zeros(int(M.sum()) + 1)
    check(lib().kdeb200_eval_batch(n, handles, iptr(M), loo.ctypes.data_as(C.POINTER(C.c_int)), fptr(q), int(precision),
                                   fptr(out)))
    res, o = [], 0
    for m in M:
        res.append(out[o:o + int(m)].copy())
        o += int(m)
    return res


def evalAvgLogL(bd1, bd2, addop=None, diffop=None):
    """src/DualTree01.jl:450-470.  bd1 is bd2 => fused leave-one-out kernel (one launch, one scalar)."""
    _require_euclidean(addop=addop, diffop=diffop)
    if bd1 is bd2:
        return -entropy(bd1)
    if isinstance(bd2, BallTreeDensity):
        L = evaluateDualTree(bd1, bd2, False, 1e-3)
        W = getWeights(bd2)
    else:
        raise KDEError("evalAvgLogL(bd1::BallTreeDensity, at::Array{Float64,1}) -- not implemented yet")
    zero = L == 0.0
    if np.any(W[zero] != 0.0):
        return -math.inf
    L = np.where(zero, 1.0, L)
    return float(np.dot(np.log(L), W))


def entropy(bd, addop=None, diffop=None):
    """src/DualTree01.jl:505-508 -- the LOO likelihood with the density's CURRENT bandwidth."""
    _require_euclidean(addop=addop, diffop=diffop)
    d = bd.bt.dims
    bw = np.ascontiguousarray(bd.bandwidthMin[:d], dtype=np.float64)
    H = C.c_double(0.0)
    check(lib().kdeb200_loo_entropy(bd._dev(stale_bw_ok=True), fptr(bw), C.byref(H)))
    return H.value


def kld(p1, p2, method="direct"):
    """src/DualTree01.jl:477-503: D_KL(p1 || p2) by :direct (p1's own points, leave-one-out for the self term) or
    :unscented (p1's points plus / minus one bandwidth per dimension, re-fitted by LOOCV; the reference's block indexing
    (i-1)*N and (2i-1)*N is kept literally, overlaps included)."""
    if method in ("direct", ":direct"):
        return evalAvgLogL(p1, p1) - evalAvgLogL(p2, p1)
    if method in ("unscented", ":unscented"):
        D, N = Ndim(p1), Npts(p1)
        ptsE = np.tile(getPoints(p1), (1, 2 * D + 1))
        bw = getBW(p1)
        for i in range(1, D + 1):
            a0, a1 = (i - 1) * N, (2 * i - 1) * N
            ptsE[i - 1, a0:a0 + N] = ptsE[i - 1, a0:a0 + N] + bw[i - 1, :]
            ptsE[i - 1, a1:a1 + N] = ptsE[i - 1, a1:a1 + N] - bw[i - 1, :]
        pE = kde(ptsE)
        return evalAvgLogL(p1, pE) - evalAvgLogL(p2, pE)
    raise KDEError("kld: method must be :direct or :unscented")


def minkld(p, q):
    return min(abs(kld(p, q)), abs(kld(q, p)))


# ----------------------------------------------- thin host wrappers over the evaluation seam ----
# (src/DualTree01.jl:512-618: out of scope as kernels -- they only call evaluateDualTree / marginal
#  and speed up for free once the seam is on the GPU; mirrored so a user of the reference finds them)
def getKDERange(bd, extend=0.1):
    """src/DualTree01.jl:512-550; bd may be one density or a list (union of the ranges)."""
    if isinstance(bd, (list, tuple)):
        r = getKDERange(bd[0], extend)
        for b in bd[1:]:
            t = getKDERange(b, extend)
            r[:, 0] = np.minimum(r[:, 0], t[:, 0])
            r[:, 1] = np.maximum(r[:, 1], t[:, 1])
        return r
    pts = getPoints(bd)
    lo, hi = pts.min(axis=1), pts.max(axis=1)
    dr = extend * (hi - lo)
    return np.stack([lo - dr, hi + dr], axis=1)


def getKDERangeLinspace(bd, extend=0.1, N=200):
    """src/DualTree01.jl:552-556 (v[1], v[2] are linear indices into the d x 2 range matrix, as in the reference)."""
    v = getKDERange(bd, extend).ravel(order="F")
    return np.linspace(v[0], v[1], N)


def getKDEMax(p, N=200):
    """src/DualTree01.jl:558-569: per-dimension argmax of the marginal on an N-point grid.  The reference builds one
    marginal tree per dimension and evaluates it; here all d marginals are evaluated on their grids in one launch
    (kdeb200_eval_marginals), straight from the d-dimensional density."""
    d = Ndim(p)
    pts = getPoints(p)
    lo, hi = pts.min(axis=1), pts.max(axis=1)          # getKDERange(marginal(p,[i])) with extend = 0.1
    dr = 0.1 * (hi - lo)
    X = np.stack([np.linspace(lo[i] - dr[i], hi[i] + dr[i], N) for i in range(d)])
    Y = eval_marginals(p, X)
    return np.array([X[i, int(np.argmax(Y[i]))] for i in range(d)])


def eval_marginals(p, grids):
    """Densities of every 1-D marginal of p on its own grid: grids is d x G (row k = abscissae of dimension k)."""
    g = np.ascontiguousarray(grids, dtype=np.float64)
    if g.ndim != 2 or g.shape[0] != Ndim(p):
        raise KDEError("eval_marginals: grids must be a %d x G matrix" % Ndim(p))
    out = np.zeros_like(g)
    check(lib().kdeb200_eval_marginals(p._dev(), fptr(g), g.shape[1], fptr(out)))
    return out


def getKDEMean(p):
    """src/DualTree01.jl:571-574"""
    return getPoints(p).mean(axis=1)


def getKDEfit(p):
    """src/DualTree01.jl:575-578 with distribution=MvNormal: maximum-likelihood (mean, covariance)."""
    pts = getPoints(p)
    mu = pts.mean(axis=1)
    c = (pts - mu[:, None]) @ (pts - mu[:, None]).T / pts.shape[1]
    return mu, c


def intersIntgAppxIS(p, q, N=201):
    """src/DualTree01.jl:581-618: grid approximation of the integral of p*q (1-D and 2-D only)."""
    nd = Ndim(p)
    if nd > 2:
        raise KDEError("Can't do higher dimensions yet")
    LD = [getKDERangeLinspace(marginal(p, [k + 1]), N=N, extend=0.3) for k in range(nd)]
    dx = [ld[1] - ld[0] for ld in LD]
    xx = np.zeros((nd, N))
    xx[0, :] = LD[0]
    if nd == 1:
        yy = evaluateDualTree(p, xx) * evaluateDualTree(q, xx)
        return float(np.sum(yy) * dx[0])
    # the reference evaluates row by row (2 N calls of N points, src/DualTree01.jl:605-613); one call per density over
    # the whole N x N grid gives the same values, then the same row-wise accumulation
    grid = np.empty((2, N * N))
    grid[0] = np.tile(LD[0], N)
    grid[1] = np.repeat(LD[1], N)
    yy = (evaluateDualTree(p, grid) * evaluateDualTree(q, grid)).reshape(N, N)
    acc = 0.0
    for i in range(N):
        acc += (dx[0] * float(np.sum(yy[i]))) * dx[1]
    return acc


def to_string(d):
    """Base.string(::BallTreeDensity) (src/StringSerialization.jl:1-5): "KDE:N:[bw]:[pts]" """
    pts = getPoints(d)
    bw = getBW(d)[:, 0]
    rows = ["%s" % " ".join(repr(float(v)) for v in row) for row in pts]
    return "KDE:%d:[%s]:[%s]" % (pts.shape[1], ", ".join(repr(float(v)) for v in bw), "; ".join(rows))


def from_string(text):
    """convert(BallTreeDensity, ::String) (src/StringSerialization.jl:13-26)"""
    if "KDE:" not in text:
        raise KDEError("not a KDE string")
    parts = [t.strip() for t in text.split(":")]
    N = int(parts[1])
    vec = lambda t, sep: [float(x) for x in t.strip().split("[")[-1].split("]")[0].split(sep) if x.strip()]
    bw = vec(parts[2], ",")
    rows = parts[3].split(";")
    if len(rows) != len(bw):
        raise KDEError("KDE string: %d bandwidths but %d point rows" % (len(bw), len(rows)))
    pts = np.zeros((len(bw), N))
    for i, r in enumerate(rows):
        pts[i, :] = vec(r, None)
    return kde(pts, bw)


# ------------------------------------------------------------------------- LOOCV -------------
def updateBandwidth(bd, bw):
    """updateBandwidth! (src/CrossValidation.jl:5-12).  The device records are marked stale: the next
    evaluation / Gibbs call re-uploads the density with the new bandwidth (entropy / nLOO_LL instead
    send the d leaf variances with each kdeb200_loo_entropy call and keep the resident points)."""
    if bd.multibandwidth != 0:
        raise KDEError("updateBandwidth! -- multibandwidth==0 ELSE not implemented yet")
    N, d = bd.bt.num_points, bd.bt.dims
    bw = np.ascontiguousarray(bw, dtype=np.float64).ravel()
    if bw.size != 2 * N * d:
        raise KDEError("updateBandwidth!: expected the full 2*N*d bandwidth array")
    bd.bandwidth = bw
    bd.bandwidthMax = bd.bandwidthMin = bd.bandwidth[N * d:].copy()
    bd._bw_dirty = True


def nLOO_LL(alpha, bd, addop=None, diffop=None, _entropy=None):
    """src/CrossValidation.jl:15-24 -- multiply, evaluate, divide back (ulp drift included).
    _entropy replaces entropy(bd) (dist.kde_sharded: rows partitioned over the ranks)."""
    alpha = alpha * alpha
    updateBandwidth(bd, bd.bandwidth * alpha)
    H = entropy(bd, addop, diffop) if _entropy is None else _entropy(bd)
    updateBandwidth(bd, bd.bandwidth / alpha)
    return H


def golden(bd, ax, bx, cx, tol, addop=None, diffop=None, _count=None, _entropy=None):
    """Golden-section minimisation of nLOO_LL (src/CrossValidation.jl:44-98); host scalar loop."""
    Cc = (3.0 - math.sqrt(5.0)) / 2.0
    R = 1.0 - Cc
    x0, x3 = ax, cx
    if abs(cx - bx) > abs(bx - ax):
        x1, x2 = bx, bx + Cc * (cx - bx)
    else:
        x1, x2 = bx - Cc * (bx - ax), bx
    f1 = nLOO_LL(x1, bd, addop, diffop, _entropy)
    f2 = nLOO_LL(x2, bd, addop, diffop, _entropy)
    n = 2
    while abs(x3 - x0) > tol * (abs(x1) + abs(x2)):
        if f2 < f1:
            x0, x1 = x1, x2
            x2 = R * x1 + Cc * x3
            f1 = f2
            f2 = nLOO_LL(x2, bd, addop, diffop, _entropy)
        else:
            x3, x2 = x2, x1
            x1 = R * x2 + Cc * x0
            f2 = f1
            f1 = nLOO_LL(x1, bd, addop, diffop, _entropy)
        n += 1
    if _count is not None:
        _count.append(n)
    return (x1, f1) if f1 < f2 else (x2, f2)


def neighborMinMax(bd):
    """src/CrossValidation.jl:100-108"""
    N, d = bd.bt.num_points, bd.bt.dims
    rang = bd.bt.ranges[:N * d].reshape(N, d)
    nrm = np.sqrt(np.sum((2.0 * rang) ** 2, axis=1))
    maxm = float(nrm[0])
    minm = max(float(np.min(nrm[:N - 1])), 1e-6)
    return minm, maxm


def ksize(bd, addop=None, diffop=None, _count=None, _entropy=None):
    """src/CrossValidation.jl:110-120"""
    _require_euclidean(addop=addop, diffop=diffop)
    minm, maxm = neighborMinMax(bd)
    p = kde(getPoints(bd), [(minm + maxm) / 2.0], getWeights(bd))
    ks, _ = golden(p, 2.0 * minm / (minm + maxm), 1.0, 2.0 * maxm / (minm + maxm), 1e-2, _count=_count,
                   _entropy=_entropy)
    ks = ks * (minm + maxm) / 2.0
    return kde(getPoints(p), [ks], getWeights(p))


# ------------------------------------------------------------------------- MS Gibbs ----------
def _handles(trees):
    arr = (_lib.tree_t * len(trees))()
    for i, t in enumerate(trees):
        arr[i] = t._dev(gibbs=True)
    return arr


def gibbs_sizes(trees, Niter):
    """(Nlevels, uniforms per sample, normals per sample, kernel evaluations per sample)"""
    L, pu, pn, ev = C.c_int(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
    check(lib().kdeb200_gibbs_sizes(_handles(trees), len(trees), int(Niter), C.byref(L), C.byref(pu), C.byref(pn),
                                    C.byref(ev)))
    return L.value, pu.value, pn.value, ev.value


def philox_streams(seed, Np, perU, perN):
    """The variates the kernel draws when no streams are injected, as (randU, randN) arrays."""
    U = np.zeros(Np * perU)
    G = np.zeros(Np * perN)
    check(lib().kdeb200_philox_streams(int(seed), Np, perU, perN, fptr(U), fptr(G)))
    return U, G


def prodAppxMSGibbsS(npd0, trees, anFcns=None, anParams=None, Niter=3, addop=None, diffop=None, getMu=None,
                     getLambda=None, glbs=None, addEntropy=True, ndims=None, Ndens=None, Np=None, randU=None,
                     randN=None, partialDimMask=None, seed=None, s0=0, s1=None, recordLabels=False):
    """prodAppxMSGibbsS(npd0, trees, anFcns, anParams; Niter=3, ...) (src/MSGibbs01.jl:645-703).

    Returns (points d x Np, indices Ndens x Np) with indices = permutation + 1 (the reference's
    label convention, :612-616).  randU / randN inject the random streams exactly like the
    reference's keyword arguments; without them the kernel draws from Philox4x32-10(seed).
    s0, s1 restrict the call to samples [s0, s1) of the Np-sample run (multi-GPU sharding); the
    returned arrays then hold only that range.  recordLabels=True (the reference's
    glbs.recordChoosen) adds a third result: labelsChoosen as an int64 array [n, Ndens, Nlevels].  Ndens: 1..64
    (more than 16 densities run in FP64 whatever set_gibbs_precision says, and refuse degenerate bandwidths)."""
    _require_euclidean(addop=addop, diffop=diffop, getMu=getMu, getLambda=getLambda)
    trees = list(trees)
    M = len(trees) if Ndens is None else int(Ndens)
    if M != len(trees) or M < 1:
        raise KDEError("prodAppxMSGibbsS: Ndens must equal length(trees) >= 1")
    d = max(Ndim(t) for t in trees)
    if ndims is not None and int(ndims) != d:
        raise KDEError("prodAppxMSGibbsS: ndims must equal the trees' dimension")
    for t in trees:
        if Ndim(t) != d:
            raise KDEError("kdes must have same dimension")
    if Np is None:
        if npd0 is None:
            raise KDEError("prodAppxMSGibbsS: pass npd0 (its Npts is the number of samples) or Np")
        Np = Npts(npd0)
    Np = int(Np)
    if Np < 0 or not (0 <= s0 <= (Np if s1 is None else s1) <= Np):
        raise KDEError("prodAppxMSGibbsS: bad sample range")
    s1 = Np if s1 is None else int(s1)
    n = s1 - s0
    mask = None
    if partialDimMask is not None:
        mask = np.ascontiguousarray(np.asarray(partialDimMask, dtype=bool).reshape(M, d).astype(np.uint8))
    if (randU is None) != (randN is None):
        raise KDEError("prodAppxMSGibbsS: pass both randU and randN or neither")
    if randU is not None:
        randU = np.ascontiguousarray(randU, dtype=np.float64).ravel()
        randN = np.ascontiguousarray(randN, dtype=np.float64).ravel()
    if seed is None:
        seed = int.from_bytes(os.urandom(8), "little")
    points = np.zeros((n, d))
    indices = np.ones((n, M), dtype=np.int64)
    rec = None
    if recordLabels:
        rec = np.zeros((n, M, gibbs_sizes(trees, Niter)[0]), dtype=np.int64)
    check(lib().kdeb200_gibbs(_handles(trees), M, Np, int(Niter), int(bool(addEntropy)),
                              None if mask is None else mask.ctypes.data_as(_lib.u8p), fptr(randU),
                              0 if randU is None else randU.size, fptr(randN), 0 if randN is None else randN.size,
                              int(seed) & 0xFFFFFFFFFFFFFFFF, int(s0), s1, fptr(points), iptr(indices), iptr(rec)))
    if recordLabels:
        return points.T, indices.T, rec
    return points.T, indices.T


def prod(trees, glbs=None, addEntropy=True, seed=None, recordLabels=False):
    """*(trees::Vector{BallTreeDensity}) (src/MSGibbs01.jl:707-726).  recordLabels=True mirrors
    `glbs.recordChoosen = true` (examples/ExtractingLabels.jl) and returns (density, labelsChoosen).  Up to 64
    densities, as prodAppxMSGibbsS."""
    trees = list(trees)
    if len(trees) == 1 and not addEntropy:
        return kde(getPoints(trees[0]).copy())
    numpts = int(round(float(np.mean([Npts(t) for t in trees]))))
    d = max(Ndim(t) for t in trees)
    for p in trees:
        if d != Ndim(p):
            raise KDEError("kdes must have same dimension")
    if recordLabels or numpts < 2:
        res = prodAppxMSGibbsS(None, trees, None, None, Niter=5, addEntropy=addEntropy, Np=numpts, seed=seed,
                               recordLabels=recordLabels)
        return (kde(res[0]), res[2]) if recordLabels else kde(res[0])
    # Gibbs + the LOOCV refit kde!(pGM) in ONE library call; up to 512 samples never leave the device in between
    if seed is None:
        seed = int.from_bytes(os.urandom(8), "little")
    pts = np.zeros((numpts, d))
    bw = np.zeros(d)
    check(lib().kdeb200_product_kde(_handles(trees), len(trees), numpts, 5, int(bool(addEntropy)), None,
                                    int(seed) & 0xFFFFFFFFFFFFFFFF, fptr(pts), None, fptr(bw), None))
    return kde(pts.T, bw)


def _batch_handles(tree_lists):
    lists = [list(t) for t in tree_lists]
    ndens = np.array([len(t) for t in lists], dtype=np.int32)
    flat = [t for ts in lists for t in ts]
    for i, ts in enumerate(lists):
        if ts and any(Ndim(t) != Ndim(ts[0]) for t in ts):
            raise KDEError("problem %d: kdes must have same dimension" % i)
    dims = [Ndim(ts[0]) if ts else 0 for ts in lists]
    return lists, ndens, _handles(flat), dims


def _seeds(seeds, n):
    if seeds is None:
        return np.frombuffer(os.urandom(8 * n), dtype=np.uint64).copy() if n else np.zeros(0, dtype=np.uint64)
    s = np.array([int(x) & 0xFFFFFFFFFFFFFFFF for x in seeds], dtype=np.uint64)
    if s.size != n:
        raise KDEError("need one seed per problem")
    return s


def prodAppxMSGibbsS_batch(tree_lists, Np, Niter=3, addEntropy=True, partialDimMasks=None, randU=None, randN=None,
                           seeds=None):
    """Many independent prodAppxMSGibbsS problems in one library call (kdeb200_gibbs_batch, one launch per dimension).

    tree_lists[i] are the densities of problem i and Np[i] its number of samples.  partialDimMasks, randU, randN are
    None or one entry per problem (an entry may be None: all dimensions, resp. Philox(seeds[i])).  Returns a list of
    (points d x Np, indices Ndens x Np), each equal to what prodAppxMSGibbsS returns for that problem alone."""
    lists, ndens, handles, dims = _batch_handles(tree_lists)
    n = len(lists)
    Np = np.array([int(x) for x in Np], dtype=np.int64)
    if Np.size != n:
        raise KDEError("need one Np per problem")
    mask = None
    if partialDimMasks is not None:
        if len(partialDimMasks) != n:
            raise KDEError("need one partialDimMask (or None) per problem")
        mask = np.concatenate([np.ones(ndens[i] * dims[i], dtype=np.uint8) if m is None else
                               np.asarray(m, dtype=bool).reshape(ndens[i], dims[i]).astype(np.uint8).ravel()
                               for i, m in enumerate(partialDimMasks)] or [np.zeros(0, dtype=np.uint8)])
    U = G = nU = nN = None
    if (randU is None) != (randN is None):
        raise KDEError("prodAppxMSGibbsS_batch: pass both randU and randN or neither")
    if randU is not None:
        if len(randU) != n or len(randN) != n:
            raise KDEError("need one randU / randN entry (or None) per problem")
        us = [np.zeros(0) if u is None else np.ascontiguousarray(u, dtype=np.float64).ravel() for u in randU]
        gs = [np.zeros(0) if g is None else np.ascontiguousarray(g, dtype=np.float64).ravel() for g in randN]
        nU = np.array([u.size for u in us], dtype=np.int64)
        nN = np.array([g.size for g in gs], dtype=np.int64)
        U = np.concatenate(us + [np.zeros(1)])
        G = np.concatenate(gs + [np.zeros(1)])
    sd = _seeds(seeds, n)
    points = np.zeros(int(sum(dims[i] * Np[i] for i in range(n))) + 1)
    indices = np.zeros(int(sum(ndens[i] * Np[i] for i in range(n))) + 1, dtype=np.int64)
    check(lib().kdeb200_gibbs_batch(n, ndens.ctypes.data_as(C.POINTER(C.c_int)), handles, iptr(Np), int(Niter),
                                    int(bool(addEntropy)), None if mask is None else mask.ctypes.data_as(_lib.u8p),
                                    fptr(U), iptr(nU), fptr(G), iptr(nN), sd.ctypes.data_as(C.POINTER(C.c_uint64)),
                                    fptr(points), iptr(indices)))
    out, p0, i0 = [], 0, 0
    for i in range(n):
        d, M, m = dims[i], int(ndens[i]), int(Np[i])
        out.append((points[p0:p0 + d * m].reshape(m, d).T.copy(), indices[i0:i0 + M * m].reshape(m, M).T.copy()))
        p0 += d * m
        i0 += M * m
    return out


def prod_batch(tree_lists, addEntropy=True, seeds=None):
    """[prod(trees, addEntropy=addEntropy, seed=s) for trees, s in zip(tree_lists, seeds)] with the Gibbs steps and the
    LOOCV refits of all problems in one library call (kdeb200_product_kde_batch).  The problems prod answers on the host
    (one density without entropy, fewer than two product samples) are answered the same way here."""
    lists = [list(t) for t in tree_lists]
    n = len(lists)
    sd = _seeds(seeds, n)
    res = [None] * n
    dev = []
    for i, ts in enumerate(lists):
        numpts = int(round(float(np.mean([Npts(t) for t in ts])))) if ts else 0
        if (len(ts) == 1 and not addEntropy) or numpts < 2:
            res[i] = prod(ts, addEntropy=addEntropy, seed=int(sd[i]))
        else:
            dev.append((i, numpts))
    if dev:
        lists_d, ndens, handles, dims = _batch_handles([lists[i] for i, _ in dev])
        Np = np.array([m for _, m in dev], dtype=np.int64)
        sdd = np.ascontiguousarray(sd[[i for i, _ in dev]])
        pts = np.zeros(int(sum(dims[k] * Np[k] for k in range(len(dev)))))
        bw = np.zeros(int(sum(dims)))
        check(lib().kdeb200_product_kde_batch(len(dev), ndens.ctypes.data_as(C.POINTER(C.c_int)), handles, iptr(Np), 5,
                                              int(bool(addEntropy)), None, sdd.ctypes.data_as(C.POINTER(C.c_uint64)),
                                              fptr(pts), None, fptr(bw), None))
        p0 = b0 = 0
        for k, (i, m) in enumerate(dev):
            d = dims[k]
            res[i] = kde(pts[p0:p0 + d * m].reshape(m, d).T, bw[b0:b0 + d])
            p0 += d * m
            b0 += d
    return res


def gibbs_batch_split():
    """(host checks + planning + packing, host-to-device copy, device-to-host copies) of the last batch call, in ms."""
    a, b, c = C.c_double(0), C.c_double(0), C.c_double(0)
    check(lib().kdeb200_gibbs_batch_split(C.byref(a), C.byref(b), C.byref(c)))
    return a.value, b.value, c.value


# ------------------------------------------------------------------------- measurement -------
def pipe_peak(which, iters=20000):
    """(lane-ops per second, ms) of a dependency-free DFMA (0) / FFMA (1) / MUFU.EX2 (2) stream."""
    r, ms = C.c_double(0), C.c_double(0)
    check(lib().kdeb200_pipe_peak(int(which), int(iters), C.byref(r), C.byref(ms)))
    return r.value, ms.value


def last_kernel_ms():
    ms, n = C.c_double(0), C.c_int(0)
    check(lib().kdeb200_last_kernel_ms(C.byref(ms), C.byref(n)))
    return ms.value, n.value
