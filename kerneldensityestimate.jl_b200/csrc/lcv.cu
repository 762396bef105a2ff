// lcv.cu -- kde!(points): per-dimension bandwidth selection by leave-one-out likelihood cross
// validation, natively behind one C call.
//
// Computes what the loop of kde!(points) src/KDE01.jl:13-23 computes for every dimension i:
//   pp = ksize(marginal(p, [i]));  bwds[i] = getBW(pp)[1]
// i.e. marginal :143-153 (1-D tree on points[i,:] with renormalised weights), neighborMinMax
// src/CrossValidation.jl:100-108, the working density of ksize :110-120, golden :44-98 over
// nLOO_LL :15-24 (multiply / evaluate / divide back, ulp drift included) and the final scaling.
//
// Two device paths, bit-identical to each other and to the per-call kdeb200_loo_entropy route:
//   N <= LCV_FUSED_MAX : ONE launch for all dimensions; CTA i runs the whole golden-section search of
//                        dimension i on chip (points in shared memory, one thread per row, the same
//                        sequential leaf-order sums and the same 1024-slot reduction tree as eval.cu)
//   larger N           : host golden loop over the tiled LOO kernel of eval.cu, one scalar back per step
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

#include "eval_shared.cuh"
#include "lcv.cuh"
#include "tree.cuh"

namespace kdeb200 {

int tree_build_host(int d, int64_t N, const double *points, const double *weights, const double *bw_var,
                    double *centers, double *ranges, double *wout, double *means, double *bandwidth,
                    int64_t *left, int64_t *right, int64_t *lowest, int64_t *highest, int64_t *perm);
int tree_create(int d, int64_t N, const double *means, const double *bandwidth, const double *weights,
                const int64_t *left, const int64_t *right, const int64_t *perm, bool gibbs_records,
                kdeb200_tree_t *out);
int tree_destroy(kdeb200_tree_t t);
int tree_on(kdeb200_tree_t t, int slot, kdeb200_tree_t *out);
int loo_partial_device(kdeb200_tree_t bd, const double *bw_var, int64_t j0, int64_t j1, double *d_sum, int *d_flag,
                       cudaStream_t st, int *launches);
bool loo_sym_shardable(const kdeb200_tree_s *bd);
int loo_sym_device(kdeb200_tree_t bd, const double *bw_var, double *d_L, cudaStream_t st, int *launches, int part,
                   int nparts, double *d_tot);
int loo_sym_combine_device(kdeb200_tree_t bd, const double *bw_var, const double *d_tots, int nparts, double *d_L,
                           cudaStream_t st, int *launches);
int loglik_reduce_device(kdeb200_tree_t bd, const double *d_L, int64_t q0, int64_t n, double *d_sum, int *d_flag,
                         cudaStream_t st, int *launches);

constexpr int LCV_THREADS = 1024;   // == the block of loglik_reduce_kernel (same reduction tree)

struct LcvDim {
  double b0;      // leaf variance of the working density, ((minm + maxm) / 2)^2
  double ax, cx;  // golden bracket [2 minm / (minm + maxm), 1, 2 maxm / (minm + maxm)]
};

struct LcvParams {
  const double *leaf;  // [dim][N][2]: leaf-ordered (x, w) records of every dimension's working density
  const LcvDim *dims;
  double *out;         // [dim][3]: xmin, fmin, number of nLOO_LL calls
  const double *exptab;
  ExpConsts ec;
  int N;
  double norm0, tol, Cg, Rg;  // (2 pi)^(1/2); golden constants computed on the host
};

// nLOO_LL(alpha) for the CTA's dimension; every thread returns the same H and updates its copy of b identically
__device__ __forceinline__ double lcv_nloo(double alpha, double &b, const double *__restrict__ rec, int N,
                                           const double *__restrict__ tab, const ExpConsts &ec, double norm0,
                                           double *sh, int *shf) {
  const double a2 = alpha * alpha;  // src/CrossValidation.jl:17
  b = b * a2;                       // updateBandwidth!(bd, bd.bandwidth * alpha)
  const double ich = -0.5 / b;
  const double norm = norm0 * sqrt(b);
  const int j = threadIdx.x;
  double s = 0.0;
  int f = 0;
  if (j < N) {
    const double x = rec[2 * j], wj = rec[2 * j + 1];
    double sum = 0.0;
#pragma unroll 4
    for (int i = 0; i < N; ++i) {  // evalDirect, leaf order, i != j (src/DualTree01.jl:130-162)
      const double2 r = *reinterpret_cast<const double2 *>(rec + 2 * i);
      const double df = __dadd_rn(x, -r.x);
      const double e = kde_exp_flush(__fma_rn(__dmul_rn(df, df), ich, 0.0), tab, ec);
      if (i != j) sum = __fma_rn(e, r.y, sum);
    }
    if (sum < EV_TINY) sum = exact_row(rec, 2, 1, N, &x, &ich, j);
    double v = 0.5 * (sum + sum) / norm;
    v = v / (1.0 - wj);
    loglik_term(v, wj, s, f);
  }
  __syncthreads();  // everyone has consumed the previous H
  loglik_block_reduce(s, f, sh, shf);
  const double H = shf[0] ? INFINITY : -sh[0];  // entropy = -evalAvgLogL, -Inf under the zero rule
  b = b / a2;                                   // updateBandwidth!(bd, bd.bandwidth / alpha)
  return H;
}

// golden (src/CrossValidation.jl:44-98), executed redundantly (and identically) by every thread of the CTA
__device__ __forceinline__ void lcv_golden_run(const LcvDim D, const double *__restrict__ rec, int N, const double *__restrict__ tab,
                                               const ExpConsts &ec, double norm0, double tol, double Cg, double Rg, double *sh,
                                               int *shf, double *out3) {
  double b = D.b0;
  const double ax = D.ax, bx = 1.0, cx = D.cx;
  double x0 = ax, x3 = cx, x1, x2;
  if (fabs(cx - bx) > fabs(bx - ax)) {
    x1 = bx;
    x2 = __dadd_rn(bx, __dmul_rn(Cg, cx - bx));  // explicit roundings: no FMA contraction, like the host loop
  } else {
    x1 = __dadd_rn(bx, -__dmul_rn(Cg, bx - ax));
    x2 = bx;
  }
  double f1 = lcv_nloo(x1, b, rec, N, tab, ec, norm0, sh, shf);
  double f2 = lcv_nloo(x2, b, rec, N, tab, ec, norm0, sh, shf);
  int n = 2;
  while (fabs(x3 - x0) > tol * (fabs(x1) + fabs(x2))) {
    if (f2 < f1) {
      x0 = x1;
      x1 = x2;
      x2 = __dadd_rn(__dmul_rn(Rg, x1), __dmul_rn(Cg, x3));
      f1 = f2;
      f2 = lcv_nloo(x2, b, rec, N, tab, ec, norm0, sh, shf);
    } else {
      x3 = x2;
      x2 = x1;
      x1 = __dadd_rn(__dmul_rn(Rg, x2), __dmul_rn(Cg, x0));
      f2 = f1;
      f1 = lcv_nloo(x1, b, rec, N, tab, ec, norm0, sh, shf);
    }
    ++n;
    if (n > 4096) break;  // NaN-proofing: the reference would spin forever
  }
  if (threadIdx.x == 0) {
    out3[0] = (f1 < f2) ? x1 : x2;
    out3[1] = (f1 < f2) ? f1 : f2;
    out3[2] = (double)n;
  }
}

__global__ void __launch_bounds__(LCV_THREADS) lcv_golden_kernel(const __grid_constant__ LcvParams P) {
  __shared__ __align__(16) double tab[KDE_EXP_TAB];
  __shared__ __align__(16) double rec[2 * LCV_FUSED_MAX];
  __shared__ double sh[LCV_THREADS];
  __shared__ int shf[LCV_THREADS];
  const int dim = blockIdx.x, N = P.N;
  for (int i = threadIdx.x; i < KDE_EXP_TAB; i += LCV_THREADS) tab[i] = P.exptab[i];
  for (int i = threadIdx.x; i < 2 * N; i += LCV_THREADS) rec[i] = P.leaf[(size_t)dim * 2 * N + i];
  __syncthreads();
  lcv_golden_run(P.dims[dim], rec, N, tab, P.ec, P.norm0, P.tol, P.Cg, P.Rg, sh, shf, P.out + dim * 3);
}

// The same search on points that are ALREADY ON THE DEVICE (the product samples of `*`, src/MSGibbs01.jl:723-725:
// kde!(pGM) right after the Gibbs kernel, SURVEY.md 8f.2): the per-dimension 1-D ball tree of ksize is never built on
// the host.  CTA `dim` sorts its coordinate in shared memory (in 1-D the tree's leaf order IS the sorted order; equal
// points carry equal weights, so their mutual order cannot matter), rebuilds the node statistics the bracket needs --
// centre and half-range of every node of the median-split tree, bottom-up with the reference's arithmetic
// (calcStatsBall!, src/BallTree01.jl:282-336), laid out as an implicit heap -- takes neighborMinMax
// (src/CrossValidation.jl:100-108) from them and runs the golden-section search above.  Bit-identical to the host route.
struct LcvPointsParams {
  const double *pts;  // N points, point i at pts + i * d
  double *out;        // [dim][5]: xmin, fmin, number of nLOO_LL calls, minm, maxm
  const double *exptab;
  ExpConsts ec;
  int N, d;
  double w2;          // the (uniform) weight of the working density of ksize, renormalised twice like the host route
  double norm0, tol, Cg, Rg;
};

// the whole search for dimension `dim` of the points at P.pts, by one CTA of LCV_THREADS threads
__device__ __forceinline__ void lcv_golden_points_cta(const LcvPointsParams &P, int dim) {
  __shared__ __align__(16) double tab[KDE_EXP_TAB];  // prologue: the heap (centres | half-ranges), then the exp table
  __shared__ __align__(16) double rec[2 * LCV_FUSED_MAX];
  __shared__ double sh[LCV_THREADS];
  __shared__ int shf[LCV_THREADS];
  const int N = P.N, tid = threadIdx.x;
  // ---- sort (bitonic, 512 slots padded with +inf)
  double *sb = sh;
  if (tid < LCV_FUSED_MAX) sb[tid] = (tid < N) ? P.pts[(size_t)tid * P.d + dim] : INFINITY;
  __syncthreads();
  for (int k = 2; k <= LCV_FUSED_MAX; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (tid < LCV_FUSED_MAX) {
        const int ixj = tid ^ j;
        if (ixj > tid) {
          const double a = sb[tid], c = sb[ixj];
          const bool up = (tid & k) == 0;
          if ((a > c) == up) {
            sb[tid] = c;
            sb[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  // ---- node statistics on the implicit heap: node h covers the leaf interval reached from [0, N-1] by the bits of h
  double *hc = tab, *hr = tab + 1024;
  const int h = tid + 1;  // 1..1024; ids >= 1024 cannot exist for N <= 512
  int lvl = 31 - __clz(h), lo = 0, hi = N - 1;
  bool valid = h < 1024;
  for (int bit = lvl - 1; bit >= 0 && valid; --bit) {
    if (lo == hi) {
      valid = false;
      break;
    }
    const int split = (lo + hi) / 2;
    if ((h >> bit) & 1) lo = split + 1; else hi = split;
  }
  const bool internal = valid && lo < hi;
  if (valid && lo == hi) {
    hc[h] = sb[lo];
    hr[h] = 0.0;
  }
  __syncthreads();
  for (int depth = 9; depth >= 0; --depth) {
    if (internal && lvl == depth) {
      const double cl = hc[2 * h], rl = hr[2 * h], cr = hc[2 * h + 1], rr = hr[2 * h + 1];
      const double hiL = __dadd_rn(cl, rl), hiR = __dadd_rn(cr, rr);
      const double maxi = hiL > hiR ? hiL : hiR;
      const double loL = __dadd_rn(cl, -rl), loR = __dadd_rn(cr, -rr);
      const double mini = loL < loR ? loL : loR;
      const double half = __ddiv_rn(__dadd_rn(maxi, -mini), 2.0);
      hr[h] = half;
      hc[h] = __dadd_rn(mini, half);
    }
    __syncthreads();
  }
  // ---- the working density's records, neighborMinMax, the bracket
  for (int i = tid; i < N; i += LCV_THREADS) {
    rec[2 * i] = sb[i];
    rec[2 * i + 1] = P.w2;
  }
  double nrm = INFINITY;
  if (internal) {
    const double t = __dmul_rn(2.0, hr[h]);
    nrm = __dsqrt_rn(__dmul_rn(t, t));
  }
  const double root_nrm = [&] {
    const double t = __dmul_rn(2.0, hr[1]);
    return __dsqrt_rn(__dmul_rn(t, t));
  }();
  __syncthreads();  // sb (= sh) has been copied out
  sh[tid] = nrm;
  __syncthreads();
  for (int off = LCV_THREADS / 2; off > 0; off >>= 1) {
    if (tid < off) sh[tid] = fmin(sh[tid], sh[tid + off]);
    __syncthreads();
  }
  const double minm = fmax(sh[0], 1e-6), maxm = root_nrm;
  __syncthreads();
  for (int i = tid; i < KDE_EXP_TAB; i += LCV_THREADS) tab[i] = P.exptab[i];  // the heap is no longer needed
  __syncthreads();
  LcvDim D;
  const double hh = __ddiv_rn(__dadd_rn(minm, maxm), 2.0);
  D.b0 = __dmul_rn(hh, hh);
  D.ax = __ddiv_rn(__dmul_rn(2.0, minm), __dadd_rn(minm, maxm));
  D.cx = __ddiv_rn(__dmul_rn(2.0, maxm), __dadd_rn(minm, maxm));
  lcv_golden_run(D, rec, N, tab, P.ec, P.norm0, P.tol, P.Cg, P.Rg, sh, shf, P.out + dim * 5);
  if (tid == 0) {
    P.out[dim * 5 + 3] = minm;
    P.out[dim * 5 + 4] = maxm;
  }
}

__global__ void __launch_bounds__(LCV_THREADS) lcv_golden_points_kernel(const __grid_constant__ LcvPointsParams P) {
  lcv_golden_points_cta(P, blockIdx.x);
}

// The same for many point sets in one launch (kdeb200_product_kde_batch): CTA b runs dimension items[b].dim of
// problem items[b].  Every item carries its own points, N, d, w2 and output block; the constants are the launch's.
__global__ void __launch_bounds__(LCV_THREADS) lcv_golden_points_batch_kernel(const LcvBatchItem *__restrict__ items,
                                                                              const __grid_constant__ LcvPointsParams C) {
  const LcvBatchItem it = items[blockIdx.x];
  LcvPointsParams P = C;
  P.pts = it.pts;
  P.out = it.out;
  P.N = it.N;
  P.d = it.d;
  P.w2 = it.w2;
  lcv_golden_points_cta(P, it.dim);
}

namespace {

// everything ksize needs from one dimension's marginal, in the reference's order of operations
struct Marginal {
  std::vector<double> leaf;  // N x (x, w2) in leaf order
  std::vector<double> means, weights;
  std::vector<int64_t> perm;
  double minm = 0, maxm = 0;
};

int build_marginal(int64_t N, const double *x, const std::vector<double> &w1, Marginal &m) {
  const int64_t NN = 2 * N;
  std::vector<double> centers(NN), ranges(NN), wout(NN), bandwidth(NN);
  std::vector<int64_t> left(NN), right(NN), lowest(NN), highest(NN);
  m.means.assign(NN, 0.0);
  m.perm.assign(NN, 0);
  const double one = 1.0;  // marginal(): getBW(bd, [1]) of kde!(points, [1.0])
  if (int rc = tree_build_host(1, N, x, w1.data(), &one, centers.data(), ranges.data(), wout.data(), m.means.data(),
                               bandwidth.data(), left.data(), right.data(), lowest.data(), highest.data(),
                               m.perm.data()))
    return rc;
  // neighborMinMax (src/CrossValidation.jl:100-108) in 1-D
  auto nrm = [&](int64_t i) { const double t = 2.0 * ranges[i]; return std::sqrt(t * t); };
  m.maxm = nrm(0);
  double mn = nrm(0);
  for (int64_t i = 1; i < N - 1; ++i) mn = std::fmin(mn, nrm(i));
  m.minm = std::fmax(mn, 1e-6);
  // ksize: p = kde!(getPoints(bd), [(minm+maxm)/2], getWeights(bd)) -- same points => same tree, the weights are
  // renormalised once more by kde! (sequential sum in original order)
  std::vector<double> w_orig(N);
  for (int64_t s = 0; s < N; ++s) w_orig[m.perm[N + s] - 1] = wout[N + s];
  double ssum = 0.0;
  for (int64_t i = 0; i < N; ++i) ssum += w_orig[i];
  m.weights.assign(NN, 0.0);
  m.leaf.resize(2 * N);
  for (int64_t s = 0; s < N; ++s) {
    const double w2 = w_orig[m.perm[N + s] - 1] / ssum;
    m.weights[N + s] = w2;
    m.leaf[2 * s] = centers[N + s];
    m.leaf[2 * s + 1] = w2;
  }
  return 0;
}

struct Golden {
  double Cg, Rg;
  Golden() {
    Cg = (3.0 - std::sqrt(5.0)) / 2.0;
    Rg = 1.0 - Cg;
  }
};

// the launch constants of the device-points search (everything but the points, N, d and w2)
LcvPointsParams lcv_points_consts() {
  const Golden G_;
  LcvPointsParams P;
  std::memset(&P, 0, sizeof(P));
  P.exptab = ctx().d_exptab;
  P.ec = make_exp_consts();
  P.norm0 = std::pow(2.0 * M_PI, 0.5);
  P.tol = 1e-2;
  P.Cg = G_.Cg;
  P.Rg = G_.Rg;
  return P;
}

}  // namespace

// kde!(points) bandwidths for N <= LCV_FUSED_MAX points resident on the device (point i at d_points + i * d): one launch on
// `st`, the d x 5 result block stays in d_out5 (xmin, fmin, calls, minm, maxm per dimension) for the caller to fetch
// together with its other results; lcv_points_finish turns it into the standard deviations.
int kde_lcv_points_device(int d, int64_t N, const double *d_points, double *d_out5, cudaStream_t st) {
  if (N < 2 || N > LCV_FUSED_MAX) KDE_FAIL(3, "kde_lcv (device points): needs 2 <= N <= %d", LCV_FUSED_MAX);
  LcvPointsParams P = lcv_points_consts();
  P.pts = d_points;
  P.out = d_out5;
  P.N = (int)N;
  P.d = d;
  P.w2 = lcv_points_w2(N);
  lcv_golden_points_kernel<<<d, LCV_THREADS, 0, st>>>(P);
  KDE_CUDA(cudaGetLastError());
  return 0;
}

double lcv_points_w2(int64_t N) {
  // the weights of the working density, exactly as the host route derives them: kde!(points, [1.0]) -> 1/N, marginal()
  // renormalises by the sequential sum, ksize's kde! renormalises once more
  double w1 = 1.0 / (double)N;
  {
    double ssum = 0.0;
    for (int64_t i = 0; i < N; ++i) ssum += w1;
    w1 = w1 / ssum;
  }
  double w2;
  {
    double ssum = 0.0;
    for (int64_t i = 0; i < N; ++i) ssum += w1;
    w2 = w1 / ssum;
  }
  return w2;
}

int kde_lcv_points_batch_device(int nitems, const LcvBatchItem *d_items, cudaStream_t st) {
  if (nitems <= 0) return 0;
  lcv_golden_points_batch_kernel<<<nitems, LCV_THREADS, 0, st>>>(d_items, lcv_points_consts());
  KDE_CUDA(cudaGetLastError());
  return 0;
}

void lcv_points_finish(int d, const double *out5, double *bw_std_out, int *ncalls_out) {
  for (int k = 0; k < d; ++k) {
    const double xmin = out5[5 * k], minm = out5[5 * k + 3], maxm = out5[5 * k + 4];
    const double ks = xmin * (minm + maxm) / 2.0;  // src/CrossValidation.jl:117
    bw_std_out[k] = std::sqrt(ks * ks);
    if (ncalls_out) ncalls_out[k] = (int)out5[5 * k + 2];
  }
}

// j0, j1 and allreduce: this process owns the leaf rows [j0, j1) of every nLOO_LL evaluation and the callback sums the
// partial likelihood (and ORs the zero flag) over the processes -- the multi-GPU split of SURVEY.md 8e.  allreduce ==
// nullptr: single process, all rows.  Small N runs the fused kernel redundantly on every process (no exchange needed).
int kde_lcv(int d, int64_t N, const double *points, int64_t j0, int64_t j1, kdeb200_allreduce_v_fn allreduce,
            void *user, double *bw_std_out, int *ncalls_out) {
  if (int rc = ensure_init()) return rc;
  const double t_enter = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
  if (d < 1) KDE_FAIL(3, "kde_lcv: d must be >= 1");
  if (N < 2) KDE_FAIL(3, "kde_lcv: at least two points are needed for cross validation");
  if (2 * N >= (int64_t)std::numeric_limits<int32_t>::max()) KDE_FAIL(3, "kde_lcv: N too large");
  if (!allreduce) {
    j0 = 0;
    j1 = N;
  }
  if (j0 < 0 || j1 > N || j0 > j1) KDE_FAIL(3, "kde_lcv: bad row range [%lld,%lld) of %lld", (long long)j0, (long long)j1, (long long)N);
  Context &c = ctx();
  const Golden G_;
  const double tol = 1e-2;

  // kde!(points, [1.0]): weights ones(N) / N; marginal(): renormalised by their sequential sum
  std::vector<double> w1(N, 1.0 / (double)N);
  {
    double ssum = 0.0;
    for (int64_t i = 0; i < N; ++i) ssum += w1[i];
    for (int64_t i = 0; i < N; ++i) w1[i] = w1[i] / ssum;
  }
  // the d marginal trees are independent: one host thread each (the builder is a pure function of its arguments)
  std::vector<Marginal> margs(d);
  {
    std::vector<int> rcs(d, 0);
    auto work = [&](int k) {
      std::vector<double> x(N);
      for (int64_t i = 0; i < N; ++i) x[i] = points[i * d + k];
      rcs[k] = build_marginal(N, x.data(), w1, margs[k]);
    };
    if (d == 1 || N < 4096) {
      for (int k = 0; k < d; ++k) work(k);
    } else {
      std::vector<std::thread> th;
      for (int k = 0; k < d; ++k) th.emplace_back(work, k);
      for (auto &t : th) t.join();
    }
    for (int k = 0; k < d; ++k)
      if (rcs[k]) KDE_FAIL(rcs[k], "kde_lcv: building the marginal tree of dimension %d failed", k + 1);
  }
  auto finish = [&](int k, double xmin) {
    const Marginal &m = margs[k];
    const double ks = xmin * (m.minm + m.maxm) / 2.0;  // src/CrossValidation.jl:117
    bw_std_out[k] = std::sqrt(ks * ks);                // getBW of kde!(.., [ks]) (variance ks^2)
  };
  c.last_launches = 0;

  if (N <= LCV_FUSED_MAX) {
    std::vector<double> leaf((size_t)d * 2 * N);
    std::vector<LcvDim> dims(d);
    for (int k = 0; k < d; ++k) {
      const Marginal &m = margs[k];
      std::copy(m.leaf.begin(), m.leaf.end(), leaf.begin() + (size_t)k * 2 * N);
      const double h = (m.minm + m.maxm) / 2.0;
      dims[k].b0 = h * h;
      dims[k].ax = 2.0 * m.minm / (m.minm + m.maxm);
      dims[k].cx = 2.0 * m.maxm / (m.minm + m.maxm);
    }
    const size_t b_leaf = sizeof(double) * leaf.size(), b_dims = sizeof(LcvDim) * d, b_out = sizeof(double) * 3 * d;
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    char *base = nullptr;
    KDE_CUDA(cudaMallocAsync(&base, up(b_leaf) + up(b_dims) + up(b_out), c.stream));
    LcvParams P;
    P.leaf = reinterpret_cast<double *>(base);
    P.dims = reinterpret_cast<LcvDim *>(base + up(b_leaf));
    P.out = reinterpret_cast<double *>(base + up(b_leaf) + up(b_dims));
    P.exptab = c.d_exptab;
    P.ec = make_exp_consts();
    P.N = (int)N;
    P.norm0 = std::pow(2.0 * M_PI, 0.5);  // src/DualTree01.jl:325 with d = 1
    P.tol = tol;
    P.Cg = G_.Cg;
    P.Rg = G_.Rg;
    std::vector<double> out(3 * d);
    cudaError_t e = cudaMemcpyAsync(base, leaf.data(), b_leaf, cudaMemcpyHostToDevice, c.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(base + up(b_leaf), dims.data(), b_dims, cudaMemcpyHostToDevice, c.stream);
    if (e == cudaSuccess) {
      cudaEventRecord(c.ev0, c.stream);
      lcv_golden_kernel<<<d, LCV_THREADS, 0, c.stream>>>(P);
      e = cudaGetLastError();
      cudaEventRecord(c.ev1, c.stream);
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out.data(), P.out, b_out, cudaMemcpyDeviceToHost, c.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
    cudaFreeAsync(base, c.stream);
    if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "kde_lcv: fused golden-section kernel: %s", cudaGetErrorString(e));
    float ms = 0;
    cudaEventElapsedTime(&ms, c.ev0, c.ev1);
    c.last_ms = ms;
    c.last_launches = 1;
    for (int k = 0; k < d; ++k) {
      finish(k, out[3 * k]);
      if (ncalls_out) ncalls_out[k] = (int)out[3 * k + 2];
    }
    return 0;
  }

  // Large N: the d golden-section searches are independent, so they advance in LOCK-STEP: every step queues the tiled
  // LOO launches of all unfinished dimensions back to back -- on every GPU of the in-process set, each owning a block
  // of this process's leaf rows -- then ONE synchronisation per GPU brings the partial likelihoods back (and, between
  // processes, ONE vector all-reduce).  ~20 round trips instead of ~20 d, and d times more work in flight per step.
  struct Search {  // golden (src/CrossValidation.jl:44-98) as a state machine: next() -> alpha to evaluate, feed(H)
    double x0, x1, x2, x3, f1 = 0, f2 = 0, Cg, Rg, tol;
    int phase = 0, ncalls = 0;  // 0: f1 pending, 1: f2 pending, 2: loop
    bool want_f2 = false, done = false;
    double pending() const { return (phase == 0) ? x1 : (phase == 1 ? x2 : (want_f2 ? x2 : x1)); }
    void advance() {  // decide the next evaluation of the loop, or finish
      if (!(std::fabs(x3 - x0) > tol * (std::fabs(x1) + std::fabs(x2))) || ncalls > 4096) {
        done = true;
        return;
      }
      if (f2 < f1) {
        x0 = x1;
        x1 = x2;
        x2 = Rg * x1 + Cg * x3;
        f1 = f2;
        want_f2 = true;
      } else {
        x3 = x2;
        x2 = x1;
        x1 = Rg * x2 + Cg * x0;
        f2 = f1;
        want_f2 = false;
      }
    }
    void feed(double H) {
      ++ncalls;
      if (phase == 0) {
        f1 = H;
        phase = 1;
      } else if (phase == 1) {
        f2 = H;
        phase = 2;
        advance();
      } else {
        if (want_f2) f2 = H; else f1 = H;
        advance();
      }
    }
    double xmin() const { return (f1 < f2) ? x1 : x2; }
  };
  int G = (j1 - j0 >= 8192 * (int64_t)multi_count()) ? multi_count() : 1;
  std::vector<kdeb200_tree_t> trees(d, nullptr);
  std::vector<Search> S(d);
  std::vector<double> b(d);
  int rc = 0, launches = 0;
  for (int k = 0; k < d && rc == 0; ++k) {
    Marginal &m = margs[k];
    const double h = (m.minm + m.maxm) / 2.0;
    b[k] = h * h;
    std::vector<double> bandwidth(2 * N, b[k]);
    rc = tree_create(1, N, m.means.data(), bandwidth.data(), m.weights.data(), nullptr, nullptr, m.perm.data(), false, &trees[k]);
    const double ax = 2.0 * m.minm / (m.minm + m.maxm), bx = 1.0, cx = 2.0 * m.maxm / (m.minm + m.maxm);
    Search &s = S[k];
    s.Cg = G_.Cg; s.Rg = G_.Rg; s.tol = tol;
    s.x0 = ax; s.x3 = cx;
    if (std::fabs(cx - bx) > std::fabs(bx - ax)) {
      s.x1 = bx;
      s.x2 = bx + G_.Cg * (cx - bx);
    } else {
      s.x1 = bx - G_.Cg * (bx - ax);
      s.x2 = bx;
    }
  }
  // per GPU: result slots [d] of (sum, flag) in one small device buffer, replicas of the d trees
  struct PerGpu {
    double *d_res = nullptr;  // d x 2 doubles: sum, flag (int in the low word)
    std::vector<kdeb200_tree_t> t;
    std::vector<double> h_res;
    int64_t r0 = 0, r1 = 0;
  };
  std::vector<PerGpu> gp(G);
  for (int g = 0; g < G && rc == 0; ++g) {
    ScopedDevice sd(g);
    Context &cg = ctx();
    const int64_t n = j1 - j0, base = n / G, rem = n % G;
    gp[g].r0 = j0 + g * base + (g < rem ? g : rem);
    gp[g].r1 = gp[g].r0 + base + (g < rem ? 1 : 0);
    gp[g].t.assign(d, nullptr);
    gp[g].h_res.assign(2 * d, 0.0);
    cudaError_t e = cudaMallocAsync(&gp[g].d_res, sizeof(double) * 2 * d, cg.stream);
    if (e != cudaSuccess) {
      set_error("kde_lcv: cudaMallocAsync: %s", cudaGetErrorString(e));
      rc = 100 + (int)e;
    }
    for (int k = 0; k < d && rc == 0; ++k) rc = tree_on(trees[k], g, &gp[g].t[k]);
  }
  // In-process multi-GPU with all rows in this process and densities in the symmetric kernel's range: the devices share
  // the TRIANGLE of pairs instead of the rows.  Device g evaluates the row blocks b = g (mod G) once per unordered pair
  // and sends its contribution to every row (N doubles) straight into the primary's memory over NVLink (peer copy on its
  // own stream + an event the primary's stream waits on); the primary folds the G vectors in device order and reduces
  // the likelihood.  No host round trip between the devices, one synchronisation (of the primary) per step.
  const bool sym_multi = rc == 0 && G > 1 && !allreduce && j0 == 0 && j1 == N && loo_sym_shardable(trees[0]);
  std::vector<double *> d_tot(G, nullptr);
  std::vector<cudaEvent_t> ev(G, nullptr);
  double *d_all0 = nullptr, *d_L0 = nullptr;
  if (sym_multi) {
    for (int g = 0; g < G && rc == 0; ++g) {
      ScopedDevice sd(g);
      cudaError_t e = cudaMallocAsync(&d_tot[g], sizeof(double) * (size_t)d * N, ctx().stream);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev[g], cudaEventDisableTiming);
      if (e != cudaSuccess) {
        set_error("kde_lcv: multi-GPU buffers: %s", cudaGetErrorString(e));
        rc = 100 + (int)e;
      }
    }
    if (rc == 0) {
      ScopedDevice sd(0);
      cudaError_t e = cudaMallocAsync(&d_all0, sizeof(double) * (size_t)d * G * N, ctx().stream);
      if (e == cudaSuccess) e = cudaMallocAsync(&d_L0, sizeof(double) * (size_t)N, ctx().stream);
      if (e != cudaSuccess) {
        set_error("kde_lcv: multi-GPU buffers: %s", cudaGetErrorString(e));
        rc = 100 + (int)e;
      }
    }
  }
  std::vector<int> active;
  std::vector<double> sums(d);
  std::vector<int> flags(d);
  const bool trace = getenv("KDEB200_TRACE") != nullptr;
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_loop = now();
  double t_queue = 0.0;
  int nsteps = 0;
  while (rc == 0) {
    const double t_s0 = now();
    ++nsteps;
    active.clear();
    for (int k = 0; k < d; ++k)
      if (!S[k].done) active.push_back(k);
    if (active.empty()) break;
    std::vector<double> a2(d, 1.0);
    for (int k : active) {
      const double alpha = S[k].pending();
      a2[k] = alpha * alpha;  // src/CrossValidation.jl:17
      b[k] = b[k] * a2[k];    // updateBandwidth!(bd, bd.bandwidth * alpha)
    }
    if (sym_multi) {
      // one host thread per device queues that device's launches (a dozen per dimension: boxes, mask, order, kernel,
      // partial sums, peer copy); queued from a single thread they cost as much as the kernels at 8 GPUs
      std::vector<int> rcs(G, 0), nl(G, 0);
      std::vector<std::string> errs(G);
      auto queue_device = [&](int g) {
        ScopedDevice sd(g);
        Context &cg = ctx();
        for (int k : active) {
          double *tot = d_tot[g] + (size_t)k * N;
          int r = loo_sym_device(gp[g].t[k], &b[k], nullptr, cg.stream, &nl[g], g, G, tot);
          if (!r) {
            cudaError_t e = cudaMemcpyPeerAsync(d_all0 + ((size_t)k * G + g) * N, ctx_at(0).device, tot, cg.device,
                                                sizeof(double) * (size_t)N, cg.stream);
            if (e != cudaSuccess) {
              set_error("kde_lcv: peer copy from GPU slot %d: %s", g, cudaGetErrorString(e));
              r = 100 + (int)e;
            }
          }
          if (r) {
            rcs[g] = r;
            errs[g] = get_error();
            return;
          }
        }
        if (cudaEventRecord(ev[g], cg.stream) != cudaSuccess) rcs[g] = 100;
      };
      {
        std::vector<std::thread> th;
        for (int g = 1; g < G; ++g) th.emplace_back(queue_device, g);
        queue_device(0);
        for (auto &t : th) t.join();
      }
      for (int g = 0; g < G; ++g) {
        launches += nl[g];
        if (rcs[g] && !rc) {
          set_error("GPU slot %d: %s", g, errs[g].c_str());
          rc = rcs[g];
        }
      }
      t_queue += now() - t_s0;
      if (!rc) {
        ScopedDevice sd(0);
        Context &c0 = ctx();
        for (int g = 1; g < G; ++g) cudaStreamWaitEvent(c0.stream, ev[g], 0);
        for (int k : active) {
          rc = loo_sym_combine_device(gp[0].t[k], &b[k], d_all0 + (size_t)k * G * N, G, d_L0, c0.stream, &launches);
          if (!rc)
            rc = loglik_reduce_device(gp[0].t[k], d_L0, 0, N, gp[0].d_res + 2 * k, reinterpret_cast<int *>(gp[0].d_res + 2 * k + 1),
                                      c0.stream, &launches);
          if (rc) break;
        }
        if (!rc) {
          cudaError_t e = cudaMemcpyAsync(gp[0].h_res.data(), gp[0].d_res, sizeof(double) * 2 * d, cudaMemcpyDeviceToHost, c0.stream);
          if (e == cudaSuccess) e = cudaStreamSynchronize(c0.stream);
          if (e != cudaSuccess) {
            set_error("kde_lcv: LOO kernels (multi-GPU, symmetric): %s", cudaGetErrorString(e));
            rc = 100 + (int)e;
          }
        }
      }
      if (rc) break;
      for (int k : active) {
        int f;
        std::memcpy(&f, &gp[0].h_res[2 * k + 1], sizeof(int));
        const double H = f ? std::numeric_limits<double>::infinity() : -gp[0].h_res[2 * k];
        b[k] = b[k] / a2[k];
        S[k].feed(H);
      }
      continue;
    }
    for (int g = 0; g < G && rc == 0; ++g) {  // queue everything, no host wait in between
      ScopedDevice sd(g);
      Context &cg = ctx();
      if (gp[g].r1 > gp[g].r0) {
        for (int k : active) {
          rc = loo_partial_device(gp[g].t[k], &b[k], gp[g].r0, gp[g].r1, gp[g].d_res + 2 * k,
                                  reinterpret_cast<int *>(gp[g].d_res + 2 * k + 1), cg.stream, &launches);
          if (rc) break;
        }
      }
    }
    for (int g = 0; g < G && rc == 0; ++g) {  // only now wait: a pageable D2H blocks the host until the stream drains
      ScopedDevice sd(g);
      if (gp[g].r1 <= gp[g].r0) continue;
      cudaError_t e = cudaMemcpyAsync(gp[g].h_res.data(), gp[g].d_res, sizeof(double) * 2 * d, cudaMemcpyDeviceToHost, ctx().stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx().stream);
      if (e != cudaSuccess) {
        set_error("kde_lcv: LOO kernels on GPU slot %d: %s", g, cudaGetErrorString(e));
        rc = 100 + (int)e;
      }
    }
    if (rc) break;
    int na = 0;
    for (int k : active) {  // partial sums of the row blocks in block order
      double sum = 0.0;
      int flag = 0;
      for (int g = 0; g < G; ++g)
        if (gp[g].r1 > gp[g].r0) {
          sum += gp[g].h_res[2 * k];
          int f;
          std::memcpy(&f, &gp[g].h_res[2 * k + 1], sizeof(int));
          flag |= f;
        }
      sums[na] = sum;
      flags[na] = flag;
      ++na;
    }
    if (allreduce) {
      if (int r = allreduce(sums.data(), flags.data(), na, user)) {
        set_error("kde_lcv: the all-reduce callback failed (%d)", r);
        rc = 9;
        break;
      }
    }
    na = 0;
    for (int k : active) {
      const double H = flags[na] ? std::numeric_limits<double>::infinity() : -sums[na];
      ++na;
      b[k] = b[k] / a2[k];  // updateBandwidth!(bd, bd.bandwidth / alpha): the ulp drift is part of the reference
      S[k].feed(H);
    }
  }
  if (trace)
    fprintf(stderr, "[kdeb200] kde_lcv N=%lld d=%d G=%d sym_multi=%d: setup %.1f ms, %d lock-step rounds in %.1f ms (host queueing %.1f ms)\n",
            (long long)N, d, G, (int)sym_multi, t_loop - t_enter, nsteps, now() - t_loop, t_queue);
  for (int g = 0; g < G; ++g) {
    ScopedDevice sd(g);
    if (sym_multi) cudaStreamSynchronize(ctx().stream);  // peers may still be copying into the primary's buffers
    if (gp[g].d_res) cudaFreeAsync(gp[g].d_res, ctx().stream);
    if (d_tot[g]) cudaFreeAsync(d_tot[g], ctx().stream);
    if (ev[g]) cudaEventDestroy(ev[g]);
  }
  {
    ScopedDevice sd(0);
    if (d_all0) cudaFreeAsync(d_all0, ctx().stream);
    if (d_L0) cudaFreeAsync(d_L0, ctx().stream);
  }
  for (int k = 0; k < d; ++k)
    if (trees[k]) tree_destroy(trees[k]);
  if (rc) return rc;
  for (int k = 0; k < d; ++k) {
    finish(k, S[k].xmin());
    if (ncalls_out) ncalls_out[k] = S[k].ncalls;
  }
  ctx_at(0).last_launches = launches;
  return 0;
}

}  // namespace kdeb200
