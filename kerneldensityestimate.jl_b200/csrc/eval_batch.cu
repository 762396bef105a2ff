// eval_batch.cu -- K2b: many independent brute-force evaluations in one blocking call (kdeb200_eval_batch), and the
// kde!(points) bandwidths of many independent point sets in one call (kdeb200_kde_lcv_batch).
//
// Evaluation.  Every problem is checked as kdeb200_eval checks it before anything runs.  Each problem gets exactly the
// (query block, component split) grid a lone FP64 kdeb200_eval would launch for it (eval_device in eval.cu); the
// batch flattens those grids into one list of work items per (d, loo) class and launches one kernel per class, each
// CTA reading its item and its problem's descriptor.  Problems with S == 1 finish in the kernel, the partial sums of
// problems with S > 1 are summed in split order by one finalize launch for the whole batch.  Descriptors, work items
// and query points travel in ONE copy from the context's pinned staging buffer (batch_stage, gibbs_batch.cu); all outputs come back in one copy.
// A problem's values are therefore those of the single call on the brute-force kernel, bit for bit.
//
// Bandwidths.  Point sets of N <= LCV_FUSED_MAX go in one copy and one lcv_golden_points_batch_kernel launch (one CTA
// per (problem, dimension)); larger ones take kde_lcv's host route one by one afterwards.
#include <chrono>
#include <cmath>
#include <cstring>
#include <limits>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "eval_shared.cuh"
#include "gibbs.cuh"
#include "lcv.cuh"
#include "tree.cuh"

namespace kdeb200 {

#ifndef EV_R
#define EV_R 2
#endif
// query points per thread: must stay in step with ev_q in eval.cu (same macros, same defaults), since the number of
// query blocks decides a problem's component split and so its summation order
#ifndef EV_Q1
#define EV_Q1 6
#endif
#ifndef EV_Q2
#define EV_Q2 4
#endif
#ifndef EV_Q4
#define EV_Q4 2
#endif
#ifndef EV_Q6
#define EV_Q6 2
#endif
constexpr int evb_q(int d) { return d == 1 ? EV_Q1 : (d == 2 ? EV_Q2 : (d <= 4 ? EV_Q4 : (d <= 6 ? EV_Q6 : 1))); }

// one evaluation problem: what eval_device puts in EvalParams for a single call (q0 = 0, scatter on)
struct EvalBatchProb {
  const double *comps;    // N leaf records, stride SE
  const double *queries;  // query i at queries + i * qstride (LOO: comps)
  const int64_t *perm;    // LOO: leaf -> original index (output scatter); null otherwise
  double *out;            // M results in the caller's order ...
  double *partial;        // ... and, when S > 1, S x M partial sums
  int64_t N, M, chunk;
  int qstride, S, tile_nodes, SE;  // SE: record stride of comps
  double ich[KDEB200_MAX_DIM];  // -0.5 / variance_k
  double norm;                  // (2 pi)^(d/2) prod sqrt(variance_k)
};

struct EvalBatchItem {  // one CTA of a class launch: (problem, query block, component split)
  int prob, qb, y, pad_;
};

struct EvalBatchParams {
  const EvalBatchProb *probs;
  const EvalBatchItem *items;  // this launch's items
  const double *exptab;
  ExpConsts ec;
};

// The loop body and epilogue below are eval_kernel's (eval.cu) with the problem's fields read from its descriptor:
// keep them in step with eval_kernel.  Only the order of the FMAs matters for the bits, and it is the same: component
// order within the split, S partials summed in split order by the finalize kernel.
template <int D, int Q, bool LOO>
__global__ void __launch_bounds__(EV_THREADS) eval_batch_kernel(const __grid_constant__ EvalBatchParams B) {
  constexpr int SE = Rec<D>::SE;
  constexpr int R = EV_R;  // component records per loop trip
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double *tiles = reinterpret_cast<double *>(smem_raw);
  __shared__ __align__(16) double tab[KDE_EXP_TAB];
  __shared__ __align__(8) uint64_t bars[EV_STAGES];

  const EvalBatchItem it = B.items[blockIdx.x];
  const EvalBatchProb *P = B.probs + it.prob;
  const double *comps = P->comps;
  const double *queries = P->queries;
  const int64_t N = P->N, M = P->M, chunk = P->chunk;
  const int qstride = P->qstride, S = P->S, TN = P->tile_nodes;
  double ich[D];
#pragma unroll
  for (int k = 0; k < D; ++k) ich[k] = P->ich[k];

  const int tid = threadIdx.x;
  for (int i = tid; i < KDE_EXP_TAB; i += EV_THREADS) tab[i] = B.exptab[i];
  if (tid == 0) {
    for (int s = 0; s < EV_STAGES; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  const int64_t c0 = (int64_t)it.y * chunk;
  const int64_t c1 = (c0 + chunk < N) ? c0 + chunk : N;
  const int ntiles = (int)((c1 - c0 + TN - 1) / TN);

  auto issue = [&](int t) {
    const int64_t a = c0 + (int64_t)t * TN;
    const int64_t cnt = (c1 - a < TN) ? (c1 - a) : TN;
    const uint32_t bytes = (uint32_t)(cnt * SE * sizeof(double));
    uint64_t *bar = &bars[t % EV_STAGES];
    mbar_expect_tx(bar, bytes);
    tma_bulk_g2s(tiles + (size_t)(t % EV_STAGES) * (EV_TILE_BYTES / 8), comps + a * SE, bytes, bar);
  };
  if (tid == 0)
    for (int t = 0; t < EV_STAGES && t < ntiles; ++t) issue(t);

  // this thread's queries
  const int64_t qbase = (int64_t)it.qb * (EV_THREADS * Q);
  double x[Q][D];
  double sum[Q];
  int64_t self[Q];
#pragma unroll
  for (int i = 0; i < Q; ++i) {
    int64_t qi = qbase + tid + (int64_t)i * EV_THREADS;
    const bool ok = qi < M;
    if (!ok) qi = M - 1;
    const double *src = queries + qi * (int64_t)qstride;
#pragma unroll
    for (int k = 0; k < D; ++k) x[i][k] = src[k];
    sum[i] = 0.0;
    self[i] = LOO ? qi : -1;
  }

  // does the CTA's own index range overlap this split? (warp-uniform; only then test i == j)
  const int64_t qlo = qbase, qhi = qlo + EV_THREADS * Q;

  for (int t = 0; t < ntiles; ++t) {
    const int64_t a = c0 + (int64_t)t * TN;
    const int cnt = (int)((c1 - a < TN) ? (c1 - a) : TN);
    mbar_wait(&bars[t % EV_STAGES], (uint32_t)((t / EV_STAGES) & 1));
    const double *rec = tiles + (size_t)(t % EV_STAGES) * (EV_TILE_BYTES / 8);
    const bool check = LOO && (a < qhi) && (a + cnt > qlo);
    if (!check) {
      int c = 0;
      for (; c + R <= cnt; c += R) {
        double rr[R][SE], e[R][Q];
#pragma unroll
        for (int r = 0; r < R; ++r) load_rec<SE>(rec + (c + r) * SE, rr[r]);
#pragma unroll
        for (int i = 0; i < Q; ++i) {
#pragma unroll
          for (int r = 0; r < R; ++r) e[r][i] = kde_exp_flush(quad<D>(x[i], rr[r], ich), tab, B.ec);
        }
#pragma unroll
        for (int i = 0; i < Q; ++i) {
#pragma unroll
          for (int r = 0; r < R; ++r) sum[i] = __fma_rn(e[r][i], rr[r][D], sum[i]);  // component order
        }
      }
      for (; c < cnt; ++c) {
        double ra[SE];
        load_rec<SE>(rec + c * SE, ra);
#pragma unroll
        for (int i = 0; i < Q; ++i) sum[i] = __fma_rn(kde_exp_flush(quad<D>(x[i], ra, ich), tab, B.ec), ra[D], sum[i]);
      }
    } else {
      for (int c = 0; c < cnt; ++c) {
        double ra[SE];
        load_rec<SE>(rec + c * SE, ra);
#pragma unroll
        for (int i = 0; i < Q; ++i) {
          const double e = kde_exp_flush(quad<D>(x[i], ra, ich), tab, B.ec);
          if (a + c != self[i]) sum[i] = __fma_rn(e, ra[D], sum[i]);  // leave-one-out (src/DualTree01.jl:146)
        }
      }
    }
    __syncthreads();  // everyone is done with this stage
    if (tid == 0 && t + EV_STAGES < ntiles) issue(t + EV_STAGES);
  }

#pragma unroll
  for (int i = 0; i < Q; ++i) {
    const int64_t qi = qbase + tid + (int64_t)i * EV_THREADS;
    if (qi >= M) continue;
    if (S > 1) {
      P->partial[(int64_t)it.y * M + qi] = sum[i];
    } else {
      double sv = sum[i];
      if (sv < EV_TINY) sv = exact_row(comps, SE, D, N, queries + qi * (int64_t)qstride, P->ich, LOO ? qi : -1);
      double v = 0.5 * (sv + sv) / P->norm;  // 0.5*(pMin+pMax)/norm, :335-339
      if (LOO) v = v / (1.0 - comps[qi * SE + D]);
      const int64_t o = (LOO && P->perm) ? P->perm[qi] : qi;
      P->out[o] = v;
    }
  }
}

// eval_finalize_kernel for every S > 1 problem of the batch: block b sums rows [256 b.y, 256 b.y + 256) of problem b.x
struct EvalBatchFin {
  int prob, blk, d, loo;
};
__global__ void eval_batch_finalize_kernel(const EvalBatchProb *probs, const EvalBatchFin *fins) {
  const EvalBatchFin f = fins[blockIdx.x];
  const EvalBatchProb *P = probs + f.prob;
  const int64_t qi = (int64_t)f.blk * blockDim.x + threadIdx.x;
  const int64_t M = P->M;
  if (qi >= M) return;
  const int SE = P->SE;
  double s = 0.0;
  for (int y = 0; y < P->S; ++y) s += P->partial[(int64_t)y * M + qi];
  if (s < EV_TINY) s = exact_row(P->comps, SE, f.d, P->N, P->queries + qi * (int64_t)P->qstride, P->ich, f.loo ? qi : -1);
  double v = 0.5 * (s + s) / P->norm;
  if (f.loo) v = v / (1.0 - P->comps[qi * SE + f.d]);
  const int64_t o = (f.loo && P->perm) ? P->perm[qi] : qi;
  P->out[o] = v;
}

// ---------------------------------------------------------------- host side --------------
template <int D, bool LOO>
static cudaError_t launch_eval_batch_d(const EvalBatchParams &B, int nitems, cudaStream_t st) {
  constexpr int Q = evb_q(D);
  auto kern = eval_batch_kernel<D, Q, LOO>;
  const size_t smem = EV_STAGES * EV_TILE_BYTES;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return e;
  kern<<<nitems, EV_THREADS, smem, st>>>(B);
  return cudaGetLastError();
}

template <bool LOO>
static cudaError_t launch_eval_batch(int d, const EvalBatchParams &B, int nitems, cudaStream_t st) {
  switch (d) {
    case 1: return launch_eval_batch_d<1, LOO>(B, nitems, st);
    case 2: return launch_eval_batch_d<2, LOO>(B, nitems, st);
    case 3: return launch_eval_batch_d<3, LOO>(B, nitems, st);
    case 4: return launch_eval_batch_d<4, LOO>(B, nitems, st);
    case 5: return launch_eval_batch_d<5, LOO>(B, nitems, st);
    case 6: return launch_eval_batch_d<6, LOO>(B, nitems, st);
    case 7: return launch_eval_batch_d<7, LOO>(B, nitems, st);
    case 8: return launch_eval_batch_d<8, LOO>(B, nitems, st);
  }
  return cudaErrorInvalidValue;
}

namespace {
size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }

struct Drain {  // an error return after the first enqueue waits for the enqueued work: the staging buffer is reused
  cudaStream_t st;
  ~Drain() { cudaStreamSynchronize(st); }
};
}  // namespace

int eval_batch(int nprob, const kdeb200_tree_t *trees, const int64_t *Min, const int *loo, const double *pos,
               int precision, double *p_out) {
  Context &c = ctx();
  const char *fn = "eval_batch";
  if (nprob < 0) KDE_FAIL(3, "%s: nprob=%d < 0", fn, nprob);
  if (precision < KDEB200_F64 || precision > KDEB200_F32_BOUNDED) KDE_FAIL(3, "%s: unknown precision %d", fn, precision);
  if (precision != KDEB200_F64) KDE_FAIL(3, "%s: only KDEB200_F64 is batched (precision %d)", fn, precision);
  if (nprob == 0) return 0;
  if (!trees || !Min || !p_out) KDE_FAIL(2, "%s: NULL argument", fn);

  // ---- every problem checked as kdeb200_eval checks it; nothing runs unless all pass
  struct Prob {
    int d, S, nqb;
    bool loo;
    int64_t M, offQ, offO, chunk;
    double norm, ich[KDEB200_MAX_DIM];
  };
  std::vector<Prob> pr(nprob);
  int64_t offQ = 0, offO = 0, offPart = 0;
  for (int i = 0; i < nprob; ++i) {
    Prob &p = pr[i];
    const kdeb200_tree_t bd = trees[i];
    if (!bd) KDE_FAIL(2, "%s: problem %d: NULL tree", fn, i);
    p.loo = loo && loo[i] != 0;
    p.d = bd->d;
    p.M = p.loo ? bd->N : Min[i];
    if (p.M < 0) KDE_FAIL(3, "%s: problem %d: M=%lld < 0", fn, i, (long long)p.M);
    if (!p.loo && !pos && p.M > 0) KDE_FAIL(2, "%s: problem %d: pos is NULL", fn, i);
    if (bd->slot != c.slot)
      KDE_FAIL(3, "%s: problem %d: the tree lives on another GPU of the set than the primary", fn, i);
    p.offQ = offQ;
    p.offO = offO;
    p.S = 0;
    p.nqb = 0;
    if (!p.loo) offQ += (int64_t)p.d * p.M;
    offO += p.M;
    if (p.M == 0) continue;  // the single call returns before it looks at the bandwidth
    // eval_device's normalisation and split, verbatim
    double norm = std::pow(2.0 * M_PI, (double)p.d / 2.0);  // src/DualTree01.jl:325-330
    for (int k = 0; k < p.d; ++k) {
      const double v = bd->hvar[k];
      if (!(v > 0.0) || !std::isfinite(v))
        KDE_FAIL(5, "%s: problem %d: bandwidth variance must be finite and > 0 (dim %d: %g)", fn, i, k + 1, v);
      p.ich[k] = -0.5 / v;
      norm *= std::sqrt(v);
    }
    p.norm = norm;
    const int SE = bd->SE;
    int TN = 1;
    while (TN * 2 * SE * 8 <= EV_TILE_BYTES) TN *= 2;
    const int bq = EV_THREADS * evb_q(p.d);
    const int64_t nqb = (p.M + bq - 1) / bq;
    const int64_t ntile_total = (bd->N + TN - 1) / TN;
    int64_t S = (8LL * c.sm_count + nqb - 1) / nqb;
    if (S > ntile_total) S = ntile_total;
    if (S > 65535) S = 65535;
    if (S < 1) S = 1;
    int64_t chunk = ((ntile_total + S - 1) / S) * TN;
    S = (bd->N + chunk - 1) / chunk;
    if (nqb * S >= ((int64_t)1 << 31)) KDE_FAIL(3, "%s: problem %d: 2^31 work items or more", fn, i);
    p.S = (int)S;
    p.nqb = (int)nqb;
    p.chunk = chunk;
    if (S > 1) offPart += S * p.M;
  }

  // ---- launch classes (d, loo) and their work items; finalize blocks of the S > 1 problems
  std::map<std::pair<int, bool>, std::vector<int>> classes;
  for (int i = 0; i < nprob; ++i)
    if (pr[i].M > 0) classes[{pr[i].d, pr[i].loo}].push_back(i);
  int64_t nitems = 0, nfin = 0;
  for (int i = 0; i < nprob; ++i) {
    nitems += (int64_t)pr[i].nqb * pr[i].S;
    if (pr[i].S > 1) nfin += (pr[i].M + 255) / 256;
  }
  if (nitems >= ((int64_t)1 << 31) || nfin >= ((int64_t)1 << 31)) KDE_FAIL(3, "%s: 2^31 work items or more", fn);

  // ---- one staging area: descriptors | work items | finalize blocks | query points
  size_t bytes = 0;
  const size_t prob_at = bytes;
  bytes += up256(sizeof(EvalBatchProb) * nprob);
  const size_t item_at = bytes;
  bytes += up256(sizeof(EvalBatchItem) * nitems);
  const size_t fin_at = bytes;
  bytes += up256(sizeof(EvalBatchFin) * nfin);
  const size_t q_at = bytes;
  bytes += up256(sizeof(double) * offQ);
  char *h = nullptr;
  if (int rc = batch_stage(bytes, &h)) return rc;
  DevBuf dBlob(c.stream), dO(c.stream), dPart(c.stream);
  KDE_CUDA(dBlob.alloc(bytes));
  KDE_CUDA(dO.alloc(sizeof(double) * offO));
  if (offPart) KDE_CUDA(dPart.alloc(sizeof(double) * offPart));
  char *dv = dBlob.as<char>();
  const double *d_q = reinterpret_cast<const double *>(dv + q_at);

  EvalBatchProb *hp = reinterpret_cast<EvalBatchProb *>(h + prob_at);
  int64_t part = 0;
  for (int i = 0; i < nprob; ++i) {
    const Prob &p = pr[i];
    const kdeb200_tree_t bd = trees[i];
    EvalBatchProb &b = hp[i];
    std::memset(&b, 0, sizeof(b));
    b.comps = bd->d_leaf;
    b.queries = p.loo ? bd->d_leaf : d_q + p.offQ;
    b.qstride = p.loo ? bd->SE : p.d;
    b.perm = p.loo ? bd->d_perm : nullptr;
    b.out = dO.as<double>() + p.offO;
    b.N = bd->N;
    b.M = p.M;
    b.chunk = p.chunk;
    b.S = p.S;
    int TN = 1;
    while (TN * 2 * bd->SE * 8 <= EV_TILE_BYTES) TN *= 2;
    b.tile_nodes = TN;
    b.SE = bd->SE;
    for (int k = 0; k < p.d; ++k) b.ich[k] = p.ich[k];
    b.norm = p.norm;
    if (p.S > 1) {
      b.partial = dPart.as<double>() + part;
      part += (int64_t)p.S * p.M;
    }
  }
  struct Launch {
    int d, n;
    bool loo;
    EvalBatchParams B;
  };
  std::vector<Launch> launches_k2b;
  EvalBatchItem *hi = reinterpret_cast<EvalBatchItem *>(h + item_at);
  int64_t ni = 0;
  for (auto &cl : classes) {
    Launch L;
    L.d = cl.first.first;
    L.loo = cl.first.second;
    L.B.probs = reinterpret_cast<const EvalBatchProb *>(dv + prob_at);
    L.B.items = reinterpret_cast<const EvalBatchItem *>(dv + item_at) + ni;
    L.B.exptab = c.d_exptab;
    L.B.ec = make_exp_consts();
    const int64_t n0 = ni;
    for (int i : cl.second)
      for (int y = 0; y < pr[i].S; ++y)
        for (int qb = 0; qb < pr[i].nqb; ++qb) hi[ni++] = EvalBatchItem{i, qb, y, 0};
    L.n = (int)(ni - n0);
    launches_k2b.push_back(L);
  }
  EvalBatchFin *hf = reinterpret_cast<EvalBatchFin *>(h + fin_at);
  int64_t nf = 0;
  for (int i = 0; i < nprob; ++i)
    if (pr[i].S > 1)
      for (int64_t blk = 0; blk < (pr[i].M + 255) / 256; ++blk) hf[nf++] = EvalBatchFin{i, (int)blk, pr[i].d, pr[i].loo};
  for (int i = 0; i < nprob; ++i) {
    const Prob &p = pr[i];
    if (!p.loo && p.M > 0) std::memcpy(h + q_at + sizeof(double) * p.offQ, pos + p.offQ, sizeof(double) * p.d * p.M);
  }

  // ---- one copy in, the launches, one copy back, one synchronise
  Drain drain{c.stream};
  KDE_CUDA(cudaMemcpyAsync(dv, h, bytes, cudaMemcpyHostToDevice, c.stream));
  KDE_CUDA(cudaEventRecord(c.ev0, c.stream));
  int launches = 0;
  for (const Launch &L : launches_k2b) {
    const cudaError_t e = L.loo ? launch_eval_batch<true>(L.d, L.B, L.n, c.stream)
                                : launch_eval_batch<false>(L.d, L.B, L.n, c.stream);
    if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "%s: K2b launch: %s", fn, cudaGetErrorString(e));
    ++launches;
  }
  if (nfin) {
    eval_batch_finalize_kernel<<<(unsigned)nfin, 256, 0, c.stream>>>(reinterpret_cast<const EvalBatchProb *>(dv + prob_at),
                                                                       reinterpret_cast<const EvalBatchFin *>(dv + fin_at));
    KDE_CUDA(cudaGetLastError());
    ++launches;
  }
  KDE_CUDA(cudaEventRecord(c.ev1, c.stream));
  if (offO) KDE_CUDA(cudaMemcpyAsync(p_out, dO.p, sizeof(double) * offO, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c.ev0, c.ev1);
  c.last_ms = ms;
  c.last_launches = launches;
  return 0;
}

int kde_lcv_batch(int nprob, const int *d, const int64_t *N, const double *points, double *bw_std_out, int *nloo_out) {
  if (int rc = ensure_init()) return rc;
  Context &c = ctx();
  const char *fn = "kde_lcv_batch";
  if (nprob < 0) KDE_FAIL(3, "%s: nprob=%d < 0", fn, nprob);
  if (nprob == 0) return 0;
  if (!d || !N || !points || !bw_std_out) KDE_FAIL(2, "%s: NULL argument", fn);

  // ---- every problem checked as kde_lcv checks it
  std::vector<int64_t> offP(nprob), offB(nprob), out5_at(nprob, -1);
  int64_t np = 0, nb = 0, nsmall = 0, nitems = 0, n5 = 0;
  for (int i = 0; i < nprob; ++i) {
    if (d[i] < 1) KDE_FAIL(3, "%s: problem %d: d must be >= 1", fn, i);
    if (N[i] < 2) KDE_FAIL(3, "%s: problem %d: at least two points are needed for cross validation", fn, i);
    if (2 * N[i] >= (int64_t)std::numeric_limits<int32_t>::max()) KDE_FAIL(3, "%s: problem %d: N too large", fn, i);
    offP[i] = np;
    offB[i] = nb;
    if (N[i] <= LCV_FUSED_MAX) {
      out5_at[i] = n5;
      n5 += 5 * d[i];
      nsmall += (int64_t)d[i] * N[i];
      nitems += d[i];
    }
    np += (int64_t)d[i] * N[i];
    nb += d[i];
  }
  if (nitems >= ((int64_t)1 << 31)) KDE_FAIL(3, "%s: 2^31 (point set, dimension) items or more", fn);

  // ---- the small point sets: one staging area (items | points), one copy, one launch, one copy back
  double kernel_ms = 0.0;
  int launches = 0;
  if (nitems) {
    const size_t item_at = 0;
    size_t bytes = up256(sizeof(LcvBatchItem) * nitems);
    const size_t p_at = bytes;
    bytes += up256(sizeof(double) * nsmall);
    char *h = nullptr;
    if (int rc = batch_stage(bytes, &h)) return rc;
    DevBuf dBlob(c.stream), dO(c.stream);
    KDE_CUDA(dBlob.alloc(bytes));
    KDE_CUDA(dO.alloc(sizeof(double) * n5));
    char *dv = dBlob.as<char>();
    LcvBatchItem *hi = reinterpret_cast<LcvBatchItem *>(h + item_at);
    int64_t ni = 0, ps = 0;
    for (int i = 0; i < nprob; ++i) {
      if (out5_at[i] < 0) continue;
      std::memcpy(h + p_at + sizeof(double) * ps, points + offP[i], sizeof(double) * d[i] * N[i]);
      const double w2 = lcv_points_w2(N[i]);
      for (int k = 0; k < d[i]; ++k) {
        LcvBatchItem &it = hi[ni++];
        it.pts = reinterpret_cast<const double *>(dv + p_at) + ps;
        it.out = dO.as<double>() + out5_at[i];
        it.N = (int)N[i];
        it.d = d[i];
        it.dim = k;
        it.pad_ = 0;
        it.w2 = w2;
      }
      ps += (int64_t)d[i] * N[i];
    }
    std::vector<double> out5(n5);
    Drain drain{c.stream};
    KDE_CUDA(cudaMemcpyAsync(dv, h, bytes, cudaMemcpyHostToDevice, c.stream));
    KDE_CUDA(cudaEventRecord(c.ev0, c.stream));
    if (int rc = kde_lcv_points_batch_device((int)nitems, reinterpret_cast<const LcvBatchItem *>(dv + item_at), c.stream))
      return rc;
    ++launches;
    KDE_CUDA(cudaEventRecord(c.ev1, c.stream));
    KDE_CUDA(cudaMemcpyAsync(out5.data(), dO.p, sizeof(double) * n5, cudaMemcpyDeviceToHost, c.stream));
    KDE_CUDA(cudaStreamSynchronize(c.stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c.ev0, c.ev1);
    kernel_ms = ms;
    for (int i = 0; i < nprob; ++i)
      if (out5_at[i] >= 0)
        lcv_points_finish(d[i], out5.data() + out5_at[i], bw_std_out + offB[i], nloo_out ? nloo_out + offB[i] : nullptr);
  }

  // ---- the larger point sets: kde_lcv's host route (lock-step golden searches over the tiled LOO kernels), one by one
  for (int i = 0; i < nprob; ++i) {
    if (out5_at[i] >= 0) continue;
    if (int rc = kde_lcv(d[i], N[i], points + offP[i], 0, N[i], nullptr, nullptr, bw_std_out + offB[i],
                         nloo_out ? nloo_out + offB[i] : nullptr)) {
      const std::string msg = get_error();
      KDE_FAIL(rc, "%s: problem %d: %s", fn, i, msg.c_str());
    }
    kernel_ms += c.last_ms;
    launches += c.last_launches;
  }
  c.last_ms = kernel_ms;
  c.last_launches = launches;
  return 0;
}

}  // namespace kdeb200
