// sample_batch.cu -- S4b: many independent sample(npd, Npts) problems (src/KDE01.jl:164-183) in one blocking call
// (kdeb200_sample_batch), and resample(p, Np) (src/BallTreeDensity01.jl:312-334) of many densities (kdeb200_resample_batch).
//
// Sampling.  Every problem is checked as kdeb200_sample checks it before anything runs.  The cumulative-weight tables of
// all handles that lack one are built together (sample_tables: two synchronises for the whole batch).  Problems with
// Np <= SB_MAX run in ONE launch of one CTA per problem: the CTA loads or draws its uniforms, sorts them in shared
// memory and runs sample_kernel's body (sample_one, sample.cuh) on each.  A sorted array is unique and both sorts are
// cub's stable radix sort with the same key transform, so the order -- and with it every point and index -- is the single
// call's.  Larger problems go through sample_device (the single call's device-wide sort) one by one on the same stream.
// Descriptors and injected streams travel in ONE copy from the context's pinned staging buffer (batch_stage); points and
// indices come back in one copy each.
//
// Resampling.  The samples of the problems with Np <= LCV_FUSED_MAX never leave the device: one
// lcv_golden_points_batch_kernel launch (one CTA per (problem, dimension), as kdeb200_kde_lcv_batch) reads them where
// the sampling wrote them.  Larger problems take kde_lcv's host route on the returned points, one by one.
#include <cub/block/block_radix_sort.cuh>

#include <cmath>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "gibbs.cuh"
#include "lcv.cuh"
#include "sample.cuh"
#include "tree.cuh"

namespace kdeb200 {

int sample_device(kdeb200_tree_t bd, int64_t Np, uint64_t seed, const double *d_randU, const double *d_randN,
                  double *d_points, int64_t *d_idx, cudaStream_t st, int *launches);

// 256 threads x 8 keys: 2048 doubles, 16 KB of shared memory for the sort's exchange (its largest part), so several
// CTAs share an SM; 8 keys per thread keeps the per-pass rank scan short.  Problems of the belief-propagation rounds this
// serves have 100-2000 samples; above SB_MAX the device-wide sort of the single call has enough work to be worth its
// launches.
constexpr int SB_THREADS = 256, SB_KEYS = 8, SB_MAX = SB_THREADS * SB_KEYS;

struct SampleBatchProb {
  const double *cw;         // the handle's tables (sample_tables)
  const int64_t *leaf_of;
  const double *leaf;       // leaf records, stride SE
  const double *randU;      // Np injected uniforms, or null: Philox(seed)
  const double *randN;      // d x Np injected normals, or null: Philox(seed)
  double *points;           // this problem's block of the output
  int64_t *idx;
  int64_t N, Np;
  uint64_t seed;
  int SE, d;
  double bw_std[KDEB200_MAX_DIM];  // sqrt of the leaf variances (getBW)
};

__global__ void __launch_bounds__(SB_THREADS) sample_batch_kernel(const SampleBatchProb *__restrict__ probs) {
  using Sort = cub::BlockRadixSort<double, SB_THREADS, SB_KEYS>;
  __shared__ typename Sort::TempStorage tmp;
  const SampleBatchProb *P = probs + blockIdx.x;
  const int64_t Np = P->Np;
  const double *randU = P->randU;
  const uint64_t seed = P->seed;
  // blocked input: thread t holds uniforms [t*SB_KEYS, (t+1)*SB_KEYS).  The padding is the largest key of cub's order
  // (positive, all other bits set), and it comes after every real key in input order: a stable sort puts it last.
  const double pad = __longlong_as_double(0x7FFFFFFFFFFFFFFFll);
  double u[SB_KEYS];
#pragma unroll
  for (int j = 0; j < SB_KEYS; ++j) {
    const int64_t i = (int64_t)threadIdx.x * SB_KEYS + j;
    u[j] = i >= Np ? pad : (randU ? randU[i] : philox_uniform(seed ^ 0x9E3779B97F4A7C15ull, (uint64_t)i, 0u));
  }
  Sort(tmp).SortBlockedToStriped(u);  // striped output: thread t holds sorted ranks t + j*SB_THREADS
#pragma unroll
  for (int j = 0; j < SB_KEYS; ++j) {
    const int64_t ii = (int64_t)j * SB_THREADS + threadIdx.x;
    if (ii < Np)
      sample_one(u[j], ii, P->cw, P->leaf_of, P->leaf, P->SE, P->d, P->N, P->randN, seed, P->bw_std, P->points, P->idx);
  }
}

namespace {
size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }

struct Drain {  // an error return after the first enqueue waits for the enqueued work: the staging buffer is reused
  cudaStream_t st;
  ~Drain() { cudaStreamSynchronize(st); }
};
}  // namespace

int sample_batch(bool resample, int nprob, const kdeb200_tree_t *trees, const int64_t *Np, const uint64_t *seeds,
                 const double *randU, const int64_t *nU, const double *randN, const int64_t *nN, double *points_out,
                 int64_t *ind_out, double *bw_std_out, int *nloo_out) {
  Context &c = ctx();
  const char *fn = resample ? "resample_batch" : "sample_batch";
  if (nprob < 0) KDE_FAIL(3, "%s: nprob=%d < 0", fn, nprob);
  if (nprob == 0) return 0;
  if (!trees || !Np || !points_out || (!resample && !ind_out) || (resample && !bw_std_out))
    KDE_FAIL(2, "%s: NULL argument", fn);
  if ((randU && !nU) || (randN && !nN)) KDE_FAIL(2, "%s: randU / randN given without nU / nN", fn);

  // ---- every problem checked as kdeb200_sample (and, resampling, kde_lcv) checks it; nothing runs unless all pass
  struct Prob {
    int d;
    int64_t Np, nU, nN, offP, offI, offU, offN, offB, out5;
  };
  std::vector<Prob> pr(nprob);
  int64_t offP = 0, offI = 0, offU = 0, offN = 0, offB = 0, n5 = 0, nitems = 0;
  int nsmall = 0;
  for (int i = 0; i < nprob; ++i) {
    Prob &p = pr[i];
    const kdeb200_tree_t bd = trees[i];
    if (!bd) KDE_FAIL(2, "%s: problem %d: NULL tree", fn, i);
    p.d = bd->d;
    p.Np = Np[i];
    if (p.Np < 0 || p.Np >= ((int64_t)1 << 31)) KDE_FAIL(3, "%s: problem %d: Np=%lld out of range", fn, i, (long long)p.Np);
    if (resample && p.Np < 2)
      KDE_FAIL(3, "%s: problem %d: at least two samples are needed for cross validation (Np=%lld)", fn, i, (long long)p.Np);
    if (resample && 2 * p.Np >= (int64_t)std::numeric_limits<int32_t>::max())
      KDE_FAIL(3, "%s: problem %d: Np too large for cross validation", fn, i);
    if (bd->slot != c.slot) KDE_FAIL(3, "%s: problem %d: the tree lives on another GPU of the set than the primary", fn, i);
    p.nU = nU ? nU[i] : 0;
    p.nN = nN ? nN[i] : 0;
    if (p.nU != 0 && (p.nU != p.Np || !randU))
      KDE_FAIL(7, "%s: problem %d: nU=%lld must be 0 or Np=%lld", fn, i, (long long)p.nU, (long long)p.Np);
    if (p.nN != 0 && (p.nN != (int64_t)p.d * p.Np || !randN))
      KDE_FAIL(7, "%s: problem %d: nN=%lld must be 0 or d*Np=%lld", fn, i, (long long)p.nN, (long long)p.d * p.Np);
    if (p.Np > 0) {
      for (int k = 0; k < p.d; ++k)
        if (!(bd->hvar[k] >= 0.0)) KDE_FAIL(5, "%s: problem %d: negative bandwidth variance (dim %d: %g)", fn, i, k + 1, bd->hvar[k]);
      if ((p.nU == 0 || p.nN == 0) && !seeds) KDE_FAIL(2, "%s: problem %d: NULL seeds for a Philox stream", fn, i);
    }
    p.offP = offP;
    p.offI = offI;
    p.offU = offU;
    p.offN = offN;
    p.offB = offB;
    p.out5 = -1;
    offP += (int64_t)p.d * p.Np;
    offI += p.Np;
    offU += p.nU;
    offN += p.nN;
    offB += p.d;
    if (p.Np > 0 && p.Np <= SB_MAX) ++nsmall;
    if (resample && p.Np <= LCV_FUSED_MAX) {
      p.out5 = n5;
      n5 += 5 * p.d;
      nitems += p.d;
    }
  }
  if (nitems >= ((int64_t)1 << 31)) KDE_FAIL(3, "%s: 2^31 (problem, dimension) items or more", fn);

  // ---- the cumulative-weight tables of every handle that draws and has none yet
  {
    std::vector<kdeb200_tree_t> draw;
    for (int i = 0; i < nprob; ++i)
      if (pr[i].Np > 0) draw.push_back(trees[i]);
    if (int rc = sample_tables(draw.data(), (int)draw.size())) return rc;
  }

  // ---- one staging area: descriptors | LOOCV items | injected uniforms | injected normals
  size_t bytes = 0;
  const size_t prob_at = bytes;
  bytes += up256(sizeof(SampleBatchProb) * nsmall);
  const size_t item_at = bytes;
  bytes += up256(sizeof(LcvBatchItem) * nitems);
  const size_t u_at = bytes;
  bytes += up256(sizeof(double) * offU);
  const size_t n_at = bytes;
  bytes += up256(sizeof(double) * offN);
  char *h = nullptr;
  if (int rc = batch_stage(bytes, &h)) return rc;
  DevBuf dBlob(c.stream), dP(c.stream), dI(c.stream), dO(c.stream);
  KDE_CUDA(dBlob.alloc(bytes));
  KDE_CUDA(dP.alloc(sizeof(double) * offP));
  KDE_CUDA(dI.alloc(sizeof(int64_t) * offI));
  if (n5) KDE_CUDA(dO.alloc(sizeof(double) * n5));
  char *dv = dBlob.as<char>();
  const double *d_u = reinterpret_cast<const double *>(dv + u_at);
  const double *d_n = reinterpret_cast<const double *>(dv + n_at);
  if (offU) std::memcpy(h + u_at, randU, sizeof(double) * offU);
  if (offN) std::memcpy(h + n_at, randN, sizeof(double) * offN);
  SampleBatchProb *hp = reinterpret_cast<SampleBatchProb *>(h + prob_at);
  LcvBatchItem *hi = reinterpret_cast<LcvBatchItem *>(h + item_at);
  int np = 0;
  int64_t ni = 0;
  for (int i = 0; i < nprob; ++i) {
    const Prob &p = pr[i];
    const kdeb200_tree_t bd = trees[i];
    if (p.Np > 0 && p.Np <= SB_MAX) {
      SampleBatchProb &b = hp[np++];
      std::memset(&b, 0, sizeof(b));
      b.cw = bd->d_cw;
      b.leaf_of = bd->d_leaf_of;
      b.leaf = bd->d_leaf;
      b.randU = p.nU ? d_u + p.offU : nullptr;
      b.randN = p.nN ? d_n + p.offN : nullptr;
      b.points = dP.as<double>() + p.offP;
      b.idx = dI.as<int64_t>() + p.offI;
      b.N = bd->N;
      b.Np = p.Np;
      b.seed = (p.nU && p.nN) ? 0 : seeds[i];
      b.SE = bd->SE;
      b.d = p.d;
      for (int k = 0; k < p.d; ++k) b.bw_std[k] = std::sqrt(bd->hvar[k]);  // getBW, as sample_device
    }
    if (p.out5 >= 0) {
      const double w2 = lcv_points_w2(p.Np);
      for (int k = 0; k < p.d; ++k) {
        LcvBatchItem &it = hi[ni++];
        it.pts = dP.as<double>() + p.offP;
        it.out = dO.as<double>() + p.out5;
        it.N = (int)p.Np;
        it.d = p.d;
        it.dim = k;
        it.pad_ = 0;
        it.w2 = w2;
      }
    }
  }

  // ---- one copy in, the launches, one copy back, one synchronise
  Drain drain{c.stream};
  KDE_CUDA(cudaMemcpyAsync(dv, h, bytes, cudaMemcpyHostToDevice, c.stream));
  KDE_CUDA(cudaEventRecord(c.ev0, c.stream));
  int launches = 0;
  if (nsmall) {
    sample_batch_kernel<<<nsmall, SB_THREADS, 0, c.stream>>>(reinterpret_cast<const SampleBatchProb *>(dv + prob_at));
    KDE_CUDA(cudaGetLastError());
    ++launches;
  }
  for (int i = 0; i < nprob; ++i) {  // above SB_MAX: the single call's route, same stream
    const Prob &p = pr[i];
    if (p.Np <= SB_MAX) continue;
    if (int rc = sample_device(trees[i], p.Np, p.nU && p.nN ? 0 : seeds[i], p.nU ? d_u + p.offU : nullptr,
                               p.nN ? d_n + p.offN : nullptr, dP.as<double>() + p.offP, dI.as<int64_t>() + p.offI,
                               c.stream, &launches)) {
      const std::string msg = get_error();
      KDE_FAIL(rc, "%s: problem %d: %s", fn, i, msg.c_str());
    }
  }
  if (nitems) {
    if (int rc = kde_lcv_points_batch_device((int)nitems, reinterpret_cast<const LcvBatchItem *>(dv + item_at), c.stream))
      return rc;
    ++launches;
  }
  KDE_CUDA(cudaEventRecord(c.ev1, c.stream));
  std::vector<double> out5(n5);
  if (offP) KDE_CUDA(cudaMemcpyAsync(points_out, dP.p, sizeof(double) * offP, cudaMemcpyDeviceToHost, c.stream));
  if (offI && ind_out) KDE_CUDA(cudaMemcpyAsync(ind_out, dI.p, sizeof(int64_t) * offI, cudaMemcpyDeviceToHost, c.stream));
  if (n5) KDE_CUDA(cudaMemcpyAsync(out5.data(), dO.p, sizeof(double) * n5, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c.ev0, c.ev1);
  double kernel_ms = ms;

  // ---- the bandwidths: fused results, or kde_lcv's host route on the returned points for Np > LCV_FUSED_MAX
  if (resample) {
    for (int i = 0; i < nprob; ++i) {
      const Prob &p = pr[i];
      int *calls = nloo_out ? nloo_out + p.offB : nullptr;
      if (p.out5 >= 0) {
        lcv_points_finish(p.d, out5.data() + p.out5, bw_std_out + p.offB, calls);
        continue;
      }
      if (int rc = kde_lcv(p.d, p.Np, points_out + p.offP, 0, p.Np, nullptr, nullptr, bw_std_out + p.offB, calls)) {
        const std::string msg = get_error();
        KDE_FAIL(rc, "%s: problem %d: %s", fn, i, msg.c_str());
      }
      kernel_ms += c.last_ms;
      launches += c.last_launches;
    }
  }
  c.last_ms = kernel_ms;
  c.last_launches = launches;
  return 0;
}

}  // namespace kdeb200
