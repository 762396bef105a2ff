// gibbs_f32.cu -- host side of K1f (FP32 Gibbs sampler): the FP32 pair records of a tree set under the call's shared affine
// map, the precision switch, launch.  The schedule is gibbs.cu's (cache) and gibbs_plan.cuh's (draws, chunks, tiles);
// the kernel lives in gibbs_f32_kernel.cuh and is instantiated once per dimension in gibbs_f32_d<N>.cu.
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "gibbs.cuh"
#include "gibbs_plan.cuh"

namespace kdeb200 {

#define GF_EXTERN(D) extern template cudaError_t launch_gibbs_f32_d<D>(const GibbsParams &, int, size_t, cudaStream_t, int);
GF_EXTERN(1) GF_EXTERN(2) GF_EXTERN(3) GF_EXTERN(4) GF_EXTERN(5) GF_EXTERN(6) GF_EXTERN(7) GF_EXTERN(8)
#undef GF_EXTERN

// ---- FP64 level records -> FP32 pair records ----------------------------------------------------------------
struct PrepDesc {
  const double *src;  // variant A: [m.., lnw] records; B, C: [m.., b.., lnw] records
  float *dst;
  int n, variant, src_stride, dst_stride;
};
struct PrepMap {
  double ctr[KDEB200_MAX_DIM], isig[KDEB200_MAX_DIM];
};

__global__ void gibbs_f32_prep_kernel(const PrepDesc *descs, int D, PrepMap mp) {
  const PrepDesc pd = descs[blockIdx.y];
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (2 * p >= pd.n) return;
  float *o = pd.dst + (size_t)p * pd.dst_stride;
  const float inf = __int_as_float(0x7f800000);
  for (int hh = 0; hh < 2; ++hh) {
    const int z = 2 * p + hh;
    const bool ok = z < pd.n;  // an odd level is padded with a node of probability zero
    const double *r = pd.src + (size_t)(ok ? z : 0) * pd.src_stride;
    // (clamped: a dimension masked out for this density may hold anything, and inf * 0 would poison the sum)
    for (int k = 0; k < D; ++k) o[2 * k + hh] = ok ? (float)fmin(fmax((r[k] - mp.ctr[k]) * mp.isig[k], -1e30), 1e30) : 0.f;
    if (pd.variant == VAR_A) {
      o[2 * D + hh] = ok ? (float)(-r[D] * GF_LOG2E) : inf;  // -log2 w  (w = 0: +inf -> p = 0)
    } else {
      double sl = 0.0;
      for (int k = 0; k < D; ++k) {
        const double b = fmin(fmax(r[D + k] * mp.isig[k] * mp.isig[k], 1e-30), 1e30);
        sl += log2(b);
        o[2 * (D + k) + hh] = ok ? (float)(pd.variant == VAR_B ? GF_HL2E / b : b) : (pd.variant == VAR_B ? 0.f : 1.f);
      }
      const double lw2 = r[2 * D] * GF_LOG2E;
      o[4 * D + hh] = ok ? (float)(pd.variant == VAR_B ? -(lw2 - 0.5 * sl) : -lw2) : inf;
    }
  }
  const int used = (pd.variant == VAR_A) ? 2 * (D + 1) : 2 * (2 * D + 1);
  for (int k = used; k < pd.dst_stride; ++k) o[k] = 0.f;
}

// ---- host side ---------------------------------------------------------------------------------------------------
namespace {
std::atomic<int> g_gibbs_precision{KDEB200_F64};
}  // namespace

int gibbs_precision() {
  if (const char *ev = getenv("KDEB200_GIBBS_F32")) return atoi(ev) ? KDEB200_F32 : KDEB200_F64;
  return g_gibbs_precision.load();
}
int gibbs_set_precision(int p) {
  if (p != KDEB200_F64 && p != KDEB200_F32) KDE_FAIL(3, "set_gibbs_precision: KDEB200_F64 or KDEB200_F32");
  g_gibbs_precision.store(p);
  return 0;
}

// The affine map shared by the call's densities: centre of the root means; per dimension the largest root standard
// deviation (data spread + bandwidth) pooled with the spread of the centres.  Refuses bandwidths FP32 cannot normalise.
static int make_map(const kdeb200_tree_t *trees, int M, int d, const unsigned char (*mask)[KDEB200_MAX_DIM], PrepMap &mp) {
  for (int k = 0; k < d; ++k) {
    double c = 0.0;
    int na = 0;
    for (int j = 0; j < M; ++j)
      if (mask[j][k]) c += trees[j]->root_mean[k], ++na;
    if (na == 0) {  // nobody reads this dimension (partialDimMask): any finite map will do
      mp.ctr[k] = 0.0;
      mp.isig[k] = 1.0;
      continue;
    }
    c /= na;
    double v = 0.0;
    for (int j = 0; j < M; ++j) {
      if (!mask[j][k]) continue;
      const double dv = trees[j]->root_mean[k] - c;
      const double vj = trees[j]->root_var[k] + dv * dv;
      if (vj > v) v = vj;
    }
    if (!(v > 0.0) || !std::isfinite(v) || !std::isfinite(c)) KDE_FAIL(8, "gibbs (FP32): degenerate spread in dimension %d", k + 1);
    mp.ctr[k] = c;
    mp.isig[k] = 1.0 / std::sqrt(v);
    for (int j = 0; j < M; ++j) {
      if (!mask[j][k]) continue;
      const double hn = trees[j]->hvar[k] / v;
      if (!(hn >= 1e-8))
        KDE_FAIL(8, "gibbs (FP32): the bandwidth of density %d in dimension %d is %.3g of the data spread; the FP32 sampler "
                    "needs >= 1e-4 (products of up to four normalised variances must stay normal floats); use KDEB200_F64",
                 j + 1, k + 1, std::sqrt(hn));
    }
  }
  for (int k = d; k < KDEB200_MAX_DIM; ++k) mp.ctr[k] = 0.0, mp.isig[k] = 1.0;
  return 0;
}

// the FP32 pair records of every block of the plan, under the affine map of the entry's tree set and mask
int gibbs32_build(const kdeb200_tree_t *trees, Plan &S, SchedEntry &e) {
  Context &c = ctx();
  const int d = trees[0]->d;
  PrepMap mp;
  if (int rc = make_map(trees, e.M, d, e.mask, mp)) return rc;
  std::memcpy(e.nctr, mp.ctr, sizeof(e.nctr));
  std::memcpy(e.nisig, mp.isig, sizeof(e.nisig));
  std::vector<PrepDesc> preps;
  int maxpairs = 1;
  for (const PlanBlock &b : S.blocks) {
    const kdeb200_tree_s *t = trees[b.j];
    const Level &lv = t->levels[b.level];
    PrepDesc pd;
    pd.src = t->d_buf + (b.variant == VAR_A ? lv.offA : lv.offC);
    pd.dst = e.d_rec + b.off;
    pd.n = (int)lv.n;
    pd.variant = b.variant;
    pd.src_stride = (b.variant == VAR_A) ? t->SA : t->SC;
    pd.dst_stride = gf_stride(d, b.variant);
    if ((pd.n + 1) / 2 > maxpairs) maxpairs = (pd.n + 1) / 2;
    preps.push_back(pd);
  }
  for (size_t i = 0; i < S.draws.size(); ++i) {  // K1f reads every level from its pair records
    S.draws[i].rec = reinterpret_cast<const double *>(e.d_rec + S.blocks[S.block[i]].off);
    S.draws[i].stride = gf_stride(d, S.draws[i].variant);
  }
  PrepDesc *d_prep = nullptr;
  KDE_CUDA(cudaMallocAsync(&d_prep, sizeof(PrepDesc) * preps.size(), c.stream));
  cudaError_t err = cudaMemcpyAsync(d_prep, preps.data(), sizeof(PrepDesc) * preps.size(), cudaMemcpyHostToDevice, c.stream);
  if (err == cudaSuccess) {
    gibbs_f32_prep_kernel<<<dim3((unsigned)((maxpairs + 127) / 128), (unsigned)preps.size()), 128, 0, c.stream>>>(d_prep, d, mp);
    err = cudaGetLastError();
  }
  if (err == cudaSuccess) err = cudaStreamSynchronize(c.stream);  // preps is pageable host memory
  cudaFreeAsync(d_prep, c.stream);
  if (err != cudaSuccess) KDE_FAIL(100 + (int)err, "gibbs (FP32): building the schedule: %s", cudaGetErrorString(err));
  return 0;
}

// P arrives filled by gibbs_device with the entry's schedule; this adds the affine map and the slow-draw counter
int gibbs32_launch(GibbsParams &P, const SchedEntry &E, int d, cudaStream_t st) {
  Context &c = ctx();
  unsigned long long *d_count = nullptr;
  if (int rc = gibbs_counters(&d_count)) return rc;
  P.slow_draws = d_count;
  for (int k = 0; k < KDEB200_MAX_DIM; ++k) {
    P.nctr[k] = E.nctr[k];
    P.nisig[k] = E.nisig[k];
  }
  const size_t smem = GB_STAGES * GB_TILE_BYTES;
  const cudaError_t e = with_d(d, [&](auto D) {
    return launch_gibbs_f32_d<decltype(D)::value>(P, P.nbatches, smem, st, c.sm_count);
  });
  if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "gibbs (FP32) kernel launch: %s", cudaGetErrorString(e));
  return 0;
}

}  // namespace kdeb200
