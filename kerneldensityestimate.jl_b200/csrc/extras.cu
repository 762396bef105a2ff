// extras.cu -- the callers either side of the evaluation seam that the reference runs as many small host calls
// (SURVEY.md 8f.2 / 8f.4), each as ONE launch over the resident density:
//   * eval_marginals: every 1-D marginal of a density on its own grid.  getKDEMax (src/DualTree01.jl:558-569) builds a
//     marginal tree per dimension (src/KDE01.jl:143-153) just to evaluate it on 200 grid points; a Gaussian product
//     kernel's marginal on dimension k is sum_i w_i N(x; x_ik, h_k^2), read straight off the d-dimensional leaf records.
//   * sample: sample(npd, Npts) (src/KDE01.jl:164-183) -- inverse-CDF draw of component indices from SORTED uniforms over
//     the cumulative weights in ORIGINAL point order, plus a Gaussian kernel perturbation; feeds rand / resample
//     (src/KDE01.jl:196-198, src/BallTreeDensity01.jl:312-334).
#include <cub/device/device_radix_sort.cuh>

#include <cmath>
#include <unordered_set>
#include <vector>

#include "eval_shared.cuh"
#include "gibbs.cuh"
#include "sample.cuh"
#include "tree.cuh"

namespace kdeb200 {

// ---------------------------------------------------------------- marginals on grids ------------------------
// grid: d x G (row k = the G query abscissae of dimension k); out: d x G densities of the k-th marginal
__global__ void __launch_bounds__(128) eval_marginals_kernel(const double *__restrict__ leaf, int SE, int d, int64_t N,
                                                             const double *__restrict__ grid, int64_t G,
                                                             const double *__restrict__ exptab, ExpConsts ec,
                                                             const double *__restrict__ ich, const double *__restrict__ norm,
                                                             double *__restrict__ out) {
  __shared__ __align__(16) double tab[KDE_EXP_TAB];
  for (int i = threadIdx.x; i < KDE_EXP_TAB; i += blockDim.x) tab[i] = exptab[i];
  __syncthreads();
  const int k = blockIdx.y;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool ok = g < G;
  const double x = grid[(int64_t)k * G + (ok ? g : G - 1)];
  const double c = ich[k];
  double s0 = 0.0, s1 = 0.0;  // leaf order, two interleaved chains folded at the end
  int64_t i = 0;
  for (; i + 2 <= N; i += 2) {
    const double xa = __ldg(leaf + i * SE + k), wa = __ldg(leaf + i * SE + d);
    const double xb = __ldg(leaf + (i + 1) * SE + k), wb = __ldg(leaf + (i + 1) * SE + d);
    const double da = __dadd_rn(x, -xa), db = __dadd_rn(x, -xb);
    s0 = __fma_rn(kde_exp_flush(__dmul_rn(__dmul_rn(da, da), c), tab, ec), wa, s0);
    s1 = __fma_rn(kde_exp_flush(__dmul_rn(__dmul_rn(db, db), c), tab, ec), wb, s1);
  }
  for (; i < N; ++i) {
    const double xa = __ldg(leaf + i * SE + k), wa = __ldg(leaf + i * SE + d);
    const double da = __dadd_rn(x, -xa);
    s0 = __fma_rn(kde_exp_flush(__dmul_rn(__dmul_rn(da, da), c), tab, ec), wa, s0);
  }
  double s = s0 + s1;
  if (s < EV_TINY) {  // far tail: exact, sequential (libdevice exp), like eval.cu
    s = 0.0;
    for (int64_t j = 0; j < N; ++j) {
      const double df = x - leaf[j * SE + k];
      s = __fma_rn(exp(df * df * c), leaf[j * SE + d], s);
    }
  }
  if (ok) out[(int64_t)k * G + g] = 0.5 * (s + s) / norm[k];
}

int eval_marginals_device(kdeb200_tree_t bd, const double *d_grid, int64_t G, double *d_out, cudaStream_t st, int *launches) {
  Context &c = ctx();
  if (G <= 0) return 0;
  const int d = bd->d;
  double h[2 * KDEB200_MAX_DIM];
  for (int k = 0; k < d; ++k) {
    const double v = bd->hvar[k];
    if (!(v > 0.0) || !std::isfinite(v)) KDE_FAIL(5, "eval_marginals: bandwidth variance must be finite and > 0");
    h[k] = -0.5 / v;
    h[KDEB200_MAX_DIM + k] = std::sqrt(2.0 * M_PI) * std::sqrt(v);  // (2 pi)^(1/2) sqrt(var): src/DualTree01.jl:325-330, d = 1
  }
  double *d_h = nullptr;
  KDE_CUDA(cudaMallocAsync(&d_h, sizeof(h), st));
  KDE_CUDA(cudaMemcpyAsync(d_h, h, sizeof(h), cudaMemcpyHostToDevice, st));
  KDE_CUDA(cudaStreamSynchronize(st));  // h is a stack array
  dim3 grid((unsigned)((G + 127) / 128), (unsigned)d);
  eval_marginals_kernel<<<grid, 128, 0, st>>>(bd->d_leaf, bd->SE, d, bd->N, d_grid, G, c.d_exptab, make_exp_consts(), d_h,
                                              d_h + KDEB200_MAX_DIM, d_out);
  KDE_CUDA(cudaGetLastError());
  KDE_CUDA(cudaFreeAsync(d_h, st));
  if (launches) *launches += 1;
  return 0;
}

// ---------------------------------------------------------------- sample ------------------------------------
__global__ void sample_uniforms_kernel(uint64_t seed, int64_t Np, double *__restrict__ u) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Np) u[i] = philox_uniform(seed ^ 0x9E3779B97F4A7C15ull, (uint64_t)i, 0u);
}

// t: SORTED uniforms; the body is sample_one (sample.cuh), shared with the batched kernel (sample_batch.cu)
__global__ void sample_kernel(const double *__restrict__ t, const double *__restrict__ cw, const int64_t *__restrict__ leaf_of,
                              const double *__restrict__ leaf, int SE, int d, int64_t N, int64_t Np,
                              const double *__restrict__ randn_in, uint64_t seed, const double *__restrict__ bw_std,
                              double *__restrict__ points, int64_t *__restrict__ idx) {
  const int64_t ii = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (ii >= Np) return;
  sample_one(t[ii], ii, cw, leaf_of, leaf, SE, d, N, randn_in, seed, bw_std, points, idx);
}

namespace {
struct Drain {  // an error return after the first enqueue waits for the enqueued work: the staging buffer is reused
  cudaStream_t st;
  ~Drain() { cudaStreamSynchronize(st); }
};
}  // namespace

int sample_tables(const kdeb200_tree_t *trees, int n) {
  Context &c = ctx();
  std::vector<kdeb200_tree_t> todo;
  std::unordered_set<kdeb200_tree_t> seen;
  int64_t tot = 0;
  for (int i = 0; i < n; ++i) {
    const kdeb200_tree_t t = trees[i];
    if (!t || t->d_cw || !seen.insert(t).second) continue;
    todo.push_back(t);
    tot += t->N;
  }
  if (todo.empty()) return 0;
  // pinned staging: leaf weights of every handle (tot doubles), then per handle its [cw | leaf_of] table (2 N words)
  char *h = nullptr;
  if (int rc = batch_stage(24 * (size_t)tot, &h)) return rc;
  double *w = reinterpret_cast<double *>(h);
  char *tab = h + 8 * (size_t)tot;
  Drain drain{c.stream};
  int64_t off = 0;
  for (const kdeb200_tree_t t : todo) {
    KDE_CUDA(cudaMemcpy2DAsync(w + off, sizeof(double), t->d_leaf + t->d, sizeof(double) * t->SE, sizeof(double), t->N,
                               cudaMemcpyDeviceToHost, c.stream));
    off += t->N;
  }
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  off = 0;
  for (const kdeb200_tree_t t : todo) {
    const int64_t N = t->N;
    const double *leafw = w + off;
    double *cw = reinterpret_cast<double *>(tab + 16 * (size_t)off);
    int64_t *leaf_of = reinterpret_cast<int64_t *>(tab + 16 * (size_t)off + 8 * (size_t)N);
    for (int64_t s = 0; s < N; ++s) {
      cw[t->h_perm[s]] = leafw[s];
      leaf_of[t->h_perm[s]] = s;
    }
    double run = 0.0;
    for (int64_t i = 0; i < N; ++i) {
      run += cw[i];
      cw[i] = run;
    }
    for (int64_t i = 0; i < N; ++i) cw[i] = cw[i] / run;
    off += N;
  }
  off = 0;
  for (const kdeb200_tree_t t : todo) {
    const int64_t N = t->N;
    char *base = nullptr;
    KDE_CUDA(cudaMallocAsync(&base, 16 * (size_t)N, c.stream));
    const cudaError_t e = cudaMemcpyAsync(base, tab + 16 * (size_t)off, 16 * (size_t)N, cudaMemcpyHostToDevice, c.stream);
    if (e != cudaSuccess) {
      cudaFreeAsync(base, c.stream);
      KDE_FAIL(100 + (int)e, "sample: uploading the cumulative weights: %s", cudaGetErrorString(e));
    }
    t->d_cw = reinterpret_cast<double *>(base);
    t->d_leaf_of = reinterpret_cast<int64_t *>(base + 8 * (size_t)N);
    off += N;
  }
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}

// d_cw / d_leaf_of: built on first use from the weights the tree was created with (sample_tables)
int sample_device(kdeb200_tree_t bd, int64_t Np, uint64_t seed, const double *d_randU, const double *d_randN,
                  double *d_points, int64_t *d_idx, cudaStream_t st, int *launches) {
  if (Np <= 0) return 0;
  const int d = bd->d;
  const int64_t N = bd->N;
  if (int rc = sample_tables(&bd, 1)) return rc;
  double bw[KDEB200_MAX_DIM];
  for (int k = 0; k < d; ++k) bw[k] = std::sqrt(bd->hvar[k]);  // getBW = sqrt of the leaf variances
  size_t tmp_bytes = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, (const double *)nullptr, (double *)nullptr, (int)Np, 0, 64, st);
  auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t b_u = up(8 * (size_t)Np), b_bw = 256, b_tmp = up(tmp_bytes);
  char *base = nullptr;
  KDE_CUDA(cudaMallocAsync(&base, 2 * b_u + b_bw + b_tmp, st));
  double *u_in = reinterpret_cast<double *>(base), *u_sorted = reinterpret_cast<double *>(base + b_u);
  double *d_bw = reinterpret_cast<double *>(base + 2 * b_u);
  void *d_tmp = base + 2 * b_u + b_bw;
  KDE_CUDA(cudaMemcpyAsync(d_bw, bw, sizeof(double) * d, cudaMemcpyHostToDevice, st));
  KDE_CUDA(cudaStreamSynchronize(st));  // bw is a stack array
  const double *src_u = d_randU;
  if (!d_randU) {
    sample_uniforms_kernel<<<(unsigned)((Np + 255) / 256), 256, 0, st>>>(seed, Np, u_in);
    src_u = u_in;
  }
  cudaError_t e = cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, src_u, u_sorted, (int)Np, 0, 64, st);  // uniforms are >= 0
  if (e != cudaSuccess) {
    cudaFreeAsync(base, st);
    KDE_FAIL(100 + (int)e, "sample: sorting the uniforms: %s", cudaGetErrorString(e));
  }
  sample_kernel<<<(unsigned)((Np + 255) / 256), 256, 0, st>>>(u_sorted, bd->d_cw, bd->d_leaf_of, bd->d_leaf, bd->SE, d, N, Np,
                                                              d_randN, seed, d_bw, d_points, d_idx);
  KDE_CUDA(cudaGetLastError());
  KDE_CUDA(cudaFreeAsync(base, st));
  if (launches) *launches += 3;
  return 0;
}

}  // namespace kdeb200
