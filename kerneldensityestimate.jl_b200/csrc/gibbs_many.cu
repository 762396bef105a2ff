// gibbs_many.cu -- host side of the single Gibbs call of more than KDEB200_MAX_DENS densities (DESIGN.md "K1m").
// GibbsParams, which K1, K1w, K1f and K1x take as their kernel parameter, holds KDEB200_MAX_DENS densities, and its
// layout is part of those kernels' code.  A larger product runs K1b's kernel (gibbs_batch_kernel.cuh) as a one-problem
// launch at a state capacity of 32 or 64 densities: K1's schedule from the schedule cache (route K1, the same plan),
// the per-density data in a device-memory descriptor, the sample slice [s0, s1) and the optional level labels.  The
// kernel is K1's arithmetic, so labels and points are K1's.  gibbs_many_d<N>.cu instantiate it per dimension.
#include <cstring>
#include <memory>

#include "gibbs.cuh"
#include "gibbs_batch_kernel.cuh"

namespace kdeb200 {

#define GM_EXTERN(D) extern template cudaError_t launch_gibbs_many_d<D>(const BatchParams &, bool, int, int, cudaStream_t);
GM_EXTERN(1) GM_EXTERN(2) GM_EXTERN(3) GM_EXTERN(4) GM_EXTERN(5) GM_EXTERN(6) GM_EXTERN(7) GM_EXTERN(8)
#undef GM_EXTERN

namespace {
template <int MDC>
int many_launch(const kdeb200_tree_t *trees, int ndens, int L, int64_t perU, int64_t perN, const SchedEntry &E,
                bool masked, int add_entropy, const uint8_t *dimmask, const double *d_randU, const double *d_randN,
                uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices, int64_t *d_level_labels,
                cudaStream_t st) {
  Context &c = ctx();
  const int d = trees[0]->d;
  const int64_t grid = (s1 - s0 + GB_THREADS - 1) / GB_THREADS;
  if (grid >= ((int64_t)1 << 31)) KDE_FAIL(3, "gibbs: more than 2^31 blocks of %d samples in one launch", GB_THREADS);
  using Prob = BatchProbT<MDC>;
  struct alignas(16) Blob {  // what the one copy carries: the descriptor and the block prefix {0, grid}
    Prob p;
    int block0[4];
  };
  auto h = std::make_unique<Blob>();
  std::memset(h.get(), 0, sizeof(Blob));
  Prob &b = h->p;
  b.draws = E.d_draws;
  b.tiles = E.d_tiles;
  b.randU = d_randU;
  b.randN = d_randN;
  b.points = d_points;
  b.indices = d_indices;
  b.Np = s1;  // the kernel's samples run from BatchParams::s0 to here
  b.perU = perU;
  b.perN = perN;
  b.seed = seed;
  b.ndraws = E.ndraws;
  b.ntiles = E.ntiles;
  b.M = ndens;
  b.L = L;
  b.add_entropy = add_entropy ? 1 : 0;
  for (int j = 0; j < ndens; ++j) {
    b.root_rec[j] = trees[j]->d_buf + trees[j]->levels[0].offC;
    b.labels[j] = trees[j]->d_labels;
    for (int k = 0; k < d; ++k) {
      b.hvar[j][k] = trees[j]->hvar[k];
      b.mask[j][k] = dimmask ? (dimmask[j * d + k] != 0) : 1;
    }
  }
  for (int j = 0; j < ndens; ++j)
    for (int k = 0; k < d; ++k) {
      unsigned char o = 0;
      for (int i = 0; i < ndens; ++i)
        if (i != j && b.mask[i][k]) o = 1;
      b.other[j][k] = o;
    }
  h->block0[1] = (int)grid;

  // The copy is from pageable memory: it has read the host blob when it returns, and runs in stream order before the
  // launch; the buffer is released in stream order after it.
  Blob *dv = nullptr;
  KDE_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&dv), sizeof(Blob), st));
  cudaError_t e = cudaMemcpyAsync(dv, h.get(), sizeof(Blob), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    BatchParams B;
    std::memset(&B, 0, sizeof(B));
    B.probs = &dv->p;
    B.block0 = dv->block0;
    B.nprob = 1;
    B.exptab = c.d_exptab;
    B.ec = make_exp_consts();
    B.s0 = s0;
    B.level_labels = d_level_labels;
    e = with_d(d, [&](auto D) { return launch_gibbs_many_d<decltype(D)::value>(B, masked, ndens, (int)grid, st); });
  }
  cudaFreeAsync(dv, st);
  if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "gibbs (many densities) kernel launch: %s", cudaGetErrorString(e));
  return 0;
}
}  // namespace

int gibbs_many_device(const kdeb200_tree_t *trees, int ndens, int L, int64_t perU, int64_t perN, int Niter,
                      int add_entropy, const uint8_t *dimmask, const double *d_randU, const double *d_randN,
                      uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                      int64_t *d_level_labels, cudaStream_t st, int *launches) {
  const int d = trees[0]->d;
  for (int j = 0; j < ndens; ++j)
    if (trees[j]->degenerate)
      KDE_FAIL(5, "gibbs: density %d has a zero, non-finite or out-of-range (variance outside [1e-30, 1e30]) bandwidth / "
                  "mean / weight; products of more than %d densities run the restructured arithmetic only, which "
                  "cannot evaluate it", j, KDEB200_MAX_DENS);
  bool masked = false;
  for (int j = 0; j < ndens * d && dimmask; ++j)
    if (!dimmask[j]) masked = true;

  SchedEntry key;  // K1's schedule: the same plan, so the cache may share it with K1 (the key holds M)
  key.M = ndens;
  key.T = Niter;
  key.masked = masked;
  for (int j = 0; j < ndens; ++j) key.trees[j] = trees[j];
  SchedEntry E;
  if (int rc = sched_get(ROUTE_K1, trees, L, key, &E, nullptr)) return rc;

  int rc = ndens <= 32 ? many_launch<32>(trees, ndens, L, perU, perN, E, masked, add_entropy, dimmask, d_randU, d_randN,
                                         seed, s0, s1, d_points, d_indices, d_level_labels, st)
                       : many_launch<KDEB200_MAX_DENS_LARGE>(trees, ndens, L, perU, perN, E, masked, add_entropy,
                                                             dimmask, d_randU, d_randN, seed, s0, s1, d_points,
                                                             d_indices, d_level_labels, st);
  if (rc) return rc;
  if (launches) *launches += 1;
  return 0;
}

}  // namespace kdeb200
