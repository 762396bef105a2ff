// gibbs_exact.cu -- host side of K1x (gibbs_exact_kernel.cuh): routing, the FP32 leaf records laid out for accuracy
// (per-tile centres, log-weights relative to the level's largest), the schedule over them (cached like gibbs.cu's),
// launch and the count of redone draws.
//
// The schedule construction and cache repeat gibbs.cu's build_schedule / sched_get for the internal levels: those are
// static there, and gibbs.cu is one of the sources whose Nsight Compute profile (profiles/ncu_issued.json) is keyed
// by a hash of its text.  They can fold back into one place once that profile is captured again.
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <list>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "gibbs_exact_kernel.cuh"

namespace kdeb200 {

extern std::atomic<uint64_t> g_tree_epoch;
int gibbs_precision();  // gibbs_f32.cu
int gibbs_sizes(const kdeb200_tree_t *trees, int ndens, int Niter, int *nlevels, int64_t *perU, int64_t *perN,
                int64_t *evals);  // gibbs.cu
int gibbs_device(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                 const uint8_t *dimmask, const double *d_randU, int64_t nU, const double *d_randN, int64_t nN,
                 uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                 int64_t *d_level_labels, cudaStream_t st, int *launches);  // gibbs.cu

#define GX_EXTERN(D)                                                                                       \
  extern template cudaError_t launch_gibbs_exact_d<D>(const GibbsParams &, const XParams &, int, size_t, \
                                                      cudaStream_t);                                     \
  extern template cudaError_t occupancy_gibbs_exact_d<D>(int, size_t, int *);
GX_EXTERN(1) GX_EXTERN(2) GX_EXTERN(3) GX_EXTERN(4) GX_EXTERN(5) GX_EXTERN(6) GX_EXTERN(7) GX_EXTERN(8)
#undef GX_EXTERN

// Relative error bound of ex2.approx.ftz.f32 over the exponents K1x feeds it, [-126, 0]: 2^-21 = 4.8e-7, more than three
// times the maximum measured over every float of that range on a B200, 1.44e-7 (tools/ulp_mufu.py, profiles/mufu_ulp.json).
constexpr double GX_EX2_ERR = 0x1.0p-21;

// ---- FP32 leaf records ------------------------------------------------------------------------------------------
struct XPrep {
  const double *src;  // [m.., ln w] records, stride SA
  float *dst;         // pair records, stride gf_stride(d, VAR_A)
  double *stats;      // per tile: min[MAX_DIM] | max[MAX_DIM] | max ln w  (pass a) -> centre[MAX_DIM] (pass b reads)
  int n, src_stride, tnodes;
  double lw2max;
};

// pass a: one CTA per tile, per-dimension min / max and the largest ln w of the tile's nodes
__global__ void gibbs_exact_stats_kernel(const XPrep *preps, int D) {
  const XPrep pd = preps[blockIdx.y];
  const int t = blockIdx.x;
  const int z0 = t * pd.tnodes;
  if (z0 >= pd.n) return;
  const int z1 = min(z0 + pd.tnodes, pd.n);
  __shared__ double red[2 * KDEB200_MAX_DIM + 1][4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = 0; k <= 2 * D; ++k) {
    const bool isw = k == 2 * D, ismax = k >= D;
    const int kk = isw ? D : (k % D);
    double v = ismax ? -INFINITY : INFINITY;
    for (int z = z0 + threadIdx.x; z < z1; z += blockDim.x) {
      const double x = pd.src[(size_t)z * pd.src_stride + kk];
      v = ismax ? fmax(v, x) : fmin(v, x);
    }
    for (int o = 16; o; o >>= 1) {
      const double w = __shfl_xor_sync(0xffffffffu, v, o);
      v = ismax ? fmax(v, w) : fmin(v, w);
    }
    if (lane == 0) red[k][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x <= 2 * D) {
    const int k = threadIdx.x;
    const bool ismax = k >= D;
    double v = red[k][0];
    for (int w = 1; w < 4; ++w) v = ismax ? fmax(v, red[k][w]) : fmin(v, red[k][w]);
    double *o = pd.stats + (size_t)t * (2 * KDEB200_MAX_DIM + 1);
    o[k == 2 * D ? 2 * KDEB200_MAX_DIM : (ismax ? KDEB200_MAX_DIM + k - D : k)] = v;
  }
}

// pass b: pair records [m'_0(a), m'_0(b), .., lw'(a), lw'(b), pad], m' = m - centre(tile), lw' = lw2max - log2 w >= 0
__global__ void gibbs_exact_rec_kernel(const XPrep *preps, const double *ctrs_base, const size_t *ctr_off, int D) {
  const XPrep pd = preps[blockIdx.y];
  const double *ctr = ctrs_base + ctr_off[blockIdx.y];
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (2 * p >= pd.n) return;
  const int stride = gf_stride(D, VAR_A);
  float *o = pd.dst + (size_t)p * stride;
  const double *c = ctr + (size_t)((2 * p) / pd.tnodes) * KDEB200_MAX_DIM;
  for (int hh = 0; hh < 2; ++hh) {
    const int z = 2 * p + hh;
    const bool ok = z < pd.n;  // an odd level is padded with a node of probability zero (finite: no 0 * inf)
    const double *r = pd.src + (size_t)(ok ? z : 0) * pd.src_stride;
    for (int k = 0; k < D; ++k) o[2 * k + hh] = ok ? (float)(r[k] - c[k]) : 0.f;
    o[2 * D + hh] = ok ? (float)fmax(pd.lw2max - r[D] * GF_LOG2E, 0.0) : 1e30f;
  }
  for (int k = 2 * (D + 1); k < stride; ++k) o[k] = 0.f;
}

// ---- schedule cache ---------------------------------------------------------------------------------------------
namespace {
struct SchedX {
  uint64_t epoch = 0;
  int slot = 0, M = 0, T = 0;
  kdeb200_tree_t trees[KDEB200_MAX_DENS] = {nullptr};
  char *d_base = nullptr;  // draws | xdraws | tiles | counters | centres | FP32 records
  Draw *d_draws = nullptr;
  XDraw *d_xd = nullptr;
  TileDesc *d_tiles = nullptr;
  int *d_counters = nullptr;
  int ndraws = 0, ntiles = 0;
  unsigned next_counter = 0;
};
constexpr int SX_COUNTERS = 256;
constexpr size_t SX_KEEP = 4;
std::mutex gx_mu;
std::list<SchedX> gx_sched[KDEB200_MAX_GPUS];
unsigned long long *gx_count[KDEB200_MAX_GPUS] = {nullptr};  // [0] lane-draws, [1] warp-draws redone

void sx_free(SchedX &e, cudaStream_t st) {
  if (e.d_base) cudaFreeAsync(e.d_base, st);
  e.d_base = nullptr;
}

// FP32 records of one leaf level: where they live and what the kernel needs to bound them
struct LeafBlock {
  size_t rec_off = 0, ctr_off = 0;  // floats / doubles into the record / centre areas
  int ntiles = 0, tnodes = 0;
  double rad[KDEB200_MAX_DIM] = {0};
  double lw2max = 0.0;
  bool fp32 = true;
};
}  // namespace

void gibbs_exact_drop_schedules(int slot) {
  std::lock_guard<std::mutex> lk(gx_mu);
  for (auto &e : gx_sched[slot]) sx_free(e, ctx_at(slot).stream);
  gx_sched[slot].clear();
  if (gx_count[slot]) cudaFreeAsync(gx_count[slot], ctx_at(slot).stream);
  gx_count[slot] = nullptr;
}

static int sx_build(const kdeb200_tree_t *trees, int M, int L, int T, SchedX &e) {
  Context &c = ctx();
  const int d = trees[0]->d;
  const int strideA = gf_stride(d, VAR_A);
  int tnA = 2;  // nodes per FP32 tile: the largest power of two whose pairs fit a ring stage
  while ((size_t)tnA * strideA * sizeof(float) <= GB_TILE_BYTES) tnA *= 2;

  // leaf levels the schedule touches
  std::map<std::pair<int, int>, LeafBlock> leaf;
  std::vector<std::pair<int, int>> leaf_keys;
  size_t nfloats = 0, nctr = 0;
  for (int l = 1; l <= L; ++l)
    for (int j = 0; j < M; ++j) {
      const kdeb200_tree_s *t = trees[j];
      const int li = l < t->depth ? l : t->depth;
      if (t->levels[li].cls != 0) continue;
      const auto key = std::make_pair(j, li);
      if (leaf.count(key)) continue;
      LeafBlock b;
      const int64_t n = t->levels[li].n;
      b.tnodes = tnA;
      b.ntiles = (int)((n + tnA - 1) / tnA);
      b.rec_off = nfloats;
      nfloats += (size_t)((n + 1) / 2) * strideA;
      nfloats = (nfloats + 7) & ~(size_t)7;
      b.ctr_off = nctr;
      nctr += (size_t)b.ntiles * KDEB200_MAX_DIM;
      leaf[key] = b;
      leaf_keys.push_back(key);
    }
  size_t nstats = 0;
  for (auto &k : leaf_keys) nstats += (size_t)leaf[k].ntiles * (2 * KDEB200_MAX_DIM + 1);

  // the draws (internal levels exactly as gibbs.cu's build_schedule with masked = literal = false)
  std::vector<Draw> draws;
  std::vector<XDraw> xds;
  struct TileRef { bool f32; const double *src64; size_t off; uint32_t bytes; };
  std::vector<TileRef> tiles;
  std::vector<std::pair<int, int>> draw_leaf;
  for (int l = 1; l <= L; ++l)
    for (int pass = 0; pass <= T; ++pass)
      for (int j = 0; j < M; ++j) {
        const kdeb200_tree_s *t = trees[j];
        const int li = l < t->depth ? l : t->depth;
        const Level &lv = t->levels[li];
        Draw dr;
        std::memset(&dr, 0, sizeof(dr));
        XDraw xd;
        std::memset(&xd, 0, sizeof(xd));
        dr.j = (short)j;
        dr.kind = pass == 0 ? 0 : 1;
        dr.level = (short)l;
        dr.new_level = (pass == 0 && j == 0) ? 1 : 0;
        dr.n = (int)lv.n;
        dr.wts = t->d_buf + lv.offW;
        dr.levperm = t->d_levperm + lv.offP;
        dr.tile0 = (int)tiles.size();
        if (lv.cls == 0) {
          dr.variant = VAR_A;
          dr.rec = t->d_buf + lv.offA;  // FP64 records: chain state and the FP64 redo
          dr.stride = t->SA;
          dr.rec_state = dr.rec;
          dr.state_stride = t->SA;
          dr.state_has_bw = 0;
          int G = 2;
          while ((int64_t)G * GB_MAXCK < lv.n) G *= 2;
          const int want = 4 * gf_unr(d, VAR_A);
          if (G < want && lv.n >= 2 * want) G = want;
          xd.G = G;
          xd.nchunks = (int)((lv.n + G - 1) / G);
          dr.G = G;
          dr.nchunks = xd.nchunks;
          dr.tnodes = tnA;
          dr.ntiles = (int)((lv.n + tnA - 1) / tnA);
          const LeafBlock &b = leaf[std::make_pair(j, li)];
          for (int qq = 0; qq < dr.ntiles; ++qq) {
            const int64_t a = (int64_t)qq * tnA;
            const int64_t cnt = (lv.n - a < tnA) ? (lv.n - a) : tnA;
            tiles.push_back(TileRef{true, nullptr, b.rec_off + (size_t)(a / 2) * strideA,
                                    (uint32_t)(((cnt + 1) / 2) * strideA * sizeof(float))});
          }
          draw_leaf.push_back(std::make_pair(j, li));
        } else {
          dr.variant = pass == 0 ? VAR_B : VAR_C;
          dr.rec = t->d_buf + (dr.variant == VAR_B ? lv.offB : lv.offC);
          dr.stride = t->SC;
          dr.rec_state = t->d_buf + lv.offC;
          dr.state_stride = t->SC;
          dr.state_has_bw = 1;
          int G = 1;
          while ((int64_t)G * GB_MAXCK < lv.n) G *= 2;
          const int dg = gb_dg(d, dr.variant);
          if (G < dg && lv.n >= 2 * dg) G = dg;
          dr.G = G;
          dr.nchunks = (int)((lv.n + G - 1) / G);
          int tn = 1;
          while (tn * 2 * dr.stride * 8 <= GB_TILE_BYTES) tn *= 2;
          dr.tnodes = tn;
          dr.ntiles = (int)((lv.n + tn - 1) / tn);
          for (int qq = 0; qq < dr.ntiles; ++qq) {
            const int64_t a = (int64_t)qq * tn;
            const int64_t cnt = (lv.n - a < tn) ? (lv.n - a) : tn;
            tiles.push_back(TileRef{false, dr.rec + a * dr.stride, 0, (uint32_t)(cnt * dr.stride * sizeof(double))});
          }
          draw_leaf.push_back(std::make_pair(-1, -1));
        }
        draws.push_back(dr);
        xds.push_back(xd);
      }

  auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t b_draws = up(sizeof(Draw) * draws.size()), b_xd = up(sizeof(XDraw) * xds.size()),
               b_tiles = up(sizeof(TileDesc) * tiles.size()), b_cnt = up(sizeof(int) * SX_COUNTERS),
               b_ctr = up(sizeof(double) * (nctr + 1)), b_rec = up(sizeof(float) * (nfloats + 8));
  KDE_CUDA(cudaMallocAsync(&e.d_base, b_draws + b_xd + b_tiles + b_cnt + b_ctr + b_rec, c.stream));
  char *p = e.d_base;
  e.d_draws = reinterpret_cast<Draw *>(p);
  e.d_xd = reinterpret_cast<XDraw *>(p += b_draws);
  e.d_tiles = reinterpret_cast<TileDesc *>(p += b_xd);
  e.d_counters = reinterpret_cast<int *>(p += b_tiles);
  double *d_ctr = reinterpret_cast<double *>(p += b_cnt);
  float *d_rec = reinterpret_cast<float *>(p += b_ctr);

  // pass a on the device, centres / radii / largest weights on the host, pass b on the device
  cudaError_t err = cudaSuccess;
  if (!leaf_keys.empty()) {
    double *d_stats = nullptr;
    XPrep *d_prep = nullptr;
    size_t *d_coff = nullptr;
    std::vector<XPrep> preps;
    std::vector<size_t> soff, coff;
    int maxt = 1, maxpairs = 1;
    size_t so = 0;
    for (auto &k : leaf_keys) {
      const kdeb200_tree_s *t = trees[k.first];
      const Level &lv = t->levels[k.second];
      LeafBlock &b = leaf[k];
      XPrep xp;
      xp.src = t->d_buf + lv.offA;
      xp.dst = d_rec + b.rec_off;
      xp.stats = nullptr;
      xp.n = (int)lv.n;
      xp.src_stride = t->SA;
      xp.tnodes = b.tnodes;
      xp.lw2max = 0.0;
      preps.push_back(xp);
      soff.push_back(so);
      coff.push_back(b.ctr_off);
      so += (size_t)b.ntiles * (2 * KDEB200_MAX_DIM + 1);
      if (b.ntiles > maxt) maxt = b.ntiles;
      if ((lv.n + 1) / 2 > maxpairs) maxpairs = (int)((lv.n + 1) / 2);
    }
    err = cudaMallocAsync(&d_stats, sizeof(double) * nstats + up(sizeof(XPrep) * preps.size()) + sizeof(size_t) * coff.size(), c.stream);
    if (err == cudaSuccess) {
      d_prep = reinterpret_cast<XPrep *>(reinterpret_cast<char *>(d_stats) + sizeof(double) * nstats);
      d_coff = reinterpret_cast<size_t *>(reinterpret_cast<char *>(d_prep) + up(sizeof(XPrep) * preps.size()));
      for (size_t i = 0; i < preps.size(); ++i) preps[i].stats = d_stats + soff[i];
      err = cudaMemcpyAsync(d_prep, preps.data(), sizeof(XPrep) * preps.size(), cudaMemcpyHostToDevice, c.stream);
      if (err == cudaSuccess) {
        gibbs_exact_stats_kernel<<<dim3((unsigned)maxt, (unsigned)preps.size()), 128, 0, c.stream>>>(d_prep, d);
        err = cudaGetLastError();
      }
      std::vector<double> st(nstats);
      if (err == cudaSuccess) err = cudaMemcpyAsync(st.data(), d_stats, sizeof(double) * nstats, cudaMemcpyDeviceToHost, c.stream);
      if (err == cudaSuccess) err = cudaStreamSynchronize(c.stream);
      std::vector<double> ctr(nctr + 1, 0.0);
      if (err == cudaSuccess) {
        for (size_t i = 0; i < leaf_keys.size(); ++i) {
          LeafBlock &b = leaf[leaf_keys[i]];
          double lwmax = -INFINITY;
          for (int tt = 0; tt < b.ntiles; ++tt) {
            const double *sv = &st[soff[i] + (size_t)tt * (2 * KDEB200_MAX_DIM + 1)];
            for (int k = 0; k < d; ++k) {
              const double lo = sv[k], hi = sv[KDEB200_MAX_DIM + k];
              const double cc = 0.5 * lo + 0.5 * hi;
              ctr[b.ctr_off + (size_t)tt * KDEB200_MAX_DIM + k] = cc;
              // |m - c| <= max(hi - c, c - lo), each rounded: a relative 1e-15 and an absolute ulp of c cover both
              const double r = std::fmax(hi - cc, cc - lo) * (1.0 + 1e-15) + std::fabs(cc) * 0x1.0p-51;
              if (!(r <= 1e20)) b.fp32 = false;  // outside FP32's comfortable range: FP64 redo for the whole level
              if (r > b.rad[k]) b.rad[k] = r;
            }
            lwmax = std::fmax(lwmax, sv[2 * KDEB200_MAX_DIM]);
          }
          b.lw2max = lwmax * GF_LOG2E;
          if (!std::isfinite(b.lw2max)) b.fp32 = false, b.lw2max = 0.0;
          preps[i].lw2max = b.lw2max;
        }
        err = cudaMemcpyAsync(d_ctr, ctr.data(), sizeof(double) * (nctr + 1), cudaMemcpyHostToDevice, c.stream);
      }
      if (err == cudaSuccess) err = cudaMemcpyAsync(d_prep, preps.data(), sizeof(XPrep) * preps.size(), cudaMemcpyHostToDevice, c.stream);
      if (err == cudaSuccess) err = cudaMemcpyAsync(d_coff, coff.data(), sizeof(size_t) * coff.size(), cudaMemcpyHostToDevice, c.stream);
      if (err == cudaSuccess) {
        gibbs_exact_rec_kernel<<<dim3((unsigned)((maxpairs + 127) / 128), (unsigned)preps.size()), 128, 0, c.stream>>>(
            d_prep, d_ctr, d_coff, d);
        err = cudaGetLastError();
      }
      if (err == cudaSuccess) err = cudaStreamSynchronize(c.stream);  // host vectors above are pageable
      cudaFreeAsync(d_stats, c.stream);
    }
  }
  if (err == cudaSuccess) {
    std::vector<TileDesc> tds(tiles.size());
    for (size_t i = 0; i < tiles.size(); ++i) {
      tds[i].src = tiles[i].f32 ? reinterpret_cast<const double *>(d_rec + tiles[i].off) : tiles[i].src64;
      tds[i].bytes = tiles[i].bytes;
      tds[i].pad = 0;
    }
    for (size_t i = 0; i < draws.size(); ++i) {
      if (draw_leaf[i].first < 0) continue;
      const LeafBlock &b = leaf[draw_leaf[i]];
      xds[i].rec32 = d_rec + b.rec_off;
      xds[i].ctr = d_ctr + b.ctr_off;
      for (int k = 0; k < KDEB200_MAX_DIM; ++k) xds[i].rad[k] = b.rad[k];
      xds[i].lw2max = b.lw2max;
      xds[i].fp32 = b.fp32 ? 1 : 0;
    }
    err = cudaMemcpyAsync(e.d_draws, draws.data(), sizeof(Draw) * draws.size(), cudaMemcpyHostToDevice, c.stream);
    if (err == cudaSuccess) err = cudaMemcpyAsync(e.d_xd, xds.data(), sizeof(XDraw) * xds.size(), cudaMemcpyHostToDevice, c.stream);
    if (err == cudaSuccess) err = cudaMemcpyAsync(e.d_tiles, tds.data(), sizeof(TileDesc) * tds.size(), cudaMemcpyHostToDevice, c.stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(e.d_counters, 0, b_cnt, c.stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(c.stream);
  }
  if (err != cudaSuccess) {
    cudaFreeAsync(e.d_base, c.stream);
    e.d_base = nullptr;
    KDE_FAIL(100 + (int)err, "gibbs (exact): building the schedule: %s", cudaGetErrorString(err));
  }
  e.ndraws = (int)draws.size();
  e.ntiles = (int)tiles.size();
  return 0;
}

static int sx_get(const kdeb200_tree_t *trees, int M, int L, int T, SchedX *out, int **counter) {
  Context &c = ctx();
  std::lock_guard<std::mutex> lk(gx_mu);
  auto &lst = gx_sched[c.slot];
  const uint64_t epoch = g_tree_epoch.load();
  for (auto it = lst.begin(); it != lst.end();) {  // entries from before the last tree_destroy may point at freed records
    if (it->epoch != epoch) {
      sx_free(*it, c.stream);
      it = lst.erase(it);
    } else {
      ++it;
    }
  }
  for (auto it = lst.begin(); it != lst.end(); ++it) {
    if (it->M != M || it->T != T) continue;
    bool same = true;
    for (int j = 0; j < M; ++j) same = same && it->trees[j] == trees[j];
    if (!same) continue;
    lst.splice(lst.begin(), lst, it);
    *counter = it->d_counters + (it->next_counter++ % SX_COUNTERS);
    *out = *it;
    return 0;
  }
  SchedX e;
  if (int rc = sx_build(trees, M, L, T, e)) return rc;
  e.epoch = epoch;
  e.slot = c.slot;
  e.M = M;
  e.T = T;
  for (int j = 0; j < M; ++j) e.trees[j] = trees[j];
  lst.push_front(e);
  while (lst.size() > SX_KEEP) {
    cudaDeviceSynchronize();  // an evicted entry may still be read by a kernel in flight
    sx_free(lst.back(), c.stream);
    lst.pop_back();
  }
  *counter = lst.front().d_counters + (lst.front().next_counter++ % SX_COUNTERS);
  *out = lst.front();
  return 0;
}

// redo counters of the calling context (atomics: launches in flight on several streams may share them)
static int sx_counter(unsigned long long **count) {
  Context &c = ctx();
  std::lock_guard<std::mutex> lk(gx_mu);
  if (!gx_count[c.slot]) {
    KDE_CUDA(cudaMallocAsync(&gx_count[c.slot], 2 * sizeof(unsigned long long), c.stream));
    KDE_CUDA(cudaMemsetAsync(gx_count[c.slot], 0, 2 * sizeof(unsigned long long), c.stream));
    KDE_CUDA(cudaStreamSynchronize(c.stream));  // the caller's stream must see a finished buffer
  }
  *count = gx_count[c.slot];
  return 0;
}

// lane-draws and warp-draws redone in FP64 on the calling context's device since the last call (synchronises)
int gibbs_exact_redone(unsigned long long *lanes, unsigned long long *warps) {
  unsigned long long *d = nullptr;
  if (int rc = sx_counter(&d)) return rc;
  unsigned long long h[2] = {0, 0};
  KDE_CUDA(cudaDeviceSynchronize());
  KDE_CUDA(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
  KDE_CUDA(cudaMemset(d, 0, sizeof(h)));
  if (lanes) *lanes = h[0];
  if (warps) *warps = h[1];
  return 0;
}

static bool exact_enabled() {
  const char *ev = getenv("KDEB200_GIBBS_EXACT");
  return !(ev && atoi(ev) == 0);
}

// K1x takes a call K1 would run (thread per chain, F64, every dimension of every density, no literal arithmetic)
// and that it has been measured to win; everything else goes to gibbs_device unchanged.
static bool exact_eligible(const kdeb200_tree_t *trees, int ndens, const uint8_t *dimmask, int64_t s0, int64_t s1) {
  if (!exact_enabled() || gibbs_precision() != KDEB200_F64) return false;
  if (ndens < 2 || ndens > KDEB200_MAX_DENS || !trees) return false;
  Context &c = ctx();
  for (int j = 0; j < ndens; ++j)
    if (!trees[j] || !trees[j]->gibbs_ready || trees[j]->degenerate || trees[j]->slot != c.slot || trees[j]->d != trees[0]->d)
      return false;
  const int d = trees[0]->d;
  if (d != 3) return false;  // the only dimension measured so far (C4: 904 -> 776 ms per 1M samples, DESIGN.md K1x)
  if (dimmask)
    for (int i = 0; i < ndens * d; ++i)
      if (!dimmask[i]) return false;
  // the warp-per-chain range of gibbs_device
  int nmax = 1;
  for (int j = 0; j < ndens; ++j)
    if (trees[j]->levels[trees[j]->depth].n > nmax) nmax = (int)trees[j]->levels[trees[j]->depth].n;
  int64_t warp_max = (int64_t)24 * c.sm_count;
  if (const char *ev = getenv("KDEB200_GIBBS_WARP_MAX")) warp_max = atoll(ev);
  if (s1 - s0 <= warp_max && gibbs_warp_smem(d, nmax) <= 96 * 1024) return false;
  // FP32 range guard: leaf bandwidths whose s_k = sqrt(0.5 log2 e / c_k) stays a normal float
  for (int j = 0; j < ndens; ++j)
    for (int k = 0; k < d; ++k)
      if (!(trees[j]->hvar[k] >= 1e-20 && trees[j]->hvar[k] <= 1e20)) return false;
  return true;
}

int gibbs_exact_device(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                       const uint8_t *dimmask, const double *d_randU, int64_t nU, const double *d_randN, int64_t nN,
                       uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                       int64_t *d_level_labels, cudaStream_t st, int *launches) {
  if (!exact_eligible(trees, ndens, dimmask, s0, s1))
    return gibbs_device(trees, ndens, Np, Niter, add_entropy, dimmask, d_randU, nU, d_randN, nN, seed, s0, s1, d_points,
                        d_indices, d_level_labels, st, launches);
  Context &c = ctx();
  int L = 0;
  int64_t perU = 0, perN = 0;
  if (int rc = gibbs_sizes(trees, ndens, Niter, &L, &perU, &perN, nullptr)) return rc;
  const int d = trees[0]->d;
  if (Np < 0 || s0 < 0 || s1 > Np || s0 > s1) KDE_FAIL(3, "gibbs: bad sample range [%lld,%lld) of %lld", (long long)s0, (long long)s1, (long long)Np);
  if (s1 == s0) return 0;
  if ((d_randU == nullptr) != (d_randN == nullptr)) KDE_FAIL(3, "gibbs: randU and randN must be given together");
  if (d_randU) {
    if (s1 * perU > nU + 1) KDE_FAIL(7, "gibbs: randU too short (%lld < %lld)", (long long)nU, (long long)(s1 * perU - 1));
    if (s1 * perN > nN) KDE_FAIL(7, "gibbs: randN too short (%lld < %lld)", (long long)nN, (long long)(s1 * perN));
  }
  GibbsParams P;
  std::memset(&P, 0, sizeof(P));
  for (int j = 0; j < ndens; ++j)
    for (int k = 0; k < d; ++k) P.mask[j][k] = 1, P.other[j][k] = 1;
  SchedX E;
  int *d_counter = nullptr;
  if (int rc = sx_get(trees, ndens, L, Niter, &E, &d_counter)) return rc;
  P.draws = E.d_draws;
  P.tiles = E.d_tiles;
  P.counter = d_counter;
  P.exptab = c.d_exptab;
  P.ec = make_exp_consts();
  P.randU = d_randU;
  P.randN = d_randN;
  P.points = d_points;
  P.indices = d_indices;
  P.level_labels = d_level_labels;
  P.s0 = s0;
  P.s1 = s1;
  P.perU = perU;
  P.perN = perN;
  P.seed = seed;
  P.ndraws = E.ndraws;
  P.ntiles = E.ntiles;
  P.M = ndens;
  P.L = L;
  P.T = Niter;
  P.add_entropy = add_entropy ? 1 : 0;
  P.nbatches = (int)((s1 - s0 + GB_THREADS - 1) / GB_THREADS);
  for (int j = 0; j < ndens; ++j) {
    const kdeb200_tree_s *t = trees[j];
    P.root_rec[j] = t->d_buf + t->levels[0].offC;
    P.labels[j] = t->d_labels;
    for (int k = 0; k < d; ++k) P.hvar[j][k] = t->hvar[k];
  }

  const size_t smem = GB_STAGES * GB_TILE_BYTES;
  int per_sm = 0;
  cudaError_t e = cudaErrorInvalidValue;
  switch (d) {
    case 1: e = occupancy_gibbs_exact_d<1>(ndens, smem, &per_sm); break;
    case 2: e = occupancy_gibbs_exact_d<2>(ndens, smem, &per_sm); break;
    case 3: e = occupancy_gibbs_exact_d<3>(ndens, smem, &per_sm); break;
    case 4: e = occupancy_gibbs_exact_d<4>(ndens, smem, &per_sm); break;
    case 5: e = occupancy_gibbs_exact_d<5>(ndens, smem, &per_sm); break;
    case 6: e = occupancy_gibbs_exact_d<6>(ndens, smem, &per_sm); break;
    case 7: e = occupancy_gibbs_exact_d<7>(ndens, smem, &per_sm); break;
    case 8: e = occupancy_gibbs_exact_d<8>(ndens, smem, &per_sm); break;
  }
  if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "gibbs (exact) occupancy: %s", cudaGetErrorString(e));
  if (per_sm < 1) per_sm = 1;
  int grid = per_sm * c.sm_count;
  if (grid > P.nbatches) grid = P.nbatches;

  XParams X;
  X.xd = E.d_xd;
  X.ex2_err = GX_EX2_ERR;
  X.inflate = 1.0;
  if (const char *ev = getenv("KDEB200_GIBBS_EXACT_INFLATE")) X.inflate = atof(ev);  // tests: force the FP64 redo
  unsigned long long *d_count = nullptr;
  if (int rc = sx_counter(&d_count)) return rc;
  X.redone = d_count;
  X.warp_redone = d_count + 1;
  // The redo scratch belongs to this launch alone, stream-ordered on `st`: launches on other streams may be in flight
  // at the same time, and a warp that shared its (block, warp) slot with another launch would sum foreign terms.
  X.scratch = nullptr;
  KDE_CUDA(cudaMallocAsync(&X.scratch, sizeof(double) * (size_t)grid * (GB_THREADS / 32) * GX_SCR, st));
  switch (d) {
    case 1: e = launch_gibbs_exact_d<1>(P, X, grid, smem, st); break;
    case 2: e = launch_gibbs_exact_d<2>(P, X, grid, smem, st); break;
    case 3: e = launch_gibbs_exact_d<3>(P, X, grid, smem, st); break;
    case 4: e = launch_gibbs_exact_d<4>(P, X, grid, smem, st); break;
    case 5: e = launch_gibbs_exact_d<5>(P, X, grid, smem, st); break;
    case 6: e = launch_gibbs_exact_d<6>(P, X, grid, smem, st); break;
    case 7: e = launch_gibbs_exact_d<7>(P, X, grid, smem, st); break;
    case 8: e = launch_gibbs_exact_d<8>(P, X, grid, smem, st); break;
  }
  cudaFreeAsync(X.scratch, st);  // released once the kernel ahead of it on `st` has finished
  if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "gibbs (exact) kernel launch: %s", cudaGetErrorString(e));
  if (launches) *launches += 1;
  return 0;
}

// ---- bound probe (tests) ------------------------------------------------------------------------------------------
// For query conditionals (mu, Calmost) of one variant-A draw: every node's FP32 term as K1x computes it, its bound, K1's
// FP64 term, K1's prefix sums, and the intervals K1x would claim for them -- per node as xa_decide forms them, and at
// checkpoints as xa_pass1 forms them (trip sums in FP32, Q in FP32 per chunk).  One CTA per query.
// out per query: [A, B, aabs, ok, lw2max, n, G, 0] then per node [p32, acc32, p64, S64, lo, hi, lo_ck, hi_ck]
// (lo_ck / hi_ck are NaN except at chunk ends).
constexpr int GX_PROBE_HDR = 8, GX_PROBE_NODE = 8;

template <int D>
__global__ void gibbs_exact_probe_kernel(Draw dr, XDraw xd, const double *mu_all, const double *cadd_all, GibbsParams P,
                                         int j, double *out_all) {
  constexpr int stride = gf_stride(D, VAR_A);
  constexpr int UNR = gf_unr(D, VAR_A);
  const int qi = blockIdx.x;
  double *out = out_all + (size_t)qi * (GX_PROBE_HDR + (size_t)GX_PROBE_NODE * dr.n);
  double mu[D];
  Hoist<D, false> h;
  float s32[D];
  for (int k = 0; k < D; ++k) {  // the expressions of gibbs_exact_kernel
    mu[k] = mu_all[qi * D + k];
    h.mu[k] = mu[k];
    h.cadd[k] = cadd_all[qi * D + k];
    h.act[k] = true;
    const double c = P.hvar[j][k] + h.cadd[k];
    h.ich[k] = sqrt(0.5 / c);
    s32[k] = (float)sqrt(GF_HL2E / c);
  }
  const XBound bd = xa_bound<D>(xd, s32, dr.n, GX_EX2_ERR, 1.0);
  Hoist32<D> g;
  for (int k = 0; k < D; ++k) g.a[k] = gf_pack(s32[k], s32[k]);
  for (int z = threadIdx.x; z < dr.n; z += blockDim.x) {
    xa_tile_hoist<D>(xd.ctr + (size_t)(z / dr.tnodes) * KDEB200_MAX_DIM, mu, s32, g);
    f32x2 acc, sc;
    gf_pre<D, VAR_A, true>(xd.rec32 + (size_t)(z >> 1) * stride, g, acc, sc);
    float al, ah;
    gf_unpack(acc, al, ah);
    const float a = (z & 1) ? ah : al;
    double *o = out + GX_PROBE_HDR + (size_t)GX_PROBE_NODE * z;
    o[0] = (double)gf_ex2_neg(a);
    o[1] = (double)a;
    o[2] = eval_node<D, false, VAR_A, true>(dr.rec + (size_t)z * dr.stride, h, P.exptab, P.ec);
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  out[0] = bd.A;
  out[1] = bd.B;
  out[2] = bd.aabs;
  out[3] = bd.ok ? 1.0 : 0.0;
  out[4] = xd.lw2max;
  out[5] = dr.n;
  out[6] = xd.G;
  out[7] = 0.0;
  double S64 = 0.0, S = 0.0, Q = 0.0, S1 = 0.0, Q1 = 0.0;
  float s = 0.f, qf = 0.f;
  int intrip = 0;
  for (int z = 0; z < dr.n; ++z) {
    double *o = out + GX_PROBE_HDR + (size_t)GX_PROBE_NODE * z;
    const double p32 = o[0], a = o[1];
    S64 = __dadd_rn(S64, o[2]);  // K1's node-order sum
    S = __dadd_rn(S, p32);       // xa_decide's per-node intervals
    Q = __fma_rn(p32, a, Q);
    const double E = xa_err(bd, S, Q, z + 1);
    o[3] = S64;
    o[4] = (S - E) * (1.0 - bd.eta);
    o[5] = (S + E) * (1.0 + bd.eta);
    // xa_pass1: FP32 trip sums of 2 UNR nodes from zero folded into FP64, Q in FP32 over the chunk
    s = __fadd_rn(s, (float)p32);
    qf = __fmaf_rn((float)p32, (float)a, qf);
    const bool chunk_end = ((z + 1) % xd.G == 0) || z + 1 == dr.n;
    if (++intrip == 2 * UNR || chunk_end) {
      S1 = __dadd_rn(S1, (double)s);
      s = 0.f;
      intrip = 0;
    }
    o[6] = o[7] = __longlong_as_double(0x7ff8000000000000LL);
    if (chunk_end) {
      Q1 = __dadd_rn(Q1, (double)qf);
      qf = 0.f;
      const double Qc = (double)__double2float_ru(Q1);
      const double E1 = xa_err(bd, S1, Qc, z + 1);
      o[6] = (S1 - E1) * (1.0 - bd.eta);
      o[7] = (S1 + E1) * (1.0 + bd.eta);
    }
  }
}

int gibbs_exact_probe(const kdeb200_tree_t *trees, int ndens, int Niter, int j, int level, const double *mu,
                      const double *cadd, int nq, double *out, int64_t out_len) {
  if (!trees || ndens < 1 || ndens > KDEB200_MAX_DENS || j < 0 || j >= ndens || nq < 1 || !mu || !cadd || !out)
    KDE_FAIL(3, "gibbs_exact_probe: bad arguments");
  const int d = trees[0]->d;
  if (d != 3) KDE_FAIL(3, "gibbs_exact_probe: d = 3 only (the dimension K1x serves)");
  Context &c = ctx();
  int L = 0;
  if (int rc = gibbs_sizes(trees, ndens, Niter, &L, nullptr, nullptr, nullptr)) return rc;
  SchedX E;
  int *d_counter = nullptr;
  if (int rc = sx_get(trees, ndens, L, Niter, &E, &d_counter)) return rc;
  std::vector<Draw> draws(E.ndraws);
  std::vector<XDraw> xds(E.ndraws);
  KDE_CUDA(cudaMemcpy(draws.data(), E.d_draws, sizeof(Draw) * E.ndraws, cudaMemcpyDeviceToHost));
  KDE_CUDA(cudaMemcpy(xds.data(), E.d_xd, sizeof(XDraw) * E.ndraws, cudaMemcpyDeviceToHost));
  int di = -1;
  for (int i = 0; i < E.ndraws && di < 0; ++i)
    if (draws[i].j == j && draws[i].level == level && draws[i].variant == VAR_A) di = i;
  if (di < 0) KDE_FAIL(3, "gibbs_exact_probe: level %d of density %d is not a leaf level", level, j + 1);
  const size_t per = GX_PROBE_HDR + (size_t)GX_PROBE_NODE * draws[di].n;
  if ((int64_t)(per * nq) > out_len) KDE_FAIL(3, "gibbs_exact_probe: out needs %lld doubles", (long long)(per * nq));
  GibbsParams P;
  std::memset(&P, 0, sizeof(P));
  P.exptab = c.d_exptab;
  P.ec = make_exp_consts();
  for (int k = 0; k < d; ++k) P.hvar[j][k] = trees[j]->hvar[k];
  double *d_mu = nullptr, *d_out = nullptr;
  KDE_CUDA(cudaMalloc(&d_mu, sizeof(double) * 2 * nq * d));
  KDE_CUDA(cudaMalloc(&d_out, sizeof(double) * per * nq));
  cudaError_t err = cudaMemcpy(d_mu, mu, sizeof(double) * nq * d, cudaMemcpyHostToDevice);
  if (err == cudaSuccess) err = cudaMemcpy(d_mu + nq * d, cadd, sizeof(double) * nq * d, cudaMemcpyHostToDevice);
  if (err == cudaSuccess) {
    gibbs_exact_probe_kernel<3><<<nq, 128, 0, c.stream>>>(draws[di], xds[di], d_mu, d_mu + nq * d, P, j, d_out);
    err = cudaGetLastError();
  }
  if (err == cudaSuccess) err = cudaStreamSynchronize(c.stream);
  if (err == cudaSuccess) err = cudaMemcpy(out, d_out, sizeof(double) * per * nq, cudaMemcpyDeviceToHost);
  cudaFree(d_mu);
  cudaFree(d_out);
  if (err != cudaSuccess) KDE_FAIL(100 + (int)err, "gibbs_exact_probe: %s", cudaGetErrorString(err));
  return 0;
}

}  // namespace kdeb200
