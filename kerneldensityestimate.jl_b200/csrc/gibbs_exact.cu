// gibbs_exact.cu -- host side of K1x (gibbs_exact_kernel.cuh): every draw is certified; its FP32 records laid out for
// accuracy (per-tile centres, log-weights relative to the level's largest), the XDraws over them, launch, and the bound
// probe.  Routing is gibbs_device's (gibbs.cu), the schedule
// gibbs.cu's (cache) and gibbs_plan.cuh's (draws, chunks, tiles), which gibbs_exact_plan adjusts.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "gibbs.cuh"
#include "gibbs_exact_kernel.cuh"
#include "gibbs_plan.cuh"

namespace kdeb200 {

#define GX_EXTERN(D)                                                                                       \
  extern template cudaError_t launch_gibbs_exact_d<D>(const GibbsParams &, const XParams &, int, size_t, \
                                                      cudaStream_t);                                     \
  extern template cudaError_t occupancy_gibbs_exact_d<D>(int, size_t, int *);
GX_EXTERN(1) GX_EXTERN(2) GX_EXTERN(3) GX_EXTERN(4) GX_EXTERN(5) GX_EXTERN(6) GX_EXTERN(7) GX_EXTERN(8)
#undef GX_EXTERN

// Relative error bound of ex2.approx.ftz.f32 over the exponents K1x feeds it, [-126, 0]: 2^-21 = 4.8e-7, more than three
// times the maximum measured over every float of that range on a B200, 1.44e-7 (tools/ulp_mufu.py, profiles/mufu_ulp.json).
constexpr double GX_EX2_ERR = 0x1.0p-21;
// The same margin for rsqrt.approx.ftz.f32 over every positive normal float: measured maximum 1.25e-7 (same sources).
constexpr double GX_RSQ_ERR = 0x1.0p-21;

// ---- FP32 records -------------------------------------------------------------------------------------------------
struct XPrep {
  const double *src;  // A: [m.., ln w], B: [m.., -0.5/b.., ln w - 0.5 sum ln b], C: [m.., b.., ln w] records
  float *dst;         // pair records, stride gf_stride(d, var)
  double *stats;      // per tile (GX_STATS doubles): min m | max m | min b | max b (B: of -0.5/b; C) | max of the last column
  int n, src_stride, tnodes, var;
  double lw2max;
};
constexpr int GX_STATS = 4 * KDEB200_MAX_DIM + 1;

// pass a: one CTA per tile, per-dimension min / max of the means (and, variants B and C, of the variance columns) and
// the largest log-weight column
__global__ void gibbs_exact_stats_kernel(const XPrep *preps, int D) {
  const XPrep pd = preps[blockIdx.y];
  const int t = blockIdx.x;
  const int z0 = t * pd.tnodes;
  if (z0 >= pd.n) return;
  const int z1 = min(z0 + pd.tnodes, pd.n);
  const int nb = pd.var != VAR_A ? 2 * D : 0;  // min / max of the variance column
  const int nq = 2 * D + nb + 1;
  __shared__ double red[GX_STATS][4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = 0; k < nq; ++k) {
    const bool isw = k == nq - 1, ismax = isw || (k % (2 * D)) >= D;
    const int col = isw ? (pd.var != VAR_A ? 2 * D : D) : (k < 2 * D ? k % D : D + k % D);
    double v = ismax ? -INFINITY : INFINITY;
    for (int z = z0 + threadIdx.x; z < z1; z += blockDim.x) {
      const double x = pd.src[(size_t)z * pd.src_stride + col];
      v = ismax ? fmax(v, x) : fmin(v, x);
    }
    for (int o = 16; o; o >>= 1) {
      const double w = __shfl_xor_sync(0xffffffffu, v, o);
      v = ismax ? fmax(v, w) : fmin(v, w);
    }
    if (lane == 0) red[k][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x < nq) {
    const int k = threadIdx.x;
    const bool isw = k == nq - 1, ismax = isw || (k % (2 * D)) >= D;
    double v = red[k][0];
    for (int w = 1; w < 4; ++w) v = ismax ? fmax(v, red[k][w]) : fmin(v, red[k][w]);
    // slot: the (2 k / D)-th block of KDEB200_MAX_DIM, dimension k % D
    pd.stats[(size_t)t * GX_STATS + (isw ? 4 * KDEB200_MAX_DIM : (k / D) * KDEB200_MAX_DIM + k % D)] = v;
  }
}

// pass b: pair records, m' = m - centre(tile), lw' = lw2max - log2 w >= 0:
//   A: [m'_0(a), m'_0(b), .., lw'(a), lw'(b), pad];  C: [m'_0(a), m'_0(b), .., b_0(a), b_0(b), .., lw'(a), lw'(b), pad];
//   B: as C with 0.5 log2e / b_k in place of b_k and log2 w - 0.5 sum log2 b_k in place of log2 w, both from K1's own
//   record values (-0.5/b_k and ln w - 0.5 sum ln b_k, times -log2e and log2e)
__global__ void gibbs_exact_rec_kernel(const XPrep *preps, const double *ctrs_base, const size_t *ctr_off, int D) {
  const XPrep pd = preps[blockIdx.y];
  const double *ctr = ctrs_base + ctr_off[blockIdx.y];
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (2 * p >= pd.n) return;
  const int stride = gf_stride(D, pd.var);
  const int nb = pd.var != VAR_A ? D : 0;
  float *o = pd.dst + (size_t)p * stride;
  const double *c = ctr + (size_t)((2 * p) / pd.tnodes) * KDEB200_MAX_DIM;
  for (int hh = 0; hh < 2; ++hh) {
    const int z = 2 * p + hh;
    const bool ok = z < pd.n;  // an odd level is padded with a node of probability zero (finite: no 0 * inf)
    const double *r = pd.src + (size_t)(ok ? z : 0) * pd.src_stride;
    for (int k = 0; k < D; ++k) o[2 * k + hh] = ok ? (float)(r[k] - c[k]) : 0.f;
    for (int k = 0; k < nb; ++k)
      o[2 * (D + k) + hh] = ok ? (float)(pd.var == VAR_B ? -r[D + k] * GF_LOG2E : r[D + k]) : (pd.var == VAR_B ? 0.f : 1.f);
    o[2 * (D + nb) + hh] = ok ? (float)fmax(pd.lw2max - r[D + nb] * GF_LOG2E, 0.0) : 1e30f;
  }
  for (int k = 2 * (D + nb + 1); k < stride; ++k) o[k] = 0.f;
}

// ---- schedule ---------------------------------------------------------------------------------------------------
// plan_schedule(.., b_records = true, f32_leaf = true, f32_internal = false) gives every leaf draw FP32 records; this
// moves every internal draw (variants B and C) onto FP32 records as well, with K1f's chunk and tile rule, and rebuilds
// the tile stream.  The draws keep K1's FP64 records in `rec`: the FP64 redo reads them.
void gibbs_exact_plan(const kdeb200_tree_t *trees, Plan &S) {
  const int d = trees[0]->d;
  const int stride = gf_stride(d, VAR_C);  // == gf_stride(d, VAR_B)
  std::vector<PlanTile> tiles;
  for (size_t i = 0; i < S.draws.size(); ++i) {
    Draw &dr = S.draws[i];
    const int t0 = dr.tile0;
    dr.tile0 = (int)tiles.size();
    if (S.block[i] >= 0) {
      tiles.insert(tiles.end(), S.tiles.begin() + t0, S.tiles.begin() + t0 + dr.ntiles);
      continue;
    }
    const kdeb200_tree_s *t = trees[dr.j];
    int G = 2;
    while ((int64_t)G * GB_MAXCK < dr.n) G *= 2;
    const int want = 4 * gf_unr(d, dr.variant);
    if (G < want && dr.n >= 2 * want) G = want;
    int tn = 2;
    while ((size_t)tn * stride * sizeof(float) <= GB_TILE_BYTES) tn *= 2;
    dr.G = G;
    dr.tnodes = tn;
    dr.nchunks = (dr.n + G - 1) / G;
    dr.ntiles = (dr.n + tn - 1) / tn;
    const int blk = plan_block(S, dr.j, dr.level < t->depth ? dr.level : t->depth, dr.variant, dr.n, stride, tn);
    S.block[i] = blk;
    for (int a = 0; a < dr.n; a += tn) {
      const int cnt = (dr.n - a < tn) ? (dr.n - a) : tn;
      tiles.push_back(PlanTile{nullptr, S.blocks[blk].off + (size_t)(a / 2) * stride,
                               (uint32_t)(((cnt + 1) / 2) * stride * sizeof(float))});
    }
  }
  S.tiles.swap(tiles);
}

// Every block of the plan holds FP32 records (a leaf level, or an internal level's B or C records).  Pass a on the device, tile
// centres / radii / variance ranges / largest weights on the host, pass b on the device; the persistent XDraws and
// centres go to e.d_extra.
int gibbs_exact_build(const kdeb200_tree_t *trees, Plan &S, SchedEntry &e) {
  Context &c = ctx();
  const int d = trees[0]->d;
  const size_t SW = GX_STATS;
  struct XBlock {
    size_t ctr_off = 0, stats_off = 0;  // doubles into the centres / statistics
    int ntiles = 0;
    double rad[KDEB200_MAX_DIM] = {0};
    double bmin[KDEB200_MAX_DIM] = {0};
    double lw2max = 0.0;
    bool fp32 = true;
  };
  std::vector<XBlock> blk(S.blocks.size());
  std::vector<XPrep> preps(S.blocks.size());
  std::vector<size_t> coff(S.blocks.size());
  size_t nctr = 0, nstats = 0;
  int maxt = 1, maxpairs = 1;
  for (size_t i = 0; i < S.blocks.size(); ++i) {
    const kdeb200_tree_s *t = trees[S.blocks[i].j];
    const Level &lv = t->levels[S.blocks[i].level];
    const int var = S.blocks[i].variant;
    XBlock &b = blk[i];
    b.ntiles = (int)((lv.n + S.blocks[i].tnodes - 1) / S.blocks[i].tnodes);
    b.ctr_off = coff[i] = nctr;
    b.stats_off = nstats;
    nctr += (size_t)b.ntiles * KDEB200_MAX_DIM;
    nstats += (size_t)b.ntiles * SW;
    XPrep &xp = preps[i];
    xp.src = t->d_buf + (var == VAR_A ? lv.offA : var == VAR_B ? lv.offB : lv.offC);
    xp.dst = e.d_rec + S.blocks[i].off;
    xp.stats = nullptr;
    xp.n = (int)lv.n;
    xp.src_stride = var == VAR_A ? t->SA : t->SC;
    xp.tnodes = S.blocks[i].tnodes;
    xp.var = S.blocks[i].variant;
    xp.lw2max = 0.0;
    if (b.ntiles > maxt) maxt = b.ntiles;
    if ((lv.n + 1) / 2 > maxpairs) maxpairs = (int)((lv.n + 1) / 2);
  }
  auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t b_xd = up(sizeof(XDraw) * S.draws.size());
  KDE_CUDA(cudaMallocAsync(&e.d_extra, b_xd + sizeof(double) * (nctr + 1), c.stream));
  e.d_xd = reinterpret_cast<XDraw *>(e.d_extra);
  double *d_ctr = reinterpret_cast<double *>(e.d_extra + b_xd);

  cudaError_t err = cudaSuccess;
  if (!preps.empty()) {
    double *d_stats = nullptr;
    err = cudaMallocAsync(&d_stats, sizeof(double) * nstats + up(sizeof(XPrep) * preps.size()) + sizeof(size_t) * coff.size(), c.stream);
    if (err == cudaSuccess) {
      XPrep *d_prep = reinterpret_cast<XPrep *>(reinterpret_cast<char *>(d_stats) + sizeof(double) * nstats);
      size_t *d_coff = reinterpret_cast<size_t *>(reinterpret_cast<char *>(d_prep) + up(sizeof(XPrep) * preps.size()));
      for (size_t i = 0; i < preps.size(); ++i) preps[i].stats = d_stats + blk[i].stats_off;
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
        for (size_t i = 0; i < blk.size(); ++i) {
          XBlock &b = blk[i];
          double lwmax = -INFINITY;
          if (preps[i].var != VAR_A)
            for (int k = 0; k < d; ++k) b.bmin[k] = INFINITY;
          for (int tt = 0; tt < b.ntiles; ++tt) {
            const double *sv = &st[b.stats_off + (size_t)tt * SW];
            for (int k = 0; k < d; ++k) {
              const double lo = sv[k], hi = sv[KDEB200_MAX_DIM + k];
              const double cc = 0.5 * lo + 0.5 * hi;
              ctr[b.ctr_off + (size_t)tt * KDEB200_MAX_DIM + k] = cc;
              // |m - c| <= max(hi - c, c - lo), each rounded: a relative 1e-15 and an absolute ulp of c cover both
              const double r = std::fmax(hi - cc, cc - lo) * (1.0 + 1e-15) + std::fabs(cc) * 0x1.0p-51;
              if (!(r <= 1e20)) b.fp32 = false;  // outside FP32's comfortable range: FP64 redo for the whole level
              if (r > b.rad[k]) b.rad[k] = r;
              if (preps[i].var != VAR_A) {
                // c_k = b_k + Calmost_k in FP32 needs b_k in (0, 2^29]; the kernel checks Calmost per chain.  Variant B
                // keeps b_k in the same range; its records hold -0.5/b_k, whose smallest value belongs to the smallest b_k
                double bl = sv[2 * KDEB200_MAX_DIM + k], bh = sv[3 * KDEB200_MAX_DIM + k];
                if (preps[i].var == VAR_B) bl = -0.5 / bl, bh = -0.5 / bh;
                if (!(bl > 0.0) || !(bh > 0.0) || !(bh <= 0x1.0p29)) b.fp32 = false;
                b.bmin[k] = std::fmin(b.bmin[k], bl);
              }
            }
            lwmax = std::fmax(lwmax, sv[4 * KDEB200_MAX_DIM]);
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
  std::vector<XDraw> xds(S.draws.size());
  std::memset(xds.data(), 0, sizeof(XDraw) * xds.size());
  for (size_t i = 0; i < S.draws.size(); ++i) {
    if (S.block[i] < 0) continue;
    const XBlock &b = blk[S.block[i]];
    XDraw &xd = xds[i];
    xd.rec32 = e.d_rec + S.blocks[S.block[i]].off;
    xd.ctr = d_ctr + b.ctr_off;
    for (int k = 0; k < KDEB200_MAX_DIM; ++k) xd.rad[k] = b.rad[k], xd.bmin[k] = b.bmin[k];
    xd.lw2max = b.lw2max;
    xd.G = S.draws[i].G;
    xd.nchunks = S.draws[i].nchunks;
    xd.fp32 = b.fp32 ? 1 : 0;
    const int nb = (S.draws[i].n + GX_SCR - 1) / GX_SCR;
    if (nb > e.redo_blocks) e.redo_blocks = nb;
  }
  if (err == cudaSuccess) err = cudaMemcpyAsync(e.d_xd, xds.data(), sizeof(XDraw) * xds.size(), cudaMemcpyHostToDevice, c.stream);
  if (err == cudaSuccess) err = cudaStreamSynchronize(c.stream);
  if (err != cudaSuccess) KDE_FAIL(100 + (int)err, "gibbs (exact): building the schedule: %s", cudaGetErrorString(err));
  return 0;
}

// P arrives filled by gibbs_device with the entry's schedule; this sizes the grid, adds the XDraws, the redo counters
// and the launch's redo scratch
int gibbs_exact_launch(GibbsParams &P, const SchedEntry &E, int d, cudaStream_t st) {
  Context &c = ctx();
  const size_t smem = GB_STAGES * GB_TILE_BYTES;
  int per_sm = 0;
  cudaError_t e = with_d(d, [&](auto D) { return occupancy_gibbs_exact_d<decltype(D)::value>(P.M, smem, &per_sm); });
  if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "gibbs (exact) occupancy: %s", cudaGetErrorString(e));
  if (per_sm < 1) per_sm = 1;
  int grid = per_sm * c.sm_count;
  if (grid > P.nbatches) grid = P.nbatches;

  XParams X;
  X.xd = E.d_xd;
  X.ex2_err = GX_EX2_ERR;
  X.rsq_err = GX_RSQ_ERR;
  X.inflate = 1.0;
  if (const char *ev = getenv("KDEB200_GIBBS_EXACT_INFLATE")) X.inflate = atof(ev);  // tests: force the FP64 tiers
  unsigned long long *d_count = nullptr;
  if (int rc = gibbs_counters(&d_count)) return rc;
  X.redone = d_count + 1;
  X.warp_redone = d_count + 2;
  X.redone_int = d_count + 3;
  X.warp_redone_int = d_count + 4;
  X.redone_b = d_count + 5;
  X.warp_redone_b = d_count + 6;
  X.tier3 = d_count + 7;
  X.warp_tier3 = d_count + 8;
  X.scr_stride = GX_SCR + E.redo_blocks;
  // The redo scratch belongs to this launch alone, stream-ordered on `st`: launches on other streams may be in flight
  // at the same time, and a warp that shared its (block, warp) slot with another launch would sum foreign terms.
  X.scratch = nullptr;
  KDE_CUDA(cudaMallocAsync(&X.scratch, sizeof(double) * (size_t)grid * (GB_THREADS / 32) * X.scr_stride, st));
  e = with_d(d, [&](auto D) { return launch_gibbs_exact_d<decltype(D)::value>(P, X, grid, smem, st); });
  cudaFreeAsync(X.scratch, st);  // released once the kernel ahead of it on `st` has finished
  if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "gibbs (exact) kernel launch: %s", cudaGetErrorString(e));
  return 0;
}

// ---- bound probe (tests) ------------------------------------------------------------------------------------------
// For query conditionals (mu, Calmost) of one certified draw (the leaf draw, variant A; on an internal level the first
// sampleIndex draw, variant C, or with pass0 the sampleIndices! draw, variant B, which ignores Calmost): every node's FP32 term as K1x computes it, its bound, K1's FP64 term, K1's prefix sums,
// and the intervals K1x would claim for them -- per node as xa_decide forms them, and at checkpoints as xa_pass1 forms
// them (trip sums in FP32, Q in FP32 per chunk).  One CTA per query.
// out per query: [A, B, aabs, ok, lw2max, n, G, W] then per node [p32, acc32, p64, S64, lo, hi, lo_ck, hi_ck]
// (lo_ck / hi_ck are NaN except at chunk ends; the intervals bound S64 / W).
constexpr int GX_PROBE_HDR = 8, GX_PROBE_NODE = 8;

template <int D, int VAR>
__global__ void gibbs_exact_probe_kernel(Draw dr, XDraw xd, const double *mu_all, const double *cadd_all, GibbsParams P,
                                         int j, double *out_all) {
  constexpr int stride = gf_stride(D, VAR);
  constexpr int UNR = gf_unr(D, VAR);
  const int qi = blockIdx.x;
  double *out = out_all + (size_t)qi * (GX_PROBE_HDR + (size_t)GX_PROBE_NODE * dr.n);
  double mu[D];
  Hoist<D, false> h;
  double cadd[D];
  for (int k = 0; k < D; ++k) {  // the expressions of gibbs_exact_kernel
    mu[k] = mu_all[qi * D + k];
    h.mu[k] = mu[k];
    cadd[k] = VAR == VAR_B ? 0.0 : cadd_all[qi * D + k];
    h.cadd[k] = cadd[k];
    h.act[k] = true;
    h.ich[k] = sqrt(0.5 / (P.hvar[j][k] + h.cadd[k]));
  }
  Hoist32<D> g;
  float ks[D], sv[D];
  double rsmax;
  const bool rok = x_chain<D, VAR>(xd, cadd, P.hvar[j], ks, sv, g, rsmax);
  XBound bd = xa_bound<D, VAR>(xd, ks, rsmax, dr.n, GX_EX2_ERR, GX_RSQ_ERR, 1.0);
  bd.ok = bd.ok && rok;
  for (int z = threadIdx.x; z < dr.n; z += blockDim.x) {
    xa_tile_hoist<D, VAR>(xd.ctr + (size_t)(z / dr.tnodes) * KDEB200_MAX_DIM, mu, sv, g);
    float al, ah, pa, pb;
    xa_pair<D, VAR, true>(xd.rec32 + (size_t)(z >> 1) * stride, g, pa, pb, al, ah);
    double *o = out + GX_PROBE_HDR + (size_t)GX_PROBE_NODE * z;
    o[0] = (double)((z & 1) ? pb : pa);
    o[1] = (double)((z & 1) ? ah : al);
    o[2] = eval_node<D, false, VAR, true>(dr.rec + (size_t)z * dr.stride, h, P.exptab, P.ec);
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
  out[7] = exp2(xd.lw2max);
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

int gibbs_exact_probe(const kdeb200_tree_t *trees, int ndens, int Niter, int j, int level, int pass0, const double *mu,
                      const double *cadd, int nq, double *out, int64_t out_len) {
  if (!trees || ndens < 1 || ndens > KDEB200_MAX_DENS || j < 0 || j >= ndens || nq < 1 || !mu || !cadd || !out)
    KDE_FAIL(3, "gibbs_exact_probe: bad arguments");
  const int d = trees[0]->d;
  if (d != 3) KDE_FAIL(3, "gibbs_exact_probe: d = 3 only (the dimension K1x serves)");
  Context &c = ctx();
  int L = 0;
  if (int rc = gibbs_sizes(trees, ndens, Niter, &L, nullptr, nullptr, nullptr)) return rc;
  SchedEntry key, E;  // K1x's key: the tree set and Niter
  key.M = ndens;
  key.T = Niter;
  for (int i = 0; i < ndens; ++i) key.trees[i] = trees[i];
  if (int rc = sched_get(ROUTE_K1X, trees, L, key, &E, nullptr)) return rc;
  std::vector<Draw> draws(E.ndraws);
  std::vector<XDraw> xds(E.ndraws);
  KDE_CUDA(cudaMemcpy(draws.data(), E.d_draws, sizeof(Draw) * E.ndraws, cudaMemcpyDeviceToHost));
  KDE_CUDA(cudaMemcpy(xds.data(), E.d_xd, sizeof(XDraw) * E.ndraws, cudaMemcpyDeviceToHost));
  int di = -1;
  for (int i = 0; i < E.ndraws && di < 0; ++i)
    if (draws[i].j == j && draws[i].level == level && (draws[i].variant == VAR_A || draws[i].kind == (pass0 ? 0 : 1)))
      di = i;
  if (di < 0) KDE_FAIL(3, "gibbs_exact_probe: level %d of density %d has no certified draw", level, j + 1);
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
    if (draws[di].variant == VAR_A)
      gibbs_exact_probe_kernel<3, VAR_A><<<nq, 128, 0, c.stream>>>(draws[di], xds[di], d_mu, d_mu + nq * d, P, j, d_out);
    else if (draws[di].variant == VAR_B)
      gibbs_exact_probe_kernel<3, VAR_B><<<nq, 128, 0, c.stream>>>(draws[di], xds[di], d_mu, d_mu + nq * d, P, j, d_out);
    else
      gibbs_exact_probe_kernel<3, VAR_C><<<nq, 128, 0, c.stream>>>(draws[di], xds[di], d_mu, d_mu + nq * d, P, j, d_out);
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
