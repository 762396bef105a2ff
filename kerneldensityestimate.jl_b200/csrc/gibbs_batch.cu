// gibbs_batch.cu -- host side of K1b (kdeb200_gibbs_batch, kdeb200_product_kde_batch): many independent
// prodAppxMSGibbsS problems in one blocking call.  Every problem is checked as a single call checks it before anything
// is launched; each distinct (tree set, masked) is planned once with K1's own planner; draws, tiles, problem
// descriptors and injected streams travel in ONE copy from a pinned staging buffer of the context; one K1b launch per
// (d, masked) class; problems with degenerate bandwidths take the single-call route (K1w's verbatim arithmetic) on the
// same stream; one device buffer and one copy back per output kind.  The batched schedules are not kept in the
// single-call cache, which holds a handful of entries and drains the device on eviction (hundreds of tree sets per
// call would turn that into a sync per problem).  Instead each tree keeps the draws K1's planner makes for it alone
// (TreeDraws), and a problem's schedule is assembled from its trees' templates: K1's plan, without planning it again.
#include <chrono>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "gibbs.cuh"
#include "gibbs_batch_kernel.cuh"
#include "gibbs_plan.cuh"
#include "lcv.cuh"

namespace kdeb200 {

#define GBB_EXTERN(D) extern template cudaError_t launch_gibbs_batch_d<D>(const BatchParams &, bool, int, int, cudaStream_t);
GBB_EXTERN(1) GBB_EXTERN(2) GBB_EXTERN(3) GBB_EXTERN(4) GBB_EXTERN(5) GBB_EXTERN(6) GBB_EXTERN(7) GBB_EXTERN(8)
#undef GBB_EXTERN

// The draws K1's planner (gibbs_plan.cuh) makes for one tree alone, per tree level li = 1..depth and pass kind (0:
// sampleIndices!, 1: sampleIndex), with their tiles.  A draw of a tree set depends on its density's tree, li =
// min(level, depth) and the kind, except for j, level, new_level and tile0; so plan_schedule(trees, M, L, T, b_records,
// false, false) is these templates in the planner's order (level, pass, density) with those four fields set.
struct TreeDraws {
  std::vector<Draw> draws;      // [(li - 1) * 2 + kind]; tile0 indexes `tiles`
  std::vector<TileDesc> tiles;
};

const TreeDraws &tree_draws(kdeb200_tree_t t, bool b_records) {
  std::shared_ptr<TreeDraws> &sp = t->batch_draws[b_records ? 1 : 0];
  if (!sp) {
    Plan S;
    plan_schedule(&t, 1, t->depth, 1, b_records, false, false, S);
    auto td = std::make_shared<TreeDraws>();
    td->draws = S.draws;
    td->tiles.resize(S.tiles.size());
    for (size_t i = 0; i < S.tiles.size(); ++i) td->tiles[i] = TileDesc{S.tiles[i].src, S.tiles[i].bytes, 0};
    sp = td;
  }
  return *sp;
}

// tiles of plan_schedule(trees, M, L, T, b_records, false, false); its draws number L (T + 1) M
int64_t assembled_tiles(const kdeb200_tree_t *trees, int M, int L, int T, bool b_records) {
  int64_t nt = 0;
  for (int j = 0; j < M; ++j) {
    const TreeDraws &td = tree_draws(trees[j], b_records);
    for (int l = 1; l <= L; ++l) {
      const int li = l < trees[j]->depth ? l : trees[j]->depth;
      nt += td.draws[(li - 1) * 2].ntiles + (int64_t)T * td.draws[(li - 1) * 2 + 1].ntiles;
    }
  }
  return nt;
}

// writes plan_schedule(trees, M, L, T, b_records, false, false)'s draws and tile descriptors
void assemble_schedule(const kdeb200_tree_t *trees, int M, int L, int T, bool b_records, Draw *draws, TileDesc *tiles) {
  const TreeDraws *td[KDEB200_MAX_DENS];
  for (int j = 0; j < M; ++j) td[j] = &tree_draws(trees[j], b_records);
  int nd = 0, nt = 0;
  for (int l = 1; l <= L; ++l)
    for (int pass = 0; pass <= T; ++pass)
      for (int j = 0; j < M; ++j) {
        const int li = l < trees[j]->depth ? l : trees[j]->depth;
        const Draw &src = td[j]->draws[(li - 1) * 2 + (pass == 0 ? 0 : 1)];
        Draw &dr = draws[nd++];
        dr = src;
        dr.j = (short)j;
        dr.level = (short)l;
        dr.new_level = (pass == 0 && j == 0) ? 1 : 0;
        dr.tile0 = nt;
        std::memcpy(tiles + nt, td[j]->tiles.data() + src.tile0, sizeof(TileDesc) * src.ntiles);
        nt += src.ntiles;
      }
}

namespace {
struct BatchState {  // per context: the pinned staging buffer and the split of the last call
  char *stage = nullptr;
  size_t stage_bytes = 0;
  cudaEvent_t ev_h2d = nullptr, ev_d2h = nullptr;
  double plan_ms = 0.0, h2d_ms = 0.0, d2h_ms = 0.0;
};
BatchState g_batch[KDEB200_MAX_GPUS];

size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }
size_t up16(size_t b) { return (b + 15) & ~(size_t)15; }

struct Prob {
  int t0, M, d, L, sched;
  int64_t Np, perU, perN, offP, offI, offU, offN, offM, offB;
  bool injected, literal, masked;
};
}  // namespace

void gibbs_batch_drop(int slot) {
  BatchState &b = g_batch[slot];
  if (b.stage) cudaFreeHost(b.stage);
  if (b.ev_h2d) cudaEventDestroy(b.ev_h2d);
  if (b.ev_d2h) cudaEventDestroy(b.ev_d2h);
  b = BatchState();
}

int batch_stage(size_t bytes, char **out) {
  BatchState &bs = g_batch[ctx().slot];
  if (bs.stage_bytes < bytes) {
    if (bs.stage) cudaFreeHost(bs.stage);
    bs.stage = nullptr;
    bs.stage_bytes = 0;
    KDE_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&bs.stage), bytes, cudaHostAllocDefault));
    bs.stage_bytes = bytes;
  }
  *out = bs.stage;
  return 0;
}

int gibbs_batch_split(double *plan_ms, double *h2d_ms, double *d2h_ms) {
  const BatchState &b = g_batch[ctx().slot];
  if (plan_ms) *plan_ms = b.plan_ms;
  if (h2d_ms) *h2d_ms = b.h2d_ms;
  if (d2h_ms) *d2h_ms = b.d2h_ms;
  return 0;
}

int gibbs_batch(const GibbsBatchArgs &a, double *points_out, int64_t *indices_out, double *bw_std_out, int *nloo_out) {
  const auto t_enter = std::chrono::steady_clock::now();
  Context &c = ctx();
  BatchState &bs = g_batch[c.slot];
  const bool product = bw_std_out != nullptr;
  const char *fn = product ? "product_kde_batch" : "gibbs_batch";
  const int n = a.nprob;
  if (n < 0) KDE_FAIL(3, "%s: nprob=%d < 0", fn, n);
  if ((a.randU == nullptr) != (a.randN == nullptr)) KDE_FAIL(3, "%s: randU and randN must be given together", fn);
  if (a.randU && (!a.nU || !a.nN)) KDE_FAIL(2, "%s: randU / randN given without nU / nN", fn);

  // ---- every problem checked as the single call checks it; nothing runs unless all pass
  std::vector<Prob> pr(n);
  int64_t tt = 0, offP = 0, offI = 0, offU = 0, offN = 0, offM = 0, offB = 0;
  for (int i = 0; i < n; ++i) {
    Prob &p = pr[i];
    p.M = a.ndens[i];
    if (p.M < 1 || p.M > KDEB200_MAX_DENS)
      KDE_FAIL(3, "%s: problem %d: ndens=%d outside 1..%d", fn, i, p.M, KDEB200_MAX_DENS);
    const kdeb200_tree_t *trees = a.trees + tt;
    if (int rc = gibbs_sizes(trees, p.M, a.Niter, &p.L, &p.perU, &p.perN, nullptr)) {
      const std::string msg = get_error();
      KDE_FAIL(rc, "%s: problem %d: %s", fn, i, msg.c_str());
    }
    p.t0 = (int)tt;
    p.d = trees[0]->d;
    p.Np = a.Np[i];
    p.sched = -1;
    if (p.Np < 0) KDE_FAIL(3, "%s: problem %d: Np=%lld < 0", fn, i, (long long)p.Np);
    if (product && p.Np < 2)
      KDE_FAIL(3, "%s: problem %d: at least two product samples are needed for cross validation", fn, i);
    const int64_t nu = a.randU ? a.nU[i] : 0, nn = a.randN ? a.nN[i] : 0;
    if (nu < 0 || nn < 0) KDE_FAIL(3, "%s: problem %d: negative stream length", fn, i);
    p.injected = nu > 0 || nn > 0;
    if (p.injected) {  // the reference would throw BoundsError
      if (p.Np * p.perU > nu + 1)
        KDE_FAIL(7, "%s: problem %d: randU too short (%lld < %lld)", fn, i, (long long)nu, (long long)(p.Np * p.perU - 1));
      if (p.Np * p.perN > nn)
        KDE_FAIL(7, "%s: problem %d: randN too short (%lld < %lld)", fn, i, (long long)nn, (long long)(p.Np * p.perN));
    } else if (p.Np > 0 && !a.seeds) {
      KDE_FAIL(2, "%s: problem %d draws from Philox but seeds is NULL", fn, i);
    }
    p.literal = false;
    p.masked = p.M == 1;  // a lone density has no "other" dims: handled by the mask logic
    int nmax = 1;
    for (int j = 0; j < p.M; ++j) {
      if (trees[j]->slot != c.slot)
        KDE_FAIL(3, "%s: problem %d: tree %d lives on another GPU of the set than the calling context", fn, i, j);
      if (trees[j]->degenerate) p.literal = true;
      if (trees[j]->levels[trees[j]->depth].n > nmax) nmax = (int)trees[j]->levels[trees[j]->depth].n;
      for (int k = 0; k < p.d; ++k)
        if (a.dimmask && !a.dimmask[offM + j * p.d + k]) p.masked = true;
    }
    if (p.literal && gibbs_warp_smem(p.d, nmax) > 96 * 1024)  // gibbs_device's limit of the verbatim arithmetic
      KDE_FAIL(8, "%s: problem %d: a density has a zero, non-finite or out-of-range bandwidth / mean / weight and more "
                  "than ~2900 components: the verbatim-arithmetic kernel cannot hold its level lists", fn, i);
    p.offP = offP;
    p.offI = offI;
    p.offU = offU;
    p.offN = offN;
    p.offM = offM;
    p.offB = offB;
    tt += p.M;
    offP += p.d * p.Np;
    offI += p.M * p.Np;
    offU += nu;
    offN += nn;
    offM += (int64_t)p.M * p.d;
    offB += p.d;
  }

  // ---- plans (one per distinct tree set and mask class) and launch classes (one per d and mask class)
  std::map<std::vector<const void *>, int> plan_of;
  std::vector<int> plan_src;  // per plan: the first problem that uses it
  std::map<std::pair<int, bool>, std::vector<int>> classes;
  int nitems = 0;
  for (int i = 0; i < n; ++i) {
    Prob &p = pr[i];
    if (product && p.Np <= LCV_FUSED_MAX) nitems += p.d;
    if (p.Np == 0 || p.literal) continue;
    std::vector<const void *> key(a.trees + p.t0, a.trees + p.t0 + p.M);
    key.push_back(reinterpret_cast<const void *>((uintptr_t)p.masked));
    auto it = plan_of.emplace(key, (int)plan_src.size()).first;
    if (it->second == (int)plan_src.size()) plan_src.push_back(i);
    p.sched = it->second;
    classes[{p.d, p.masked}].push_back(i);
  }
  const size_t nplans = plan_src.size();
  std::vector<int> plan_draws(nplans), plan_tiles(nplans);
  for (size_t k = 0; k < nplans; ++k) {
    const Prob &p = pr[plan_src[k]];
    plan_draws[k] = p.L * (a.Niter + 1) * p.M;
    const int64_t nt = assembled_tiles(a.trees + p.t0, p.M, p.L, a.Niter, /*b_records=*/!p.masked);
    if (nt >= ((int64_t)1 << 31)) KDE_FAIL(3, "%s: problem %d: schedule of 2^31 tiles or more", fn, plan_src[k]);
    plan_tiles[k] = (int)nt;
  }

  // ---- one staging area: draws | tiles | descriptors | block prefixes | LOOCV items | randU | randN
  std::vector<size_t> draw_at(nplans), tile_at(nplans);
  size_t bytes = 0;
  for (size_t k = 0; k < nplans; ++k) {
    draw_at[k] = bytes;
    bytes += up16(sizeof(Draw) * plan_draws[k]);
    tile_at[k] = bytes;
    bytes += up16(sizeof(TileDesc) * plan_tiles[k]);
  }
  bytes = up256(bytes);
  size_t nactive = 0;
  for (auto &cl : classes) nactive += cl.second.size();
  const size_t prob_at = bytes;
  bytes += up256(sizeof(BatchProb) * nactive);
  const size_t block_at = bytes;
  bytes += up256(sizeof(int) * (nactive + classes.size()));
  const size_t item_at = bytes;
  bytes += up256(sizeof(LcvBatchItem) * nitems);
  const size_t u_at = bytes;
  bytes += up256(sizeof(double) * offU);
  const size_t n_at = bytes;
  bytes += up256(sizeof(double) * offN);

  char *h = nullptr;
  if (int rc = batch_stage(bytes, &h)) return rc;
  if (!bs.ev_h2d) KDE_CUDA(cudaEventCreate(&bs.ev_h2d));
  if (!bs.ev_d2h) KDE_CUDA(cudaEventCreate(&bs.ev_d2h));
  DevBuf dBlob(c.stream), dP(c.stream), dI(c.stream), dO(c.stream);
  KDE_CUDA(dBlob.alloc(bytes));
  KDE_CUDA(dP.alloc(sizeof(double) * offP));
  KDE_CUDA(dI.alloc(sizeof(int64_t) * offI));
  KDE_CUDA(dO.alloc(sizeof(double) * 5 * offB));
  char *dv = dBlob.as<char>();
  const double *d_U = reinterpret_cast<const double *>(dv + u_at), *d_N = reinterpret_cast<const double *>(dv + n_at);

  for (size_t k = 0; k < nplans; ++k) {
    const Prob &p = pr[plan_src[k]];
    assemble_schedule(a.trees + p.t0, p.M, p.L, a.Niter, /*b_records=*/!p.masked,
                      reinterpret_cast<Draw *>(h + draw_at[k]), reinterpret_cast<TileDesc *>(h + tile_at[k]));
  }
  BatchProb *hp = reinterpret_cast<BatchProb *>(h + prob_at);
  int *hb = reinterpret_cast<int *>(h + block_at);
  struct Launch {
    int d, maxM, grid;
    bool masked;
    BatchParams B;
  };
  std::vector<Launch> launches_k1b;
  size_t np_at = 0, nb_at = 0;
  std::vector<std::pair<int, int>> slot;  // (descriptor, problem)
  for (auto &cl : classes) {
    Launch L;
    L.d = cl.first.first;
    L.masked = cl.first.second;
    L.maxM = 0;
    L.B.probs = reinterpret_cast<const BatchProb *>(dv + prob_at) + np_at;
    L.B.block0 = reinterpret_cast<const int *>(dv + block_at) + nb_at;
    L.B.nprob = (int)cl.second.size();
    L.B.exptab = c.d_exptab;
    L.B.ec = make_exp_consts();
    int64_t blocks = 0;
    for (int i : cl.second) {
      const Prob &p = pr[i];
      slot.push_back({(int)np_at++, i});
      hb[nb_at++] = (int)blocks;
      blocks += (p.Np + GB_THREADS - 1) / GB_THREADS;
      if (p.M > L.maxM) L.maxM = p.M;
    }
    if (blocks >= ((int64_t)1 << 31)) KDE_FAIL(3, "%s: more than 2^31 blocks of %d samples in one launch", fn, GB_THREADS);
    hb[nb_at++] = (int)blocks;
    L.grid = (int)blocks;
    launches_k1b.push_back(L);
  }
  for (size_t q = 0; q < slot.size(); ++q) {
    const int i = slot[q].second;
    const Prob &p = pr[i];
    const kdeb200_tree_t *trees = a.trees + p.t0;
    BatchProb &b = hp[slot[q].first];
    std::memset(&b, 0, sizeof(b));
    b.draws = reinterpret_cast<const Draw *>(dv + draw_at[p.sched]);
    b.tiles = reinterpret_cast<const TileDesc *>(dv + tile_at[p.sched]);
    b.randU = p.injected ? d_U + p.offU : nullptr;
    b.randN = p.injected ? d_N + p.offN : nullptr;
    b.points = dP.as<double>() + p.offP;
    b.indices = dI.as<int64_t>() + p.offI;
    b.Np = p.Np;
    b.perU = p.perU;
    b.perN = p.perN;
    b.seed = a.seeds ? a.seeds[i] : 0;
    b.ndraws = plan_draws[p.sched];
    b.ntiles = plan_tiles[p.sched];
    b.M = p.M;
    b.L = p.L;
    b.add_entropy = a.add_entropy ? 1 : 0;
    for (int j = 0; j < p.M; ++j) {
      b.root_rec[j] = trees[j]->d_buf + trees[j]->levels[0].offC;
      b.labels[j] = trees[j]->d_labels;
      for (int k = 0; k < p.d; ++k) {
        b.hvar[j][k] = trees[j]->hvar[k];
        b.mask[j][k] = a.dimmask ? (a.dimmask[p.offM + j * p.d + k] != 0) : 1;
      }
    }
    for (int j = 0; j < p.M; ++j)
      for (int k = 0; k < p.d; ++k) {
        unsigned char o = 0;
        for (int i2 = 0; i2 < p.M; ++i2)
          if (i2 != j && b.mask[i2][k]) o = 1;
        b.other[j][k] = o;
      }
  }
  LcvBatchItem *hi = reinterpret_cast<LcvBatchItem *>(h + item_at);
  std::vector<int64_t> out5_at(n, -1);
  {
    int64_t at5 = 0, ni = 0;
    for (int i = 0; i < n && product; ++i) {
      const Prob &p = pr[i];
      if (p.Np > LCV_FUSED_MAX) continue;
      out5_at[i] = at5;
      const double w2 = lcv_points_w2(p.Np);
      for (int k = 0; k < p.d; ++k) {
        LcvBatchItem &it = hi[ni++];
        it.pts = dP.as<double>() + p.offP;
        it.out = dO.as<double>() + at5;
        it.N = (int)p.Np;
        it.d = p.d;
        it.dim = k;
        it.pad_ = 0;
        it.w2 = w2;
      }
      at5 += 5 * p.d;
    }
  }
  if (offU) std::memcpy(h + u_at, a.randU, sizeof(double) * offU);
  if (offN) std::memcpy(h + n_at, a.randN, sizeof(double) * offN);
  bs.plan_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_enter).count();

  // ---- one copy in, the launches, one copy back per output kind, one synchronise
  struct Drain {  // an error return after this point waits for the enqueued work: the staging buffer is reused
    cudaStream_t st;
    ~Drain() { cudaStreamSynchronize(st); }
  } drain{c.stream};
  KDE_CUDA(cudaEventRecord(bs.ev_h2d, c.stream));
  KDE_CUDA(cudaMemcpyAsync(dv, h, bytes, cudaMemcpyHostToDevice, c.stream));
  KDE_CUDA(cudaEventRecord(c.ev0, c.stream));
  int launches = 0;
  for (const Launch &L : launches_k1b) {
    const cudaError_t e = with_d(L.d, [&](auto D) {
      return launch_gibbs_batch_d<decltype(D)::value>(L.B, L.masked, L.maxM, L.grid, c.stream);
    });
    if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "%s: K1b launch: %s", fn, cudaGetErrorString(e));
    ++launches;
  }
  for (int i = 0; i < n; ++i) {  // degenerate bandwidths: the single call's verbatim route, one call each
    const Prob &p = pr[i];
    if (!p.literal || p.Np == 0) continue;
    if (int rc = gibbs_device(a.trees + p.t0, p.M, p.Np, a.Niter, a.add_entropy, a.dimmask ? a.dimmask + p.offM : nullptr,
                              p.injected ? d_U + p.offU : nullptr, p.injected ? a.nU[i] : 0,
                              p.injected ? d_N + p.offN : nullptr, p.injected ? a.nN[i] : 0, a.seeds ? a.seeds[i] : 0, 0,
                              p.Np, dP.as<double>() + p.offP, dI.as<int64_t>() + p.offI, nullptr, c.stream, &launches)) {
      const std::string msg = get_error();
      KDE_FAIL(rc, "%s: problem %d: %s", fn, i, msg.c_str());
    }
  }
  if (nitems) {
    if (int rc = kde_lcv_points_batch_device(nitems, reinterpret_cast<const LcvBatchItem *>(dv + item_at), c.stream))
      return rc;
    ++launches;
  }
  KDE_CUDA(cudaEventRecord(c.ev1, c.stream));
  std::vector<double> out5(5 * offB);
  if (offP) KDE_CUDA(cudaMemcpyAsync(points_out, dP.p, sizeof(double) * offP, cudaMemcpyDeviceToHost, c.stream));
  if (offI && indices_out)
    KDE_CUDA(cudaMemcpyAsync(indices_out, dI.p, sizeof(int64_t) * offI, cudaMemcpyDeviceToHost, c.stream));
  if (nitems) KDE_CUDA(cudaMemcpyAsync(out5.data(), dO.p, sizeof(double) * 5 * offB, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaEventRecord(bs.ev_d2h, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, bs.ev_h2d, c.ev0);
  bs.h2d_ms = ms;
  cudaEventElapsedTime(&ms, c.ev1, bs.ev_d2h);
  bs.d2h_ms = ms;
  cudaEventElapsedTime(&ms, c.ev0, c.ev1);
  double kernel_ms = ms;

  // ---- the LOOCV bandwidths: fused results, or the host bandwidth loop for Np > LCV_FUSED_MAX (as kdeb200_product_kde)
  for (int i = 0; i < n && product; ++i) {
    const Prob &p = pr[i];
    if (out5_at[i] >= 0) {
      lcv_points_finish(p.d, out5.data() + out5_at[i], bw_std_out + p.offB, nloo_out ? nloo_out + p.offB : nullptr);
    } else {
      if (int rc = kde_lcv(p.d, p.Np, points_out + p.offP, 0, p.Np, nullptr, nullptr, bw_std_out + p.offB,
                           nloo_out ? nloo_out + p.offB : nullptr)) {
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
