// gibbs.cu -- host side of the Gibbs sampler: argument checks, routing (K1w, K1f, K1x, K1, K1m), the schedule cache of the
// thread-per-chain kernels, the launches of K1 and K1w, Philox stream materialisation.  K1's kernels live in
// gibbs_kernel.cuh and are instantiated once per dimension in gibbs_d<N>.cu; the schedule is planned in gibbs_plan.cuh.
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <list>
#include <mutex>
#include <vector>

#include "gibbs.cuh"
#include "gibbs_plan.cuh"

namespace kdeb200 {

#define GB_EXTERN(D)                                                                                      \
  extern template cudaError_t launch_gibbs_d<D>(const GibbsParams &, bool, int, size_t, cudaStream_t, int); \
  extern template cudaError_t launch_gibbs_warp_d<D>(const GibbsParams &, bool, int, cudaStream_t);
GB_EXTERN(1) GB_EXTERN(2) GB_EXTERN(3) GB_EXTERN(4) GB_EXTERN(5) GB_EXTERN(6) GB_EXTERN(7) GB_EXTERN(8)
#undef GB_EXTERN

__global__ void philox_streams_kernel(uint64_t seed, int64_t Np, int64_t perU, int64_t perN, double *U, double *G) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nu = Np * perU, nn = Np * perN;
  if (i < nu) {
    // array slot g (0-based) is read by sample s = (g+1) / perU at call c = (g+1) % perU
    const int64_t g1 = i + 1;
    U[i] = philox_uniform(seed, (uint64_t)(g1 / perU), (uint32_t)(g1 % perU));
  }
  if (i < nn) G[i] = philox_normal(seed, (uint64_t)(i / perN), (uint32_t)(i % perN));
}

// ---------------------------------------------------------------- host side --------------
int gibbs_nlevels(const kdeb200_tree_t *trees, int ndens) {
  int64_t maxNp = 0;
  for (int j = 0; j < ndens; ++j)
    if (maxNp < trees[j]->N) maxNp = trees[j]->N;
  return (int)std::floor((std::log((double)maxNp) / std::log(2.0)) + 1.0);  // src/MSGibbs01.jl:568
}

int gibbs_sizes(const kdeb200_tree_t *trees, int ndens, int Niter, int *nlevels, int64_t *perU, int64_t *perN,
                int64_t *evals) {
  if (ndens < 1 || ndens > KDEB200_MAX_DENS_LARGE)
    KDE_FAIL(3, "gibbs: ndens=%d outside 1..%d", ndens, KDEB200_MAX_DENS_LARGE);
  if (Niter < 0) KDE_FAIL(3, "gibbs: Niter must be >= 0");
  for (int j = 0; j < ndens; ++j) {
    if (!trees[j]) KDE_FAIL(3, "gibbs: tree %d is NULL", j);
    if (!trees[j]->gibbs_ready)
      KDE_FAIL(7, "gibbs: tree %d was created by kdeb200_tree_create_eval (leaf records only); use kdeb200_tree_create", j);
    if (trees[j]->d != trees[0]->d) KDE_FAIL(6, "kdes must have same dimension");  // src/MSGibbs01.jl:721
  }
  const int L = gibbs_nlevels(trees, ndens);
  if (nlevels) *nlevels = L;
  if (perU) *perU = (int64_t)ndens * (1 + (int64_t)L * (1 + Niter));
  if (perN) *perN = (int64_t)trees[0]->d * (L + 1);
  if (evals) {
    int64_t e = 0;
    for (int j = 0; j < ndens; ++j)
      for (int l = 1; l <= L; ++l) e += trees[j]->levels[l < trees[j]->depth ? l : trees[j]->depth].n;
    *evals = e * (1 + Niter);
  }
  return 0;
}

// ---- schedule cache -----------------------------------------------------------------------------------------
// The static schedule (draws + tile list, and K1f's / K1x's FP32 records) depends only on the tree set, Niter and the
// route's key (SchedEntry).  It used to be rebuilt, allocated, uploaded and SYNCHRONISED on every call -- irrelevant at
// 1M samples, but it was the difference between a 0.34 ms kernel and a 0.39 ms call at the small configurations, and it
// made kdeb200_gibbs_device block.  K1m (gibbs_many.cu, more than KDEB200_MAX_DENS densities) uses route K1's entries.  Entries are invalidated wholesale whenever any tree is destroyed (a global epoch);
// each context keeps the most recent ones of each route (K1 8, K1f 4, K1x 4).  Batch counters come from a ring of 256
// slots per entry, zeroed once at creation and reset by the LAST CTA of each launch.
std::atomic<uint64_t> g_tree_epoch{1};
void gibbs_invalidate_schedules() { g_tree_epoch.fetch_add(1); }

namespace {
constexpr int SCHED_COUNTERS = 256;
constexpr size_t SCHED_KEEP[NROUTES] = {8, 4, 4};
std::mutex g_sched_mu;
std::list<SchedEntry> g_sched[NROUTES][KDEB200_MAX_GPUS];
unsigned long long *g_counters[KDEB200_MAX_GPUS] = {nullptr};
constexpr int NCOUNTERS = 9;

void sched_free(SchedEntry &e, cudaStream_t st) {
  if (e.d_base) cudaFreeAsync(e.d_base, st);
  if (e.d_extra) cudaFreeAsync(e.d_extra, st);
  e.d_base = e.d_extra = nullptr;
}

bool same_key(const SchedEntry &a, const SchedEntry &b) {
  if (a.M != b.M || a.T != b.T || a.masked != b.masked || a.literal != b.literal ||
      std::memcmp(a.mask, b.mask, sizeof(a.mask)) != 0)
    return false;
  for (int j = 0; j < a.M; ++j)
    if (a.trees[j] != b.trees[j]) return false;
  return true;
}

size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }

// plan, allocate, run the route's part, upload; the upload runs on the library stream of this context and is complete
// before the entry is published, so the caller's stream only ever sees finished buffers
int sched_build(Route r, const kdeb200_tree_t *trees, int L, SchedEntry &e) {
  Context &c = ctx();
  Plan S;
  plan_schedule(trees, e.M, L, e.T, !e.masked && !e.literal, r != ROUTE_K1, r == ROUTE_K1F, S);
  if (r == ROUTE_K1X) gibbs_exact_plan(trees, S);
  const size_t b_draws = up256(sizeof(Draw) * S.draws.size()), b_tiles = up256(sizeof(TileDesc) * S.tiles.size()),
               b_cnt = up256(sizeof(int) * SCHED_COUNTERS),
               b_rec = S.blocks.empty() ? 0 : up256(sizeof(float) * (S.nfloats + 8));
  KDE_CUDA(cudaMallocAsync(&e.d_base, b_draws + b_tiles + b_cnt + b_rec, c.stream));
  e.d_draws = reinterpret_cast<Draw *>(e.d_base);
  e.d_tiles = reinterpret_cast<TileDesc *>(e.d_base + b_draws);
  e.d_counters = reinterpret_cast<int *>(e.d_base + b_draws + b_tiles);
  e.d_rec = b_rec ? reinterpret_cast<float *>(e.d_base + b_draws + b_tiles + b_cnt) : nullptr;
  if (r == ROUTE_K1F)
    if (int rc = gibbs32_build(trees, S, e)) return rc;
  if (r == ROUTE_K1X)
    if (int rc = gibbs_exact_build(trees, S, e)) return rc;
  std::vector<TileDesc> tds(S.tiles.size());
  for (size_t i = 0; i < S.tiles.size(); ++i) {
    tds[i].src = S.tiles[i].src ? S.tiles[i].src : reinterpret_cast<const double *>(e.d_rec + S.tiles[i].off);
    tds[i].bytes = S.tiles[i].bytes;
    tds[i].pad = 0;
  }
  e.ndraws = (int)S.draws.size();
  e.ntiles = (int)tds.size();
  cudaError_t err = cudaMemcpyAsync(e.d_draws, S.draws.data(), sizeof(Draw) * S.draws.size(), cudaMemcpyHostToDevice, c.stream);
  if (err == cudaSuccess) err = cudaMemcpyAsync(e.d_tiles, tds.data(), sizeof(TileDesc) * tds.size(), cudaMemcpyHostToDevice, c.stream);
  if (err == cudaSuccess) err = cudaMemsetAsync(e.d_counters, 0, b_cnt, c.stream);
  if (err == cudaSuccess) err = cudaStreamSynchronize(c.stream);  // the host vectors are pageable memory
  if (err != cudaSuccess) KDE_FAIL(100 + (int)err, "gibbs: uploading the schedule: %s", cudaGetErrorString(err));
  return 0;
}
}  // namespace

void gibbs_drop_schedules(int slot) {
  std::lock_guard<std::mutex> lk(g_sched_mu);
  for (auto &lst : g_sched) {
    for (auto &e : lst[slot]) sched_free(e, ctx_at(slot).stream);
    lst[slot].clear();
  }
  if (g_counters[slot]) cudaFreeAsync(g_counters[slot], ctx_at(slot).stream);
  g_counters[slot] = nullptr;
}

int sched_get(Route r, const kdeb200_tree_t *trees, int L, const SchedEntry &key, SchedEntry *out, int **counter) {
  Context &c = ctx();
  std::lock_guard<std::mutex> lk(g_sched_mu);
  auto &lst = g_sched[r][c.slot];
  const uint64_t epoch = g_tree_epoch.load();
  for (auto it = lst.begin(); it != lst.end();) {  // entries from before the last tree_destroy may point at freed records
    if (it->epoch != epoch) {
      sched_free(*it, c.stream);
      it = lst.erase(it);
    } else {
      ++it;
    }
  }
  auto it = lst.begin();
  while (it != lst.end() && !same_key(*it, key)) ++it;
  if (it != lst.end()) {
    lst.splice(lst.begin(), lst, it);  // most recently used first
  } else {
    SchedEntry e = key;
    e.epoch = epoch;
    if (int rc = sched_build(r, trees, L, e)) {
      sched_free(e, c.stream);
      return rc;
    }
    lst.push_front(e);
    while (lst.size() > SCHED_KEEP[r]) {
      // an evicted entry may still be read by a kernel in flight on a caller stream: release it only after the device
      // has drained (rare: more distinct tree sets alternating than the route keeps)
      cudaDeviceSynchronize();
      sched_free(lst.back(), c.stream);
      lst.pop_back();
    }
  }
  if (counter) *counter = lst.front().d_counters + (lst.front().next_counter++ % SCHED_COUNTERS);
  *out = lst.front();
  return 0;
}

int gibbs_counters(unsigned long long **out) {
  Context &c = ctx();
  std::lock_guard<std::mutex> lk(g_sched_mu);
  if (!g_counters[c.slot]) {
    KDE_CUDA(cudaMallocAsync(&g_counters[c.slot], NCOUNTERS * sizeof(unsigned long long), c.stream));
    KDE_CUDA(cudaMemsetAsync(g_counters[c.slot], 0, NCOUNTERS * sizeof(unsigned long long), c.stream));
    KDE_CUDA(cudaStreamSynchronize(c.stream));  // the caller's stream must see a finished buffer
  }
  *out = g_counters[c.slot];
  return 0;
}

// counters [first, first + n) of the calling context's device, reset to zero (synchronises the device)
static int take_counters(int first, int n, unsigned long long *h) {
  unsigned long long *d = nullptr;
  if (int rc = gibbs_counters(&d)) return rc;
  KDE_CUDA(cudaDeviceSynchronize());
  KDE_CUDA(cudaMemcpy(h, d + first, n * sizeof(*h), cudaMemcpyDeviceToHost));
  KDE_CUDA(cudaMemset(d + first, 0, n * sizeof(*h)));
  return 0;
}

// K1f draws redone in FP64 since the last call
int gibbs32_slow_draws(unsigned long long *out) { return take_counters(0, 1, out); }

// K1x lane-draws and warp-draws redone in FP64 since the last call: leaf levels, sampleIndex draws of internal levels,
// sampleIndices! draws of internal levels
int gibbs_exact_redone(unsigned long long *lanes, unsigned long long *warps) {
  unsigned long long h[2] = {0, 0};
  if (int rc = take_counters(1, 2, h)) return rc;
  if (lanes) *lanes = h[0];
  if (warps) *warps = h[1];
  return 0;
}
int gibbs_exact_redone_internal(unsigned long long *lanes, unsigned long long *warps) {
  unsigned long long h[2] = {0, 0};
  if (int rc = take_counters(3, 2, h)) return rc;
  if (lanes) *lanes = h[0];
  if (warps) *warps = h[1];
  return 0;
}
int gibbs_exact_redone_b(unsigned long long *lanes, unsigned long long *warps) {
  unsigned long long h[2] = {0, 0};
  if (int rc = take_counters(5, 2, h)) return rc;
  if (lanes) *lanes = h[0];
  if (warps) *warps = h[1];
  return 0;
}
// of those, the ones the warp-parallel FP64 sum could not decide either (every class)
int gibbs_exact_tier3(unsigned long long *lanes, unsigned long long *warps) {
  unsigned long long h[2] = {0, 0};
  if (int rc = take_counters(7, 2, h)) return rc;
  if (lanes) *lanes = h[0];
  if (warps) *warps = h[1];
  return 0;
}

// K1x takes the thread-per-chain FP64 calls that it has been measured to win: every dimension of every density (no
// partial-dimension mask, no lone density), no literal arithmetic, d = 3 (the only dimension measured so far; C4: 904
// -> 776 ms per 1M samples, DESIGN.md K1x), and leaf bandwidths whose FP32 scale s_k = sqrt(0.5 log2 e / c_k) stays a
// normal float.  KDEB200_GIBBS_EXACT=0 forces K1.
static bool exact_eligible(const kdeb200_tree_t *trees, int ndens, bool masked, bool literal) {
  const char *ev = getenv("KDEB200_GIBBS_EXACT");
  if ((ev && atoi(ev) == 0) || ndens < 2 || masked || literal || trees[0]->d != 3) return false;
  for (int j = 0; j < ndens; ++j)
    for (int k = 0; k < trees[0]->d; ++k)
      if (!(trees[j]->hvar[k] >= 1e-20 && trees[j]->hvar[k] <= 1e20)) return false;
  return true;
}

int gibbs_device(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                 const uint8_t *dimmask, const double *d_randU, int64_t nU, const double *d_randN, int64_t nN,
                 uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                 int64_t *d_level_labels, cudaStream_t st, int *launches) {
  Context &c = ctx();
  int L = 0;
  int64_t perU = 0, perN = 0;
  if (int rc = gibbs_sizes(trees, ndens, Niter, &L, &perU, &perN, nullptr)) return rc;
  const int d = trees[0]->d;
  if (Np < 0 || s0 < 0 || s1 > Np || s0 > s1) KDE_FAIL(3, "gibbs: bad sample range [%lld,%lld) of %lld", (long long)s0, (long long)s1, (long long)Np);
  if (s1 == s0) return 0;
  if ((d_randU == nullptr) != (d_randN == nullptr)) KDE_FAIL(3, "gibbs: randU and randN must be given together");
  if (d_randU) {  // the reference would throw BoundsError
    if (s1 * perU > nU + 1) KDE_FAIL(7, "gibbs: randU too short (%lld < %lld)", (long long)nU, (long long)(s1 * perU - 1));
    if (s1 * perN > nN) KDE_FAIL(7, "gibbs: randN too short (%lld < %lld)", (long long)nN, (long long)(s1 * perN));
  }
  // Densities the restructured arithmetic cannot take (zero / non-finite / out-of-range variances, non-finite means or
  // weights) run through the warp-per-chain kernel with the reference's arithmetic verbatim, NaN / Inf rules included
  // (src/MSGibbs01.jl:287-315) -- as long as their level lists fit that kernel's shared memory.
  bool literal = false;
  for (int j = 0; j < ndens; ++j) {
    if (trees[j]->degenerate) literal = true;
    if (trees[j]->slot != c.slot) KDE_FAIL(3, "gibbs: tree %d lives on another GPU of the set than the calling context", j);
  }
  if (ndens > KDEB200_MAX_DENS)  // more densities than GibbsParams holds: K1m at every Np and precision (gibbs_many.cu)
    return gibbs_many_device(trees, ndens, L, perU, perN, Niter, add_entropy, dimmask, d_randU, d_randN, seed, s0, s1,
                             d_points, d_indices, d_level_labels, st, launches);

  GibbsParams P;
  std::memset(&P, 0, sizeof(P));
  bool masked = (ndens == 1);  // a lone density has no "other" dims: handled by the mask logic
  for (int j = 0; j < ndens; ++j)
    for (int k = 0; k < d; ++k) {
      P.mask[j][k] = dimmask ? (dimmask[j * d + k] != 0) : 1;
      if (!P.mask[j][k]) masked = true;
    }
  for (int j = 0; j < ndens; ++j)
    for (int k = 0; k < d; ++k) {
      unsigned char o = 0;
      for (int i = 0; i < ndens; ++i)
        if (i != j && P.mask[i][k]) o = 1;
      P.other[j][k] = o;
    }
  if (literal) masked = true;  // the literal evaluation reads the activity flags in every mode

  // Few chains: one warp per chain (K1w).  The thread-per-chain kernel needs ~128 x 4 x SMs chains to fill the chip and
  // costs the same 0.3 - 3 ms whether it runs 100 chains or 10 000; measured crossover (tools/gibbs_kernel_crossover.py,
  // profiles/r02_gibbs_crossover.json): ~4 000 chains for 2 - 6 densities of 100 - 1000 components, so the warp
  // kernel takes calls of up to 24 chains per SM (KDEB200_GIBBS_WARP_MAX overrides; 0 disables it).  Its prefix sums
  // live in shared memory, which bounds the level size.
  int nmax = 1;
  for (int j = 0; j < ndens; ++j)
    if (trees[j]->levels[trees[j]->depth].n > nmax) nmax = (int)trees[j]->levels[trees[j]->depth].n;
  int64_t warp_max = (int64_t)24 * c.sm_count;
  if (const char *ev = getenv("KDEB200_GIBBS_WARP_MAX")) warp_max = atoll(ev);
  const bool warp_fits = gibbs_warp_smem(d, nmax) <= 96 * 1024;
  if (literal && !warp_fits)
    KDE_FAIL(8, "gibbs: a density has a zero, non-finite or out-of-range (variance outside [1e-30, 1e30]) bandwidth / mean / "
                "weight and more than ~2900 components: the verbatim-arithmetic kernel cannot hold its level lists "
                "(no CPU fallback)");
  const bool warp = warp_fits && (literal || s1 - s0 <= warp_max);

  Route r = ROUTE_K1;
  if (!warp && gibbs_precision() == KDEB200_F32)
    r = ROUTE_K1F;  // FP32 label probabilities (statistical mode only)
  else if (!warp && exact_eligible(trees, ndens, masked, literal))
    r = ROUTE_K1X;
  SchedEntry key;
  key.M = ndens;
  key.T = Niter;
  for (int j = 0; j < ndens; ++j) key.trees[j] = trees[j];
  if (r != ROUTE_K1X) key.masked = masked;
  if (r == ROUTE_K1) key.literal = literal;
  if (r == ROUTE_K1F) std::memcpy(key.mask, P.mask, sizeof(key.mask));
  SchedEntry E;
  int *d_counter = nullptr;
  if (int rc = sched_get(r, trees, L, key, &E, &d_counter)) return rc;

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
  P.literal = literal ? 1 : 0;
  P.nbatches = (int)((s1 - s0 + GB_THREADS - 1) / GB_THREADS);
  for (int j = 0; j < ndens; ++j) {
    const kdeb200_tree_s *t = trees[j];
    P.root_rec[j] = t->d_buf + t->levels[0].offC;
    P.labels[j] = t->d_labels;
    for (int k = 0; k < d; ++k) P.hvar[j][k] = t->hvar[k];
  }

  if (r == ROUTE_K1F) {
    if (int rc = gibbs32_launch(P, E, d, st)) return rc;
  } else if (r == ROUTE_K1X) {
    if (int rc = gibbs_exact_launch(P, E, d, st)) return rc;
  } else if (warp) {
    const cudaError_t e = with_d(d, [&](auto D) { return launch_gibbs_warp_d<decltype(D)::value>(P, masked, nmax, st); });
    if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "gibbs (warp per chain) kernel launch: %s", cudaGetErrorString(e));
  } else {
    const size_t smem = GB_STAGES * GB_TILE_BYTES;
    const cudaError_t e = with_d(d, [&](auto D) {
      return launch_gibbs_d<decltype(D)::value>(P, masked, P.nbatches, smem, st, c.sm_count);
    });
    if (e != cudaSuccess) KDE_FAIL(100 + (int)e, "gibbs kernel launch: %s", cudaGetErrorString(e));
  }
  if (launches) *launches += 1;
  return 0;
}

int philox_streams_device(uint64_t seed, int64_t Np, int64_t perU, int64_t perN, double *d_U, double *d_G,
                          cudaStream_t st) {
  const int64_t n = (Np * perU > Np * perN) ? Np * perU : Np * perN;
  if (n <= 0) return 0;
  philox_streams_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(seed, Np, perU, perN, d_U, d_G);
  KDE_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace kdeb200
