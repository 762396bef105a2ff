// gibbs.cuh -- host-side declarations of the Gibbs sampler: its entry points, and what the host files of the
// thread-per-chain kernels share -- K1 and K1w in gibbs.cu (which also routes every call), K1f in gibbs_f32.cu, K1x in
// gibbs_exact.cu: one schedule cache, the per-context counters and the dimension dispatch.
#pragma once
#include <type_traits>

#include "tree.cuh"

namespace kdeb200 {

struct Draw;
struct TileDesc;
struct XDraw;
struct GibbsParams;
struct Plan;

int gibbs_sizes(const kdeb200_tree_t *trees, int ndens, int Niter, int *nlevels, int64_t *perU, int64_t *perN,
                int64_t *evals);
int gibbs_device(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                 const uint8_t *dimmask, const double *d_randU, int64_t nU, const double *d_randN, int64_t nN,
                 uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                 int64_t *d_level_labels, cudaStream_t st, int *launches);
// K1m, the call of more than KDEB200_MAX_DENS densities (gibbs_many.cu); gibbs_device checks the arguments and routes
int gibbs_many_device(const kdeb200_tree_t *trees, int ndens, int L, int64_t perU, int64_t perN, int Niter,
                      int add_entropy, const uint8_t *dimmask, const double *d_randU, const double *d_randN,
                      uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                      int64_t *d_level_labels, cudaStream_t st, int *launches);
int philox_streams_device(uint64_t seed, int64_t Np, int64_t perU, int64_t perN, double *d_U, double *d_G,
                          cudaStream_t st);
int gibbs_precision();
int gibbs_set_precision(int p);
int gibbs32_slow_draws(unsigned long long *out);
int gibbs_exact_redone(unsigned long long *lanes, unsigned long long *warps);
int gibbs_exact_redone_internal(unsigned long long *lanes, unsigned long long *warps);
int gibbs_exact_redone_b(unsigned long long *lanes, unsigned long long *warps);
int gibbs_exact_tier3(unsigned long long *lanes, unsigned long long *warps);
int gibbs_exact_probe(const kdeb200_tree_t *trees, int ndens, int Niter, int j, int level, int pass0, const double *mu,
                      const double *cadd, int nq, double *out, int64_t out_len);
void gibbs_invalidate_schedules();  // a tree is destroyed: cached schedules point into tree records
void gibbs_drop_schedules(int slot);  // a context goes away: frees its schedules and counters

// ---- batched problems (gibbs_batch.cu): the arguments of kdeb200_gibbs_batch, problem by problem
struct GibbsBatchArgs {
  int nprob;
  const int *ndens;
  const kdeb200_tree_t *trees;
  const int64_t *Np;
  int Niter, add_entropy;
  const uint8_t *dimmask;
  const double *randU;
  const int64_t *nU;
  const double *randN;
  const int64_t *nN;
  const uint64_t *seeds;
};
// Blocking, on the calling context.  bw_std_out != null adds the LOOCV refit of kdeb200_product_kde_batch.
int gibbs_batch(const GibbsBatchArgs &a, double *points_out, int64_t *indices_out, double *bw_std_out, int *nloo_out);
int gibbs_batch_split(double *plan_ms, double *h2d_ms, double *d2h_ms);  // of the context's last batch
void gibbs_batch_drop(int slot);  // a context goes away: frees its staging buffer
// the calling context's pinned staging buffer of the batch calls (gibbs_batch.cu, eval_batch.cu), at least `bytes` long;
// a batch call synchronises its stream before it returns, so the next call may reuse it
int batch_stage(size_t bytes, char **out);

// ---- the schedule cache (gibbs.cu) ------------------------------------------------------------------------------
enum Route : int { ROUTE_K1 = 0, ROUTE_K1F = 1, ROUTE_K1X = 2, NROUTES = 3 };  // K1 also serves K1w

// A cached schedule.  The key fields are what the route's schedule depends on; a route leaves the others zero:
// K1 compares masked and literal, K1f masked and the mask bytes (its affine map depends on them), K1x neither.
struct SchedEntry {
  uint64_t epoch = 0;
  int M = 0, T = 0;
  bool masked = false, literal = false;
  unsigned char mask[KDEB200_MAX_DENS][KDEB200_MAX_DIM] = {};  // K1f only, which serves M <= KDEB200_MAX_DENS
  kdeb200_tree_t trees[KDEB200_MAX_DENS_LARGE] = {nullptr};    // K1 also caches K1m's schedules (gibbs_many.cu)
  char *d_base = nullptr;   // draws | tiles | counters | FP32 records, one allocation on the context's device
  char *d_extra = nullptr;  // K1x: XDraws | tile centres
  Draw *d_draws = nullptr;
  TileDesc *d_tiles = nullptr;
  int *d_counters = nullptr;
  float *d_rec = nullptr;
  XDraw *d_xd = nullptr;
  int ndraws = 0, ntiles = 0;
  int redo_blocks = 0;  // K1x: blocks of its FP64 redo on the largest certified level
  unsigned next_counter = 0;
  double nctr[KDEB200_MAX_DIM] = {0}, nisig[KDEB200_MAX_DIM] = {0};  // K1f: the affine map of its FP32 records
};

// The schedule of `key` for route r on the calling context, built on a miss; *counter (if wanted) is the batch counter
// of one launch.
int sched_get(Route r, const kdeb200_tree_t *trees, int L, const SchedEntry &key, SchedEntry *out, int **counter);

// The route-specific part of a schedule build, run once the plan is made and the entry's memory is allocated: K1f's
// affine map and FP32 records (gibbs_f32.cu), K1x's record statistics, FP32 records and XDraws (gibbs_exact.cu).
// gibbs_exact_plan runs before the allocation: it moves K1x's internal draws onto FP32 records.
int gibbs32_build(const kdeb200_tree_t *trees, Plan &S, SchedEntry &e);
void gibbs_exact_plan(const kdeb200_tree_t *trees, Plan &S);
int gibbs_exact_build(const kdeb200_tree_t *trees, Plan &S, SchedEntry &e);
int gibbs32_launch(GibbsParams &P, const SchedEntry &E, int d, cudaStream_t st);
int gibbs_exact_launch(GibbsParams &P, const SchedEntry &E, int d, cudaStream_t st);

// Counters of the calling context, zeroed at allocation: [0] K1f draws redone in FP64, [1] K1x leaf lane-draws and [2]
// K1x leaf warp-draws redone in FP64, [3] and [4] the same for K1x's internal sampleIndex draws, [5] and [6] for its
// internal sampleIndices! draws (atomics: launches in flight on several streams may share them).
int gibbs_counters(unsigned long long **out);

// f(std::integral_constant<int, d>()) for the instantiated dimensions: 1..8, or 3 alone in the tuning builds
// (GB_ONLY_D3 / GF_ONLY_D3 link one instantiation, tools/sweep_build*.py)
template <class F>
cudaError_t with_d(int d, F &&f) {
  switch (d) {
    case 3: return f(std::integral_constant<int, 3>());
#if !defined(GB_ONLY_D3) && !defined(GF_ONLY_D3)
    case 1: return f(std::integral_constant<int, 1>());
    case 2: return f(std::integral_constant<int, 2>());
    case 4: return f(std::integral_constant<int, 4>());
    case 5: return f(std::integral_constant<int, 5>());
    case 6: return f(std::integral_constant<int, 6>());
    case 7: return f(std::integral_constant<int, 7>());
    case 8: return f(std::integral_constant<int, 8>());
#endif
  }
  return cudaErrorInvalidValue;
}

}  // namespace kdeb200
