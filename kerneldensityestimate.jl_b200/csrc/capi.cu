// capi.cu -- the extern "C" entry points declared in include/kdeb200.h.
// Host-buffer variants stage through device memory inside the call (H2D / D2H included), the
// *_device variants are asynchronous on the caller's stream.
#include <cmath>
#include <limits>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "tree.cuh"

namespace kdeb200 {
int tree_build_host(int d, int64_t N, const double *points, const double *weights, const double *bw_var,
                    double *centers, double *ranges, double *wout, double *means, double *bandwidth,
                    int64_t *left, int64_t *right, int64_t *lowest, int64_t *highest, int64_t *perm);
int tree_create(int d, int64_t N, const double *means, const double *bandwidth, const double *weights,
                const int64_t *left, const int64_t *right, const int64_t *perm, bool gibbs_records,
                kdeb200_tree_t *out);
int tree_destroy(kdeb200_tree_t t);
int kde_lcv(int d, int64_t N, const double *points, int64_t j0, int64_t j1, kdeb200_allreduce_v_fn allreduce, void *user,
            double *bw_std_out, int *ncalls_out);
int eval_device(kdeb200_tree_t bd, const double *d_pos, int64_t M, int loo, int64_t q0, bool scatter,
                const double *bw_var, double *d_out, cudaStream_t st, int *launches, int prune);
int kde_lcv_points_device(int d, int64_t N, const double *d_points, double *d_out5, cudaStream_t st);
void lcv_points_finish(int d, const double *out5, double *bw_std_out, int *ncalls_out);
int eval_marginals_device(kdeb200_tree_t bd, const double *d_grid, int64_t G, double *d_out, cudaStream_t st, int *launches);
int sample_device(kdeb200_tree_t bd, int64_t Np, uint64_t seed, const double *d_randU, const double *d_randN,
                  double *d_points, int64_t *d_idx, cudaStream_t st, int *launches);
bool loo_sym_shardable(const kdeb200_tree_s *bd);
int eval_pruned_f32_device(kdeb200_tree_t bd, const double *d_pos, int64_t M, double *d_out, cudaStream_t st, int *launches);
void set_prune_mode(int m);
int get_prune_mode();
int pruned_last_stats(double *kept_fraction, int64_t *redo_rows);
// precision argument of the evaluation entry points -> (is FP32, prune argument of eval_device)
static inline int prune_for(int precision) {
  if (precision == KDEB200_F64_BOUNDED) return 2;
  return get_prune_mode() >= 2 ? 1 : 0;
}
int eval_device_f32(kdeb200_tree_t bd, const double *d_pos, int64_t M, int loo, double *d_out, cudaStream_t st,
                    int *launches);
int loo_partial_device(kdeb200_tree_t bd, const double *bw_var, int64_t j0, int64_t j1, double *d_sum, int *d_flag,
                       cudaStream_t st, int *launches);
int gibbs_sizes(const kdeb200_tree_t *trees, int ndens, int Niter, int *nlevels, int64_t *perU, int64_t *perN,
                int64_t *evals);
int gibbs_device(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                 const uint8_t *dimmask, const double *d_randU, int64_t nU, const double *d_randN, int64_t nN,
                 uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                 int64_t *d_level_labels, cudaStream_t st, int *launches);
int gibbs_exact_device(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                       const uint8_t *dimmask, const double *d_randU, int64_t nU, const double *d_randN, int64_t nN,
                       uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                       int64_t *d_level_labels, cudaStream_t st, int *launches);
int gibbs_exact_redone(unsigned long long *lanes, unsigned long long *warps);
int gibbs_exact_probe(const kdeb200_tree_t *trees, int ndens, int Niter, int j, int level, const double *mu,
                      const double *cadd, int nq, double *out, int64_t out_len);
int philox_streams_device(uint64_t seed, int64_t Np, int64_t perU, int64_t perN, double *d_U, double *d_G,
                          cudaStream_t st);
int gibbs_set_precision(int p);
int gibbs32_slow_draws(unsigned long long *out);
int pipe_peak(int which, int iters, double *lane_ops_per_s, double *ms_out);
int dfma_probe(int ilp, int blocks_per_sm, int threads, int iters, double *lane_ops_per_s);

// The reference is single-threaded with module-level state; the library keeps one stream and one
// event pair per process, so compute entry points are serialised (recursive: loo_entropy -> loo_partial).
static std::recursive_mutex g_call_mu;
#define KDE_SERIALISE() std::lock_guard<std::recursive_mutex> kde_lock__(::kdeb200::g_call_mu)

// RAII device buffer on a stream
struct DevBuf {
  void *p = nullptr;
  cudaStream_t st;
  explicit DevBuf(cudaStream_t s) : st(s) {}
  cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes ? bytes : 16, st); }
  ~DevBuf() {
    if (p) cudaFreeAsync(p, st);
  }
  template <class T>
  T *as() { return static_cast<T *>(p); }
};

struct Timer {  // CUDA-event bracket on the library stream, result readable via kdeb200_last_kernel_ms
  Context &c;
  explicit Timer(Context &cc) : c(cc) {
    c.last_launches = 0;
    cudaEventRecord(c.ev0, c.stream);
  }
  void stop() {
    cudaEventRecord(c.ev1, c.stream);
    cudaEventSynchronize(c.ev1);
    float ms = 0;
    cudaEventElapsedTime(&ms, c.ev0, c.ev1);
    c.last_ms = ms;
  }
};

// ---- in-process multi-GPU: block partition + one host thread per device --------------------------------------------
static inline void shard_range(int64_t n, int g, int G, int64_t &a, int64_t &b) {  // first n % G blocks get one extra unit
  const int64_t base = n / G, rem = n % G;
  a = g * base + (g < rem ? g : rem);
  b = a + base + (g < rem ? 1 : 0);
}

// GPUs to use for `units` independent units when each GPU should get at least `min_per_gpu`
static inline int gpus_for(int64_t units, int64_t min_per_gpu) {
  int G = multi_count();
  if (G > 1 && units < (int64_t)G * min_per_gpu) G = (int)(units / min_per_gpu);
  return G < 1 ? 1 : G;
}

// fn(slot) on slots 0..G-1: slot 0 on the calling thread, the others on their own host threads bound to their device.
// Error strings are thread-local, so the first failing worker's message is copied to the caller.
template <class F>
static int for_each_gpu(int G, F fn) {
  if (G <= 1) return fn(0);
  std::vector<int> rc(G, 0);
  std::vector<std::string> err(G);
  std::vector<std::thread> th;
  for (int g = 1; g < G; ++g)
    th.emplace_back([&, g] {
      ScopedDevice sd(g);
      rc[g] = fn(g);
      if (rc[g]) err[g] = get_error();
    });
  {
    ScopedDevice sd(0);
    rc[0] = fn(0);
    if (rc[0]) err[0] = get_error();
  }
  for (auto &t : th) t.join();
  for (int g = 0; g < G; ++g)
    if (rc[g]) {
      set_error("GPU slot %d: %s", g, err[g].c_str());
      return rc[g];
    }
  return 0;
}

// samples [a, b) of the run on the GPU of the calling thread's context: staging, launch, D2H into the caller's buffers
// (points_out / indices_out / level_labels_out point at sample a's slot)
static int gibbs_host_block(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                            const uint8_t *dimmask, const double *randU, const double *randN, uint64_t seed, int64_t a,
                            int64_t b, int L, int64_t perU, int64_t perN, double *points_out, int64_t *indices_out,
                            int64_t *level_labels_out, double *ms_out, int *launches_out) {
  Context &c = ctx();
  const int d = trees[0]->d;
  const int64_t n = b - a;
  if (n <= 0) return 0;
  kdeb200_tree_t loc[KDEB200_MAX_DENS];
  for (int j = 0; j < ndens; ++j)
    if (int rc = tree_on(trees[j], c.slot, &loc[j])) return rc;
  DevBuf dU(c.stream), dN(c.stream), dP(c.stream), dI(c.stream), dR(c.stream);
  if (randU) {
    // only the slices this range touches travel: [a*perU - 1, b*perU - 1) and [a*perN, b*perN)
    KDE_CUDA(dU.alloc(sizeof(double) * n * perU));
    KDE_CUDA(dN.alloc(sizeof(double) * n * perN));
    const int64_t ulo = a * perU > 0 ? a * perU - 1 : 0;  // slot -1 of sample 0 is never read
    const int64_t skip = a * perU > 0 ? 0 : 1;
    KDE_CUDA(cudaMemcpyAsync(dU.as<double>() + skip, randU + ulo, sizeof(double) * (n * perU - skip),
                             cudaMemcpyHostToDevice, c.stream));
    KDE_CUDA(cudaMemcpyAsync(dN.p, randN + a * perN, sizeof(double) * n * perN, cudaMemcpyHostToDevice, c.stream));
  }
  KDE_CUDA(dP.alloc(sizeof(double) * d * n));
  KDE_CUDA(dI.alloc(sizeof(int64_t) * ndens * n));
  int64_t *d_rec = nullptr;
  if (level_labels_out) {  // never-written entries (Niter == 0) stay -1
    KDE_CUDA(dR.alloc(sizeof(int64_t) * ndens * n * L));
    KDE_CUDA(cudaMemsetAsync(dR.p, 0xFF, sizeof(int64_t) * ndens * n * L, c.stream));
    d_rec = dR.as<int64_t>();
  }
  Timer tm(c);
  int launches = 0;
  int rc;
  if (randU) {
    // device slices are re-based: sample s reads U[(s-a)*perU + c - 1 + 1] => pass pointer + 1
    rc = gibbs_exact_device(loc, ndens, n, Niter, add_entropy, dimmask, dU.as<double>() + 1, n * perU - 1, dN.as<double>(),
                      n * perN, seed, 0, n, dP.as<double>(), dI.as<int64_t>(), d_rec, c.stream, &launches);
  } else {
    rc = gibbs_exact_device(loc, ndens, Np, Niter, add_entropy, dimmask, nullptr, 0, nullptr, 0, seed, a, b, dP.as<double>(),
                      dI.as<int64_t>(), d_rec, c.stream, &launches);
  }
  if (rc) return rc;
  tm.stop();
  c.last_launches = launches;
  if (ms_out) *ms_out = c.last_ms;
  if (launches_out) *launches_out = launches;
  KDE_CUDA(cudaMemcpyAsync(points_out, dP.p, sizeof(double) * d * n, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaMemcpyAsync(indices_out, dI.p, sizeof(int64_t) * ndens * n, cudaMemcpyDeviceToHost, c.stream));
  if (level_labels_out)
    KDE_CUDA(cudaMemcpyAsync(level_labels_out, dR.p, sizeof(int64_t) * ndens * n * L, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}

// query rows [a, b) on the calling thread's GPU; LOO rows come back in LEAF order (the caller scatters through h_perm)
static int eval_host_block(kdeb200_tree_t bd, const double *pos, int64_t a, int64_t b, int loo, int precision,
                           bool scatter, double *out_block, double *ms_out, int *launches_out) {
  Context &c = ctx();
  const int64_t n = b - a;
  if (n <= 0) return 0;
  kdeb200_tree_t loc;
  if (int rc = tree_on(bd, c.slot, &loc)) return rc;
  DevBuf dQ(c.stream), dO(c.stream);
  if (!loo) {
    KDE_CUDA(dQ.alloc(sizeof(double) * bd->d * n));
    KDE_CUDA(cudaMemcpyAsync(dQ.p, pos + a * bd->d, sizeof(double) * bd->d * n, cudaMemcpyHostToDevice, c.stream));
  }
  KDE_CUDA(dO.alloc(sizeof(double) * n));
  Timer tm(c);
  int launches = 0;
  int rc;
  if (precision == KDEB200_F32_BOUNDED && !loo)
    rc = eval_pruned_f32_device(loc, dQ.as<double>(), n, dO.as<double>(), c.stream, &launches);
  else if (precision == KDEB200_F32 || precision == KDEB200_F32_BOUNDED)
    rc = eval_device_f32(loc, dQ.as<double>(), n, loo, dO.as<double>(), c.stream, &launches);
  else
    rc = eval_device(loc, dQ.as<double>(), n, loo, a, scatter, nullptr, dO.as<double>(), c.stream, &launches,
                     prune_for(precision));
  if (rc) return rc;
  tm.stop();
  c.last_launches = launches;
  if (ms_out) *ms_out = c.last_ms;
  if (launches_out) *launches_out = launches;
  KDE_CUDA(cudaMemcpyAsync(out_block, dO.p, sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}

static int loo_partial_block(kdeb200_tree_t bd, const double *bw_var, int64_t j0, int64_t j1, double *sum_out,
                             int *zero_flag_out, double *ms_out, int *launches_out) {
  Context &c = ctx();
  *sum_out = 0.0;
  *zero_flag_out = 0;
  if (j0 >= j1) return 0;
  kdeb200_tree_t loc;
  if (int rc = tree_on(bd, c.slot, &loc)) return rc;
  DevBuf dS(c.stream), dF(c.stream);
  KDE_CUDA(dS.alloc(sizeof(double)));
  KDE_CUDA(dF.alloc(sizeof(int)));
  Timer tm(c);
  int launches = 0;
  if (int rc = loo_partial_device(loc, bw_var, j0, j1, dS.as<double>(), dF.as<int>(), c.stream, &launches)) return rc;
  tm.stop();
  c.last_launches = launches;
  if (ms_out) *ms_out = c.last_ms;
  if (launches_out) *launches_out = launches;
  KDE_CUDA(cudaMemcpyAsync(sum_out, dS.p, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaMemcpyAsync(zero_flag_out, dF.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}

// kernel time of a sharded call = the slowest device; launches = the sum
static void publish_timing(const std::vector<double> &ms, const std::vector<int> &launches) {
  double m = 0.0;
  int l = 0;
  for (double v : ms) m = v > m ? v : m;
  for (int v : launches) l += v;
  ctx_at(0).last_ms = m;
  ctx_at(0).last_launches = l;
}
}  // namespace kdeb200

using namespace kdeb200;

extern "C" {

int kdeb200_tree_build_host(int d, int64_t N, const double *points, const double *weights, const double *bw_var,
                            double *centers, double *ranges, double *weights_out, double *means, double *bandwidth,
                            int64_t *left_child, int64_t *right_child, int64_t *lowest_leaf, int64_t *highest_leaf,
                            int64_t *permutation) {
  if (!points || !weights || !bw_var || !centers || !ranges || !weights_out || !means || !bandwidth || !left_child ||
      !right_child || !lowest_leaf || !highest_leaf || !permutation)
    KDE_FAIL(2, "tree_build_host: NULL argument");
  return tree_build_host(d, N, points, weights, bw_var, centers, ranges, weights_out, means, bandwidth, left_child,
                         right_child, lowest_leaf, highest_leaf, permutation);
}

int kdeb200_tree_create(int d, int64_t N, const double *means, const double *bandwidth, const double *weights,
                        const int64_t *left_child, const int64_t *right_child, const int64_t *permutation,
                        kdeb200_tree_t *out) {
  KDE_SERIALISE();
  if (!means || !bandwidth || !weights || !left_child || !right_child || !permutation)
    KDE_FAIL(2, "tree_create: NULL argument");
  return tree_create(d, N, means, bandwidth, weights, left_child, right_child, permutation, true, out);
}

int kdeb200_tree_create_eval(int d, int64_t N, const double *means, const double *bandwidth, const double *weights,
                             const int64_t *permutation, kdeb200_tree_t *out) {
  KDE_SERIALISE();
  if (!means || !bandwidth || !weights || !permutation) KDE_FAIL(2, "tree_create_eval: NULL argument");
  return tree_create(d, N, means, bandwidth, weights, nullptr, nullptr, permutation, false, out);
}

int kdeb200_tree_destroy(kdeb200_tree_t t) {
  KDE_SERIALISE();
  return tree_destroy(t);
}

int kdeb200_tree_info(kdeb200_tree_t t, int *d, int64_t *N, int *nlevels, int64_t *device_bytes) {
  KDE_SERIALISE();
  if (!t) KDE_FAIL(2, "tree_info: NULL tree");
  if (d) *d = t->d;
  if (N) *N = t->N;
  if (nlevels) *nlevels = t->depth;
  if (device_bytes) *device_bytes = (int64_t)t->device_bytes;
  return 0;
}

int kdeb200_gibbs_sizes(const kdeb200_tree_t *trees, int ndens, int Niter, int *nlevels, int64_t *uniforms_per_sample,
                        int64_t *normals_per_sample, int64_t *kernel_evals_per_sample) {
  if (!trees) KDE_FAIL(2, "gibbs_sizes: NULL trees");
  return gibbs_sizes(trees, ndens, Niter, nlevels, uniforms_per_sample, normals_per_sample, kernel_evals_per_sample);
}

int kdeb200_gibbs_device(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                         const uint8_t *dimmask, const double *d_randU, int64_t nU, const double *d_randN, int64_t nN,
                         uint64_t seed, int64_t s0, int64_t s1, double *d_points, int64_t *d_indices,
                         int64_t *d_level_labels, void *stream) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!trees || !d_points || !d_indices) KDE_FAIL(2, "gibbs_device: NULL argument");
  int launches = 0;
  int rc = gibbs_exact_device(trees, ndens, Np, Niter, add_entropy, dimmask, d_randU, nU, d_randN, nN, seed, s0, s1,
                        d_points, d_indices, d_level_labels, (cudaStream_t)stream, &launches);
  ctx().last_launches = launches;
  return rc;
}

int kdeb200_gibbs(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                  const uint8_t *dimmask, const double *randU, int64_t nU, const double *randN, int64_t nN,
                  uint64_t seed, int64_t s0, int64_t s1, double *points_out, int64_t *indices_out,
                  int64_t *level_labels_out) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!trees || !points_out || !indices_out) KDE_FAIL(2, "gibbs: NULL argument");
  int L;
  int64_t perU, perN;
  if (int rc = gibbs_sizes(trees, ndens, Niter, &L, &perU, &perN, nullptr)) return rc;
  if (Np < 0 || s0 < 0 || s1 > Np || s0 > s1) KDE_FAIL(3, "gibbs: bad sample range");
  const int d = trees[0]->d;
  const int64_t n = s1 - s0;
  if (n == 0) return 0;
  if ((randU == nullptr) != (randN == nullptr)) KDE_FAIL(3, "gibbs: randU and randN must be given together");
  if (randU) {
    if (s1 * perU > nU + 1) KDE_FAIL(7, "gibbs: randU too short (%lld < %lld)", (long long)nU, (long long)(s1 * perU - 1));
    if (s1 * perN > nN) KDE_FAIL(7, "gibbs: randN too short (%lld < %lld)", (long long)nN, (long long)(s1 * perN));
  }
  // in-process multi-GPU: contiguous sample blocks, one per device; every device copies its shard straight into the
  // caller's buffers (chains are addressed by global sample index => the result does not depend on the split)
  const int G = gpus_for(n, 2048);
  std::vector<double> ms(G, 0.0);
  std::vector<int> nl(G, 0);
  int rc = for_each_gpu(G, [&](int g) {
    int64_t a, b;
    shard_range(n, g, G, a, b);
    a += s0;
    b += s0;
    return gibbs_host_block(trees, ndens, Np, Niter, add_entropy, dimmask, randU, randN, seed, a, b, L, perU, perN,
                            points_out + (a - s0) * d, indices_out + (a - s0) * ndens,
                            level_labels_out ? level_labels_out + (a - s0) * ndens * L : nullptr, &ms[g], &nl[g]);
  });
  if (rc) return rc;
  publish_timing(ms, nl);
  return 0;
}

int kdeb200_philox_streams(uint64_t seed, int64_t Np, int64_t perU, int64_t perN, double *randU_out,
                           double *randN_out) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!randU_out || !randN_out || Np < 0 || perU < 1 || perN < 1) KDE_FAIL(2, "philox_streams: bad argument");
  Context &c = ctx();
  DevBuf dU(c.stream), dN(c.stream);
  KDE_CUDA(dU.alloc(sizeof(double) * Np * perU));
  KDE_CUDA(dN.alloc(sizeof(double) * Np * perN));
  if (int rc = philox_streams_device(seed, Np, perU, perN, dU.as<double>(), dN.as<double>(), c.stream)) return rc;
  KDE_CUDA(cudaMemcpyAsync(randU_out, dU.p, sizeof(double) * Np * perU, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaMemcpyAsync(randN_out, dN.p, sizeof(double) * Np * perN, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}

int kdeb200_eval_device(kdeb200_tree_t bd, const double *d_pos, int64_t M, int loo, int precision, double *d_out,
                        void *stream) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!bd || !d_out) KDE_FAIL(2, "eval_device: NULL argument");
  if (!loo && !d_pos) KDE_FAIL(2, "eval_device: pos is NULL");
  if (loo) M = bd->N;
  int launches = 0;
  int rc;
  if (precision == KDEB200_F64 || precision == KDEB200_F64_BOUNDED)
    rc = eval_device(bd, d_pos, M, loo, 0, true, nullptr, d_out, (cudaStream_t)stream, &launches, prune_for(precision));
  else if (precision == KDEB200_F32_BOUNDED && !loo)
    rc = eval_pruned_f32_device(bd, d_pos, M, d_out, (cudaStream_t)stream, &launches);
  else if (precision == KDEB200_F32 || precision == KDEB200_F32_BOUNDED)
    rc = eval_device_f32(bd, d_pos, M, loo, d_out, (cudaStream_t)stream, &launches);
  else
    KDE_FAIL(3, "eval: unknown precision %d", precision);
  ctx().last_launches = launches;
  return rc;
}

int kdeb200_eval(kdeb200_tree_t bd, const double *pos, int64_t M, int loo, int precision, double *p_out) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!bd || !p_out) KDE_FAIL(2, "eval: NULL argument");
  if (!loo && !pos && M > 0) KDE_FAIL(2, "eval: pos is NULL");
  if (precision < KDEB200_F64 || precision > KDEB200_F32_BOUNDED) KDE_FAIL(3, "eval: unknown precision %d", precision);
  if (loo) M = bd->N;
  if (M <= 0) return 0;
  // in-process multi-GPU: query rows block-partitioned.  LOO rows are leaf rows: each device returns its block in leaf
  // order and the host scatters through the permutation.  (FP32 LOO has no row-range form: one device.)
  const bool f32_loo = loo && (precision == KDEB200_F32 || precision == KDEB200_F32_BOUNDED);
  const int G = f32_loo ? 1 : gpus_for(M, 4096);
  std::vector<double> ms(G, 0.0);
  std::vector<int> nl(G, 0);
  std::vector<double> rows;
  const bool scatter_on_host = loo && G > 1;
  if (scatter_on_host) rows.resize(M);
  int rc = for_each_gpu(G, [&](int g) {
    int64_t a, b;
    shard_range(M, g, G, a, b);
    return eval_host_block(bd, pos, a, b, loo, precision, /*scatter=*/!scatter_on_host,
                           scatter_on_host ? rows.data() + a : (loo ? p_out : p_out + a), &ms[g], &nl[g]);
  });
  if (rc) return rc;
  if (scatter_on_host)
    for (int64_t j = 0; j < M; ++j) p_out[bd->h_perm[j]] = rows[j];
  publish_timing(ms, nl);
  return 0;
}

int kdeb200_loo_partial(kdeb200_tree_t bd, const double *bw_var, int64_t j0, int64_t j1, double *sum_out,
                        int *zero_flag_out) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!bd || !sum_out || !zero_flag_out) KDE_FAIL(2, "loo_partial: NULL argument");
  if (j0 < 0 || j1 > bd->N || j0 > j1) KDE_FAIL(3, "loo_partial: bad row range");
  double ms = 0.0;
  int nl = 0;
  ScopedDevice sd(0);
  if (int rc = loo_partial_block(bd, bw_var, j0, j1, sum_out, zero_flag_out, &ms, &nl)) return rc;
  return 0;
}

int kdeb200_loo_entropy(kdeb200_tree_t bd, const double *bw_var, double *H_out) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!bd || !H_out) KDE_FAIL(2, "loo_entropy: NULL argument");
  // in-process multi-GPU: leaf rows block-partitioned, partial sums added in block order -- unless the density is in
  // the range of the symmetric each-pair-once kernel, which on one device beats row shards on a few (the bandwidth loop
  // kdeb200_kde_lcv shares the triangle of pairs over the devices instead)
  const int G = loo_sym_shardable(bd) ? 1 : gpus_for(bd->N, 8192);
  std::vector<double> sums(G, 0.0), ms(G, 0.0);
  std::vector<int> flags(G, 0), nl(G, 0);
  int rc = for_each_gpu(G, [&](int g) {
    int64_t a, b;
    shard_range(bd->N, g, G, a, b);
    return loo_partial_block(bd, bw_var, a, b, &sums[g], &flags[g], &ms[g], &nl[g]);
  });
  if (rc) return rc;
  double s = 0.0;
  int flag = 0;
  for (int g = 0; g < G; ++g) {
    s += sums[g];
    flag |= flags[g];
  }
  publish_timing(ms, nl);
  // evalAvgLogL returns -Inf under the zero rule; entropy = -evalAvgLogL
  *H_out = flag ? std::numeric_limits<double>::infinity() : -s;
  return 0;
}

int kdeb200_kde_lcv(int d, int64_t N, const double *points, double *bw_std_out, int *nloo_calls_out) {
  KDE_SERIALISE();
  if (!points || !bw_std_out) KDE_FAIL(2, "kde_lcv: NULL argument");
  return kde_lcv(d, N, points, 0, N, nullptr, nullptr, bw_std_out, nloo_calls_out);
}

int kdeb200_kde_lcv_sharded_v(int d, int64_t N, const double *points, int64_t j0, int64_t j1,
                              kdeb200_allreduce_v_fn allreduce, void *user, double *bw_std_out, int *nloo_calls_out) {
  KDE_SERIALISE();
  if (!points || !bw_std_out || !allreduce) KDE_FAIL(2, "kde_lcv_sharded: NULL argument");
  return kde_lcv(d, N, points, j0, j1, allreduce, user, bw_std_out, nloo_calls_out);
}

namespace {
struct ScalarExchange {  // the scalar callback form on top of the vector exchange: one call per entry
  kdeb200_allreduce_fn fn;
  void *user;
};
int scalar_exchange_adapter(double *sums, int *flags, int count, void *user) {
  ScalarExchange *x = static_cast<ScalarExchange *>(user);
  for (int i = 0; i < count; ++i)
    if (int r = x->fn(&sums[i], &flags[i], x->user)) return r;
  return 0;
}
}  // namespace

int kdeb200_kde_lcv_sharded(int d, int64_t N, const double *points, int64_t j0, int64_t j1,
                            kdeb200_allreduce_fn allreduce, void *user, double *bw_std_out, int *nloo_calls_out) {
  KDE_SERIALISE();
  if (!points || !bw_std_out || !allreduce) KDE_FAIL(2, "kde_lcv_sharded: NULL argument");
  ScalarExchange x{allreduce, user};
  return kde_lcv(d, N, points, j0, j1, scalar_exchange_adapter, &x, bw_std_out, nloo_calls_out);
}

int kdeb200_product_kde(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                        const uint8_t *dimmask, uint64_t seed, double *points_out, int64_t *indices_out,
                        double *bw_std_out, int *nloo_calls_out) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!trees || !points_out || !bw_std_out) KDE_FAIL(2, "product_kde: NULL argument");
  if (Np < 2) KDE_FAIL(3, "product_kde: at least two product samples are needed for cross validation");
  int L;
  int64_t perU, perN;
  if (int rc = gibbs_sizes(trees, ndens, Niter, &L, &perU, &perN, nullptr)) return rc;
  ScopedDevice sd(0);
  Context &c = ctx();
  const int d = trees[0]->d;
  DevBuf dP(c.stream), dI(c.stream), dO(c.stream);
  KDE_CUDA(dP.alloc(sizeof(double) * d * Np));
  KDE_CUDA(dI.alloc(sizeof(int64_t) * ndens * Np));
  KDE_CUDA(dO.alloc(sizeof(double) * 5 * d));
  Timer tm(c);
  int launches = 0;
  if (int rc = gibbs_exact_device(trees, ndens, Np, Niter, add_entropy, dimmask, nullptr, 0, nullptr, 0, seed, 0, Np,
                            dP.as<double>(), dI.as<int64_t>(), nullptr, c.stream, &launches))
    return rc;
  const bool fused = Np <= 512;  // the samples never leave the device between the two kernels
  if (fused) {
    if (int rc = kde_lcv_points_device(d, Np, dP.as<double>(), dO.as<double>(), c.stream)) return rc;
    ++launches;
  }
  tm.stop();
  c.last_launches = launches;
  double out5[5 * KDEB200_MAX_DIM];
  KDE_CUDA(cudaMemcpyAsync(points_out, dP.p, sizeof(double) * d * Np, cudaMemcpyDeviceToHost, c.stream));
  if (indices_out)
    KDE_CUDA(cudaMemcpyAsync(indices_out, dI.p, sizeof(int64_t) * ndens * Np, cudaMemcpyDeviceToHost, c.stream));
  if (fused) KDE_CUDA(cudaMemcpyAsync(out5, dO.p, sizeof(double) * 5 * d, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  if (fused) {
    lcv_points_finish(d, out5, bw_std_out, nloo_calls_out);
    return 0;
  }
  // larger products: the bandwidth loop over the tiled LOO kernels (marginal trees on the host)
  const double ms_gibbs = c.last_ms;
  int rc = kde_lcv(d, Np, points_out, 0, Np, nullptr, nullptr, bw_std_out, nloo_calls_out);
  c.last_ms += ms_gibbs;
  return rc;
}

int kdeb200_eval_marginals(kdeb200_tree_t bd, const double *grids, int64_t G, double *out) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!bd || !grids || !out) KDE_FAIL(2, "eval_marginals: NULL argument");
  if (G <= 0) return 0;
  Context &c = ctx();
  DevBuf dG(c.stream), dO(c.stream);
  const size_t bytes = sizeof(double) * (size_t)bd->d * G;
  KDE_CUDA(dG.alloc(bytes));
  KDE_CUDA(dO.alloc(bytes));
  KDE_CUDA(cudaMemcpyAsync(dG.p, grids, bytes, cudaMemcpyHostToDevice, c.stream));
  Timer tm(c);
  int launches = 0;
  if (int rc = eval_marginals_device(bd, dG.as<double>(), G, dO.as<double>(), c.stream, &launches)) return rc;
  tm.stop();
  c.last_launches = launches;
  KDE_CUDA(cudaMemcpyAsync(out, dO.p, bytes, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}

int kdeb200_sample(kdeb200_tree_t bd, int64_t Np, uint64_t seed, const double *randU, const double *randN,
                   double *points_out, int64_t *ind_out) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  if (!bd || !points_out || !ind_out) KDE_FAIL(2, "sample: NULL argument");
  if (Np < 0 || Np >= ((int64_t)1 << 31)) KDE_FAIL(3, "sample: Np out of range");
  if (Np == 0) return 0;
  for (int k = 0; k < bd->d; ++k)
    if (!(bd->hvar[k] >= 0.0)) KDE_FAIL(5, "sample: negative bandwidth variance");
  Context &c = ctx();
  const int d = bd->d;
  DevBuf dU(c.stream), dN(c.stream), dP(c.stream), dI(c.stream);
  if (randU) {
    KDE_CUDA(dU.alloc(sizeof(double) * Np));
    KDE_CUDA(cudaMemcpyAsync(dU.p, randU, sizeof(double) * Np, cudaMemcpyHostToDevice, c.stream));
  }
  if (randN) {
    KDE_CUDA(dN.alloc(sizeof(double) * d * Np));
    KDE_CUDA(cudaMemcpyAsync(dN.p, randN, sizeof(double) * d * Np, cudaMemcpyHostToDevice, c.stream));
  }
  KDE_CUDA(dP.alloc(sizeof(double) * d * Np));
  KDE_CUDA(dI.alloc(sizeof(int64_t) * Np));
  Timer tm(c);
  int launches = 0;
  if (int rc = sample_device(bd, Np, seed, randU ? dU.as<double>() : nullptr, randN ? dN.as<double>() : nullptr,
                             dP.as<double>(), dI.as<int64_t>(), c.stream, &launches))
    return rc;
  tm.stop();
  c.last_launches = launches;
  KDE_CUDA(cudaMemcpyAsync(points_out, dP.p, sizeof(double) * d * Np, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaMemcpyAsync(ind_out, dI.p, sizeof(int64_t) * Np, cudaMemcpyDeviceToHost, c.stream));
  KDE_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}

int kdeb200_set_pruning(int mode) {
  KDE_SERIALISE();
  if (mode < 0 || mode > 2) KDE_FAIL(3, "set_pruning: mode must be 0, 1 or 2");
  set_prune_mode(mode);
  return 0;
}

int kdeb200_set_gibbs_precision(int precision) {
  KDE_SERIALISE();
  return gibbs_set_precision(precision);
}

int kdeb200_gibbs_f32_slow_draws(unsigned long long *count_out) {
  KDE_SERIALISE();
  if (!count_out) KDE_FAIL(2, "gibbs_f32_slow_draws: NULL argument");
  if (int rc = ensure_init()) return rc;
  return gibbs32_slow_draws(count_out);
}

int kdeb200_gibbs_exact_redone(unsigned long long *lanes_out, unsigned long long *warps_out) {
  KDE_SERIALISE();
  if (!lanes_out) KDE_FAIL(2, "gibbs_exact_redone: NULL argument");
  if (int rc = ensure_init()) return rc;
  return gibbs_exact_redone(lanes_out, warps_out);
}

int kdeb200_gibbs_exact_bound_probe(const kdeb200_tree_t *trees, int ndens, int Niter, int density, int level,
                                    const double *mu, const double *cadd, int nq, double *out, int64_t out_len) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  return gibbs_exact_probe(trees, ndens, Niter, density, level, mu, cadd, nq, out, out_len);
}

int kdeb200_pruned_stats(double *kept_fraction, int64_t *redo_rows) {
  KDE_SERIALISE();
  if (int rc = ensure_init()) return rc;
  return pruned_last_stats(kept_fraction, redo_rows);
}

int kdeb200_pipe_peak(int which, int iters, double *lane_ops_per_s, double *ms) {
  KDE_SERIALISE();
  return pipe_peak(which, iters, lane_ops_per_s, ms);
}

int kdeb200_dfma_probe(int ilp, int blocks_per_sm, int threads, int iters, double *lane_ops_per_s) {
  KDE_SERIALISE();
  return dfma_probe(ilp, blocks_per_sm, threads, iters, lane_ops_per_s);
}

}  // extern "C"
