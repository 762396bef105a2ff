/*
 * kdeb200.h -- C-ABI of libkdeb200.so: the B200 (sm_100a) implementation of the data-parallel
 * hot path of KernelDensityEstimate.jl (multiscale Gibbs KDE-product sampler, brute-force
 * Gaussian-kernel evaluation, leave-one-out likelihood).
 *
 * This is the drop-in boundary: the reference is pure Julia with no FFI of its own, so each
 * entry point below names the reference function it replaces (paths relative to the reference
 * repo) -- that is the call a maintainer re-points with `ccall` (INTEGRATION.md shows the
 * Julia binding; kerneldensityestimate.jl_b200/_lib.py is the ctypes mirror used by the tests).
 *
 * Conventions
 *   - every function returns 0 on success, nonzero on error; kdeb200_last_error() returns the
 *     message for the calling thread (the reference raises ErrorException via error(...):
 *     src/DualTree01.jl:311,382,414, src/MSGibbs01.jl:721 -- the binding turns nonzero into that).
 *   - matrices are column-major exactly as Julia passes them (d x N => point i at [i*d, i*d+d)).
 *   - indices inside tree arrays are the reference's 1-based node ids (NO_CHILD = -1).
 *   - host buffers are owned by the caller and never retained; `_device` variants take device
 *     pointers plus a cudaStream_t (as void*) and do not synchronise.
 *   - Euclidean (+,-) manifolds only, d <= KDEB200_MAX_DIM, uniform bandwidth (multibandwidth
 *     == 0, the only case the reference's typed constructors produce).  Anything else is an
 *     error: there is no CPU fallback.
 */
#ifndef KDEB200_H
#define KDEB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KDEB200_MAX_DIM 8
#define KDEB200_MAX_DENS 16
#define KDEB200_MAX_GPUS 16

#define KDEB200_F64 0 /* FP64 arithmetic (parity mode: 1e-12 eval, exact labels) */
#define KDEB200_F32 1 /* FP32 arithmetic with MUFU ex2 (evaluation only, 1e-5; far-tail values flush to 0) */
#define KDEB200_F64_BOUNDED 2 /* FP64, tile-pruned with a guaranteed bound: every value within 1e-13 relative of the
                                 brute-force sum (the counterpart of the reference's dual-tree evaluation) */
#define KDEB200_F32_BOUNDED 3 /* FP32 arithmetic through the same pruning (window 8.6 bandwidths, rows below the bound
                                 recomputed in FP64): 1e-5 like KDEB200_F32; leave-one-out calls run unpruned */

typedef struct kdeb200_tree_s *kdeb200_tree_t; /* opaque device-resident BallTreeDensity */

/* ---- library / device ----------------------------------------------------------------- */
const char *kdeb200_last_error(void);
int kdeb200_version(void);
int kdeb200_device_count(int *count);
/* Binds the calling process to CUDA device `device` (one process per GPU). */
int kdeb200_init(int device);
/* In-process multi-GPU (SURVEY.md 8b S0 / 8e): one host process drives `ngpus` devices (<= 0: every visible one;
 * the device bound by kdeb200_init, or device 0, stays the primary).  Afterwards the HOST-BUFFER entry points
 * kdeb200_gibbs, kdeb200_eval, kdeb200_loo_entropy and kdeb200_kde_lcv shard their independent units (samples, query
 * points, leaf rows) over the set: trees are replicated to every device on first use (peer copies over NVLink), each
 * device runs its block on its own stream from its own host thread and copies its shard straight into the caller's
 * host buffer -- no gather and no collective, because the consumer is host memory.  Results do not depend on the
 * number of GPUs (units are addressed by global index; likelihood partials are summed in block order).  The
 * *_device entry points keep running on the device that owns their pointers.  kdeb200_init_multi(1) switches back. */
int kdeb200_init_multi(int ngpus);
/* Explicit device list (devices[0] = primary).  A device may be listed more than once: several contexts then share
 * that GPU (no speed-up; exercises the whole sharding path on a single-GPU box). */
int kdeb200_init_multi_devices(const int *devices, int n);
int kdeb200_multi_count(int *ngpus);
int kdeb200_shutdown(void);
int kdeb200_device_props(int *sm_count, int *cc_major, int *cc_minor, int *clock_khz, size_t *free_bytes);

/* ---- S0: tree handle --------------------------------------------------------------------
 * Replaces nothing in the reference by itself: it is the hand-over of a host-built
 * BallTreeDensity (src/BallTree01.jl:10-28, src/BallTreeDensity01.jl:11-24).  The arrays are the
 * struct fields verbatim: means / bandwidth are 2N*d, weights / left / right / perm are 2N.
 * The library flattens them into level-ordered device records (DESIGN.md "HBM layout"). */
int kdeb200_tree_create(int d, int64_t N, const double *means, const double *bandwidth, const double *weights,
                        const int64_t *left_child, const int64_t *right_child, const int64_t *permutation,
                        kdeb200_tree_t *out);
/* Evaluation-only hand-over: uploads the leaf records alone (8*(d+2)*N bytes instead of the
 * ~5x larger level records), for trees that only meet kdeb200_eval* / kdeb200_loo_* -- e.g. the
 * marginals that nLOO_LL / ksize (src/CrossValidation.jl:15-24, 65-83) build once per dimension.
 * A Gibbs call on such a handle fails with code 7. */
int kdeb200_tree_create_eval(int d, int64_t N, const double *means, const double *bandwidth,
                             const double *weights, const int64_t *permutation, kdeb200_tree_t *out);
int kdeb200_tree_destroy(kdeb200_tree_t t);
int kdeb200_tree_info(kdeb200_tree_t t, int *d, int64_t *N, int *nlevels, int64_t *device_bytes);

/* Host-side construction of the reference's tree arrays (makeBallTreeDensity,
 * src/BallTreeDensity01.jl:192-231 -> buildTree! src/BallTree01.jl:415-434).  For hosts without
 * Julia (the python mirror) and as the fast path for SURVEY.md 8f.1; a Julia caller keeps using
 * its own builder and passes the arrays to kdeb200_tree_create.  All outputs are caller-allocated:
 * centers, ranges, means, bandwidth: 2N*d; weights_out, left, right, lowest, highest, perm: 2N. */
int kdeb200_tree_build_host(int d, int64_t N, const double *points, const double *weights, const double *bw_var,
                            double *centers, double *ranges, double *weights_out, double *means,
                            double *bandwidth, int64_t *left_child, int64_t *right_child,
                            int64_t *lowest_leaf, int64_t *highest_leaf, int64_t *permutation);

/* ---- S1: multiscale Gibbs product sampler -------------------------------------------------
 * Replaces gibbs1(Ndens, trees, Np, Niter, pts, ind, randU, randN; ...) src/MSGibbs01.jl:527-629
 * as called by prodAppxMSGibbsS :697-700 and `*` :724.
 *   dimmask   ndens*d bytes, dimmask[j*d+k] != 0 <=> partialDimMask[j][k]; NULL = all active.
 *   randU/N   injected streams exactly as the reference's keyword arguments (:661-662); when
 *             randU == NULL both streams come from counter-based Philox4x32-10 keyed by `seed`
 *             and addressed by (sample, draw) so results do not depend on sharding.
 *   s0, s1    compute samples s in [s0, s1) of the Np-sample run (0-based); outputs hold only
 *             that range: points_out d x (s1-s0), indices_out ndens x (s1-s0) (= permutation + 1,
 *             the reference's label convention, :612-616).
 *   level_labels_out  optional (NULL = off): glbs.recordChoosen / labelsChoosen[sample][density][level]
 *             (:29-31,109-112) as int64 [(s1-s0)][ndens][Nlevels]: permutation of the node selected by
 *             the last sampleIndex call of each level (0 for internal nodes, -1 if Niter == 0).
 */
int kdeb200_gibbs(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                  const uint8_t *dimmask, const double *randU, int64_t nU, const double *randN, int64_t nN,
                  uint64_t seed, int64_t s0, int64_t s1, double *points_out, int64_t *indices_out,
                  int64_t *level_labels_out);
/* Same, outputs (and the optional injected streams) in device memory, asynchronous on `stream`. */
int kdeb200_gibbs_device(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                         const uint8_t *dimmask, const double *d_randU, int64_t nU, const double *d_randN,
                         int64_t nN, uint64_t seed, int64_t s0, int64_t s1, double *d_points,
                         int64_t *d_indices, int64_t *d_level_labels, void *stream);
/* `*` in one call (src/MSGibbs01.jl:707-726): Np product samples by prodAppxMSGibbsS (Philox(seed)) and, without the
 * samples leaving the device, the LOOCV bandwidths of kde!(pGM) (src/KDE01.jl:13-23): for Np <= 512 the Gibbs kernel is
 * followed by ONE kernel that sorts every coordinate, rebuilds the 1-D ball-tree statistics of ksize / neighborMinMax on
 * chip and runs all golden-section searches (bit-identical to kdeb200_gibbs + kdeb200_kde_lcv); larger Np fall back to that
 * two-step route inside the call.  The caller builds the product density as kde!(points_out, bw_std_out).
 * indices_out (ndens x Np) and nloo_calls_out (d) may be NULL. */
int kdeb200_product_kde(const kdeb200_tree_t *trees, int ndens, int64_t Np, int Niter, int add_entropy,
                        const uint8_t *dimmask, uint64_t seed, double *points_out, int64_t *indices_out,
                        double *bw_std_out, int *nloo_calls_out);
/* Arithmetic of the label probabilities in kdeb200_gibbs / _gibbs_device / _product_kde (process-wide; default KDEB200_F64;
 * the environment variable KDEB200_GIBBS_F32=1/0 overrides):
 *   KDEB200_F64  parity mode (a): labels identical to the reference under injected variates.
 *   KDEB200_F32  statistical mode (b) only: makeFasterSampleIndex! (src/MSGibbs01.jl:250-328) evaluated in packed FP32
 *                with MUFU ex2 / rsqrt (2^-22 relative per term) on calls large enough for the thread-per-chain kernel;
 *                chain state, samplePoint! and the output points stay FP64.  With the same seed a chain follows the FP64
 *                kernel until a uniform lands within ~1e-6 of a CDF edge.  A draw whose FP32 total under/overflows is
 *                redone in FP64 with the reference's literal arithmetic (kdeb200_gibbs_f32_slow_draws counts them since
 *                its last call).  Refused (code 8) when a bandwidth is below 1e-4 of the data spread. */
int kdeb200_set_gibbs_precision(int precision);
int kdeb200_gibbs_f32_slow_draws(unsigned long long *count_out);
/* KDEB200_F64 calls of the thread-per-chain sampler decide the leaf-level labels from FP32 prefix sums with a proven
 * error bound and redo in FP64 only the draws the bound cannot decide; the labels and points are those of the FP64
 * arithmetic bit for bit (KDEB200_GIBBS_EXACT=0 forces the all-FP64 kernel).  Counts the redone lane-draws and the
 * warp-draws that contained one (warps_out may be NULL) on the calling context's device since the last call. */
int kdeb200_gibbs_exact_redone(unsigned long long *lanes_out, unsigned long long *warps_out);
/* Diagnostic for tests of the bound above (d = 3): for nq query conditionals (mu, Calmost: nq x d each, row-major) of the
 * leaf-level draw of density `density` (0-based) on schedule level `level` (1-based), writes per query a header
 * [A, B, aabs, ok, log2 w_max, n, G, 0] and per node [p32, acc32, p64, S64, lo, hi, lo_ck, hi_ck]: the FP32 term and its
 * exponent, the FP64 term and prefix sum, and the intervals claimed for S64 / w_max per node and at checkpoints
 * (NaN between checkpoints).  out_len: capacity of out in doubles. */
int kdeb200_gibbs_exact_bound_probe(const kdeb200_tree_t *trees, int ndens, int Niter, int density, int level,
                                    const double *mu, const double *cadd, int nq, double *out, int64_t out_len);
/* glbs.Nlevels (src/MSGibbs01.jl:555-568) and the per-sample stream consumption. */
int kdeb200_gibbs_sizes(const kdeb200_tree_t *trees, int ndens, int Niter, int *nlevels,
                        int64_t *uniforms_per_sample, int64_t *normals_per_sample,
                        int64_t *kernel_evals_per_sample);
/* The Philox streams as arrays (what the kernel draws when randU == NULL), for parity tests. */
int kdeb200_philox_streams(uint64_t seed, int64_t Np, int64_t uniforms_per_sample, int64_t normals_per_sample,
                           double *randU_out, double *randN_out);

/* ---- S2: brute-force evaluation ------------------------------------------------------------
 * Replaces evaluate(bd, locations, p, maxErr, addop, diffop) src/DualTree01.jl:303-346 with
 * FORCE_EVAL_DIRECT (evalDirect :130-162, distGauss! :14-47), i.e. what evaluateDualTree :370-421
 * and the functor :431-446 compute.  pos is d x M (original order); loo != 0 ignores pos and
 * evaluates bd at its own points leaving each one out (bd === locations), output in original
 * point order. */
int kdeb200_eval(kdeb200_tree_t bd, const double *pos, int64_t M, int loo, int precision, double *p_out);
/* Pruning policy (replaces setForceEvalDirect! / FORCE_EVAL_DIRECT src/DualTree01.jl:3-9, and the dual-tree recursion
 * evaluate :248-299 + recurseMinMax :164-242 it switches on).  The pruned kernel drops (query block, component tile)
 * pairs whose bounding boxes are so far apart that each kernel value is below 1e-26, and recomputes over all
 * components every row whose kept sum is too small for that to mean 1e-13 relative: results are within 1e-13 of the
 * brute-force sum (the reference's dual tree: errTol = 1e-3).
 *   0  brute force everywhere
 *   1  (default) pruned kernel for the leave-one-out likelihood (kdeb200_loo_*, kdeb200_kde_lcv*), brute force for
 *      kdeb200_eval unless precision == KDEB200_F64_BOUNDED
 *   2  pruned kernel also for every FP64 kdeb200_eval (= setForceEvalDirect!(false))
 * kdeb200_pruned_stats: fraction of (block, tile) pairs the last pruned call on this device kept, and how many rows
 * it recomputed exactly. */
int kdeb200_set_pruning(int mode);
int kdeb200_pruned_stats(double *kept_fraction, int64_t *redo_rows);
int kdeb200_eval_device(kdeb200_tree_t bd, const double *d_pos, int64_t M, int loo, int precision, double *d_out,
                        void *stream);

/* Every 1-D marginal of bd evaluated on its own grid in ONE launch, straight from the d-dimensional records: replaces
 * the per-dimension `mm = marginal(p,[i]); mm(X)` of getKDEMax (src/DualTree01.jl:558-569, marginal src/KDE01.jl:143-153),
 * which builds a 1-D tree per dimension to evaluate 200 points.  grids and out are d x G, row k = dimension k. */
int kdeb200_eval_marginals(kdeb200_tree_t bd, const double *grids, int64_t G, double *out);

/* sample(npd, Npts) (src/KDE01.jl:164-183; rand :196-198, resample src/BallTreeDensity01.jl:312-334): component indices
 * by inverse CDF from SORTED uniforms over the cumulative weights in original point order, plus the Gaussian kernel
 * perturbation bw .* randn.  randU (Np uniforms, any order -- they are sorted like the reference's sort(rand(Npts))) and
 * randN (d x Np, column-major) inject the variates; NULL draws them from Philox4x32-10(seed).  ind_out is 1-based. */
int kdeb200_sample(kdeb200_tree_t bd, int64_t Np, uint64_t seed, const double *randU, const double *randN,
                   double *points_out, int64_t *ind_out);

/* ---- S3: leave-one-out likelihood (fused) --------------------------------------------------
 * Replaces entropy(bd) src/DualTree01.jl:505-508 / evalAvgLogL :450-470 as called from
 * nLOO_LL src/CrossValidation.jl:15-24.  bw_var (d variances) overrides the tree's leaf
 * bandwidth for this call (the caller applies alpha^2 like updateBandwidth! :5-12); NULL keeps
 * the tree's.  H_out = -(sum_j W_j log L_j), or +Inf under the reference's zero rule. */
int kdeb200_loo_entropy(kdeb200_tree_t bd, const double *bw_var, double *H_out);
/* Rows [j0, j1) of the leaf-ordered LOO sum only: partial sum_j W_j log L_j and zero flag, for
 * the multi-GPU split (all-reduce the two scalars). */
int kdeb200_loo_partial(kdeb200_tree_t bd, const double *bw_var, int64_t j0, int64_t j1, double *sum_out,
                        int *zero_flag_out);

/* kde!(points) bandwidth selection in one call: the per-dimension loop of src/KDE01.jl:13-23,
 *   bwds[i] = getBW(ksize(marginal(p, [i])))[1]
 * i.e. marginal (src/KDE01.jl:143-153), neighborMinMax, ksize and golden over nLOO_LL
 * (src/CrossValidation.jl:15-24, 44-120).  points is d x N column-major; bw_std_out receives the d
 * standard deviations to hand to kde!(points, bwds); nloo_calls_out (d entries, may be NULL) the
 * number of nLOO_LL evaluations per dimension.  N <= 512 runs every dimension's whole
 * golden-section search in ONE kernel launch; larger N loops on the host over the tiled LOO
 * kernel.  Both give the bits of the call-by-call route through kdeb200_loo_entropy. */
int kdeb200_kde_lcv(int d, int64_t N, const double *points, double *bw_std_out, int *nloo_calls_out);

/* The same with the leaf rows [j0, j1) of every nLOO_LL evaluation owned by this process (one process
 * per GPU): after each partial evaluation the library calls allreduce(&sum, &zero_flag, user), which
 * must replace sum by its total over the processes and zero_flag by its maximum (MPI_Allreduce, an NCCL
 * all-reduce on two scalars, ...) and return 0.  Every process runs the same golden-section loop on the
 * same totals and gets the same bandwidths.  N <= 512 is computed redundantly by every process. */
typedef int (*kdeb200_allreduce_fn)(double *sum, int *zero_flag, void *user);
int kdeb200_kde_lcv_sharded(int d, int64_t N, const double *points, int64_t j0, int64_t j1,
                            kdeb200_allreduce_fn allreduce, void *user, double *bw_std_out,
                            int *nloo_calls_out);
/* Vector form of the exchange: the d golden-section searches advance in lock-step (every step evaluates the current
 * alpha of every unfinished dimension, the launches of all dimensions queued back to back), so ONE call
 * allreduce(sums, zero_flags, count, user) per step carries the `count` (<= d) partial likelihoods and flags of that
 * step -- one small all-reduce instead of d.  Same bandwidths as the scalar form. */
typedef int (*kdeb200_allreduce_v_fn)(double *sums, int *zero_flags, int count, void *user);
int kdeb200_kde_lcv_sharded_v(int d, int64_t N, const double *points, int64_t j0, int64_t j1,
                              kdeb200_allreduce_v_fn allreduce, void *user, double *bw_std_out,
                              int *nloo_calls_out);

/* ---- measurement ----------------------------------------------------------------------------
 * Pipe-rate microbenchmarks for the roofline denominators (SURVEY.md 8d): dependent-free DFMA,
 * FFMA and MUFU.EX2 loops over the whole chip.  which: 0 = DFMA, 1 = FFMA, 2 = MUFU.EX2.
 * Returns achieved instructions/s (per thread-lane) and the elapsed ms. */
int kdeb200_pipe_peak(int which, int iters, double *lane_ops_per_s, double *ms);
/* DFMA latency / throughput probe: `ilp` independent dependent chains per thread (1,2,4,8,16) at
 * a chosen occupancy; used to size the kernels' ILP x warps product (DESIGN.md). */
int kdeb200_dfma_probe(int ilp, int blocks_per_sm, int threads, int iters, double *lane_ops_per_s);
/* Milliseconds spent in the kernels of the last call on this thread (CUDA events). */
int kdeb200_last_kernel_ms(double *ms, int *launches);

#ifdef __cplusplus
}
#endif
#endif
