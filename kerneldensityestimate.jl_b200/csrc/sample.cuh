// sample.cuh -- what the sample kernels of extras.cu (one density per call) and sample_batch.cu (many) share: the
// per-sample body after the sort, and the builder of the cumulative-weight tables.
#pragma once
#include "common.cuh"

namespace kdeb200 {

#ifdef __CUDACC__
// Sample ii of sample(npd, Npts) (src/KDE01.jl:164-183) from its SORTED uniform tv.  cw: cumulative weights in original
// point order, normalised (cw[N-1] == 1); the reference's scan picks the first i with cw[i] > tv (:176-181).  Both
// kernels call this one body, so r[k] + bw_std[k] * g contracts to the same FMA in both.
__device__ __forceinline__ void sample_one(double tv, int64_t ii, const double *__restrict__ cw,
                                           const int64_t *__restrict__ leaf_of, const double *__restrict__ leaf, int SE,
                                           int d, int64_t N, const double *__restrict__ randn_in, uint64_t seed,
                                           const double *__restrict__ bw_std, double *__restrict__ points,
                                           int64_t *__restrict__ idx) {
  int64_t lo = 0, hi = N - 1;  // first i with cw[i] > tv; cw[N-1] = 1 > tv always (tv < 1)
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (cw[mid] > tv) hi = mid; else lo = mid + 1;
  }
  const double *r = leaf + leaf_of[lo] * SE;
  for (int k = 0; k < d; ++k) {
    const double g = randn_in ? randn_in[ii * d + k] : philox_normal(seed, (uint64_t)ii, (uint32_t)k);
    points[ii * d + k] = r[k] + bw_std[k] * g;
  }
  idx[ii] = lo + 1;  // 1-based like the reference
}
#endif

// Builds the d_cw / d_leaf_of tables of every handle in trees[0..n) that has none yet (NULL entries and repeats are
// skipped), on the calling context's stream: every leaf-weight copy is queued before ONE synchronise, the host
// sequential cumsum runs per handle (the reference's cumsum(w) ./ w[end]), every table copy is queued before one more.
int sample_tables(const kdeb200_tree_t *trees, int n);

}  // namespace kdeb200
