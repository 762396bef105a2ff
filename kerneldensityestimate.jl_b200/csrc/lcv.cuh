// lcv.cuh -- what lcv.cu (kde!(points) bandwidths by leave-one-out cross validation) offers the other host files.
#pragma once
#include "common.cuh"

namespace kdeb200 {

constexpr int LCV_FUSED_MAX = 512;  // one row per thread and a single component tile: the sums of eval.cu at S = 1

// One (point set, dimension) of a batched device-points search: one CTA of lcv_golden_points_batch_kernel.
struct LcvBatchItem {
  const double *pts;  // N points, point i at pts + i * d
  double *out;        // the point set's [dim][5] block: xmin, fmin, number of nLOO_LL calls, minm, maxm
  int N, d, dim, pad_;
  double w2;          // lcv_points_w2(N)
};

int kde_lcv(int d, int64_t N, const double *points, int64_t j0, int64_t j1, kdeb200_allreduce_v_fn allreduce, void *user,
            double *bw_std_out, int *ncalls_out);
int kde_lcv_points_device(int d, int64_t N, const double *d_points, double *d_out5, cudaStream_t st);
// the uniform weight of ksize's working density for N points, as the host route computes it
double lcv_points_w2(int64_t N);
// one launch, one CTA per item (2 <= N <= LCV_FUSED_MAX each); d_items in device memory
int kde_lcv_points_batch_device(int nitems, const LcvBatchItem *d_items, cudaStream_t st);
void lcv_points_finish(int d, const double *out5, double *bw_std_out, int *ncalls_out);

}  // namespace kdeb200
