// gibbs_exact_d7.cu -- explicit instantiation of the certified-FP32 Gibbs kernel (K1x) for d = 7.
#include "gibbs_exact_kernel.cuh"
namespace kdeb200 {
template cudaError_t launch_gibbs_exact_d<7>(const GibbsParams &, const XParams &, int, size_t, cudaStream_t);
template cudaError_t occupancy_gibbs_exact_d<7>(int, size_t, int *);
}
