// gibbs_many_d4.cu -- explicit instantiation of the many-density Gibbs kernel (K1m, MD = 32 and 64) for d = 4.
#include "gibbs_batch_kernel.cuh"
namespace kdeb200 {
template cudaError_t launch_gibbs_many_d<4>(const BatchParams &, bool, int, int, cudaStream_t);
}
