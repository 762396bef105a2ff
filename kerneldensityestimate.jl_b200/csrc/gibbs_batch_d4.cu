// gibbs_batch_d4.cu -- explicit instantiation of the batched Gibbs kernel (K1b) for d = 4.
#include "gibbs_batch_kernel.cuh"
namespace kdeb200 {
template cudaError_t launch_gibbs_batch_d<4>(const BatchParams &, bool, int, int, cudaStream_t);
}
