// gibbs_batch_d1.cu -- explicit instantiation of the batched Gibbs kernel (K1b) for d = 1.
#include "gibbs_batch_kernel.cuh"
namespace kdeb200 {
template cudaError_t launch_gibbs_batch_d<1>(const BatchParams &, bool, int, int, cudaStream_t);
}
