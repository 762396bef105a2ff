// gibbs_batch_d8.cu -- explicit instantiation of the batched Gibbs kernel (K1b) for d = 8.
#include "gibbs_batch_kernel.cuh"
namespace kdeb200 {
template cudaError_t launch_gibbs_batch_d<8>(const BatchParams &, bool, int, int, cudaStream_t);
}
