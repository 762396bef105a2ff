// gibbs_batch_d3.cu -- explicit instantiation of the batched Gibbs kernel (K1b) for d = 3.
#include "gibbs_batch_kernel.cuh"
namespace kdeb200 {
template cudaError_t launch_gibbs_batch_d<3>(const BatchParams &, bool, int, int, cudaStream_t);
}
