// mufu_err.cu -- exhaustive relative error of ex2.approx.ftz.f32 on [-126, 0] and rsqrt.approx.ftz.f32 on every positive
// normal float, against FP64 references (tools/ulp_mufu.py builds and runs it).
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

__device__ unsigned long long g_max[2];  // bit patterns of the largest relative errors (non-negative doubles order as integers)

__global__ void ex2_err(uint32_t lo, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float x = __uint_as_float(lo + i);  // -0 .. -126 as increasing bit patterns of negative floats
    if (!(x >= -126.0f && x <= 0.0f)) continue;
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
    const double ref = exp2((double)x);
    const double r = fabs((double)e - ref) / ref;
    atomicMax(&g_max[0], (unsigned long long)__double_as_longlong(r));
  }
}
__global__ void rsqrt_err(uint32_t lo, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float x = __uint_as_float(lo + i);
    float e;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
    const double ref = 1.0 / sqrt((double)x);
    const double r = fabs((double)e - ref) / ref;
    atomicMax(&g_max[1], (unsigned long long)__double_as_longlong(r));
  }
}
int main() {
  const uint32_t neg0 = 0x80000000u, neg126 = 0xC2FC0000u;  // -0.0f .. -126.0f
  ex2_err<<<4096, 256>>>(neg0, neg126 - neg0 + 1);
  const uint32_t pmin = 0x00800000u, pmax = 0x7F7FFFFFu;    // positive normal floats
  rsqrt_err<<<4096, 256>>>(pmin, pmax - pmin + 1);
  unsigned long long h[2];
  if (cudaMemcpyFromSymbol(h, g_max, sizeof(h)) != cudaSuccess) return 1;
  double r[2];
  for (int k = 0; k < 2; ++k) r[k] = *reinterpret_cast<double *>(&h[k]);
  printf("{\"ex2_approx_ftz_f32_max_rel_err\": %.6e, \"ex2_range\": \"[-126, 0], every float\", "
         "\"rsqrt_approx_ftz_f32_max_rel_err\": %.6e, \"rsqrt_range\": \"every positive normal float\"}\n", r[0], r[1]);
  return 0;
}
