// Element-wise copies with a type conversion between the caller's row-major [N,k] tensors and the handle's state.
#pragma once
#include <cuda_runtime.h>

namespace so101 {

__global__ void int_to_float_kernel(const int *__restrict__ src, float *__restrict__ dst, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (float)src[i];
}
template <typename A, typename B>
__global__ void cast_copy_kernel(const A *__restrict__ src, B *__restrict__ dst, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (B)src[i];
}
template <typename A, typename B>
inline void launch_cast_copy(const A *src, B *dst, size_t n, cudaStream_t s) {
  cast_copy_kernel<A, B><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, dst, n);
}
inline void launch_int_to_float(const int *src, float *dst, int n, cudaStream_t s) {
  int_to_float_kernel<<<(n + 255) / 256, 256, 0, s>>>(src, dst, n);
}

}  // namespace so101
