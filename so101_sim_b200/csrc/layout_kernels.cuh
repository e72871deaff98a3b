// Element-wise copies with a type conversion between the caller's row-major [N,k] tensors and the handle's state.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

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
// rows i of a row-major [n][width] float array with mask[i] != 0 (every row when mask is null) -> 0
__global__ void zero_rows_kernel(float *__restrict__ rows, const uint8_t *__restrict__ mask, int n, int width) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)n * width) return;
  if (!mask || mask[i / width]) rows[i] = 0.f;
}
inline void launch_zero_rows(float *rows, const uint8_t *mask, int n, int width, cudaStream_t s) {
  const size_t total = (size_t)n * width;
  zero_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(rows, mask, n, width);
}
inline void launch_int_to_float(const int *src, float *dst, int n, cudaStream_t s) {
  int_to_float_kernel<<<(n + 255) / 256, 256, 0, s>>>(src, dst, n);
}

}  // namespace so101
