// Deterministic reduction of per-CTA partial tensors: out[i] = sum_p partials[p][i], p in a
// fixed order.  Every weight-gradient kernel writes partials; nothing uses float atomics.
#include "common.cuh"

namespace arl {

// many elements, few partials (fc wgrad: 663 552 x 7): one thread per element
__global__ void reduce_partials_kernel(const float* __restrict__ partials, float* __restrict__ out,
                                       int num_partials, int n, float alpha) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  if (i >= n) return;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int p = 0;
  for (; p + 4 <= num_partials; p += 4) {
    a0 += partials[(size_t)p * n + i];
    a1 += partials[(size_t)(p + 1) * n + i];
    a2 += partials[(size_t)(p + 2) * n + i];
    a3 += partials[(size_t)(p + 3) * n + i];
  }
  for (; p < num_partials; ++p) a0 += partials[(size_t)p * n + i];
  out[i] = ((a0 + a1) + (a2 + a3)) * alpha;
}

// few elements, many partials (conv wgrads: 4096 / 8192 x 148; conv bias grads: 16 / 32 x 2368):
// a block owns 32 elements; 32 slices of the partial index are summed in parallel (slice s takes
// p = s, s+32, ...) and combined by a fixed-order tree, so the result does not depend on timing
__global__ void __launch_bounds__(1024)
reduce_partials_wide_kernel(const float* __restrict__ partials, float* __restrict__ out,
                            int num_partials, int n, float alpha) {
  __shared__ float red[32][33];
  const int e = threadIdx.x & 31, s = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + e;
  pdl_wait();
  // eight loads in flight per thread: the bias-gradient reductions are ONE block walking 2368
  // partials (74 per thread); with two loads in flight they took 17 and 36 us (ncu launch list)
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (i < n) {
    int p = s;
    for (; p + 7 * 32 < num_partials; p += 8 * 32) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = partials[(size_t)(p + 32 * u) * n + i];
#pragma unroll
      for (int u = 0; u < 8; ++u) acc[u] += v[u];
    }
    for (int u = 0; p < num_partials; p += 32, ++u) acc[u] += partials[(size_t)p * n + i];
  }
  red[s][e] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
  __syncthreads();
#pragma unroll
  for (int h = 16; h > 0; h >>= 1) {
    if (s < h) red[s][e] += red[s + h][e];
    __syncthreads();
  }
  if (s == 0 && i < n) out[i] = red[0][e] * alpha;
}

// out = alpha * sum of the partials (alpha = 1 / tensor_scale: the gradients handed from layer to
// layer carry a power-of-two factor so that they sit in the middle of the fp16 range, see
// arl_backward; a power of two scales exactly)
int reduce_partials_scaled(const float* partials, float* out, int num_partials, int n, float alpha,
                           cudaStream_t stream) {
  if (n >= 65536 || num_partials < 16)
    ARL_CUDA(launch_pdl(reduce_partials_kernel, dim3((n + 255) / 256), dim3(256), 0, stream, partials, out,
                        num_partials, n, alpha));
  else
    ARL_CUDA(launch_pdl(reduce_partials_wide_kernel, dim3((n + 31) / 32), dim3(1024), 0, stream, partials, out,
                        num_partials, n, alpha));
  ARL_LAUNCH_CHECK("reduce_partials_kernel");
  return ARL_OK;
}
int reduce_partials(const float* partials, float* out, int num_partials, int n,
                    cudaStream_t stream) {
  return reduce_partials_scaled(partials, out, num_partials, n, 1.0f, stream);
}

// reduce_partials_kernel's sums over partials [P][rows][2w], written as two matrices: columns < w to
// out0 [rows][w], the others to out1 (the dueling streams' fc weight gradient: l4_w and la_w)
__global__ void reduce_partials_cols_kernel(const float* __restrict__ partials, float* __restrict__ out0,
                                            float* __restrict__ out1, int num_partials, int n, int w, float alpha) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  if (i >= n) return;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int p = 0;
  for (; p + 4 <= num_partials; p += 4) {
    a0 += partials[(size_t)p * n + i];
    a1 += partials[(size_t)(p + 1) * n + i];
    a2 += partials[(size_t)(p + 2) * n + i];
    a3 += partials[(size_t)(p + 3) * n + i];
  }
  for (; p < num_partials; ++p) a0 += partials[(size_t)p * n + i];
  const int r = i / (2 * w), c = i - r * 2 * w;
  (c < w ? out0 + (size_t)r * w + c : out1 + (size_t)r * w + (c - w))[0] = ((a0 + a1) + (a2 + a3)) * alpha;
}

int reduce_partials_cols(const float* partials, float* out0, float* out1, int num_partials, int rows, int w,
                         float alpha, cudaStream_t stream) {
  const int n = rows * 2 * w;
  ARL_CUDA(launch_pdl(reduce_partials_cols_kernel, dim3((n + 255) / 256), dim3(256), 0, stream, partials, out0, out1,
                      num_partials, n, w, alpha));
  ARL_LAUNCH_CHECK("reduce_partials_cols_kernel");
  return ARL_OK;
}

int conv_init() { return ARL_OK; }

}  // namespace arl
