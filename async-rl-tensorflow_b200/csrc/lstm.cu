// The A3C LSTM agent's recurrent layer (include/asyncrl_b200_lstm.h): 256 LSTM cells between fc256 and
// the heads, stepped once per env step in the rollout and trained by truncated BPTT over the rollout.
// Both contractions run on the tcgen05 tensor cores through gemm_tc.cuh's BulkGemm (bf16x3 split
// operands in HBM, fp32 TMEM accumulation), as fc256 does:
//   forward : z [B,1024]   = xh [B,512] . lstm_w            A = xh (K-major), B = lstm_w^T (K-major)
//   dgrad   : dxh [B,512]  = dz [B,1024] . lstm_w^T         A = dz (K-major), B = lstm_w (K-major)
//   wgrad   : dW [512,1024] = xh^T . dz over T*B samples    A = xh (MN-major), B = dz (MN-major);
//             split-K over samples, partials summed in a fixed order
// The elementwise parts (packing [x | keep*h_prev] into a split block, the cell, the cell backward,
// the hand-over of dx to arl_fc_backward) are small kernels around them.
#include <string.h>

#include "gemm_tc.cuh"
#include "../../include/asyncrl_b200_lstm.h"

namespace arl {

int reduce_partials_scaled(const float* partials, float* out, int num_partials, int n, float alpha,
                           cudaStream_t stream);
template <class Draw, bool Dueling, bool Streams = false>
int heads_forward(const float* params, int action_size, const float* h, float* logits, float* probs, float* value,
                  int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev, uint64_t seed,
                  int64_t num_samples, int wait_first, Draw draw, cudaStream_t st);

constexpr int kCells = 256, kGates = 4 * kCells, kXH = 2 * kCells;

// lstm_w, lstm_b follow q_b; the ten tensors before them keep their offsets
enum { T_LSTMW = ARL_NUM_TENSORS, T_LSTMB };
constexpr int kLstmTensors = ARL_NUM_TENSORS + 2;
struct LstmLayout {
  int64_t off[kLstmTensors + 1];
};
inline LstmLayout lstm_layout(int A) {
  const ParamLayout P = param_layout(A);
  LstmLayout L;
  for (int i = 0; i <= ARL_NUM_TENSORS; ++i) L.off[i] = P.off[i];
  L.off[T_LSTMW + 1] = L.off[T_LSTMW] + (int64_t)kXH * kGates;
  L.off[T_LSTMB + 1] = L.off[T_LSTMB] + kGates;
  return L;
}
// prepared images: the plain ones at the plain offsets, then
constexpr int64_t kPrepLstmWT = kPrepBytes;                             // lstm_w^T [1024 rows][512] split block
constexpr int64_t kPrepLstmW = kPrepLstmWT + (int64_t)kXH * kGates * 4; // lstm_w [512 rows][1024] split block
constexpr int64_t kPrepLstmBytes = kPrepLstmW + (int64_t)kXH * kGates * 4;

// one GEMM shape serves all three contractions: 128-column N tiles, K in 32-wide stages
using LstmGemm = tc::BulkGemm<128, 32, false, false, tc::EPI_PLAIN, 4>;
using LstmWgrad = tc::BulkGemm<128, 32, true, true, tc::EPI_PLAIN, 4>;
constexpr int kWgradSplits = 4;           // 4 m tiles x 8 n tiles x 4 slices = 128 work items

__device__ __forceinline__ float sigm(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ void store_split8(uint8_t* d, int64_t lo_off, const float (&x)[8]) {
  uint4 h, l;
  tc::split2(x[0], x[1], h.x, l.x);
  tc::split2(x[2], x[3], h.y, l.y);
  tc::split2(x[4], x[5], h.z, l.z);
  tc::split2(x[6], x[7], h.w, l.w);
  *reinterpret_cast<uint4*>(d) = h;
  *reinterpret_cast<uint4*>(d + lo_off) = l;
}

// W fp32 [rows][8*chunks] at any 4-byte alignment (lstm_w follows q_b) -> one split block
// [part][chunk][row][8].  Thread = (chunk, row), rows fastest: the stores are coalesced.
__global__ void split_rows_any_kernel(const float* __restrict__ W, int rows, int chunks, uint8_t* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)rows * chunks) return;
  const int c = (int)(idx / rows), row = (int)(idx - (int64_t)c * rows);
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = __ldg(W + (int64_t)row * chunks * 8 + c * 8 + e);
  store_split8(out + idx * 16, (int64_t)rows * chunks * 16, x);
}
// W fp32 [cols][rows] -> the split block of its transpose [rows][cols]; thread = (chunk, row), rows
// fastest: the loads are coalesced over rows
__global__ void split_cols_any_kernel(const float* __restrict__ W, int rows, int chunks, uint8_t* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)rows * chunks) return;
  const int c = (int)(idx / rows), row = (int)(idx - (int64_t)c * rows);
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = __ldg(W + (int64_t)(c * 8 + e) * rows + row);
  store_split8(out + idx * 16, (int64_t)rows * chunks * 16, x);
}

// [x | keep * h_prev] -> the step's split block xh [part][64 chunks][n rows][8].  Thread = (chunk, row),
// rows fastest.
__global__ void lstm_pack_kernel(const float* __restrict__ x, const float* __restrict__ h_prev,
                                 const uint8_t* __restrict__ reset, uint8_t* __restrict__ xh, int n) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  if (idx >= (int64_t)n * (kXH / 8)) return;
  const int c = (int)(idx / n), row = (int)(idx - (int64_t)c * n);
  const bool from_h = c >= kCells / 8;
  const float* src = from_h ? h_prev + (int64_t)row * kCells + (c - kCells / 8) * 8 : x + (int64_t)row * kCells + c * 8;
  const float keep = from_h && reset != nullptr && reset[row] != 0 ? 0.f : 1.f;
  const float4 a = tc::ldg4(src), b = tc::ldg4(src + 4);
  const float v[8] = {a.x * keep, a.y * keep, a.z * keep, a.w * keep, b.x * keep, b.y * keep, b.z * keep, b.w * keep};
  store_split8(xh + idx * 16, (int64_t)n * kXH * 2, v);
}

// the cell: thread = (row, cell)
__global__ void lstm_cell_kernel(const float* __restrict__ z, const float* __restrict__ bias,
                                 float* __restrict__ state_h, float* __restrict__ state_c,
                                 const uint8_t* __restrict__ reset, int advance, float* __restrict__ gates,
                                 float* __restrict__ c_prev_out, float* __restrict__ c_out, float* __restrict__ h_out,
                                 int n) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  if (idx >= (int64_t)n * kCells) return;
  const int64_t row = idx / kCells;
  const int k = (int)(idx - row * kCells);
  const float* zr = z + row * kGates;
  const float gi = sigm(zr[k] + bias[k]);
  const float gj = tanhf(zr[kCells + k] + bias[kCells + k]);
  const float gf = sigm(zr[2 * kCells + k] + bias[2 * kCells + k] + 1.0f);   // forget_bias = 1
  const float go = sigm(zr[3 * kCells + k] + bias[3 * kCells + k]);
  const float cp = reset != nullptr && reset[row] != 0 ? 0.f : state_c[idx];
  const float c = gf * cp + gi * gj;
  const float h = go * tanhf(c);
  if (gates != nullptr) {
    float* g = gates + row * kGates;
    g[k] = gi; g[kCells + k] = gj; g[2 * kCells + k] = gf; g[3 * kCells + k] = go;
  }
  if (c_prev_out != nullptr) c_prev_out[idx] = cp;
  c_out[idx] = c;
  h_out[idx] = h;
  if (advance) {
    state_c[idx] = c;
    state_h[idx] = h;
  }
}

// The cell backward of one step.  CTA = 256 threads, thread = cell k, rows [r0, r0 + per) of the step;
// dz of kSubRows rows is staged in shared memory and leaves as 16-byte split vectors, 8 rows of one chunk
// per run.  dh = d_h_lstm + keep' * dh_rec and dc_in = keep' * dc, keep' = 1 - term_next (the reset
// of step t+1; term_next == NULL: the last step, nothing comes back).  dc is replaced by
// dc * sigmoid(f) (the gradient w.r.t. the cell state step t read).  bpart[cta][1024]: the CTA's column
// sums of dz, written at the last step (first == 1) and added to at the others, in stream order.
constexpr int kSubRows = 8, kDzLd = kGates + 4;
__global__ void __launch_bounds__(256)
lstm_cell_bwd_kernel(const float* __restrict__ d_h_lstm, const float* __restrict__ dh_rec,
                     const uint8_t* __restrict__ term_next, float* __restrict__ dc,
                     const float* __restrict__ gates, const float* __restrict__ c_prev,
                     const float* __restrict__ cst, uint8_t* __restrict__ dz, float* __restrict__ bpart,
                     int n, int per, int first) {
  __shared__ __align__(16) float st[kSubRows][kDzLd];
  const int k = threadIdx.x;
  pdl_wait();
  const int r0 = blockIdx.x * per, r1 = min(n, r0 + per);
  float b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
  const int64_t lo_off = (int64_t)n * kGates * 2;
  for (int s0 = r0; s0 < r1; s0 += kSubRows) {
    const int ns = min(kSubRows, r1 - s0);
    for (int s = 0; s < ns; ++s) {
      const int64_t row = s0 + s, e = row * kCells + k;
      float dh = d_h_lstm[e], dcn = 0.f;
      if (term_next != nullptr && term_next[row] == 0) {
        dh += dh_rec[row * kXH + kCells + k];
        dcn = dc[e];
      }
      const float* g = gates + row * kGates;
      const float gi = g[k], gj = g[kCells + k], gf = g[2 * kCells + k], go = g[3 * kCells + k];
      const float tc = tanhf(cst[e]);
      const float dcc = fmaf(dh * go, 1.0f - tc * tc, dcn);
      const float zi = dcc * gj * gi * (1.0f - gi);
      const float zj = dcc * gi * (1.0f - gj * gj);
      const float zf = dcc * c_prev[e] * gf * (1.0f - gf);
      const float zo = dh * tc * go * (1.0f - go);
      dc[e] = dcc * gf;
      st[s][k] = zi; st[s][kCells + k] = zj; st[s][2 * kCells + k] = zf; st[s][3 * kCells + k] = zo;
      b0 += zi; b1 += zj; b2 += zf; b3 += zo;
    }
    __syncthreads();
    for (int v = k; v < kSubRows * (kGates / 8); v += 256) {
      const int s = v % kSubRows, c = v / kSubRows;
      if (s < ns) {
        const float4 a = *reinterpret_cast<const float4*>(&st[s][c * 8]);
        const float4 b = *reinterpret_cast<const float4*>(&st[s][c * 8 + 4]);
        const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        store_split8(dz + ((int64_t)c * n + s0 + s) * 16, lo_off, x);
      }
    }
    __syncthreads();
  }
  float* bp = bpart + (int64_t)blockIdx.x * kGates;
  if (first) {
    bp[k] = b0; bp[kCells + k] = b1; bp[2 * kCells + k] = b2; bp[3 * kCells + k] = b3;
  } else {
    bp[k] += b0; bp[kCells + k] += b1; bp[2 * kCells + k] += b2; bp[3 * kCells + k] += b3;
  }
}

// dx (dxh's first 256 columns, times tensor_scale) masked by h_fc > 0 -> arl_fc_backward's d_h: the
// split block [hi|lo][32 chunks][N rows][8] and its transposed copy [hi|lo][ceil(N/8)][256][8 samples]
// (heads.cu heads_bwd_kernel writes the same two).  CTA = 256 threads, 32 samples, staged in shared memory.
__global__ void __launch_bounds__(256)
lstm_dx_pack_kernel(const float* __restrict__ dxh, const float* __restrict__ h_fc, uint8_t* __restrict__ dhs,
                    int64_t n) {
  __shared__ float dt[32][kCells + 1];
  const int k = threadIdx.x;
  pdl_wait();
  const int64_t s0 = (int64_t)blockIdx.x * 32;
  const int ns = (int)min((int64_t)32, n - s0);
  for (int s = 0; s < 32; ++s) {
    const int64_t row = s0 + s;
    dt[s][k] = s < ns && h_fc[row * kCells + k] > 0.f ? dxh[row * kXH + k] : 0.f;
  }
  __syncthreads();
  const int64_t lo_part = (int64_t)32 * n * 16;
  for (int v = k; v < 32 * 32; v += 256) {
    const int s = v % 32, kc = v / 32;
    if (s < ns) {
      float x[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = dt[s][kc * 8 + e];
      store_split8(dhs + ((int64_t)kc * n + s0 + s) * 16, lo_part, x);
    }
  }
  uint8_t* dhsT = dhs + n * kCells * 4;
  const int64_t lo_partT = ((n + 7) / 8) * kCells * 16;
  for (int sc = 0; sc * 8 < ns; ++sc) {
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = dt[sc * 8 + e][k];            // rows >= ns were zeroed above
    store_split8(dhsT + ((s0 / 8 + sc) * kCells + k) * 16, lo_partT, x);
  }
}

template <class K, class... Args>
static int launch_elems(K kern, int64_t n, cudaStream_t st, const char* name, Args... args) {
  if (n <= 0) return ARL_OK;
  ARL_CUDA(launch_pdl(kern, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, args...));
  ARL_LAUNCH_CHECK(name);
  return ARL_OK;
}

}  // namespace arl

using namespace arl;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

extern "C" int arl_lstm_param_layout(int action_size, int64_t* offsets) {
  ARL_REQUIRE(offsets, "arl_lstm_param_layout: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_lstm_param_layout: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  const LstmLayout L = lstm_layout(action_size);
  memcpy(offsets, L.off, sizeof(L.off));
  return ARL_OK;
}

extern "C" int64_t arl_lstm_prepared_floats(void) { return kPrepLstmBytes / 4; }

extern "C" int64_t arl_lstm_workspace_bytes(int action_size) {
  // the plain backward's (the fc wgrad partials, which also hold the LSTM wgrad's 4 x 512 x 1024), then
  // the cell backward's bias partials: up to 2 * 148 CTAs x 1024 floats
  return arl_backward_workspace_bytes(action_size) + (int64_t)2 * 160 * kGates * sizeof(float);
}

extern "C" int arl_prepare_weights_lstm(const float* params, float* prepared, int action_size, void* stream) {
  ARL_REQUIRE(params && prepared, "arl_prepare_weights_lstm: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_prepare_weights_lstm: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = arl_prepare_weights(params, prepared, stream);
  if (rc) return rc;
  const float* W = params + lstm_layout(action_size).off[T_LSTMW];
  uint8_t* P = reinterpret_cast<uint8_t*>(prepared);
  const int64_t n = (int64_t)kXH * kGates / 8;
  // lstm_w^T [1024 rows][512]: the forward's K-major B operand
  split_cols_any_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(W, kGates, kXH / 8, P + kPrepLstmWT);
  ARL_LAUNCH_CHECK("split_cols_any_kernel");
  // lstm_w [512 rows][1024]: the input gradient's K-major B operand
  split_rows_any_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(W, kXH, kGates / 8, P + kPrepLstmW);
  ARL_LAUNCH_CHECK("split_rows_any_kernel");
  return ARL_OK;
}

extern "C" int arl_lstm_step(const float* params, const float* prepared, int action_size, const float* h_fc,
                             float* state_h, float* state_c, const uint8_t* reset, int advance, float* xh, float* z,
                             float* gates, float* c_prev_out, float* c_out, float* h_out, int num_envs,
                             void* stream) {
  ARL_REQUIRE(params && prepared && h_fc && state_h && state_c && xh && z && c_out && h_out,
              "arl_lstm_step: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_lstm_step: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_envs >= 0, "arl_lstm_step: negative size");
  ARL_REQUIRE(aligned16(prepared) && aligned16(h_fc) && aligned16(state_h) && aligned16(xh) && aligned16(z),
              "arl_lstm_step: pointers must be 16-byte aligned");
  if (num_envs == 0) return ARL_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int n = num_envs;
  int rc = launch_elems(lstm_pack_kernel, (int64_t)n * (kXH / 8), st, "lstm_pack_kernel", h_fc,
                        (const float*)state_h, reset, (uint8_t*)xh, n);
  if (rc) return rc;
  tc::BulkGemmArgs g = {};
  g.A = mat(xh, n, n, kXH / 8);
  g.B = mat(reinterpret_cast<const uint8_t*>(prepared) + kPrepLstmWT, kGates, kGates, kXH / 8);
  g.mask = mat(nullptr, 0, 1, 0);
  g.D = z; g.M = n; g.N = kGates; g.K = kXH; g.ldd = kGates;
  rc = run_gemm<LstmGemm>(g, 1, st);
  if (rc) return rc;
  return launch_elems(lstm_cell_kernel, (int64_t)n * kCells, st, "lstm_cell_kernel", (const float*)z,
                      params + lstm_layout(action_size).off[T_LSTMB], state_h, state_c, reset, advance, gates,
                      c_prev_out, c_out, h_out, n);
}

extern "C" int arl_forward_lstm(const float* params, float* prepared, int refresh_prepared, int action_size,
                                const uint8_t* ring, int num_envs, int ring_slots, int first_slot, float* a1,
                                float* a2, float* h_fc, float* state_h, float* state_c, const uint8_t* reset,
                                int advance, float* xh, float* z, float* gates, float* c_prev_out, float* c_out,
                                float* h_out, float* logits, float* probs, float* value, int32_t* actions,
                                int64_t env_id_base, int64_t step, const int64_t* step_dev, uint64_t seed,
                                void* stream) {
  ARL_REQUIRE(params && prepared && ring && a1 && a2 && h_fc && logits && probs && value,
              "arl_forward_lstm: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_forward_lstm: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_envs >= 0 && env_id_base >= 0 && step >= 0, "arl_forward_lstm: negative argument");
  if (num_envs == 0) return ARL_OK;
  int rc = ARL_OK;
  if (refresh_prepared) rc = arl_prepare_weights_lstm(params, prepared, action_size, stream);
  if (rc) return rc;
  // the trunk env range by env range (arl_a2_block_rows); the LSTM and the heads over all envs
  const int chunk = (int)arl_a2_block_rows(num_envs);
  for (int off = 0; off < num_envs; off += chunk) {
    const int n = num_envs - off < chunk ? num_envs - off : chunk;
    float* a1c = a1 + (size_t)off * 3200;                       // 12 800 bytes of fp16 per sample
    float* a2c = a2 + (size_t)off * ARL_A2_ELEMS;
    rc = arl_conv1_forward(prepared, ring + (size_t)off * ring_slots * kPlane, a1c, n, ring_slots, first_slot, 1,
                           stream);
    if (rc) return rc;
    rc = arl_conv2_forward(prepared, a1c, a2c, n, stream);
    if (rc) return rc;
    rc = arl_fc_forward(params, prepared, a2c, h_fc + (size_t)off * ARL_FC, n, stream);
    if (rc) return rc;
  }
  rc = arl_lstm_step(params, prepared, action_size, h_fc, state_h, state_c, reset, advance, xh, z, gates, c_prev_out,
                     c_out, h_out, num_envs, stream);
  if (rc) return rc;
  return heads_forward<SampleDraw, false>(params, action_size, h_out, logits, probs, value, actions, env_id_base, step,
                                          step_dev, seed, num_envs, /*wait_first=*/1, SampleDraw{},
                                          (cudaStream_t)stream);
}

extern "C" int arl_lstm_backward(const float* params, const float* prepared, int action_size, int num_envs, int steps,
                                 const uint8_t* terminals, const float* h_fc, const float* xh, const float* gates,
                                 const float* c_prev, const float* c, const float* d_h_lstm, float* dz, float* dxh,
                                 float* dc, float* d_h, float* grads, void* workspace, float tensor_scale,
                                 void* stream) {
  ARL_REQUIRE(params && prepared && terminals && h_fc && xh && gates && c_prev && c && d_h_lstm && dz && dxh && dc &&
                  d_h && grads && workspace,
              "arl_lstm_backward: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_lstm_backward: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(tensor_scale > 0.f, "arl_lstm_backward: tensor_scale must be > 0");
  ARL_REQUIRE(num_envs > 0 && steps > 0 && (int64_t)num_envs * steps < (1LL << 31), "arl_lstm_backward: bad size");
  ARL_REQUIRE(aligned16(prepared) && aligned16(xh) && aligned16(dz) && aligned16(dxh) && aligned16(d_h) &&
                  aligned16(workspace),
              "arl_lstm_backward: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int B = num_envs, T = steps, N = B * T;
  const LstmLayout L = lstm_layout(action_size);
  float* part = (float*)workspace;
  float* bpart = (float*)((uint8_t*)workspace + arl_backward_workspace_bytes(action_size));
  int grid = 2 * num_sms();
  if (grid > 320) grid = 320;
  int per = (B + grid - 1) / grid;
  per = (per + kSubRows - 1) / kSubRows * kSubRows;
  grid = (B + per - 1) / per;
  const float unscale = 1.0f / tensor_scale;
  for (int t = T - 1; t >= 0; --t) {
    const int64_t o = (int64_t)t * B;
    uint8_t* dzt = reinterpret_cast<uint8_t*>(dz) + o * kGates * 4;
    const bool last = t == T - 1;
    ARL_CUDA(launch_pdl(lstm_cell_bwd_kernel, dim3(grid), dim3(256), 0, st, d_h_lstm + o * kCells,
                        last ? (const float*)nullptr : (const float*)dxh + (o + B) * kXH,
                        last ? (const uint8_t*)nullptr : terminals + o, dc, gates + o * kGates, c_prev + o * kCells,
                        c + o * kCells, dzt, bpart, B, per, last ? 1 : 0));
    ARL_LAUNCH_CHECK("lstm_cell_bwd_kernel");
    // [dx_t | dh_rec_t] = dz_t . lstm_w^T
    tc::BulkGemmArgs g = {};
    g.A = mat(dzt, B, B, kGates / 8);
    g.B = mat(reinterpret_cast<const uint8_t*>(prepared) + kPrepLstmW, kXH, kXH, kGates / 8);
    g.mask = mat(nullptr, 0, 1, 0);
    g.D = dxh + o * kXH; g.M = B; g.N = kXH; g.K = kGates; g.ldd = kXH;
    int rc = run_gemm<LstmGemm>(g, 1, st);
    if (rc) return rc;
  }
  // d lstm_w [512,1024] = xh^T . dz over the N samples (split-K), d lstm_b = column sums of dz
  tc::BulkGemmArgs g = {};
  g.A = mat(xh, N, B, kXH / 8);
  g.B = mat(dz, N, B, kGates / 8);
  g.mask = mat(nullptr, 0, 1, 0);
  g.D = part; g.M = kXH; g.N = kGates; g.K = N; g.ldd = kGates;
  int rc = run_gemm<LstmWgrad>(g, kWgradSplits, st);
  if (rc) return rc;
  rc = reduce_partials_scaled(part, grads + L.off[T_LSTMW], g.k_splits, kXH * kGates, unscale, st);
  if (rc) return rc;
  rc = reduce_partials_scaled(bpart, grads + L.off[T_LSTMB], grid, kGates, unscale, st);
  if (rc) return rc;
  // dx masked by h_fc > 0 in arl_fc_backward's form
  ARL_CUDA(launch_pdl(lstm_dx_pack_kernel, dim3((unsigned)((N + 31) / 32)), dim3(256), 0, st, (const float*)dxh, h_fc,
                      reinterpret_cast<uint8_t*>(d_h), (int64_t)N));
  ARL_LAUNCH_CHECK("lstm_dx_pack_kernel");
  return ARL_OK;
}

extern "C" int arl_backward_lstm(const float* params, const float* prepared, int action_size, const uint8_t* ring,
                                 int num_envs, int ring_slots, int first_slot, int steps, const uint8_t* terminals,
                                 const float* a1, const float* a2, const float* h_fc, const float* xh,
                                 const float* gates, const float* c_prev, const float* c, const float* h_lstm,
                                 const float* dlogits, const float* dvalue, float* d_h_lstm, float* dz, float* dxh,
                                 float* dc, float* d_h, float* d_a2, float* d_a1, float* grads, void* workspace,
                                 float tensor_scale, int allreduce, void* stream) {
  ARL_REQUIRE(tensor_scale > 0.f, "arl_backward_lstm: tensor_scale must be > 0");
  const int64_t N = (int64_t)num_envs * steps;
  const float unscale = 1.0f / tensor_scale;
  int rc = arl_heads_backward_lstm(params, action_size, h_lstm, dlogits, dvalue, d_h_lstm, grads, workspace, N,
                                   tensor_scale, stream);
  if (rc) return rc;
  rc = arl_lstm_backward(params, prepared, action_size, num_envs, steps, terminals, h_fc, xh, gates, c_prev, c,
                         d_h_lstm, dz, dxh, dc, d_h, grads, workspace, tensor_scale, stream);
  if (rc) return rc;
  rc = arl_fc_backward(prepared, a2, arl_a2_block_rows(num_envs), d_h, d_a2, grads, workspace, N, unscale, stream);
  if (rc) return rc;
  rc = arl_conv2_backward(prepared, a1, d_a2, d_a1, grads, workspace, N, unscale, stream);
  if (rc) return rc;
  rc = arl_conv1_backward(ring, d_a1, grads, workspace, num_envs, ring_slots, first_slot, steps, unscale, stream);
  if (rc || !(allreduce && arl_comm_size() > 1)) return rc;
  return arl_allreduce_grads(grads, lstm_layout(action_size).off[kLstmTensors], stream);
}
