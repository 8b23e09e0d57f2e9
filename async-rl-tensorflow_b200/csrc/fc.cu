// K3: the fc256 layer (agent.py:251, ops.py:32-46) forward and backward on the tcgen05 tensor
// cores (gemm_tc.cuh: TMEM accumulators, bf16x3 split of the fp32 values, fp32 accumulate).
// Every operand is kept in HBM as split bf16 in 16-byte chunk vectors (gemm_tc.cuh "SplitMat"):
// a2 by conv2 forward, d_h by heads backward, l4_w by arl_fc_prepare -- the kernels here move
// them with cp.async.bulk only.
//   forward : h    = relu(a2 [N,2592] . W [2592,256] + b)     A = a2s (K-major), B = Ws (MN-major)
//   dgrad   : d_a2 = (d_h [N,256] . W^T) * (a2 > 0)           A = dhs (K-major), B = Ws (K-major),
//                                                             mask = sign of a2s' hi part
//   wgrad   : dW   = a2^T [2592,N] . d_h [N,256]              A = a2s (MN-major: k = sample), B = dhsT
//             (d_h's transposed copy, K-major over samples: 4 KB runs); split-K over samples,
//             partials summed in a fixed order (deterministic)
//   bgrad   : db   = column sums of d_h
#include "gemm_tc.cuh"
#include "../../include/asyncrl_b200_dueling_streams.h"

namespace arl {

int reduce_partials(const float* partials, float* out, int num_partials, int n,
                    cudaStream_t stream);
int reduce_partials_scaled(const float* partials, float* out, int num_partials, int n, float alpha,
                           cudaStream_t stream);
template <class Draw, bool Dueling, bool Streams = false>
int heads_forward(const float* params, int action_size, const float* h, float* logits, float* probs, float* value,
                  int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev, uint64_t seed,
                  int64_t num_samples, int wait_first, Draw draw, cudaStream_t st);

// X fp32 [rows][8*chunks] (row stride ld) -> one split block [part][chunk][row][8 bf16].
// Thread = (row, chunk): reads 32 contiguous bytes, writes one hi and one lo vector.
__global__ void split_rows_kernel(const float* __restrict__ X, int64_t ld, int rows, int chunks,
                                  uint8_t* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)rows * chunks) return;
  const int row = (int)(idx / chunks), c = (int)(idx - (int64_t)row * chunks);
  const float4 x0 = tc::ldg4(X + (int64_t)row * ld + c * 8), x1 = tc::ldg4(X + (int64_t)row * ld + c * 8 + 4);
  uint4 h, l;
  tc::split2(x0.x, x0.y, h.x, l.x);
  tc::split2(x0.z, x0.w, h.y, l.y);
  tc::split2(x1.x, x1.y, h.z, l.z);
  tc::split2(x1.z, x1.w, h.w, l.w);
  uint8_t* d = out + ((int64_t)c * rows + row) * 16;
  *reinterpret_cast<uint4*>(d) = h;
  *reinterpret_cast<uint4*>(d + (int64_t)chunks * rows * 16) = l;
}
// X fp32 [cols][rows] (row stride ld; i.e. the TRANSPOSE of the matrix to split) -> one split block
// [part][chunk][row][8 bf16].  Thread = (chunk, row), rows fastest: reads are coalesced over rows.
__global__ void split_cols_kernel(const float* __restrict__ X, int64_t ld, int rows, int chunks, int cols,
                                  uint8_t* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)rows * chunks) return;
  const int c = (int)(idx / rows), row = (int)(idx - (int64_t)c * rows);
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = c * 8 + e < cols ? __ldg(X + (int64_t)(c * 8 + e) * ld + row) : 0.f;
  uint4 h, l;
  tc::split2(x[0], x[1], h.x, l.x);
  tc::split2(x[2], x[3], h.y, l.y);
  tc::split2(x[4], x[5], h.z, l.z);
  tc::split2(x[6], x[7], h.w, l.w);
  uint8_t* d = out + idx * 16;
  *reinterpret_cast<uint4*>(d) = h;
  *reinterpret_cast<uint4*>(d + (int64_t)chunks * rows * 16) = l;
}
int split_cols(const float* X, int64_t ld, int rows, int cols, void* out, cudaStream_t st) {
  const int chunks = (cols + 7) / 8;
  const int64_t n = (int64_t)rows * chunks;
  if (n == 0) return ARL_OK;
  split_cols_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(X, ld, rows, chunks, cols, (uint8_t*)out);
  ARL_LAUNCH_CHECK("split_cols_kernel");
  return ARL_OK;
}
int split_rows(const float* X, int64_t ld, int rows, int chunks, void* out, cudaStream_t st) {
  const int64_t n = (int64_t)rows * chunks;
  if (n == 0) return ARL_OK;
  split_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(X, ld, rows, chunks, (uint8_t*)out);
  ARL_LAUNCH_CHECK("split_rows_kernel");
  return ARL_OK;
}

// [X0 | X1] (two fp32 [rows][8*chunks] matrices side by side, row stride ld each) -> ONE split block of
// 2*chunks chunks [part][chunk][row][8 bf16]: the dueling streams' [l4_w | la_w] image.  Scalar loads:
// la_w follows q_b, so its offset is 4-byte aligned only
__global__ void split_rows_pair_kernel(const float* __restrict__ X0, const float* __restrict__ X1, int64_t ld,
                                      int rows, int chunks, uint8_t* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)rows * 2 * chunks) return;
  const int row = (int)(idx / (2 * chunks)), c = (int)(idx - (int64_t)row * 2 * chunks);
  const float* X = (c < chunks ? X0 : X1) + (int64_t)row * ld + (c < chunks ? c : c - chunks) * 8;
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = __ldg(X + e);
  uint4 h, l;
  tc::split2(x[0], x[1], h.x, l.x);
  tc::split2(x[2], x[3], h.y, l.y);
  tc::split2(x[4], x[5], h.z, l.z);
  tc::split2(x[6], x[7], h.w, l.w);
  uint8_t* d = out + ((int64_t)c * rows + row) * 16;
  *reinterpret_cast<uint4*>(d) = h;
  *reinterpret_cast<uint4*>(d + (int64_t)2 * chunks * rows * 16) = l;
}

// partial column sums of a split matrix [rows][256] (one block): CTA b sums its row range, warp w
// the chunks 4w..4w+3, lanes stride over the rows (512 contiguous bytes per load) -> partials[b][256]
__global__ void __launch_bounds__(256)
colsum_split256_kernel(const uint8_t* __restrict__ xs, float* __restrict__ partials, int rows) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_wait();
  const int per = (rows + gridDim.x - 1) / gridDim.x;
  const int beg = per * blockIdx.x, end = min(rows, beg + per);
  const int64_t part = (int64_t)32 * rows * 16;
  // the four chunks of a warp side by side: 8 loads in flight per lane and row (one chunk after
  // the other, two loads in flight, was latency-bound: 16 us for 21 MB)
  float acc[4][8];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[q][i] = 0.f;
  const uint8_t* p0 = xs + (int64_t)(warp * 4) * rows * 16;
  for (int r = beg + lane; r < end; r += 32) {
    uint4 h[4], l[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint8_t* p = p0 + (int64_t)q * rows * 16 + (int64_t)r * 16;
      h[q] = __ldg(reinterpret_cast<const uint4*>(p));
      l[q] = __ldg(reinterpret_cast<const uint4*>(p + part));
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t hw[4] = {h[q].x, h[q].y, h[q].z, h[q].w}, lw[4] = {l[q].x, l[q].y, l[q].z, l[q].w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[q][2 * i] += __uint_as_float(hw[i] << 16) + __uint_as_float(lw[i] << 16);
        acc[q][2 * i + 1] += __uint_as_float(hw[i] & 0xFFFF0000u) + __uint_as_float(lw[i] & 0xFFFF0000u);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[q][i] = warp_sum(acc[q][i]);
    if (lane == 0) {
      float* d = partials + (size_t)blockIdx.x * 256 + (warp * 4 + q) * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) d[i] = acc[q][i];
    }
  }
}

// the column sums of colsum_split256_kernel for each stream of the dueling streams' d_h, a split
// block [rows][512] (64 chunks): blockIdx.y = stream (chunks 32y .. 32y+31) -> partials[y][b][256]
__global__ void __launch_bounds__(256)
colsum_split512_kernel(const uint8_t* __restrict__ xs, float* __restrict__ partials, int rows) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_wait();
  const int per = (rows + gridDim.x - 1) / gridDim.x;
  const int beg = per * blockIdx.x, end = min(rows, beg + per);
  const int64_t part = (int64_t)64 * rows * 16;
  float acc[4][8];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[q][i] = 0.f;
  const uint8_t* p0 = xs + (int64_t)(blockIdx.y * 32 + warp * 4) * rows * 16;
  for (int r = beg + lane; r < end; r += 32) {
    uint4 h[4], l[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint8_t* p = p0 + (int64_t)q * rows * 16 + (int64_t)r * 16;
      h[q] = __ldg(reinterpret_cast<const uint4*>(p));
      l[q] = __ldg(reinterpret_cast<const uint4*>(p + part));
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t hw[4] = {h[q].x, h[q].y, h[q].z, h[q].w}, lw[4] = {l[q].x, l[q].y, l[q].z, l[q].w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[q][2 * i] += __uint_as_float(hw[i] << 16) + __uint_as_float(lw[i] << 16);
        acc[q][2 * i + 1] += __uint_as_float(hw[i] & 0xFFFF0000u) + __uint_as_float(lw[i] & 0xFFFF0000u);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[q][i] = warp_sum(acc[q][i]);
    if (lane == 0) {
      float* d = partials + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 256 + (warp * 4 + q) * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) d[i] = acc[q][i];
    }
  }
}

// forward: narrow N tiles (4 per row tile) so that one env step of 4096 samples fills 128 SMs.  The
// kernel is bound by the bulk-copy rate of ONE SM (~29 B/clk measured), not by L2 or the tensor
// pipe: 64 CTAs of 128 x 128 tiles move 2/3 of the bytes and take 1.6x as long (measured).
using FcFwd = tc::BulkGemm<64, 32, false, true, tc::EPI_BIAS_RELU, 8>;
using FcDgrad = tc::BulkGemm<128, 32, false, false, tc::EPI_MASK, 4>;
// wgrad: 128 x 256 tiles (all of d_h's columns: l4_w's gradient rows are read once), three N = 256
// MMAs per 16 samples; B comes from d_h's transposed copy in 4 KB runs (8 per stage) instead of 64
// runs of 1 KB: the bulk-copy unit costs ~40 cycles per copy (122 -> @ us)
using FcWgrad = tc::BulkGemm<256, 32, true, false, tc::EPI_PLAIN, 4, false>;

// forward for up to 37 row tiles (one env step): 128 x 256 tiles, split-K over a cluster of 4 CTAs.
// A CTA ingests (128 + 256) x K/4 operand rows instead of (128 + 64) x K -- half the bytes through
// its bulk-copy unit -- and in copies of 2 KB (a2 rows) and 4 KB (l4_w TRANSPOSED, K-major: a run =
// the 256 output columns of one k chunk): the unit needs ~40 cycles per copy whatever its size, so
// the MN-major l4_w image (512-B runs of 32 k) made this kernel slower than FcFwd.  Each CTA dumps its fp32 partial tile into its
// own (by then idle) pipeline stages as [float4 column][row]; after a cluster barrier CTA r sums
// column quarter r of the four partials through distributed shared memory, adds the bias,
// applies relu and writes h.
struct FcFwdCluster : tc::BulkGemm<256, 32, false, false, tc::EPI_PLAIN, 4, false> {
  static constexpr bool CUSTOM_EPI = true;
  static constexpr int CLUSTER = 4;
  static __device__ __forceinline__ void custom_epilogue(const Args&, const tc::TileCoord&, const uint8_t* res,
                                                         uint32_t taddr, int row, EpiPre&, EpiState&) {
    float4* part = reinterpret_cast<float4*>(const_cast<uint8_t*>(res) - STAGES * STAGE_BYTES);
#pragma unroll 4
    for (int c8 = 0; c8 < N_TILE / 8; ++c8) {
      float v[8];
      tc::tmem_ld8(taddr + c8 * 8, v);
      part[(2 * c8) * tc::kTileM + row] = make_float4(v[0], v[1], v[2], v[3]);
      part[(2 * c8 + 1) * tc::kTileM + row] = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
  // (Measured and rejected, round 2: multiplying the reduced hidden rows with [p_w | q_w] right here
  // and finishing softmax + Philox draw in a second cluster phase -- heads and sampling fused into
  // this kernel, parity-green -- made the launch 24.8 -> 39.5 us (ncu) and the cycle 2.164 -> 2.230 ms:
  // only the 128 epilogue threads of each CTA have the rows, one warp per scheduler, so every
  // shared-memory weight read and FMA chain runs at full latency while the other 160 threads and,
  // in the second phase, three of the four CTAs wait at the cluster barrier.  The heads stay a
  // separate warp-per-sample kernel, which now also draws the action: heads.cu.)
  static __device__ __forceinline__ void cluster_reduce(const Args& g, uint8_t* smem, int warp, int lane) {
    const uint32_t rank = tc::cluster_ctarank();
    const int row = warp * 32 + lane, m = (int)(blockIdx.x / CLUSTER) * tc::kTileM + row;
    const uint32_t base = smem_u32(smem);
    uint32_t peer[CLUSTER];
#pragma unroll
    for (int r = 0; r < CLUSTER; ++r) peer[r] = tc::dsmem_addr(base, (uint32_t)r);
    constexpr int Q4 = N_TILE / 4 / CLUSTER;                       // float4 columns per CTA
#pragma unroll 2
    for (int j = 0; j < Q4; ++j) {
      const int c4 = (int)rank * Q4 + j;
      const uint32_t off = (uint32_t)(c4 * tc::kTileM + row) * 16u;
      float4 a = tc::dsmem_ld4(peer[0] + off);
#pragma unroll
      for (int r = 1; r < CLUSTER; ++r) {                          // fixed order: deterministic
        const float4 b = tc::dsmem_ld4(peer[r] + off);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
      }
      const float4 bb = tc::ldg4(g.bias + c4 * 4);
      if (m < g.M)
        *reinterpret_cast<float4*>(g.D + (int64_t)m * g.ldd + c4 * 4) =
            make_float4(fmaxf(a.x + bb.x, 0.f), fmaxf(a.y + bb.y, 0.f), fmaxf(a.z + bb.z, 0.f),
                        fmaxf(a.w + bb.w, 0.f));
    }
  }
};

// FcFwdCluster over several N tiles of 256 (the dueling streams: n tile = stream) in one launch: the
// clusters of a row tile's streams are neighbours in the grid, so both read its a2 rows from L2 close
// together; a grid larger than the SM count runs in waves
struct FcFwdClusterStreams : FcFwdCluster {
  static constexpr bool MULTI_WAVE = true;
  static __device__ __forceinline__ void cluster_reduce(const Args& g, uint8_t* smem, int warp, int lane) {
    const uint32_t rank = tc::cluster_ctarank();
    const int tile = (int)(blockIdx.x / CLUSTER), mt = tile / g.n_tiles, n0 = (tile - mt * g.n_tiles) * N_TILE;
    const int row = warp * 32 + lane, m = mt * tc::kTileM + row;
    const uint32_t base = smem_u32(smem);
    uint32_t peer[CLUSTER];
#pragma unroll
    for (int r = 0; r < CLUSTER; ++r) peer[r] = tc::dsmem_addr(base, (uint32_t)r);
    constexpr int Q4 = N_TILE / 4 / CLUSTER;
#pragma unroll 2
    for (int j = 0; j < Q4; ++j) {
      const int c4 = (int)rank * Q4 + j;
      const uint32_t off = (uint32_t)(c4 * tc::kTileM + row) * 16u;
      float4 a = tc::dsmem_ld4(peer[0] + off);
#pragma unroll
      for (int r = 1; r < CLUSTER; ++r) {                          // fixed order: deterministic
        const float4 b = tc::dsmem_ld4(peer[r] + off);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
      }
      const float4 bb = tc::ldg4(g.bias + n0 + c4 * 4);
      if (m < g.M)
        *reinterpret_cast<float4*>(g.D + (int64_t)m * g.ldd + n0 + c4 * 4) =
            make_float4(fmaxf(a.x + bb.x, 0.f), fmaxf(a.y + bb.y, 0.f), fmaxf(a.z + bb.z, 0.f),
                        fmaxf(a.w + bb.w, 0.f));
    }
  }
};

// number of split-K slices the wgrad produces for K samples and a request of `want`
int fc_wgrad_splits(int K, int want) {
  const int kb = FcWgrad::KB;
  const int k_chunk = ((K + want - 1) / want + kb - 1) / kb * kb;
  return (K + k_chunk - 1) / k_chunk;
}

}  // namespace arl

using namespace arl;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Test hook: the three production instantiations of the tcgen05 GEMM on arbitrary shapes.  The
// fp32 operands are split into scratch buffers first (cudaMalloc + synchronise: test use only).
// variant 0/1: D = relu(A[M,K] . B[K,N] + extra[N])                      (forward instantiation)
// variant 2  : D = (A[M,K] . B[N,K]^T) masked by extra[M,N] > 0          (dgrad)
// variant 3/4: D[z] = A[K,M]^T . B[K,N] over split-K slice z (k_splits slices, M*N floats each)
extern "C" int arl_debug_gemm(int variant, const float* A, const float* B, float* D,
                              const float* extra, int M, int N, int K, int k_splits, void* stream) {
  ARL_REQUIRE(A && B && D, "arl_debug_gemm: null pointer");
  ARL_REQUIRE(variant >= 0 && variant <= 4, "arl_debug_gemm: unknown variant %d", variant);
  ARL_REQUIRE(M > 0 && N > 0 && K > 0 && N % 16 == 0 && (variant >= 3 || K % 8 == 0),
              "arl_debug_gemm: need M,N,K > 0, N %% 16 == 0, K %% 8 == 0");
  ARL_REQUIRE(variant < 3 || M % 8 == 0, "arl_debug_gemm: variants 3/4 need M %% 8 == 0");
  ARL_REQUIRE(variant == 2 || variant >= 3 || extra, "arl_debug_gemm: variants 0/1 need a bias");
  ARL_REQUIRE(variant != 2 || extra, "arl_debug_gemm: variant 2 needs a mask");
  cudaStream_t st = (cudaStream_t)stream;
  // stored shapes [rows][cols] of A, B (and the mask)
  const int ar = variant >= 3 ? K : M, ac = variant >= 3 ? M : K;
  const int br = variant == 2 ? N : K, bc = variant == 2 ? K : N;
  const int k8 = (K + 7) / 8 * 8;
  uint8_t *as = nullptr, *bs = nullptr, *ms = nullptr;
  ARL_CUDA(cudaMalloc(&as, (size_t)ar * ac * 4));
  ARL_CUDA(cudaMalloc(&bs, (size_t)(variant >= 3 ? k8 : br) * bc * 4));
  if (variant == 2) ARL_CUDA(cudaMalloc(&ms, (size_t)M * N * 4));
  int rc = split_rows(A, ac, ar, ac / 8, as, st);
  tc::BulkGemmArgs g = {};
  g.A = mat(as, ar, ar, ac / 8);
  if (variant >= 3) {          // the wgrad's B is K-major over the samples: the transposed split of B [K][N]
    if (!rc) rc = split_cols(B, N, N, K, bs, st);
    g.B = mat(bs, N, N, k8 / 8);
  } else {
    if (!rc) rc = split_rows(B, bc, br, bc / 8, bs, st);
    g.B = mat(bs, br, br, bc / 8);
  }
  if (!rc && variant == 2) rc = split_rows(extra, N, M, N / 8, ms, st);
  g.mask = mat(ms, M, M, N / 8);
  g.D = D; g.bias = extra; g.M = M; g.N = N; g.K = K; g.ldd = N;
  if (!rc) {
    if (variant <= 1) rc = run_gemm<FcFwd>(g, 1, st);
    else if (variant == 2) rc = run_gemm<FcDgrad>(g, 1, st);
    else rc = run_gemm<FcWgrad>(g, k_splits, st);
  }
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(as); cudaFree(bs); cudaFree(ms);
  if (rc) return rc;
  if (e != cudaSuccess) return cuda_fail(e, "arl_debug_gemm");
  return ARL_OK;
}

namespace arl { int conv_prepare(const float* params, void* prepared, cudaStream_t st); }

extern "C" int64_t arl_prepared_floats(void) { return kPrepBytes / 4; }

extern "C" int arl_prepare_weights(const float* params, float* prepared, void* stream) {
  ARL_REQUIRE(params && prepared, "arl_prepare_weights: null pointer");
  ARL_REQUIRE(aligned16(params) && aligned16(prepared), "arl_prepare_weights: pointers must be 16-byte aligned");
  const ParamLayout L = param_layout(1);
  // The conv images FIRST: the conv kernels copy their resident image into shared memory BEFORE
  // griddepcontrol.wait (programmatic dependent launch), which is only sound for data that was
  // complete before their immediate predecessor in the stream started.  With this order the kernel
  // a forward launched right after this call overlaps with is split_cols (a plain launch: it began
  // after build_images had completed), whose output the fc256 kernels read after their wait.
  int rc = conv_prepare(params, prepared, (cudaStream_t)stream);
  if (rc) return rc;
  rc = split_rows(params + L.off[T_L4W], ARL_FC, ARL_A2_ELEMS, ARL_FC / 8,
                  reinterpret_cast<uint8_t*>(prepared) + kPrepFcW, (cudaStream_t)stream);
  if (rc) return rc;
  // l4_w^T [256][2592] for the K-major B operand of the clustered forward
  return split_cols(params + L.off[T_L4W], ARL_FC, ARL_FC, ARL_A2_ELEMS,
                    reinterpret_cast<uint8_t*>(prepared) + kPrepFcWT, (cudaStream_t)stream);
}

static int fc_forward_impl(const float* params, const float* prepared, const float* a2, float* h,
                           int64_t num_samples, cudaStream_t st) {
  const ParamLayout L = param_layout(1);
  const int M = (int)num_samples;
  tc::BulkGemmArgs g = {};
  g.A = mat(a2, M, M, ARL_A2_ELEMS / 8);
  g.B = mat(prepared, ARL_A2_ELEMS, ARL_A2_ELEMS, ARL_FC / 8);
  g.mask = mat(nullptr, 0, 1, 0);
  g.D = h; g.bias = params + L.off[T_L4B];
  g.M = M; g.N = ARL_FC; g.K = ARL_A2_ELEMS; g.ldd = ARL_FC;
  // one env step of up to 37 row tiles: 4-CTA clusters, one split-K slice per CTA
  if ((M + tc::kTileM - 1) / tc::kTileM * FcFwdCluster::CLUSTER <= num_sms()) {
    g.B = mat(reinterpret_cast<const uint8_t*>(prepared) + kPrepFcWT, ARL_FC, ARL_FC, ARL_A2_ELEMS / 8);
    return run_gemm<FcFwdCluster>(g, FcFwdCluster::CLUSTER, st);
  }
  return run_gemm<FcFwd>(g, 1, st);
}

extern "C" int arl_fc_forward(const float* params, const float* prepared, const float* a2, float* h,
                              int64_t num_samples, void* stream) {
  ARL_REQUIRE(params && prepared && a2 && h, "arl_fc_forward: null pointer");
  ARL_REQUIRE(num_samples >= 0 && num_samples < (1LL << 31), "arl_fc_forward: bad num_samples");
  ARL_REQUIRE(aligned16(params) && aligned16(prepared) && aligned16(a2) && aligned16(h),
              "arl_fc_forward: pointers must be 16-byte aligned");
  if (num_samples == 0) return ARL_OK;
  return fc_forward_impl(params, prepared, a2, h, num_samples, (cudaStream_t)stream);
}

namespace arl {
// arl_fc_heads_forward with the action draw `draw` (common.cuh) and the head kind Dueling (heads.cu):
// the forward entries of api.cu end here
template <class Draw, bool Dueling>
int fc_heads_forward(const float* params, const float* prepared, int action_size, const float* a2, float* h,
                     float* logits, float* probs, float* value, int32_t* actions, int64_t env_id_base, int64_t step,
                     const int64_t* step_dev, uint64_t seed, int64_t num_samples, Draw draw, void* stream) {
  ARL_REQUIRE(params && prepared && a2 && h && logits && probs && value, "arl_fc_heads_forward: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_fc_heads_forward: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_samples >= 0 && num_samples < (1LL << 31), "arl_fc_heads_forward: bad num_samples");
  ARL_REQUIRE(env_id_base >= 0 && step >= 0, "arl_fc_heads_forward: negative argument");
  ARL_REQUIRE(aligned16(params) && aligned16(prepared) && aligned16(a2) && aligned16(h),
              "arl_fc_heads_forward: pointers must be 16-byte aligned");
  if (num_samples == 0) return ARL_OK;
  int rc = fc_forward_impl(params, prepared, a2, h, num_samples, (cudaStream_t)stream);
  if (rc) return rc;
  // heads + softmax + (optionally) the draw: one warp-per-sample kernel
  return heads_forward<Draw, Dueling>(params, action_size, h, logits, probs, value, actions, env_id_base, step,
                                      step_dev, seed, num_samples, /*wait_first=*/0, draw, (cudaStream_t)stream);
}
template int fc_heads_forward<SampleDraw, false>(const float*, const float*, int, const float*, float*, float*,
                                                 float*, float*, int32_t*, int64_t, int64_t, const int64_t*,
                                                 uint64_t, int64_t, SampleDraw, void*);
template int fc_heads_forward<EgreedyDraw, false>(const float*, const float*, int, const float*, float*, float*,
                                                  float*, float*, int32_t*, int64_t, int64_t, const int64_t*,
                                                  uint64_t, int64_t, EgreedyDraw, void*);
template int fc_heads_forward<SampleDraw, true>(const float*, const float*, int, const float*, float*, float*,
                                                float*, float*, int32_t*, int64_t, int64_t, const int64_t*,
                                                uint64_t, int64_t, SampleDraw, void*);
template int fc_heads_forward<EgreedyDraw, true>(const float*, const float*, int, const float*, float*, float*,
                                                 float*, float*, int32_t*, int64_t, int64_t, const int64_t*,
                                                 uint64_t, int64_t, EgreedyDraw, void*);
}  // namespace arl

extern "C" int arl_fc_heads_forward(const float* params, const float* prepared, int action_size,
                                    const float* a2, float* h, float* logits, float* probs, float* value,
                                    int32_t* actions, int64_t env_id_base, int64_t step,
                                    const int64_t* step_dev, uint64_t seed, int64_t num_samples,
                                    void* stream) {
  return fc_heads_forward<SampleDraw, false>(params, prepared, action_size, a2, h, logits, probs, value, actions,
                                             env_id_base, step, step_dev, seed, num_samples, SampleDraw{}, stream);
}

extern "C" int arl_fc_backward(const float* prepared, const float* a2, int64_t a2_block_rows,
                               const float* d_h, float* d_a2, float* grads, void* workspace,
                               int64_t num_samples, float grad_unscale, void* stream) {
  ARL_REQUIRE(prepared && a2 && d_h && d_a2 && grads && workspace, "arl_fc_backward: null pointer");
  ARL_REQUIRE(num_samples >= 0 && num_samples < (1LL << 31), "arl_fc_backward: bad num_samples");
  ARL_REQUIRE(aligned16(prepared) && aligned16(a2) && aligned16(d_h) && aligned16(d_a2) &&
                  aligned16(grads) && aligned16(workspace),
              "arl_fc_backward: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const ParamLayout L = param_layout(1);
  float* gW = grads + L.off[T_L4W];
  float* gb = grads + L.off[T_L4B];
  if (num_samples == 0) {
    ARL_CUDA(cudaMemsetAsync(gW, 0, (size_t)(ARL_A2_ELEMS + 1) * ARL_FC * sizeof(float), st));
    return ARL_OK;
  }
  ARL_REQUIRE(a2_block_rows > 0 && num_samples % a2_block_rows == 0,
              "arl_fc_backward: num_samples %lld is not a whole number of a2 blocks of %lld rows",
              (long long)num_samples, (long long)a2_block_rows);
  const int M = (int)num_samples;
  const tc::SplitMat a2s = mat(a2, M, (int)a2_block_rows, ARL_A2_ELEMS / 8);
  const tc::SplitMat dhs = mat(d_h, M, M, ARL_FC / 8);
  // the transposed copy follows the block: rows = the 256 columns of d_h, chunks = groups of 8 samples
  const tc::SplitMat dhsT = mat(reinterpret_cast<const uint8_t*>(d_h) + (size_t)M * ARL_FC * sizeof(float),
                                ARL_FC, ARL_FC, (M + 7) / 8);
  const tc::SplitMat ws = mat(prepared, ARL_A2_ELEMS, ARL_A2_ELEMS, ARL_FC / 8);
  // wgrad first (dW [2592,256] = a2^T . d_h, 7 split-K slices x 21 row tiles = 147 items), dgrad
  // LAST: the next kernel of the chain (conv2 backward) starts with the d_a2 rows dgrad wrote last
  float* part = (float*)workspace;
  tc::BulkGemmArgs g = {};
  g.A = a2s; g.B = dhsT; g.mask = mat(nullptr, 0, 1, 0);
  g.D = part; g.bias = nullptr;
  g.M = ARL_A2_ELEMS; g.N = ARL_FC; g.K = M; g.ldd = ARL_FC;
  int rc = run_gemm<FcWgrad>(g, 7, st);
  if (rc) return rc;
  rc = reduce_partials_scaled(part, gW, g.k_splits, ARL_A2_ELEMS * ARL_FC, grad_unscale, st);
  if (rc) return rc;
  // dgrad: d_a2 [M,2592] = d_h [M,256] . W^T, masked by a2 > 0
  g.A = dhs; g.B = ws; g.mask = a2s;
  g.D = d_a2;
  g.M = M; g.N = ARL_A2_ELEMS; g.K = ARL_FC; g.ldd = ARL_A2_ELEMS;
  rc = run_gemm<FcDgrad>(g, 1, st);
  if (rc) return rc;
  // bias grad
  const int grid = (int)((num_samples + 63) / 64 < num_sms() ? (num_samples + 63) / 64 : num_sms());
  ARL_CUDA(launch_pdl(colsum_split256_kernel, dim3(grid), dim3(256), 0, st, (const uint8_t*)d_h, part, M));
  ARL_LAUNCH_CHECK("colsum_split256_kernel");
  return reduce_partials_scaled(part, gb, grid, ARL_FC, grad_unscale, st);
}

// ---------------------------------------------------------------------------------------------
// Dueling streams (include/asyncrl_b200_dueling_streams.h): two fc256 layers on a2, the value
// stream's (l4_w, l4_b) and the advantage stream's (la_w, la_b), computed as ONE layer of 512
// outputs: h [N][512] = [h_v | h_a] = relu(a2 . [l4_w | la_w] + [l4_b | la_b]).  A row of h holds
// both streams of a sample (not a plane per stream): the fc256 kernels write it with ldd = 512 and
// one N tile per stream, and the heads warp of a sample reads its 2 KB in one go.
namespace arl {
int reduce_partials_cols(const float* partials, float* out0, float* out1, int num_partials, int rows, int w,
                         float alpha, cudaStream_t stream);
}

extern "C" int64_t arl_streams_prepared_floats(void) { return kPrepStreamsBytes / 4; }

extern "C" int arl_prepare_weights_streams(const float* params, float* prepared, int action_size, void* stream) {
  ARL_REQUIRE(params && prepared, "arl_prepare_weights_streams: null pointer");
  ARL_REQUIRE(aligned16(params) && aligned16(prepared),
              "arl_prepare_weights_streams: pointers must be 16-byte aligned");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_prepare_weights_streams: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  cudaStream_t st = (cudaStream_t)stream;
  const StreamsLayout L = streams_layout(action_size);
  uint8_t* prep = reinterpret_cast<uint8_t*>(prepared);
  // the conv images first and the fc256 splits last, as arl_prepare_weights (the PDL rule there)
  int rc = conv_prepare(params, prepared, st);
  if (rc) return rc;
  ARL_CUDA(cudaMemcpyAsync(prep + kPrepSB, params + L.off[T_L4B], ARL_FC * 4, cudaMemcpyDeviceToDevice, st));
  ARL_CUDA(cudaMemcpyAsync(prep + kPrepSB + ARL_FC * 4, params + L.off[T_LAB], ARL_FC * 4, cudaMemcpyDeviceToDevice,
                           st));
  // [l4_w | la_w]: the streaming forward's B (MN-major, 64 chunks) and dgrad's B (K-major, K = 512)
  const int64_t n = (int64_t)ARL_A2_ELEMS * 2 * (ARL_FC / 8);
  split_rows_pair_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(params + L.off[T_L4W], params + L.off[T_LAW],
                                                                        ARL_FC, ARL_A2_ELEMS, ARL_FC / 8,
                                                                        prep + kPrepSW);
  ARL_LAUNCH_CHECK("split_rows_pair_kernel");
  // l4_w^T and la_w^T, one behind the other: the clustered forward's B
  rc = split_cols(params + L.off[T_L4W], ARL_FC, ARL_FC, ARL_A2_ELEMS, prep + kPrepFcWT, st);
  if (rc) return rc;
  return split_cols(params + L.off[T_LAW], ARL_FC, ARL_FC, ARL_A2_ELEMS, prep + kPrepLaWT, st);
}

// Both streams in ONE launch, the stream an N tile: measured against one launch per stream on one B200
// at its 1000 W power limit (DESIGN §3.3), 38.2 / 55.6 / 185.9 us against 39.0 / 73.4 / 240.5 us at
// 4096 / 4736 / 20 480 samples -- the second launch streamed a2 again
static int fc_streams_forward_impl(const float* prepared, const float* a2, float* h, int64_t num_samples,
                                   cudaStream_t st) {
  const uint8_t* prep = reinterpret_cast<const uint8_t*>(prepared);
  const int M = (int)num_samples;
  tc::BulkGemmArgs g = {};
  g.A = mat(a2, M, M, ARL_A2_ELEMS / 8);
  g.mask = mat(nullptr, 0, 1, 0);
  g.D = h; g.bias = reinterpret_cast<const float*>(prep + kPrepSB);
  g.M = M; g.N = 2 * ARL_FC; g.K = ARL_A2_ELEMS; g.ldd = 2 * ARL_FC;
  // the row-tile count at which arl_fc_forward leaves the clustered kernel; the streams' clusters run in
  // waves above 148 CTAs
  if ((M + tc::kTileM - 1) / tc::kTileM * FcFwdCluster::CLUSTER <= num_sms()) {
    g.B = mat(prep + kPrepFcWT, 2 * ARL_FC, ARL_FC, ARL_A2_ELEMS / 8);
    return run_gemm<FcFwdClusterStreams>(g, FcFwdCluster::CLUSTER, st);
  }
  g.B = mat(prep + kPrepSW, ARL_A2_ELEMS, ARL_A2_ELEMS, 2 * ARL_FC / 8);
  return run_gemm<FcFwd>(g, 1, st);
}

extern "C" int arl_fc_forward_streams(const float* prepared, const float* a2, float* h, int64_t num_samples,
                                      void* stream) {
  ARL_REQUIRE(prepared && a2 && h, "arl_fc_forward_streams: null pointer");
  ARL_REQUIRE(num_samples >= 0 && num_samples < (1LL << 31), "arl_fc_forward_streams: bad num_samples");
  ARL_REQUIRE(aligned16(prepared) && aligned16(a2) && aligned16(h),
              "arl_fc_forward_streams: pointers must be 16-byte aligned");
  if (num_samples == 0) return ARL_OK;
  return fc_streams_forward_impl(prepared, a2, h, num_samples, (cudaStream_t)stream);
}

namespace arl {
// fc_heads_forward for the dueling streams: h [N][512], the streams' heads kind (heads.cu)
template <class Draw>
int fc_heads_forward_streams(const float* params, const float* prepared, int action_size, const float* a2, float* h,
                             float* logits, float* probs, float* value, int32_t* actions, int64_t env_id_base,
                             int64_t step, const int64_t* step_dev, uint64_t seed, int64_t num_samples, Draw draw,
                             void* stream) {
  ARL_REQUIRE(params && prepared && a2 && h && logits && probs && value, "arl_forward_streams: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_forward_streams: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_samples >= 0 && num_samples < (1LL << 31), "arl_forward_streams: bad num_samples");
  ARL_REQUIRE(aligned16(params) && aligned16(prepared) && aligned16(a2) && aligned16(h),
              "arl_forward_streams: pointers must be 16-byte aligned");
  if (num_samples == 0) return ARL_OK;
  int rc = fc_streams_forward_impl(prepared, a2, h, num_samples, (cudaStream_t)stream);
  if (rc) return rc;
  return heads_forward<Draw, true, true>(params, action_size, h, logits, probs, value, actions, env_id_base, step,
                                         step_dev, seed, num_samples, /*wait_first=*/0, draw, (cudaStream_t)stream);
}
template int fc_heads_forward_streams<SampleDraw>(const float*, const float*, int, const float*, float*, float*,
                                                  float*, float*, int32_t*, int64_t, int64_t, const int64_t*,
                                                  uint64_t, int64_t, SampleDraw, void*);
template int fc_heads_forward_streams<EgreedyDraw>(const float*, const float*, int, const float*, float*, float*,
                                                   float*, float*, int32_t*, int64_t, int64_t, const int64_t*,
                                                   uint64_t, int64_t, EgreedyDraw, void*);
}  // namespace arl

// arl_fc_backward for the dueling streams: d_h is [d_h_v | d_h_a] (heads_bwd_streams_kernel), K = 512
extern "C" int arl_fc_backward_streams(const float* prepared, const float* a2, int64_t a2_block_rows,
                                       const float* d_h, float* d_a2, float* grads, void* workspace,
                                       int64_t num_samples, float grad_unscale, int action_size, void* stream) {
  ARL_REQUIRE(prepared && a2 && d_h && d_a2 && grads && workspace, "arl_fc_backward_streams: null pointer");
  ARL_REQUIRE(num_samples >= 0 && num_samples < (1LL << 31), "arl_fc_backward_streams: bad num_samples");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_fc_backward_streams: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(aligned16(prepared) && aligned16(a2) && aligned16(d_h) && aligned16(d_a2) && aligned16(grads) &&
                  aligned16(workspace),
              "arl_fc_backward_streams: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const StreamsLayout L = streams_layout(action_size);
  float* gW = grads + L.off[T_L4W];
  float* gb = grads + L.off[T_L4B];
  float* gWa = grads + L.off[T_LAW];
  float* gba = grads + L.off[T_LAB];
  if (num_samples == 0) {
    ARL_CUDA(cudaMemsetAsync(gW, 0, (size_t)(ARL_A2_ELEMS + 1) * ARL_FC * sizeof(float), st));
    ARL_CUDA(cudaMemsetAsync(gWa, 0, (size_t)(ARL_A2_ELEMS + 1) * ARL_FC * sizeof(float), st));
    return ARL_OK;
  }
  ARL_REQUIRE(a2_block_rows > 0 && num_samples % a2_block_rows == 0,
              "arl_fc_backward_streams: num_samples %lld is not a whole number of a2 blocks of %lld rows",
              (long long)num_samples, (long long)a2_block_rows);
  const int M = (int)num_samples, F2 = 2 * ARL_FC;
  const uint8_t* prep = reinterpret_cast<const uint8_t*>(prepared);
  const tc::SplitMat a2s = mat(a2, M, (int)a2_block_rows, ARL_A2_ELEMS / 8);
  const tc::SplitMat dhs = mat(d_h, M, M, F2 / 8);
  const tc::SplitMat dhsT = mat(reinterpret_cast<const uint8_t*>(d_h) + (size_t)M * F2 * sizeof(float), F2, F2,
                                (M + 7) / 8);
  // wgrad: [dl4_w | dla_w] [2592,512] = a2^T . [d_h_v | d_h_a], two N tiles of 256 per row tile
  float* part = (float*)workspace;
  tc::BulkGemmArgs g = {};
  g.A = a2s; g.B = dhsT; g.mask = mat(nullptr, 0, 1, 0);
  g.D = part; g.bias = nullptr;
  g.M = ARL_A2_ELEMS; g.N = F2; g.K = M; g.ldd = F2;
  int rc = run_gemm<FcWgrad>(g, 7, st);
  if (rc) return rc;
  rc = reduce_partials_cols(part, gW, gWa, g.k_splits, ARL_A2_ELEMS, ARL_FC, grad_unscale, st);
  if (rc) return rc;
  // dgrad: d_a2 [M,2592] = [d_h_v | d_h_a] . [l4_w | la_w]^T (K = 512), masked by a2 > 0
  g.A = dhs; g.B = mat(prep + kPrepSW, ARL_A2_ELEMS, ARL_A2_ELEMS, F2 / 8); g.mask = a2s;
  g.D = d_a2;
  g.M = M; g.N = ARL_A2_ELEMS; g.K = F2; g.ldd = ARL_A2_ELEMS;
  rc = run_gemm<FcDgrad>(g, 1, st);
  if (rc) return rc;
  // bias grads: each stream's column sums, reduced in arl_fc_backward's order
  const int grid = (int)((num_samples + 63) / 64 < num_sms() ? (num_samples + 63) / 64 : num_sms());
  ARL_CUDA(launch_pdl(colsum_split512_kernel, dim3(grid, 2), dim3(256), 0, st, (const uint8_t*)d_h, part, M));
  ARL_LAUNCH_CHECK("colsum_split512_kernel");
  rc = reduce_partials_scaled(part, gb, grid, ARL_FC, grad_unscale, st);
  if (rc) return rc;
  return reduce_partials_scaled(part + (size_t)grid * ARL_FC, gba, grid, ARL_FC, grad_unscale, st);
}
