// K2 on the tensor cores: both convolutions, forward and backward, as implicit GEMMs on tcgen05
// (gemm_tc.cuh).  No im2col matrix ever exists in HBM, and none is built in smem either:
//
//   space-to-depth + shifted descriptors.  An 8x8 stride-4 conv over [84,84,4] is a 2x2
//   stride-1 conv over the space-to-depth tensor X[21,21,64]; a 4x4 stride-2 conv over
//   [20,20,16] is a 2x2 stride-1 conv over X2[10,10,64].  If output pixels are numbered on the
//   SAME grid as X (one garbage column/row per sample), output row P needs X rows P + a*GW + b
//   for the four taps (a,b): a constant row shift.  In the UMMA K-major no-swizzle image a row
//   shift is a 16-byte shift of the descriptor start address, so the four taps are four
//   descriptors onto ONE smem image of the tile's X rows (+ a halo).  Every input element is
//   loaded from HBM and converted exactly once per tile.
//
//   conv1 fwd  : X rows from the u8 ring (exact in bf16 -> hi image only), W1 resident
//   conv2 fwd  : X2 rows from a1 (bf16 hi+lo), W2 resident
//   conv2 bwd  : ONE kernel, one dy2 image (fp16 hi+lo) per tile serves both MMAs.  Input
//                gradient = the transposed conv: output pixels of one parity class (y&1, x&1) use
//                4 taps of dy2 on the X2 grid itself (its zero rows are the padding); the 4 classes
//                share the image and differ only in the resident weights.  Weight gradient: see
//                wgrads; its accumulator lives across the CTA's tiles.
//   wgrads     : dW[(tap,ch), co] = sum_P X[P+shift][ch] * dyz[P][co] reduces over ROWS, so the
//                same row-major images serve as MN-major operands (k = row index); tap b is a
//                second copy of the image shifted by one row, tap a a descriptor row offset.
//                Work is split over ranges of (env, step window, row tile) units (conv1) or CTAs
//                (conv2); partials are summed in a fixed order.
#include <stdlib.h>

#include "gemm_tc.cuh"

namespace arl {

int reduce_partials(const float* partials, float* out, int num_partials, int n, cudaStream_t stream);
int reduce_partials_scaled(const float* partials, float* out, int num_partials, int n, float alpha,
                           cudaStream_t stream);

namespace {
using tc::TileCoord;
using tc::kTileM;

__device__ __forceinline__ void load8(const float* p, float (&x)[8]) {
  const float4 x0 = __ldg(reinterpret_cast<const float4*>(p));
  const float4 x1 = __ldg(reinterpret_cast<const float4*>(p) + 1);
  x[0] = x0.x; x[1] = x0.y; x[2] = x0.z; x[3] = x0.w;
  x[4] = x1.x; x[5] = x1.y; x[6] = x1.z; x[7] = x1.w;
}
__device__ __forceinline__ TileCoord row_tile(int item) {
  TileCoord t;
  t.mt = item; t.nt = 0; t.ks = 0; t.k_begin = 0; t.k_end = 0;
  return t;
}

// ---- pixel-contiguous fp32 tensors scattered onto a padded row grid --------------------------
// A tensor [samples][PH*PW pixels][4*CF4 floats] (dy1, dy2) is laid on a per-sample grid of
// GROWS = rows of width GW with the pixel (py,px) at grid row (py+OFF)*GW + (px+OFF); the other
// grid rows are zero.  A stage needs the grid rows [z0, z0+ROWS).  The pixels that land there are
// ONE contiguous range of the tensor, so the producers stream that range with warp-contiguous
// float4 loads (lane = 16 consecutive bytes) and scatter each float4 to its image position;
// a second small pass zero-fills the rows no pixel maps to.  All row/pixel indices fit in int32
// (checked by the entry points).
template <int GW, int GROWS, int PH, int PW, int OFF, int CF4>
struct PixelGrid {
  static constexpr int PP = PH * PW, WIDTH = PW;
  // a pixel index that is <= the first pixel whose grid row is >= z
  static __device__ __forceinline__ int lower_pixel(int z) {
    const int n = z / GROWS, rem = z - n * GROWS, gy = rem / GW, gx = rem - gy * GW;
    const int py = min(max(gy - OFF, 0), PH - 1), px = min(max(gx - OFF, 0), PW - 1);
    return n * PP + max(py * PW + px - PW, 0);
  }
  static __device__ __forceinline__ int grid_of_pixel(int pix) {
    const int n = pix / PP, rem = pix - n * PP, py = rem / PW, px = rem - py * PW;
    return n * GROWS + (py + OFF) * GW + (px + OFF);
  }
  static __device__ __forceinline__ bool row_has_pixel(int z, int num_samples) {
    const int n = z / GROWS, rem = z - n * GROWS, gy = rem / GW, gx = rem - gy * GW;
    return n < num_samples && gy >= OFF && gy < PH + OFF && gx >= OFF && gx < PW + OFF;
  }
};

// Streams the pixels of grid rows [z0, z0+ROWS) (z0 may be negative: rows before the first sample
// are zero) into an fp16 hi + lo image pair whose 16-B vector (row r, chunk kc) sits at
// kc*PL + r*16.  U float4 loads are in flight per lane before the first one is consumed
// (U * gsize >= the whole window => one latency per stage).  acc accumulates the column sums of
// the window rows r >= SUM_FROM: a lane owns floats (glane % CF4)*4 .. +3 of every pixel it touches.
template <class G, int CF4, int ROWS, int PL, int U, int SUM_FROM>
__device__ __forceinline__ void stream_pixels(uint8_t* hi, uint8_t* lo, const float* __restrict__ src,
                                              int z0, int num_samples, int glane, int gsize,
                                              float (&acc)[4]) {
  const int p0 = G::lower_pixel(z0);
  const int p_total = num_samples * G::PP;
  constexpr int SPAN = ROWS + 2 * G::WIDTH + 2;              // lower_pixel undershoots by <= 2*PW
  constexpr int TOTAL = SPAN * CF4;
  const float4* s4 = reinterpret_cast<const float4*>(src) + (int64_t)p0 * CF4;
  const int q = glane % CF4;                                 // gsize % CF4 == 0
  for (int f0 = glane; f0 < TOTAL; f0 += U * gsize) {
    float4 x[U];
    int rr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int f = f0 + u * gsize;
      const int pix = p0 + f / CF4;
      x[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      rr[u] = -1;
      if (f < TOTAL && pix < p_total) {
        const int z = G::grid_of_pixel(pix);
        if (z >= z0 && z < z0 + ROWS) {
          rr[u] = z - z0;
          x[u] = __ldg(s4 + f);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (rr[u] < 0) continue;
      const int off = (q >> 1) * PL + rr[u] * 16 + (q & 1) * 8;
      tc::store_half_split_h(hi, lo, off, x[u]);
      if (rr[u] >= SUM_FROM) { acc[0] += x[u].x; acc[1] += x[u].y; acc[2] += x[u].z; acc[3] += x[u].w; }
    }
  }
  // rows of the window that no pixel maps to (grid padding, beyond the last sample)
  for (int r = glane; r < ROWS; r += gsize) {
    if (!G::row_has_pixel(z0 + r, num_samples)) {
#pragma unroll
      for (int kc = 0; kc < CF4 / 2; ++kc) {
        *reinterpret_cast<uint4*>(hi + kc * PL + r * 16) = make_uint4(0u, 0u, 0u, 0u);
        *reinterpret_cast<uint4*>(lo + kc * PL + r * 16) = make_uint4(0u, 0u, 0u, 0u);
      }
    }
  }
}

using GridDy2 = PixelGrid<10, 100, 9, 9, 0, 8>;       // dy2 [N,81,32] on the conv2 X2 grid

// resident operand image: built once per parameter change by arl_prepare_weights (build_image of
// the policy), copied into shared memory by the producer threads in the kernel prologue
template <int BYTES>
__device__ __forceinline__ void copy_image(uint8_t* res, const uint8_t* __restrict__ img, int ptid, int nthr) {
  static_assert(BYTES % 16 == 0, "image size");
  // eight loads in flight per thread: with one at a time the 33-KB conv2 image took ~8 us of the
  // 45-us forward kernel (ncu: 19 % of the samples at the prologue barrier)
  constexpr int N = BYTES / 16, U = 8;
  for (int i0 = ptid; i0 < N; i0 += U * nthr) {
    uint4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (i0 + u * nthr < N) v[u] = __ldg(reinterpret_cast<const uint4*>(img) + i0 + u * nthr);
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (i0 + u * nthr < N) reinterpret_cast<uint4*>(res)[i0 + u * nthr] = v[u];
  }
}

// ---- conv1 A operand: space-to-depth rows of the u8 ring ---------------------------------------
// The ring stores every 84x84 plane in 4x4 blocks (K1 writes it that way): the 16 bytes at
// plane + q*16 are block q = y'*21 + x' = frame rows 4y'..4y'+3, columns 4x'..4x'+3 = the 16
// channels plane c contributes to X row (n, y', x').  Sample n = t*num_envs + b stacks the planes
// of env b in ring slots (first_slot + t + c) mod ring_slots, c = 0..3.
struct RingGeo {
  const uint8_t* ring;
  int num_envs, ring_slots, first_slot;
};

// ---- a1 in HBM: fp16, blocked ("a1s") -----------------------------------------------------------
// conv1's output is only ever consumed as a tensor-core operand (conv2 forward / backward) and as
// the relu mask of conv2's input gradient, so it is stored the way those kernels want it -- ONE fp16 per
// value (12 800 bytes per sample, half of fp32 [20,20,16]) in space-to-depth order:
//   a1s[n][kc = (i*2+j)*2 + chalf][q = yp*10 + xp][8 channels]     (16-B vectors)
// with pixel (y,x) = (2yp+i, 2xp+j) and channels chalf*8 .. chalf*8+7.  A run of X2 rows of one
// plane kc is then contiguous: the conv2 kernels fetch their A images with cp.async.bulk and
// convert nothing.  (Round 1 kept a bf16 hi + lo pair, the bytes of fp32; tests/precision_study.py
// is the measurement behind the narrower format.)
constexpr int kA1sSample = 12800, kA1sPlane = 1600;    // bytes
__device__ __forceinline__ int a1s_offset(int y, int x, int chalf) {       // bytes inside a sample
  return (((y & 1) * 2 + (x & 1)) * 2 + chalf) * kA1sPlane + ((y >> 1) * 10 + (x >> 1)) * 16;
}

// Bulk copies of X2 grid rows [xr0, xr0 + ROWS) of plane kc into an image whose vector (row r, kc)
// sits at kc*PL + r*16; SHIFT additionally fills planes 8..15 with the image shifted by one row
// (tap b = 1 of the wgrad).  Called by the lanes that own one plane each; returns the bytes this
// lane has put in flight (it must expect_tx them BEFORE calling).
template <int ROWS, bool SHIFT>
__device__ __forceinline__ uint32_t a1s_bulk_bytes(int xr0, int num_samples) {
  // bytes one plane owner moves: every existing row once (+ once more, minus the first, if SHIFT)
  const int rows_left = num_samples * 100 - xr0;
  const int n = rows_left < ROWS ? (rows_left > 0 ? rows_left : 0) : ROWS;
  return (uint32_t)(SHIFT ? (n > 0 ? 2 * n - 1 : 0) : n) * 16u;
}
template <int ROWS, int PL, bool SHIFT>
__device__ __forceinline__ void a1s_bulk_issue(uint8_t* st, const uint8_t* a1s, int xr0, int num_samples,
                                               int kc, uint64_t* full) {
  int r = 0, n = xr0 / 100, q = xr0 - n * 100;
  while (r < ROWS && n < num_samples) {
    const int cnt = min(100 - q, ROWS - r);
    const uint8_t* src = a1s + (size_t)n * kA1sSample + kc * kA1sPlane + q * 16;
    uint8_t* dst = st + kc * PL + r * 16;
    bulk_g2s(dst, src, (uint32_t)cnt * 16u, full);
    if (SHIFT) {
      if (r > 0) bulk_g2s(dst + 8 * PL - 16, src, (uint32_t)cnt * 16u, full);
      else if (cnt > 1) bulk_g2s(dst + 8 * PL, src + 16, (uint32_t)(cnt - 1) * 16u, full);
    }
    r += cnt; q = 0; ++n;
  }
}
// rows of the window beyond the last sample (last tile only): zero, by all lanes of the group
template <int ROWS, int PL, int PLANES>
__device__ __forceinline__ void a1s_zero_tail(uint8_t* st, int xr0, int num_samples, int glane, int gsize) {
  const int valid = num_samples * 100 - xr0;
  if (valid >= ROWS) return;
  for (int c = glane; c < ROWS * PLANES; c += gsize) {
    const int r = c % ROWS, kc = c / ROWS;
    // planes 8.. (if any) hold the image shifted by one row: their row r is source row r+1
    if (r >= valid - (kc >= 8 ? 1 : 0))
      *reinterpret_cast<uint4*>(st + kc * PL + r * 16) = make_uint4(0u, 0u, 0u, 0u);
  }
}

// =================================== conv1 forward ============================================
struct Conv1FwdArgs {
  const uint8_t* w_img;  // prepared: s8 limb image of l1_w | 3 limb scales | l1_b
  RingGeo geo;
  uint8_t* a1s;          // fp16 blocked output (see a1s above), 12 800 B per sample
  int64_t rows;          // 441 * num_samples (grid rows)
  int num_samples;
};
// The ring planes ARE the tensor-core operand: a plane is 441 blocks of 16 bytes, and 16 bytes
// = 16 u8 K-values of one row is exactly the core-matrix row of the K-major no-swizzle layout for
// 8-bit operands.  So the A image of a tile is 4 x (rows x 16 B) copied verbatim by
// cp.async.bulk (no conversion, no LSU traffic), the MMA is kind::i8 (u8 x s8 -> s32, K = 32)
// and the fp32 weights enter as three s8 limbs, w = s*(L0/64 + L1/2^13 + L2/2^20) (residual
// < 5e-7 * max|w|), concatenated along N (N = 48: one MMA per K block instead of three).  The
// integer accumulation is exact; the epilogue recombines the limb sums in fp32.
struct Conv1Fwd : tc::PolicyBase {
  using Args = Conv1FwdArgs;
  static constexpr int GW = 21, GROWS = 441, TROWS = 150;
  static constexpr int PL = (TROWS + 1) * 16;                 // 2416: plane of one 16-channel chunk
  // two epilogue sets: with bulk-copied operands and 8 short MMAs per tile the accumulator
  // read-out is the longest stage of the pipeline (four sets measured: no further gain)
  static constexpr int EPI_SETS = 2, PROD_WARPS = 8, STAGES = 8, STAGE_BYTES = 4 * PL;   // u8: 4 planes
  // resident W1 image (s8): rows = limb*16 + co (N = 48), 16 k-chunk planes (tap*4 + c); then
  // the three limb scales
  static constexpr int PLB = 49 * 16, B_IMG = 16 * PLB, SCALE_OFF = B_IMG, BIAS_OFF = B_IMG + 16;
  static constexpr int RES_BYTES = B_IMG + 16 + 64;
  static constexpr int ACC_COLS = 64, OUT_COLS = 16, LO_DELTA = 16, SEG = 16;
  static constexpr bool CUSTOM_EPI = true, ACC_LIMBS3 = true;
  static __device__ __forceinline__ int acc_col(int c) { return c; }
  static __device__ __forceinline__ int num_items(const Args& g) { return (int)((g.rows + 127) / 128); }
  static __device__ __forceinline__ TileCoord coord(const Args&, int item) { return row_tile(item); }
  static __device__ __forceinline__ int num_stages(const Args&, const TileCoord&) { return 1; }
  static __device__ __forceinline__ void load_resident(const Args& g, uint8_t* res, int ptid, int nthr) {
    copy_image<RES_BYTES>(res, g.w_img, ptid, nthr);
  }
  // (arl_prepare_weights) params = the flat parameter buffer; all nthr threads of the CTA take part
  static __device__ __forceinline__ void build_image(const float* params, uint8_t* res, int ptid, int nthr) {
    struct { const float* params; } g{params};
    // (1) s = max |w1| over the tensor, by all threads (named barrier 1)
    uint32_t* smax = reinterpret_cast<uint32_t*>(res + SCALE_OFF + 12);
    if (ptid == 0) *smax = 0u;
    asm volatile("bar.sync 1, %0;" ::"r"(nthr) : "memory");
    float m = 0.f;
    for (int i = ptid; i < 4096; i += nthr) m = fmaxf(m, fabsf(g.params[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((ptid & 31) == 0) atomicMax(smax, __float_as_uint(m));      // non-negative floats order as uints
    asm volatile("bar.sync 1, %0;" ::"r"(nthr) : "memory");
    const float s = fmaxf(__uint_as_float(*smax), 1e-30f), inv = 1.0f / s;
    if (ptid == 0) {
      float* sc = reinterpret_cast<float*>(res + SCALE_OFF);
      sc[0] = s * (1.0f / 64.0f); sc[1] = s * (1.0f / 8192.0f); sc[2] = s * (1.0f / 1048576.0f);
    }
    // (2) limbs: one thread per (k-chunk plane, co): 16 K-values = block bytes e = i*4 + j
    for (int ch = ptid; ch < 16 * 16; ch += nthr) {
      const int co = ch & 15, kc = ch >> 4, tap = kc >> 2, c = kc & 3, a = tap >> 1, b = tap & 1;
      uint32_t l0[4] = {0, 0, 0, 0}, l1[4] = {0, 0, 0, 0}, l2[4] = {0, 0, 0, 0};
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        const int i = e >> 2, j = e & 3;
        const float v = g.params[(((4 * a + i) * 8 + 4 * b + j) * 4 + c) * 16 + co] * inv * 64.0f;
        const float r0 = rintf(v), f1 = (v - r0) * 128.0f, r1 = rintf(f1), r2 = rintf((f1 - r1) * 128.0f);
        l0[e >> 2] |= ((uint32_t)(int)r0 & 0xFFu) << (8 * (e & 3));
        l1[e >> 2] |= ((uint32_t)(int)r1 & 0xFFu) << (8 * (e & 3));
        l2[e >> 2] |= ((uint32_t)(int)r2 & 0xFFu) << (8 * (e & 3));
      }
      uint8_t* d = res + kc * PLB + co * 16;
      *reinterpret_cast<uint4*>(d) = make_uint4(l0[0], l0[1], l0[2], l0[3]);
      *reinterpret_cast<uint4*>(d + 16 * 16) = make_uint4(l1[0], l1[1], l1[2], l1[3]);
      *reinterpret_cast<uint4*>(d + 32 * 16) = make_uint4(l2[0], l2[1], l2[2], l2[3]);
    }
    if (ptid < 16) reinterpret_cast<float*>(res + BIAS_OFF)[ptid] = g.params[4096 + ptid];
  }
  // rows of the window that belong to no sample (only in the last tile) are zero-filled here
  static __device__ __forceinline__ void load_stage(const Args& g, const TileCoord& t, int,
                                                    uint8_t* st, int glane, int gsize, Prod&) {
    const int64_t valid = (int64_t)g.num_samples * GROWS - (int64_t)t.mt * 128;
    if (valid >= TROWS) return;
    for (int c = glane; c < TROWS * 4; c += gsize) {
      const int r = c % TROWS, kc = c / TROWS;
      if (r >= valid) *reinterpret_cast<uint4*>(st + kc * PL + r * 16) = make_uint4(0u, 0u, 0u, 0u);
    }
  }
  // lanes 0..7 own one copy each: (segment, plane) = (lane / 4, lane % 4).  At most two samples
  // intersect the window: rows [q0, 441) of n0, then rows [0, ..) of n0+1.  (One lane issuing all
  // eight copies kept the stage's turn-around -- free -> requested -- at ~1.3 us of serial address
  // arithmetic; with 0.65 us per tile and 8 stages that was on the critical path.)
  static __device__ __forceinline__ bool bulk_stage(const Args& g, const TileCoord& t, int, uint8_t* st,
                                                    int glane, int, uint64_t* full) {
    if (glane >= 8) return false;
    const int sgm = glane >> 2, c = glane & 3;
    const int xr0 = t.mt * 128;
    const int n0 = xr0 / GROWS, q0 = xr0 - n0 * GROWS;
    const int first = min(GROWS - q0, TROWS);
    const int n = n0 + sgm;
    int cnt = sgm == 0 ? first : TROWS - first;
    if (n >= g.num_samples) cnt = 0;
    mbar_expect_tx(full, (uint32_t)cnt * 16u);
    if (cnt > 0) {
      const int tt = n / g.geo.num_envs, b = n - tt * g.geo.num_envs;
      const int slot = (g.geo.first_slot + tt + c) % g.geo.ring_slots;
      const uint8_t* src = g.geo.ring + ((size_t)b * g.geo.ring_slots + slot) * kPlane + (sgm == 0 ? q0 : 0) * 16;
      bulk_g2s(st + c * PL + (sgm == 0 ? 0 : first) * 16, src, (uint32_t)cnt * 16u, full);
    }
    return true;
  }
  static __device__ __forceinline__ void issue(const Args&, const TileCoord&, int, uint32_t st,
                                               uint32_t res, uint32_t d) {
    constexpr uint32_t idesc = tc::make_idesc_i8(48);              // x(u8) . [L0 | L1 | L2](s8)
    const uint64_t da0 = tc::make_sdesc(st, PL), db0 = tc::make_sdesc(res, PLB);   // one derivation per stage
#pragma unroll
    for (int tap = 0; tap < 4; ++tap) {
#pragma unroll
      for (int k32 = 0; k32 < 2; ++k32) {
        const uint64_t da = tc::sdesc_advance(da0, ((tap >> 1) * GW + (tap & 1)) * 16 + 2 * k32 * PL);
        const uint64_t db = tc::sdesc_advance(db0, (tap * 4 + 2 * k32) * PLB);
        tc::umma_i8(d, da, db, idesc, (tap | k32) != 0 ? 1u : 0u);
      }
    }
  }
  // epilogue: lane = output pixel; limbs -> fp32 -> /255 + bias, relu -> fp16 -> two 16-B vectors
  // straight into the a1s planes (no staging: 16 consecutive lanes write 256 contiguous B)
  static __device__ __forceinline__ void custom_epilogue(const Args& g, const TileCoord& t,
                                                         const uint8_t* res, uint32_t taddr, int row,
                                                         EpiPre&, EpiState&) {
    const float* sc = reinterpret_cast<const float*>(res + SCALE_OFF);
    float v[16];
    {
      float a[8], b[8];
      tc::tmem_ld8_limbs3(taddr, taddr + 16, taddr + 32, sc[0], sc[1], sc[2], a);
      tc::tmem_ld8_limbs3(taddr + 8, taddr + 24, taddr + 40, sc[0], sc[1], sc[2], b);
#pragma unroll
      for (int e = 0; e < 8; ++e) { v[e] = a[e]; v[8 + e] = b[e]; }
    }
    const int xr = t.mt * 128 + row, n = xr / GROWS;
    const int q = xr - n * GROWS, y = q / GW, x = q - y * GW;
    if (n >= g.num_samples || y >= 20 || x >= 20) return;
    const float2* bias = reinterpret_cast<const float2*>(res + BIAS_OFF);
    uint32_t h[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float2 bb = bias[e];
      const float o0 = fmaxf(fmaf(v[2 * e], 1.0f / 255.0f, bb.x), 0.f);
      const float o1 = fmaxf(fmaf(v[2 * e + 1], 1.0f / 255.0f, bb.y), 0.f);
      h[e] = tc::pack_h2(o0, o1);
    }
    uint8_t* d = g.a1s + (size_t)n * kA1sSample + a1s_offset(y, x, 0);
    *reinterpret_cast<uint4*>(d) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(d + kA1sPlane) = make_uint4(h[4], h[5], h[6], h[7]);
  }
};

// =================================== conv2 forward ============================================
struct Conv2FwdArgs {
  const uint8_t* w_img;  // prepared: fp16 [hi | lo] image of l2_w | l2_b
  const uint8_t* a1s;    // fp16 blocked conv1 output
  uint8_t* a2s;          // split-bf16 chunked output, one block of num_samples rows (gemm_tc.cuh SplitMat)
  int64_t rows;          // 100 * num_samples
  int num_samples;
  int reverse;           // walk the row tiles from the last to the first (see serpentine())
};
struct Conv2Fwd : tc::PolicyBase {
  using Args = Conv2FwdArgs;
  static constexpr int GW = 10, GROWS = 100, TROWS = 140;
  static constexpr int PL = (TROWS + 1) * 16, IMG = 8 * PL;
  // operands arrive by cp.async.bulk straight from the a1s planes: one producer warp per stage,
  // lanes 0..7 own one plane each; two epilogue sets.  One fp16 image per stage (18 KB): six
  // stages = six tiles' worth of copies in flight per SM.
  static constexpr int EPI_SETS = 2, PROD_WARPS = 6, STAGES = 6, STAGE_BYTES = IMG;
  // resident W2 image: rows = [32 co hi | 32 co lo] (N = 64), 32 k-chunk planes
  static constexpr int PLB = 65 * 16, B_IMG = 32 * PLB, BIAS_OFF = B_IMG, RES_BYTES = B_IMG + 128;
  static constexpr int ACC_COLS = 64, OUT_COLS = 32, LO_DELTA = 32, SEG = 32;
  static constexpr bool CUSTOM_EPI = true;
  static __device__ __forceinline__ int acc_col(int c) { return c; }
  static __device__ __forceinline__ int num_items(const Args& g) { return (int)((g.rows + 127) / 128); }
  static __device__ __forceinline__ TileCoord coord(const Args& g, int item) {
    return row_tile(g.reverse ? num_items(g) - 1 - item : item);
  }
  static __device__ __forceinline__ int num_stages(const Args&, const TileCoord&) { return 1; }
  static __device__ __forceinline__ void load_resident(const Args& g, uint8_t* res, int ptid, int nthr) {
    copy_image<RES_BYTES>(res, g.w_img, ptid, nthr);
  }
  static __device__ __forceinline__ void build_image(const float* params, uint8_t* res, int ptid, int nthr) {
    const float* w2 = params + 4112;
    if (ptid < 32) reinterpret_cast<float*>(res + BIAS_OFF)[ptid] = params[4112 + 8192 + ptid];
    for (int ch = ptid; ch < 32 * 32; ch += nthr) {
      const int co = ch & 31, kc = ch >> 5;                    // kc = tap*8 + (i*2+j)*2 + chalf
      const int tap = kc >> 3, ij = (kc >> 1) & 3, chalf = kc & 1;
      const int kh = 2 * (tap >> 1) + (ij >> 1), kw = 2 * (tap & 1) + (ij & 1);
      float x[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = w2[((kh * 4 + kw) * 16 + chalf * 8 + e) * 32 + co];
      tc::store_chunk_split_h(res, res + 32 * 16, kc * PLB + co * 16, x);
    }
  }
  static __device__ __forceinline__ void load_stage(const Args& g, const TileCoord& t, int,
                                                    uint8_t* st, int glane, int gsize, Prod&) {
    a1s_zero_tail<TROWS, PL, 8>(st, t.mt * 128, g.num_samples, glane, gsize);
  }
  static __device__ __forceinline__ bool bulk_stage(const Args& g, const TileCoord& t, int, uint8_t* st,
                                                    int glane, int, uint64_t* full) {
    if (glane >= 8) return false;
    mbar_expect_tx(full, a1s_bulk_bytes<TROWS, false>(t.mt * 128, g.num_samples));
    a1s_bulk_issue<TROWS, PL, false>(st, g.a1s, t.mt * 128, g.num_samples, glane, full);
    return true;
  }
  static __device__ __forceinline__ void issue(const Args&, const TileCoord&, int, uint32_t st,
                                               uint32_t res, uint32_t d) {
    constexpr uint32_t idesc64 = tc::make_idesc_h(64);
    const uint64_t da0 = tc::make_sdesc(st, PL), db0 = tc::make_sdesc(res, PLB);   // one derivation per stage
#pragma unroll
    for (int tap = 0; tap < 4; ++tap) {
      const uint32_t aoff = ((tap >> 1) * GW + (tap & 1)) * 16;
#pragma unroll
      for (int k16 = 0; k16 < 4; ++k16) {
        const uint64_t da = tc::sdesc_advance(da0, aoff + 2 * k16 * PL);
        const uint64_t db = tc::sdesc_advance(db0, (tap * 8 + 2 * k16) * PLB);
        tc::umma_f16(d, da, db, idesc64, (tap | k16) != 0 ? 1u : 0u);      // x . [w_hi | w_lo]
      }
    }
  }
  // epilogue: lane = output pixel (n, yp, xp); its 32 channels = features (yp*9+xp)*32 .. +31 of the
  // NHWC flatten (agent.py:231-232) = chunks (yp*9+xp)*4 .. +3 of the split-bf16 a2 block
  // [part][324 chunks][num_samples][8] that the fc256 kernels consume with cp.async.bulk
  static __device__ __forceinline__ void custom_epilogue(const Args& g, const TileCoord& t, const uint8_t* res,
                                                         uint32_t taddr, int row, EpiPre&, EpiState&) {
    const int xr = t.mt * 128 + row, n = xr / GROWS;
    const int q = xr - n * GROWS, yp = q / GW, xp = q - yp * GW;
    const bool ok = n < g.num_samples && yp < 9 && xp < 9;
    const float4* bias = reinterpret_cast<const float4*>(res + BIAS_OFF);
    const int64_t plane = (int64_t)g.num_samples * 16, part = 324 * plane;
    uint8_t* d = g.a2s + (int64_t)((yp * 9 + xp) * 4) * plane + (int64_t)n * 16;
#pragma unroll
    for (int c8 = 0; c8 < 4; ++c8) {
      float v[8];
      tc::tmem_ld8_sum(taddr + c8 * 8, taddr + 32 + c8 * 8, v);          // x.w_hi + x.w_lo
      if (!ok) continue;
      const float4 b0 = bias[c8 * 2], b1 = bias[c8 * 2 + 1];
      uint4 h, l;
      tc::split2(fmaxf(v[0] + b0.x, 0.f), fmaxf(v[1] + b0.y, 0.f), h.x, l.x);
      tc::split2(fmaxf(v[2] + b0.z, 0.f), fmaxf(v[3] + b0.w, 0.f), h.y, l.y);
      tc::split2(fmaxf(v[4] + b1.x, 0.f), fmaxf(v[5] + b1.y, 0.f), h.z, l.z);
      tc::split2(fmaxf(v[6] + b1.z, 0.f), fmaxf(v[7] + b1.w, 0.f), h.w, l.w);
      *reinterpret_cast<uint4*>(d + c8 * plane) = h;
      *reinterpret_cast<uint4*>(d + part + c8 * plane) = l;
    }
  }
};

// =================================== conv2 backward ===========================================
// dy1s: the gradient w.r.t. conv1's output is only ever the B operand of the conv1 weight-gradient
// MMA (rows of the 21-wide X grid = the reduction index), so conv2 backward stores it the way that
// kernel fetches it with cp.async.bulk -- ONE fp16 per value (x tensor_scale, saturating):
//   dy1s[co group (2)][grid row n*441 + y*21 + x][8 channels]      (16-B vectors)
// with the rows y = 20 / x = 20 (no conv1 output there) written as zeros: 14 112 B per sample.
// One term is enough HERE (unlike dy2): its only consumer is l1_w (l1_b comes from the fp32 sums
// of this kernel's epilogue), 2e-4 in tests/precision_study.py's "fp16 a1 + d_a1" row; round 1
// kept a bf16 hi + lo pair (28 224 B).
constexpr int kDy1sRows = 441;

// per-lane bias sums (4 floats of every CF4-th float4) -> per-warp partial row of CF4*4 floats
template <int CF4>
__device__ __forceinline__ void bias_partial_store(float* dst_row, float (&acc)[4], int lane) {
#pragma unroll
  for (int e = 0; e < 4; ++e) {
#pragma unroll
    for (int o = 16; o >= CF4; o >>= 1) acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], o);
  }
  if (lane < CF4)
    *reinterpret_cast<float4*>(dst_row + lane * 4) = make_float4(acc[0], acc[1], acc[2], acc[3]);
}

struct Conv2BwdArgs {
  const uint8_t* w_img;   // prepared: transposed fp16 [hi | lo] image of l2_w
  const uint8_t* a1s;     // fp16 blocked conv1 output: weight-gradient operand and relu mask
  const float* dy2;       // [N, 81, 32]
  uint8_t* dy1s;          // conv1 output gradient (see dy1s above)
  float* partials;        // [grid][8192]: dW2 of each CTA's tiles
  float* bias2_partials;  // [grid * PROD_WARPS][32]: column sums of dy2 (= db2), per producer warp
  float* bias1_partials;  // [grid * 8 epilogue warps][16]: column sums of dy1 (= db1)
  int64_t rows;           // 100 * num_samples
  int num_samples;
  int reverse;            // walk the row tiles from the last to the first (see serpentine())
};
// Weight and input gradient of conv2 in one pass over 128-row tiles of the 10-wide X2 grid.  A
// stage holds the tile's X2 rows [p0, p0 + 140) (+ the copy shifted by one row), bulk-copied from
// a1s, and dy2 rows [p0 - 11, p0 + 128) converted ONCE into an fp16 hi + lo pair.  Both MMAs read
// that one dy image:
//   input gradient (transposed conv): output block (yy, xx) of parity class (dy, dx), tap (th, tw)
//     reads dy2 pixel (yy - th, xx - tw) = grid row P - 10*th - tw, with kh = dy + 2*th,
//     kw = dx + 2*tw.  Every out-of-range pixel lands on a zero row of the grid (px = 9 / py = 9 of
//     this or the previous sample, or before sample 0), so no padded grid is needed.  dy is the
//     K-major A operand (M = rows, K = co) at a row offset of 11 - 10*th - tw; the resident W2^T
//     image is B with rows part*64 + cls*16 + c (N = 128: the 4 parity classes and the lo part
//     share the A tile of a tap): z_hi . [wT_hi | wT_lo] + z_lo . wT_hi into the tile's accumulator.
//   weight gradient: dW2[(a,b) tap][ch][co] = sum_P X2[P + a*10 + b][ch] * dy2[P][co].  Tap b is
//     folded into M (planes 8..15 = the shifted copy), tap a is a row offset of the A descriptor;
//     dy rows [p0, p0 + 128) are the MN-major B operand [dy_hi | dy_lo] (N = 64), accumulated over
//     all the CTA's tiles in a CTA-lifetime accumulator that the epilogue warps drain once.
// The relu mask the input gradient's epilogue needs is a1s row P of the 8 planes = rows this CTA's
// bulk copies have just brought into L2.
struct Conv2Bwd : tc::PolicyBase {
  using Args = Conv2BwdArgs;
  struct Prod { float acc[4]; };    // running column sums of dy2 over the CTA's tiles (bias gradient)
  static constexpr int GW = 10, GROWS = 100, TROWS = 140;
  static constexpr int HALO = 11, DROWS = kTileM + HALO;           // dy rows [p0 - 11, p0 + 128)
  static constexpr int PLA = (TROWS + 1) * 16, A_IMG = 8 * PLA;    // X2: one copy = 8 channel groups
  // dy: 4 co groups per part; 142 rows: the producers' 8-byte stores of the 4 chunks of a row fall
  // into distinct banks (PLD % 128 = 96)
  static constexpr int PLD = 142 * 16, D_IMG = 4 * PLD;
  // 4 producer warps per stage stream the 159-pixel dy window in one round of 10 float4 per lane;
  // two epilogue sets: the mask loads of one tile overlap the read-out of the previous one.
  // 21 warps -> 96 registers per thread
  static constexpr int EPI_SETS = 2, PROD_WARPS = 12, STAGES = 3, STAGE_BYTES = 2 * A_IMG + 2 * D_IMG;
  static constexpr int PLB = 129 * 16, RES_BYTES = 16 * PLB;       // W2^T: 16 k-chunk planes (tap*4 + co8)
  // tile accumulator: cls*16 + c (hi products), + 64 (lo); CTA accumulator: a*64 + part*32 + co
  static constexpr int ACC_COLS = 128, OUT_COLS = 64, LO_DELTA = 64, SEG = 32, PERSIST_COLS = 128;
  static constexpr bool CUSTOM_EPI = true, PROD_PER_CTA = true;
  static __device__ __forceinline__ int acc_col(int c) { return c; }
  static __device__ __forceinline__ int num_items(const Args& g) { return (int)((g.rows + 127) / 128); }
  static __device__ __forceinline__ TileCoord coord(const Args& g, int item) {
    TileCoord t = row_tile(g.reverse ? num_items(g) - 1 - item : item);
    t.ks = item;                      // == blockIdx.x: the CTA's first tile (starts dW2 at zero)
    return t;
  }
  static __device__ __forceinline__ int num_stages(const Args&, const TileCoord&) { return 1; }
  static __device__ __forceinline__ void load_resident(const Args& g, uint8_t* res, int ptid, int nthr) {
    copy_image<RES_BYTES>(res, g.w_img, ptid, nthr);
  }
  static __device__ __forceinline__ void build_image(const float* params, uint8_t* res, int ptid, int nthr) {
    const float* w2 = params + 4112;
    for (int ch = ptid; ch < 4 * 16 * 16; ch += nthr) {
      const int c = ch & 15, kc = (ch >> 4) & 15, cls = ch >> 8;   // kc = tap*4 + co8
      const int tap = kc >> 2, co8 = kc & 3;
      const int kh = (cls >> 1) + 2 * (tap >> 1), kw = (cls & 1) + 2 * (tap & 1);
      float x[8];
      load8(w2 + ((kh * 4 + kw) * 16 + c) * 32 + co8 * 8, x);
      tc::store_chunk_split_h(res, res + 64 * 16, kc * PLB + (cls * 16 + c) * 16, x);
    }
  }
  static __device__ __forceinline__ void prod_begin(Prod& ps) {
    ps.acc[0] = ps.acc[1] = ps.acc[2] = ps.acc[3] = 0.f;
  }
  static __device__ __forceinline__ void load_stage(const Args& g, const TileCoord& t, int,
                                                    uint8_t* st, int glane, int gsize, Prod& ps) {
    const int p0 = t.mt * 128;
    // X2 rows arrive by cp.async.bulk (bulk_stage); only the rows beyond the last sample need zeros
    a1s_zero_tail<TROWS, PLA, 16>(st, p0, g.num_samples, glane, gsize);
    // dy2 on the 10-wide grid; the bias sums skip the 11 halo rows (the previous tile's)
    uint8_t* d_hi = st + 2 * A_IMG;
    stream_pixels<GridDy2, 8, DROWS, PLD, 10, HALO>(d_hi, d_hi + D_IMG, g.dy2, p0 - HALO, g.num_samples,
                                                   glane, gsize, ps.acc);
  }
  // 8 lanes of the stage's 128 (every 16th) own one a1s plane each
  static __device__ __forceinline__ bool bulk_stage(const Args& g, const TileCoord& t, int, uint8_t* st,
                                                    int glane, int, uint64_t* full) {
    if (glane % 16 != 0) return false;
    const int p0 = t.mt * 128, kc = glane / 16;                      // 0..7
    mbar_expect_tx(full, a1s_bulk_bytes<TROWS, true>(p0, g.num_samples));
    a1s_bulk_issue<TROWS, PLA, true>(st, g.a1s, p0, g.num_samples, kc, full);
    return true;
  }
  static __device__ __forceinline__ void prod_end(const Args& g, const TileCoord& t, Prod& ps, int pw,
                                                  int lane) {
    bias_partial_store<8>(g.bias2_partials + ((size_t)t.ks * PROD_WARPS + pw) * 32, ps.acc, lane);
  }
  static __device__ __forceinline__ void issue(const Args&, const TileCoord& t, int, uint32_t st,
                                               uint32_t res, uint32_t d, uint32_t dw) {
    const uint32_t dy = st + 2 * A_IMG;
    {                                                                // input gradient
      constexpr uint32_t idesc128 = tc::make_idesc_h(128), idesc64 = tc::make_idesc_h(64);
      const uint64_t da0 = tc::make_sdesc(dy, PLD), db0 = tc::make_sdesc(res, PLB);
#pragma unroll
      for (int tap = 0; tap < 4; ++tap) {
        const uint32_t aoff = (HALO - GW * (tap >> 1) - (tap & 1)) * 16;
#pragma unroll
        for (int k16 = 0; k16 < 2; ++k16) {
          const uint64_t da_hi = tc::sdesc_advance(da0, aoff + 2 * k16 * PLD);
          const uint64_t da_lo = tc::sdesc_advance(da0, aoff + D_IMG + 2 * k16 * PLD);
          const uint64_t db = tc::sdesc_advance(db0, (tap * 4 + 2 * k16) * PLB);
          tc::umma_f16(d, da_hi, db, idesc128, (tap | k16) != 0 ? 1u : 0u);  // z_hi . [wT_hi | wT_lo]
          tc::umma_f16(d, da_lo, db, idesc64, 1u);                            // z_lo . wT_hi
        }
      }
    }
    {                                                                // weight gradient
      constexpr uint32_t idesc = tc::make_idesc_h(64, true, true);   // [x ; x shifted] . [dy_hi | dy_lo]
      const uint64_t da0 = tc::make_sdesc(st, 128, PLA), db0 = tc::make_sdesc(dy + HALO * 16, 128, PLD);
      const bool first = t.ks == (int)blockIdx.x;
#pragma unroll
      for (int a = 0; a < 2; ++a) {
#pragma unroll
        for (int k16 = 0; k16 < 8; ++k16) {
          const uint64_t da = tc::sdesc_advance(da0, (a * GW + k16 * 16) * 16);
          const uint64_t db = tc::sdesc_advance(db0, k16 * 256);
          tc::umma_f16(dw + a * 64, da, db, idesc, (first && k16 == 0) ? 0u : 1u);
        }
      }
    }
  }
  // input-gradient epilogue: lane = row (yy, xx) of the 10-wide grid = the 2x2 block of dy1 pixels
  // (2yy+dy, 2xx+dx), accumulator columns cls*16 + c with cls = dy*2 + dx.  Per pixel and channel
  // half: relu mask (sign of a1, prefetched before the accumulator wait), bias-gradient sums, one
  // fp16 vector into dy1s.  The lanes of the last block row / column (yy = 9 / xx = 9) also write
  // the zero rows y = 20 / x = 20, so every byte of dy1s is written on every call.
  struct EpiPre { uint4 m[8]; };
  struct EpiState { float b[16]; };
  static __device__ __forceinline__ void epi_begin(EpiState& s) {
#pragma unroll
    for (int c = 0; c < 16; ++c) s.b[c] = 0.f;
  }
  static __device__ __forceinline__ void epi_prefetch(const Args& g, const TileCoord& t, int row, EpiPre& pre) {
    const int pr = t.mt * 128 + row, n = pr / GROWS, q = pr - n * GROWS;
    const bool ok = n < g.num_samples;
    const uint8_t* p = g.a1s + (int64_t)n * kA1sSample + q * 16;     // plane = cls*2 + chalf (fp16 a1)
#pragma unroll
    for (int i = 0; i < 8; ++i)
      pre.m[i] = ok ? __ldg(reinterpret_cast<const uint4*>(p + i * kA1sPlane)) : make_uint4(0u, 0u, 0u, 0u);
  }
  static __device__ __forceinline__ void custom_epilogue(const Args& g, const TileCoord& t, const uint8_t*,
                                                         uint32_t taddr, int row, EpiPre& pre, EpiState& st) {
    const int pr = t.mt * 128 + row, n = pr / GROWS;
    const int q = pr - n * GROWS, yy = q / GW, xx = q - yy * GW;
    const bool live = n < g.num_samples;
    const int64_t R = (int64_t)g.num_samples * kDy1sRows;
    uint8_t* d0 = g.dy1s + (int64_t)n * kDy1sRows * 16;
#pragma unroll
    for (int cls = 0; cls < 4; ++cls) {
      const int y = 2 * yy + (cls >> 1), x = 2 * xx + (cls & 1);
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float v[8];
        tc::tmem_ld8_sum(taddr + cls * 16 + half * 8, taddr + 64 + cls * 16 + half * 8, v);
        if (!live) continue;
        const uint4 m = pre.m[cls * 2 + half];
        const uint32_t w[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if ((int16_t)(w[i] & 0xFFFFu) <= 0) v[2 * i] = 0.f;        // fp16 > 0 <=> its bits as int16 > 0
          if ((int32_t)w[i] < 0x10000) v[2 * i + 1] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) st.b[half * 8 + e] += v[e];
        *reinterpret_cast<uint4*>(d0 + (half * R + y * 21 + x) * 16) =
            make_uint4(tc::pack_h2(v[0], v[1]), tc::pack_h2(v[2], v[3]), tc::pack_h2(v[4], v[5]),
                       tc::pack_h2(v[6], v[7]));
      }
    }
    if (live && (yy == 9 || xx == 9)) {
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint4* dh = reinterpret_cast<uint4*>(d0 + half * R * 16);
        if (yy == 9) { dh[20 * 21 + 2 * xx] = z; dh[20 * 21 + 2 * xx + 1] = z; }
        if (xx == 9) { dh[(2 * yy) * 21 + 20] = z; dh[(2 * yy + 1) * 21 + 20] = z; }
        if (yy == 9 && xx == 9) dh[20 * 21 + 20] = z;
      }
    }
  }
  static __device__ __forceinline__ void epi_end(const Args& g, EpiState& st, int warp, int lane) {
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const float s = warp_sum(st.b[c]);
      if (lane == 0) g.bias1_partials[((size_t)blockIdx.x * 8 + warp) * 16 + c] = s;
    }
  }
  // weight gradient, once per CTA: epilogue set a drains tap a.  Accumulator row = b*64 + ch with
  // ch = (i*2+j)*16 + cin; tap (kh = 2a+i, kw = 2b+j); columns a*64 + co (hi) and + 32 (lo)
  static __device__ __forceinline__ void persist_epilogue(const Args& g, uint32_t taddr, int row, int a) {
    const int b = row >> 6, ch = row & 63, ij = ch >> 4, cin = ch & 15;
    float* dst = g.partials + (size_t)blockIdx.x * 8192 + (size_t)a * 8 * 16 * 32 +
                 (((ij >> 1) * 4 + 2 * b + (ij & 1)) * 16 + cin) * 32;
#pragma unroll
    for (int c8 = 0; c8 < 4; ++c8) {
      float v[8];
      tc::tmem_ld8_sum(taddr + a * 64 + c8 * 8, taddr + a * 64 + 32 + c8 * 8, v);
      reinterpret_cast<float4*>(dst + c8 * 8)[0] = make_float4(v[0], v[1], v[2], v[3]);
      reinterpret_cast<float4*>(dst + c8 * 8)[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
};

struct Conv1WgradArgs {
  RingGeo geo;
  const uint8_t* dy1s;   // fp16 on the X grid, written by conv2 backward (see dy1s above)
  float* partials;       // [items][4096]
  int64_t dy1s_rows;     // 441 * num_samples: rows of one dy1s co group
  int steps, windows;    // windows = steps per env / Conv1Wgrad::S, rounded up
  int units, k_chunk, items;
};
struct Conv1Wgrad : tc::PolicyBase {
  using Args = Conv1WgradArgs;
  // dW1[(a,b) tap][ch][co] = sum_P X[P + a*21 + b][ch] * dy1[P][co] over the rows P of the X grid.
  // Both operands fp16: the u8 pixels are exact, dy1 is one fp16 per value.  Tap b is folded into M
  // (a second copy of the X image shifted by one row), tap a into N (a second copy of the dy1 image
  // shifted BACK by 21 rows: sum_Q X[Q + b][ch] * dy1[Q - 21][co]), so one N = 32 MMA per 16 rows
  // covers all four taps and the wide X tile is read from shared memory once.
  //
  // Work unit (one pipeline stage) = env b, a window of up to S consecutive steps t0 .. t0+S-1 of
  // that env, grid rows [q0, q0 + R) of each of their samples.  Sample t stacks ring planes
  // t .. t+3, so the window's S samples share S + 3 planes: the producers load and convert each of
  // them ONCE per unit (the t-major row walk of round 3 converted every plane up to 4 times).  A
  // image, cin-major: per plane c of the window, 4 chunk planes [rows 0-1 | rows 2-3 | the same
  // two shifted by one grid row]; the M = 128 rows of sample t are then the 16 chunk planes of
  // planes t .. t+3 at one uniform stride, i.e. one descriptor based at plane t.  The dy1 images
  // of each sample ([dy | dy'] x 2 co groups) arrive by cp.async.bulk from dy1s.
  // Each work item = one CTA's contiguous range of units, so a CTA's accumulator sums its range.
  // S = 5 = the flagship t_max (one window per env); R = 64 (7 row tiles, 448 rows for 441):
  // R = 32 would double the bulk copies per sample row, R = 128 would pad 441 rows to 512.
  static constexpr int GW = 21, GROWS = 441, S = 5, R = 64, TILES = (GROWS + R - 1) / R;
  static constexpr int XROWS = R + 1;                               // + the row the shifted copy needs
  static constexpr int PLA = XROWS * 16, A_IMG = (S + 3) * 4 * PLA; // u8 -> fp16, exact
  static constexpr int PLB = R * 16, B_IMG = 4 * PLB;               // per sample: [dy | dy'] x 2 co groups
  // stage = [A | B of sample 0 .. S-1]: four stages of 53 KB
  static constexpr int PROD_WARPS = 16, STAGES = 4, STAGE_BYTES = A_IMG + S * B_IMG, RES_BYTES = 0;
  // accumulator columns: a*16 + co
  static constexpr int ACC_COLS = 32, OUT_COLS = 32, LO_DELTA = 0, SEG = 16;
  struct Unit { int b, t0, ns, q0; };
  static __device__ __forceinline__ Unit unit(const Args& g, int u) {
    const int ew = u / TILES, w = ew % g.windows;
    Unit x;
    x.q0 = (u - ew * TILES) * R;
    x.b = ew / g.windows;
    x.t0 = w * S;
    x.ns = min(S, g.steps - x.t0);
    return x;
  }
  static __device__ __forceinline__ int acc_col(int c) { return c; }
  static __device__ __forceinline__ int num_items(const Args& g) { return g.items; }
  static __device__ __forceinline__ TileCoord coord(const Args& g, int item) {
    TileCoord t;
    t.mt = item; t.nt = 0; t.ks = item;
    t.k_begin = item * g.k_chunk;
    t.k_end = min(g.units, t.k_begin + g.k_chunk);
    return t;
  }
  static __device__ __forceinline__ int num_stages(const Args&, const TileCoord& t) {
    return t.k_end - t.k_begin;
  }
  static __device__ __forceinline__ void load_resident(const Args&, uint8_t*, int, int) {}
  // the u8 ring rows of the NEXT stage are requested (5 x 16 B per lane, held in registers) before
  // the producer waits for its slot: the ncu capture of round 1 showed producers 24 % of their time
  // waiting for a free stage and then another 13 % on the first use of these loads.  Load = (plane,
  // row): ONE 16-byte vector; lanes run along the rows of one plane, so a warp instruction reads
  // 512 contiguous bytes.  Rows past the sample (last row tile) load as zeros.
  static constexpr bool PREFETCH = true;
  static constexpr int XU = 5;                                      // 16 warps / 4 stages = 128 lanes x 5 >= 8 x 65
  static_assert(XU * 32 * (PROD_WARPS / STAGES) >= (S + 3) * XROWS, "one round of loads per stage");
  struct Prod { uint4 w[XU]; };
  static __device__ __forceinline__ void prefetch_stage(const Args& g, const TileCoord& t, int s, int glane,
                                                        int gsize, Prod& ps) {
    const Unit x = unit(g, t.k_begin + s);
    const uint8_t* env = g.geo.ring + (size_t)x.b * g.geo.ring_slots * kPlane;
#pragma unroll
    for (int u = 0; u < XU; ++u) {
      const int un = glane + u * gsize, c = un / XROWS, q = x.q0 + un - c * XROWS;
      ps.w[u] = make_uint4(0u, 0u, 0u, 0u);
      if (c < x.ns + 3 && q < GROWS) {
        int slot = g.geo.first_slot + x.t0 + c;                     // < 2 * ring_slots
        slot -= slot >= g.geo.ring_slots ? g.geo.ring_slots : 0;
        ps.w[u] = __ldg(reinterpret_cast<const uint4*>(env + (size_t)slot * kPlane) + q);
      }
    }
  }
  static __device__ __forceinline__ void load_stage(const Args& g, const TileCoord& t, int s,
                                                    uint8_t* st, int glane, int gsize, Prod& ps) {
    const Unit x = unit(g, t.k_begin + s);
    // A: chunk planes 4c, 4c+1 = X rows q0 .. q0+R of plane c; 4c+2, 4c+3 = the copy shifted by one
    // row (tap b = 1)
#pragma unroll
    for (int u = 0; u < XU; ++u) {
      const int un = glane + u * gsize, c = un / XROWS, r = un - c * XROWS;
      if (c >= x.ns + 3) break;
      const uint4 lo2 = tc::bytes8_to_f16(ps.w[u].x, ps.w[u].y), hi2 = tc::bytes8_to_f16(ps.w[u].z, ps.w[u].w);
      uint8_t* d = st + 4 * c * PLA + r * 16;
      *reinterpret_cast<uint4*>(d) = lo2;
      *reinterpret_cast<uint4*>(d + PLA) = hi2;
      if (r > 0) {
        *reinterpret_cast<uint4*>(d + 2 * PLA - 16) = lo2;
        *reinterpret_cast<uint4*>(d + 3 * PLA - 16) = hi2;
      }
    }
    // B of sample i, planes 4i + (0, 1) = dy1 rows q0 + r, 4i + (2, 3) = dy1 rows q0 + r - 21.  Rows
    // past the sample (last row tile) and the 21 rows before it (first row tile) are zero here;
    // bulk_stage copies the others.
    const int valid = min(R, GROWS - x.q0), lead = x.q0 == 0 ? GW : 0;
    if (valid < R || lead > 0) {
      for (int i = glane; i < x.ns * 4 * R; i += gsize) {
        const int sp = i / R, r = i - sp * R;
        if ((sp & 2) ? r < lead : r >= valid)
          *reinterpret_cast<uint4*>(st + A_IMG + sp * PLB + r * 16) = make_uint4(0u, 0u, 0u, 0u);
      }
    }
  }
  // lanes 0 .. 4*ns-1 of the stage's group own one dy1 plane each: sample i = lane / 4,
  // plane = copy*2 + co group
  static __device__ __forceinline__ bool bulk_stage(const Args& g, const TileCoord& t, int s, uint8_t* st,
                                                    int glane, int, uint64_t* full) {
    const Unit x = unit(g, t.k_begin + s);
    if (glane >= 4 * x.ns) return false;
    const int n = (x.t0 + (glane >> 2)) * g.geo.num_envs + x.b;
    int src = x.q0, dst = 0, cnt = min(R, GROWS - x.q0);
    if (glane & 2) {
      src = x.q0 - GW; cnt = R;
      if (src < 0) { dst = -src; cnt += src; src = 0; }
    }
    mbar_expect_tx(full, (uint32_t)cnt * 16u);
    bulk_g2s(st + A_IMG + glane * PLB + dst * 16,
             g.dy1s + ((glane & 1) * g.dy1s_rows + (int64_t)n * GROWS + src) * 16, (uint32_t)cnt * 16u, full);
    return true;
  }
  static __device__ __forceinline__ void issue(const Args& g, const TileCoord& t, int s, uint32_t st,
                                               uint32_t, uint32_t d) {
    constexpr uint32_t idesc = tc::make_idesc_h(32, true, true);   // [x ; x shifted] . [dy | dy']
    const int ns = unit(g, t.k_begin + s).ns;
    // one descriptor derivation per stage; sample i: A at plane i, B at its own image
    const uint64_t da0 = tc::make_sdesc(st, 128, PLA), db0 = tc::make_sdesc(st + A_IMG, 128, PLB);
#pragma unroll
    for (int i = 0; i < S; ++i) {
      if (i >= ns) break;
#pragma unroll
      for (int k16 = 0; k16 < R / 16; ++k16)
        tc::umma_f16(d, tc::sdesc_advance(da0, i * 4 * PLA + k16 * 256),
                     tc::sdesc_advance(db0, i * B_IMG + k16 * 256), idesc, (s | i | k16) != 0 ? 1u : 0u);
    }
  }
  // row = cin*32 + b*16 + i*4 + j (chunk plane 4*cin + 2b + i/2); segment a = 16 co of tap
  // (kh = 4a+i, kw = 4b+j)
  static __device__ __forceinline__ float* row_ptr(const Args& g, const TileCoord& t, int row) {
    const int cin = row >> 5, b = (row >> 4) & 1, i = (row >> 2) & 3, j = row & 3;
    const int kw = 4 * b + j;
    return g.partials + (size_t)t.ks * 4096 + ((i * 8 + kw) * 4 + cin) * 16;
  }
  static __device__ __forceinline__ int64_t seg_offset(const Args&, const TileCoord&, int a) {
    return a * 4 * 8 * 4 * 16;
  }
  static __device__ __forceinline__ float4 finish(const Args&, float4 v, float4) {
    const float s = 1.0f / 255.0f;
    return make_float4(v.x * s, v.y * s, v.z * s, v.w * s);
  }
};

// arl_prepare_weights: CTA 0 / 1 / 2 builds the resident image of conv1 fwd / conv2 fwd / conv2 bwd
// in shared memory (the same code the kernels used to run in their prologues) and writes it out
__global__ void __launch_bounds__(256) build_images_kernel(const float* __restrict__ params, uint8_t* prepared) {
  extern __shared__ __align__(128) uint8_t img[];
  const int tid = threadIdx.x;
  int bytes = 0;
  uint8_t* out = prepared;
  if (blockIdx.x == 0) {
    Conv1Fwd::build_image(params, img, tid, 256);
    bytes = Conv1Fwd::RES_BYTES; out += kPrepW1;
  } else if (blockIdx.x == 1) {
    Conv2Fwd::build_image(params, img, tid, 256);
    bytes = Conv2Fwd::RES_BYTES; out += kPrepW2F;
  } else {
    Conv2Bwd::build_image(params, img, tid, 256);
    bytes = Conv2Bwd::RES_BYTES; out += kPrepW2D;
  }
  __syncthreads();
  for (int i = tid; i < bytes / 16; i += 256) reinterpret_cast<uint4*>(out)[i] = reinterpret_cast<const uint4*>(img)[i];
}
static_assert(Conv1Fwd::RES_BYTES <= kPrepW1Bytes && Conv2Fwd::RES_BYTES <= kPrepW2FBytes &&
                  Conv2Bwd::RES_BYTES <= kPrepW2DBytes, "prepared-weight layout");

// Serpentine sweep: consecutive kernels of a chain walk the samples in OPPOSITE directions, so a
// kernel starts with the rows its predecessor touched last -- the ones still in the 126 MB L2 --
// instead of the ones evicted longest ago.  forward: conv1 up, conv2 DOWN; backward: fc dgrad up,
// conv2 backward DOWN.  (conv1 wgrad walks envs, and the samples of one env lie at a stride of
// num_envs samples across all of d_a1, so no direction starts with the rows conv2 backward wrote
// last.)  ARL_SERPENTINE=0 turns it off (A/B runs).
bool serpentine() {
  static const bool on = [] { const char* e = getenv("ARL_SERPENTINE"); return !(e && e[0] == '0'); }();
  return on;
}

}  // namespace

int conv_prepare(const float* params, void* prepared, cudaStream_t st) {
  build_images_kernel<<<3, 256, 33536, st>>>(params, (uint8_t*)prepared);
  ARL_LAUNCH_CHECK("build_images_kernel");
  return ARL_OK;
}

}  // namespace arl

using namespace arl;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

extern "C" int arl_conv1_forward(const float* prepared, const uint8_t* ring, float* a1, int num_envs,
                                 int ring_slots, int first_slot, int steps, void* stream) {
  const float* params = prepared;
  ARL_REQUIRE(params && ring && a1, "arl_conv1_forward: null pointer");
  ARL_REQUIRE(num_envs >= 0 && steps >= 0, "arl_conv1_forward: negative size");
  ARL_REQUIRE(ring_slots >= steps + 3 && first_slot >= 0 && first_slot < ring_slots,
              "arl_conv1_forward: ring_slots %d must be >= steps+3 (%d) and first_slot %d inside it",
              ring_slots, steps + 3, first_slot);
  ARL_REQUIRE(aligned16(params) && aligned16(ring) && aligned16(a1),
              "arl_conv1_forward: pointers must be 16-byte aligned");
  const int64_t N = (int64_t)num_envs * steps;
  if (N == 0) return ARL_OK;
  ARL_REQUIRE(N * 441 < (1LL << 31) - 256, "arl_conv1_forward: too many samples");
  Conv1FwdArgs g{reinterpret_cast<const uint8_t*>(prepared) + kPrepW1, {ring, num_envs, ring_slots, first_slot},
                 reinterpret_cast<uint8_t*>(a1), N * 441, (int)N};
  return tc::launch<Conv1Fwd>(g, (int)((g.rows + 127) / 128), (cudaStream_t)stream);
}

extern "C" int arl_conv2_forward(const float* prepared, const float* a1, float* a2,
                                 int64_t num_samples, void* stream) {
  const float* params = prepared;
  ARL_REQUIRE(params && a1 && a2, "arl_conv2_forward: null pointer");
  ARL_REQUIRE(num_samples >= 0 && num_samples < (1LL << 24), "arl_conv2_forward: bad num_samples");
  ARL_REQUIRE(aligned16(params) && aligned16(a1) && aligned16(a2),
              "arl_conv2_forward: pointers must be 16-byte aligned");
  if (num_samples == 0) return ARL_OK;
  Conv2FwdArgs g{reinterpret_cast<const uint8_t*>(prepared) + kPrepW2F, reinterpret_cast<const uint8_t*>(a1),
                 reinterpret_cast<uint8_t*>(a2), num_samples * 100, (int)num_samples, serpentine() ? 1 : 0};
  return tc::launch<Conv2Fwd>(g, (int)((g.rows + 127) / 128), (cudaStream_t)stream);
}

extern "C" int arl_conv1_backward(const uint8_t* ring, const float* d_a1, float* grads,
                                  void* workspace, int num_envs, int ring_slots, int first_slot,
                                  int steps, float grad_unscale, void* stream) {
  ARL_REQUIRE(ring && d_a1 && grads && workspace, "arl_conv1_backward: null pointer");
  ARL_REQUIRE(num_envs >= 0 && steps >= 0, "arl_conv1_backward: negative size");
  ARL_REQUIRE(ring_slots >= steps + 3 && first_slot >= 0 && first_slot < ring_slots,
              "arl_conv1_backward: ring geometry (slots %d, steps %d, first %d)", ring_slots,
              steps, first_slot);
  ARL_REQUIRE(aligned16(ring) && aligned16(d_a1) && aligned16(grads) && aligned16(workspace),
              "arl_conv1_backward: pointers must be 16-byte aligned");
  const int64_t N = (int64_t)num_envs * steps;
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) {
    ARL_CUDA(cudaMemsetAsync(grads, 0, 4096 * sizeof(float), st));
    return ARL_OK;
  }
  ARL_REQUIRE(N * 441 < (1LL << 31) - 256, "arl_conv1_backward: too many samples");
  Conv1WgradArgs g;
  g.geo = {ring, num_envs, ring_slots, first_slot};
  g.dy1s = reinterpret_cast<const uint8_t*>(d_a1);
  g.partials = (float*)workspace;
  g.dy1s_rows = N * 441;
  g.steps = steps;
  g.windows = (steps + Conv1Wgrad::S - 1) / Conv1Wgrad::S;
  g.units = num_envs * g.windows * Conv1Wgrad::TILES;              // <= 7 N: fits int
  // one contiguous range of units per CTA: at most num_sms() partials
  g.k_chunk = (g.units + num_sms() - 1) / num_sms();
  g.items = (g.units + g.k_chunk - 1) / g.k_chunk;
  int rc = tc::launch<Conv1Wgrad>(g, g.items, st);
  if (rc) return rc;
  return reduce_partials_scaled(g.partials, grads, g.items, 4096, grad_unscale, st);   // l1_w
}

extern "C" int arl_conv2_backward(const float* prepared, const float* a1, const float* d_a2,
                                  float* d_a1, float* grads, void* workspace, int64_t num_samples,
                                  float grad_unscale, void* stream) {
  const float* params = prepared;
  ARL_REQUIRE(params && a1 && d_a2 && d_a1 && grads && workspace,
              "arl_conv2_backward: null pointer");
  ARL_REQUIRE(num_samples >= 0 && num_samples < (1LL << 24), "arl_conv2_backward: bad num_samples");
  ARL_REQUIRE(aligned16(params) && aligned16(a1) && aligned16(d_a2) && aligned16(d_a1) &&
                  aligned16(grads) && aligned16(workspace),
              "arl_conv2_backward: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  float* g2 = grads + 4096 + 16;                                                 // l2_w | l2_b
  if (num_samples == 0) {
    ARL_CUDA(cudaMemsetAsync(grads + 4096, 0, (16 + 8192 + 32) * sizeof(float), st));   // l1_b | l2_w | l2_b
    return ARL_OK;
  }
  Conv2BwdArgs g;
  g.w_img = reinterpret_cast<const uint8_t*>(prepared) + kPrepW2D;
  g.a1s = reinterpret_cast<const uint8_t*>(a1);
  g.dy2 = d_a2;
  g.dy1s = reinterpret_cast<uint8_t*>(d_a1);
  g.rows = num_samples * 100;
  g.num_samples = (int)num_samples;
  g.reverse = serpentine() ? 1 : 0;
  const int items = (int)((g.rows + 127) / 128), grid = items < num_sms() ? items : num_sms();
  g.partials = (float*)workspace;
  g.bias2_partials = g.partials + (size_t)grid * 8192;
  g.bias1_partials = g.bias2_partials + (size_t)grid * Conv2Bwd::PROD_WARPS * 32;
  int rc = tc::launch<Conv2Bwd>(g, items, st);
  if (rc) return rc;
  rc = reduce_partials_scaled(g.partials, g2, grid, 8192, grad_unscale, st);                     // l2_w
  if (rc) return rc;
  rc = reduce_partials_scaled(g.bias2_partials, g2 + 8192, grid * Conv2Bwd::PROD_WARPS, 32, grad_unscale, st);   // l2_b
  if (rc) return rc;
  return reduce_partials_scaled(g.bias1_partials, grads + 4096, grid * 8, 16, grad_unscale, st);   // l1_b
}
