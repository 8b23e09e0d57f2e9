// tcgen05 contraction framework (sm_100a).  Every dense contraction of the net (fc256 and the
// two convolutions, forward and backward) is an instance of
//     D[128-row tile, N_TILE] (fp32, TMEM) += A[128, K] . B[N_TILE, K]^T
// where the operand tiles are BUILT IN SHARED MEMORY BY PRODUCER WARPS straight from the
// tensors in HBM (fp32 activations / u8 frames / fp32 weights): gather (im2col), split into
// bf16 hi + bf16 lo ("bf16x3": hi*hi + hi*lo + lo*hi with fp32 accumulation, relative error
// ~2^-16 instead of bf16's 2^-8; u8 pixels are exact in bf16 and need no lo part) and store in
// the UMMA canonical K-major no-swizzle layout.  A Policy supplies the gather, the tile
// decomposition and the epilogue; this file owns the pipeline.
//
// One persistent CTA per SM, 416 threads:
//   warps 0-3   epilogue : tcgen05.ld (TMEM lane quadrant = warp id) -> Policy::store -> HBM
//   warps 4-11  producers: 8/STAGES warps own each smem stage and fill it independently of the
//                          other stages (STAGES load->convert->store chains in flight);
//                          fence.proxy.async + mbarrier arrive hand the stage to the MMA warp
//   warp 12     MMA      : one thread issues tcgen05.mma (cta_group::1, kind::f16, M=128,
//                          N=N_TILE, K=16); tcgen05.commit frees the stage / publishes the
//                          accumulator (2 TMEM accumulator stages); owns tcgen05.alloc/dealloc
//
// smem operand image (bf16): element (row r, k) of a [ROWS x KB] tile sits at
//   (k/8)*LBO + r*16 + (k%8)*2,  LBO = (ROWS+pad)*16, SBO = 128 (the 8 rows of a core matrix are
//   contiguous).  Producers read HBM with WARP-CONTIGUOUS float4 loads (lane = 16 consecutive
//   bytes, a warp instruction = 512 contiguous bytes = 4 full lines) and store the converted
//   half-chunk (4 bf16 = 8 B) of hi and lo; `pad` is chosen per policy so that those 8-byte
//   stores are bank-conflict-free.
//
// Epilogue: TMEM -> registers (lane = row) -> per-warp smem staging -> coalesced float4 stores
// (SEG/4 lanes per row), so an instruction writes full 128-B lines instead of 32 x 16 B.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <atomic>

#include "common.cuh"

namespace arl {
namespace tc {

constexpr int kTileM = 128;
// per policy: EPI_SETS sets of 4 epilogue warps (set e drains accumulator stage e when there are
// two: the read-outs of consecutive tiles overlap, which hides the HBM latency of a mask-reading
// epilogue), PROD_WARPS producer warps; warp layout = [epilogue | producers | MMA]
template <class P> __host__ __device__ constexpr int epi_warps() { return 4 * P::EPI_SETS; }
template <class P> __host__ __device__ constexpr int prod_threads() { return P::PROD_WARPS * 32; }
template <class P> __host__ __device__ constexpr int cta_threads() { return (epi_warps<P>() + P::PROD_WARPS + 1) * 32; }

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// One lane of a CONVERGED warp (elect.sync over the full mask: always the same lane).  The MMA
// warp waits for its barriers converged and issues the tcgen05 instructions of a whole stage
// inside ONE `if (elect_one())`: a region the compiler knows to be single-threaded, so every
// tcgen05.mma is a bare UTCHMMA on uniform registers.  Inside `if (lane == 0)` it cannot prove
// that and wraps EVERY UTCHMMA in an ELECT / R2UR / BRA.U.ANY sequence plus a fresh descriptor
// derivation: 13-18 SASS instructions of one thread's serial chain per MMA (~8 cycles each), which
// is what bounded the wgrad kernels (ncu: MMA warp 73-83 % busy, 95-173 cycles per MMA).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// D[tmem] (+)= A[smem desc] . B[smem desc]
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (s32) (+)= A[smem desc] (u8) . B[smem desc] (s8), K = 32
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
          smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,"
      "%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
                 "=r"(r[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// three s32 limb accumulators (int8 path), 8 columns each: v = a0*s0 + a1*s1 + a2*s2
__device__ __forceinline__ void tmem_ld8_limbs3(uint32_t t0, uint32_t t1, uint32_t t2, float s0,
                                                float s1, float s2, float (&v)[8]) {
  uint32_t a[8], b[8], c[8];
#define ARL_LD8(dst, addr)                                                                       \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"          \
               : "=r"(dst[0]), "=r"(dst[1]), "=r"(dst[2]), "=r"(dst[3]), "=r"(dst[4]), "=r"(dst[5]), \
                 "=r"(dst[6]), "=r"(dst[7])                                                      \
               : "r"(addr)                                                                       \
               : "memory")
  ARL_LD8(a, t0);
  ARL_LD8(b, t1);
  ARL_LD8(c, t2);
#undef ARL_LD8
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i)
    v[i] = fmaf((float)(int)a[i], s0, fmaf((float)(int)b[i], s1, (float)(int)c[i] * s2));
}
// hi-part + lo-part accumulators, 8 columns: two loads in flight, one wait
__device__ __forceinline__ void tmem_ld8_sum(uint32_t taddr_a, uint32_t taddr_b, float (&v)[8]) {
  uint32_t r[8], q[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
                 "=r"(r[7])
               : "r"(taddr_a)
               : "memory");
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]),
                 "=r"(q[7])
               : "r"(taddr_b)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]) + __uint_as_float(q[i]);
}
// two 16-column loads in flight, one wait; v += w (hi-part + lo-part accumulators)
__device__ __forceinline__ void tmem_ld16_sum(uint32_t taddr_a, uint32_t taddr_b, float (&v)[16]) {
  uint32_t r[16], q[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,"
      "%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr_a)
      : "memory");
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,"
      "%15}, [%16];"
      : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]),
        "=r"(q[7]), "=r"(q[8]), "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]),
        "=r"(q[14]), "=r"(q[15])
      : "r"(taddr_b)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]) + __uint_as_float(q[i]);
}

// ---- thread-block clusters: barrier + distributed shared memory -------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {     // every thread of every CTA of the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t dsmem_addr(uint32_t cta_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ float dsmem_ld1(uint32_t addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float4 dsmem_ld4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// instruction descriptor: bf16 x bf16 -> f32, M=128; operands K-major unless *_mn
__host__ __device__ constexpr uint32_t make_idesc(int n, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
}
// instruction descriptor: fp16 x fp16 -> f32 (kind::f16 with both operand formats = F16), M=128
__host__ __device__ constexpr uint32_t make_idesc_h(int n, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | (0u << 7) | (0u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
}
// instruction descriptor: u8 x s8 -> s32 (kind::i8), M=128, both operands K-major
__host__ __device__ constexpr uint32_t make_idesc_i8(int n) {
  return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
}
// shared-memory matrix descriptor, SWIZZLE_NONE.  The operand images in this file place the 16-B
// vector of (index r of the 16-B-strided axis, chunk c of the other axis) at c*PLANE + r*16.
//   K-major operand : r = row (M/N), c = k/8   -> LBO = PLANE (next K chunk), SBO = 128
//   MN-major operand: r = k,         c = row/8 -> LBO = 128 (next 8 k), SBO = PLANE (next 8 rows)
__device__ __forceinline__ uint64_t make_sdesc(uint32_t smem_addr, uint32_t lbo_bytes,
                                               uint32_t sbo_bytes = 128) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) |
         ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}

// the descriptor of the same image `bytes` further on (start-address field only; the shared
// window is < 256 KB, so the 14-bit field cannot carry): one add instead of a re-derivation
__device__ __forceinline__ uint64_t sdesc_advance(uint64_t d, uint32_t bytes) {
  return (d & 0xFFFFFFFF00000000ull) | (uint64_t)((uint32_t)d + (bytes >> 4));
}

// ---- chunk helpers (a chunk = 8 consecutive k of one row = 16 B of bf16) ---------------------
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  const float2 hf = __bfloat1622float2(h);
  const __nv_bfloat162 l = __floats2bfloat162_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void store_chunk_split(uint8_t* hi_img, uint8_t* lo_img, int off,
                                                  const float (&x)[8]) {
  uint4 h, l;
  split2(x[0], x[1], h.x, l.x);
  split2(x[2], x[3], h.y, l.y);
  split2(x[4], x[5], h.z, l.z);
  split2(x[6], x[7], h.w, l.w);
  *reinterpret_cast<uint4*>(hi_img + off) = h;
  *reinterpret_cast<uint4*>(lo_img + off) = l;
}
// ---- fp16 storage (round 2: tensors that are only ever tensor-core operands are kept as ONE fp16
// value instead of a bf16 hi + lo pair: 2^-12 relative per element, measured 2.5e-4 / 4.4e-4 on
// logits / gradients against the float64 oracle -- tests/precision_study.py; plain bf16 fails the
// 1e-3 bar).  Activations are O(1); the layer-to-layer gradients carry a power-of-two factor
// (arl_backward tensor_scale) that keeps them in the middle of the fp16 range, and conversions
// saturate instead of overflowing to infinity.
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  const __half2 h = __floats2half2_rn(fminf(fmaxf(a, -65504.f), 65504.f), fminf(fmaxf(b, -65504.f), 65504.f));
  return *reinterpret_cast<const uint32_t*>(&h);
}
// 8 consecutive k of one row -> one 16-byte vector of fp16
__device__ __forceinline__ void store_chunk_h(uint8_t* img, int off, const float (&x)[8]) {
  *reinterpret_cast<uint4*>(img + off) =
      make_uint4(pack_h2(x[0], x[1]), pack_h2(x[2], x[3]), pack_h2(x[4], x[5]), pack_h2(x[6], x[7]));
}
// 4 consecutive k of one row: 8 bytes
__device__ __forceinline__ void store_half_h(uint8_t* img, int off, const float4& x) {
  *reinterpret_cast<uint2*>(img + off) = make_uint2(pack_h2(x.x, x.y), pack_h2(x.z, x.w));
}
// weights keep two fp16 terms (hi = fp16(w), lo = fp16(w - hi); the lo term of an O(0.02) weight is
// a subnormal with 2^-24 absolute precision): x . [w_hi | w_lo] as ONE MMA of width 2N
__device__ __forceinline__ void split2_h(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void store_chunk_split_h(uint8_t* hi_img, uint8_t* lo_img, int off,
                                                    const float (&x)[8]) {
  uint4 h, l;
  split2_h(x[0], x[1], h.x, l.x);
  split2_h(x[2], x[3], h.y, l.y);
  split2_h(x[4], x[5], h.z, l.z);
  split2_h(x[6], x[7], h.w, l.w);
  *reinterpret_cast<uint4*>(hi_img + off) = h;
  *reinterpret_cast<uint4*>(lo_img + off) = l;
}
// 4 consecutive k of one row as an fp16 hi + lo pair (gradients: saturating hi)
__device__ __forceinline__ void store_half_split_h(uint8_t* hi_img, uint8_t* lo_img, int off, const float4& x) {
  const float c = 65504.f;
  const float a0 = fminf(fmaxf(x.x, -c), c), a1 = fminf(fmaxf(x.y, -c), c);
  const float a2 = fminf(fmaxf(x.z, -c), c), a3 = fminf(fmaxf(x.w, -c), c);
  uint2 h, l;
  split2_h(a0, a1, h.x, l.x);
  split2_h(a2, a3, h.y, l.y);
  *reinterpret_cast<uint2*>(hi_img + off) = h;
  *reinterpret_cast<uint2*>(lo_img + off) = l;
}
__device__ __forceinline__ float4 ldg4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
// 8 bytes (two u32 words) -> 8 exact bf16
__device__ __forceinline__ uint32_t bytes2bf16x2(uint32_t w, int sel_lo, int sel_hi) {
  // 0x4B000000 | byte = 8388608 + byte as fp32; subtracting 8388608 is exact
  const float a = __uint_as_float(__byte_perm(w, 0x4B000000u, sel_lo)) - 8388608.0f;
  const float b = __uint_as_float(__byte_perm(w, 0x4B000000u, sel_hi)) - 8388608.0f;
  const __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&p);
}
__device__ __forceinline__ uint4 bytes8_to_bf16(uint32_t w0, uint32_t w1) {
  // selector: result byte0 = src byte i, bytes 1..3 = 0x00,0x00,0x4B of the magic word
  uint4 o;
  o.x = bytes2bf16x2(w0, 0x7440, 0x7441);
  o.y = bytes2bf16x2(w0, 0x7442, 0x7443);
  o.z = bytes2bf16x2(w1, 0x7440, 0x7441);
  o.w = bytes2bf16x2(w1, 0x7442, 0x7443);
  return o;
}

// 8 bytes (two u32 words) -> 8 exact fp16: 0x6400 | byte = 1024 + byte as fp16; subtracting 1024 is exact
__device__ __forceinline__ uint32_t bytes2h2(uint32_t w, int sel) {
  const uint32_t m = __byte_perm(w, 0x64646464u, sel);
  const __half2 h = __hsub2(*reinterpret_cast<const __half2*>(&m), __floats2half2_rn(1024.f, 1024.f));
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint4 bytes8_to_f16(uint32_t w0, uint32_t w1) {
  // selector: result bytes = (src byte i, 0x64, src byte i+1, 0x64)
  uint4 o;
  o.x = bytes2h2(w0, 0x4140);
  o.y = bytes2h2(w0, 0x4342);
  o.z = bytes2h2(w1, 0x4140);
  o.w = bytes2h2(w1, 0x4342);
  return o;
}

struct TileCoord {
  int mt, nt, ks;        // tile indices (meaning is the policy's)
  int k_begin, k_end;    // reduction range of this work item (meaning is the policy's)
};

// Per-thread producer state that lives across the stages of one work item (e.g. the running
// column sums of the operand a producer streams through its registers anyway = a bias gradient).
struct PolicyBase {
  static constexpr int EPI_SETS = 1;
  // policy provides custom_epilogue(g, tc, res, taddr, row, pre, state): reads its accumulator row
  // (lane = row) and writes its output itself.  EpiPre = registers filled by epi_prefetch BEFORE the
  // accumulator is waited for (operands the finishing op needs from HBM); EpiState = per-thread
  // state that lives across the tiles of the CTA (epi_begin / epi_end), e.g. running column sums
  static constexpr bool CUSTOM_EPI = false;
  // CLUSTER > 1: the CTAs of a cluster work on split-K slices of ONE tile (one work item per CTA);
  // custom_epilogue leaves each CTA's partial in its own shared memory and, after a cluster
  // barrier, cluster_reduce (epilogue warps) combines them through distributed shared memory
  static constexpr int CLUSTER = 1;
  // MULTI_WAVE (CLUSTER > 1): still one work item per CTA, but the grid may exceed the SM count and
  // run in several waves of clusters (launch() does not clamp it)
  static constexpr bool MULTI_WAVE = false;
  template <class Args>
  static __device__ __forceinline__ void cluster_reduce(const Args&, uint8_t*, int, int) {}
  // CLUSTER_PHASES == 2: after another cluster barrier cluster_reduce2 (epilogue warps) may read what
  // the peers left in their shared memory during cluster_reduce
  static constexpr int CLUSTER_PHASES = 1;
  template <class Args>
  static __device__ __forceinline__ void cluster_reduce2(const Args&, uint8_t*, int, int) {}
  struct EpiPre {};
  struct EpiState {};
  template <class Args, class Pre>
  static __device__ __forceinline__ void epi_prefetch(const Args&, const TileCoord&, int, Pre&) {}
  template <class St>
  static __device__ __forceinline__ void epi_begin(St&) {}
  template <class Args, class St>
  static __device__ __forceinline__ void epi_end(const Args&, St&, int, int) {}
  template <class Args, class Pre, class St>
  static __device__ __forceinline__ void custom_epilogue(const Args&, const TileCoord&, const uint8_t*,
                                                         uint32_t, int, Pre&, St&) {}
  template <class Args>
  static __device__ __forceinline__ float* row_ptr(const Args&, const TileCoord&, int) { return nullptr; }
  static constexpr bool ACC_LIMBS3 = false;    // accumulators are 3 s32 limb sets (int8 path)
  static constexpr int SCALE_OFF = 0;          // byte offset of the 3 limb scales in resident smem
  // Operand data that needs no conversion is moved by cp.async.bulk: the hook runs after
  // load_stage; the lane that issues copies does mbarrier.arrive.expect_tx on `full` itself and
  // returns true (the framework then skips that lane's plain arrive).
  template <class Args>
  static __device__ __forceinline__ bool bulk_stage(const Args&, const TileCoord&, int, uint8_t*, int,
                                                    int, uint64_t*) { return false; }
  // A finishing operand that is laid out like the accumulator read-out (lane = row, 8 consecutive
  // columns = one 16-byte vector): loaded ahead of the accumulator wait, applied in registers
  static constexpr bool HAS_PRE = false;
  template <class Args>
  static __device__ __forceinline__ int64_t pre_row(const Args&, const TileCoord&, int) { return 0; }
  template <class Args>
  static __device__ __forceinline__ uint4 pre_load(const Args&, const TileCoord&, int64_t, int) {
    return make_uint4(0u, 0u, 0u, 0u);
  }
  static __device__ __forceinline__ void pre_apply(float (&)[8], const uint4&) {}
  static constexpr bool HAS_AUX = false;       // finish() needs an operand from HBM (bias, relu mask)
  static constexpr bool AUX_ROW_INVARIANT = true;   // ... that depends on the column only (bias)
  struct Prod {};
  // PROD_PER_CTA: Prod lives across all the items of the CTA (prod_begin before the first,
  // prod_end after the last, with a TileCoord whose ks = blockIdx.x) instead of one item
  static constexpr bool PROD_PER_CTA = false;
  // PERSIST_COLS > 0: a second accumulator of that many TMEM columns (after the NUM_ACC per-item
  // ones) that lives across all the items of the CTA.  issue() gets its address as a 7th argument;
  // the MMA warp commits it after the CTA's last stage, and the epilogue warps then read it out
  // once: persist_epilogue(g, taddr (lane quadrant of the warp), row, epilogue set)
  static constexpr int PERSIST_COLS = 0;
  template <class Args>
  static __device__ __forceinline__ void persist_epilogue(const Args&, uint32_t, int, int) {}
  template <class Pr>
  static __device__ __forceinline__ void prod_begin(Pr&) {}
  // PREFETCH: the producer requests the global data of its NEXT stage (into registers held in
  // Prod) right after it has handed the current one over, i.e. BEFORE it waits for that stage's
  // shared-memory slot to be free: the load latency runs behind the wait instead of after it
  static constexpr bool PREFETCH = false;
  template <class Args, class Pr>
  static __device__ __forceinline__ void prefetch_stage(const Args&, const TileCoord&, int, int, int, Pr&) {}
  template <class Args, class Pr>
  static __device__ __forceinline__ void prod_end(const Args&, const TileCoord&, Pr&, int, int) {}
  template <class Args>
  static __device__ __forceinline__ bool seg_valid(const Args&, const TileCoord&, int) { return true; }
  template <class Args>
  static __device__ __forceinline__ bool col_valid(const Args&, const TileCoord&, int) { return true; }
  template <class Args>
  static __device__ __forceinline__ int64_t seg_offset(const Args&, const TileCoord&, int) { return 0; }
  template <class Args>
  static __device__ __forceinline__ float4 aux_load(const Args&, const TileCoord&, const float*, int, int64_t) {
    return make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // per-row quantity the aux loads of a row share (computed once per row, kept in smem)
  template <class Args>
  static __device__ __forceinline__ int64_t row_aux(const Args&, const TileCoord&, int) { return 0; }
  template <class Args>
  static __device__ __forceinline__ float4 finish(const Args&, float4 v, float4) { return v; }
};

// A Policy (derived from PolicyBase) provides:
//   Args; PROD_WARPS (8 or 16); STAGES (2, 4 or 8); STAGE_BYTES; RES_BYTES (resident smem, e.g. converted weights);
//   ACC_COLS (TMEM columns of one accumulator set, multiple of 16)
//   OUT_COLS (logical output columns), acc_col(c) (TMEM column of output column c, c % 16 == 0),
//   LO_DELTA (> 0: output = acc[acc_col(c)] + acc[acc_col(c) + LO_DELTA]; the bf16 lo-part of the
//   B operand is CONCATENATED to its hi-part along N so that one MMA of width 2N replaces two of
//   width N -- the A tile is read from shared memory once instead of twice, which is what bounds
//   the narrow-N (16/32) convolutions: see DESIGN.md "L1 data pipe")
//   static __device__ int num_items(const Args&)
//   static __device__ TileCoord coord(const Args&, int item)
//   static __device__ int num_stages(const Args&, const TileCoord&)          stages per item
//   static __device__ void load_resident(const Args&, uint8_t* res, int ptid, int nthreads)
//   static __device__ void load_stage(const Args&, const TileCoord&, int s, uint8_t* stage,
//                                     int glane, int gsize, Prod&)   lanes of the stage's warp group
//   optional: Prod, prod_begin(Prod&), prod_end(Args, TileCoord, Prod&, producer warp, lane)
//             called by every producer thread before the first / after the last stage of an item
//   static __device__ void issue(const Args&, const TileCoord&, int s, uint32_t stage_addr,
//                                uint32_t res_addr, uint32_t d_tmem)   all MMAs of stage s
//                                (s == 0 must start with accumulate = 0)
//   epilogue: SEG (16 or 32 floats: contiguous output run of one row), NSEG = OUT_COLS / SEG,
//     static __device__ float* row_ptr(const Args&, const TileCoord&, int row)   nullptr = skip row
//     static __device__ bool seg_valid(const Args&, const TileCoord&, int sg)    (warp-uniform)
//     static __device__ int64_t seg_offset(const Args&, const TileCoord&, int sg) floats from row_ptr
//     static __device__ bool col_valid(const Args&, const TileCoord&, int col)
//     static __device__ float4 aux_load(const Args&, const TileCoord&, const float* dst, int col)
//     static __device__ float4 finish(const Args&, float4 acc, float4 aux)
//       col = sg*SEG + 4*j: the float4's first logical output column; aux = what the finishing
//       op needs from HBM (bias, relu mask), loaded ahead of the accumulator read-out
template <class P>
struct Smem {
  static constexpr int BAR_OFF = P::STAGES * P::STAGE_BYTES + P::RES_BYTES;
  static constexpr int EPI_OFF = BAR_OFF + 512;                 // up to 2*16 + 4 mbarriers + TMEM slot
  static constexpr int EPI_ROW = (P::SEG + 4) * 4;              // staged row, padded: conflict-free
  static constexpr int EPI_WARP = 32 * EPI_ROW + 32 * 8 + 32 * 8;   // staging + 32 row pointers + 32 row aux offsets
  // a custom epilogue writes its output itself and never touches the staging area
  static constexpr int TOTAL = EPI_OFF + (P::CUSTOM_EPI ? 0 : epi_warps<P>() * EPI_WARP);
};

template <class P>
__global__ void __launch_bounds__(cta_threads<P>(), 1) tc_kernel(typename P::Args g) {
  using S = Smem<P>;
  constexpr int STAGES = P::STAGES, WPS = P::PROD_WARPS / STAGES;  // producer warps per stage
  constexpr int kEpiWarps = epi_warps<P>();
  constexpr int kMmaWarp = kEpiWarps + P::PROD_WARPS;
  static_assert(P::PROD_WARPS % STAGES == 0, "producer warps must divide evenly over the stages");
  static_assert(STAGES >= 2 && STAGES <= 16, "STAGES");
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* res = smem + STAGES * P::STAGE_BYTES;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::BAR_OFF);
  uint64_t* empty = full + STAGES;
  // accumulator stages: one per epilogue set (at least two)
  constexpr int NUM_ACC = P::EPI_SETS > 2 ? P::EPI_SETS : 2;
  uint64_t* tfull = empty + STAGES;      // [NUM_ACC]
  uint64_t* tempty = tfull + NUM_ACC;    // [NUM_ACC]
  uint64_t* pfull = tempty + NUM_ACC;    // PERSIST_COLS > 0: the CTA-lifetime accumulator is final
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(pfull + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int kAccCols = NUM_ACC * P::ACC_COLS + P::PERSIST_COLS;
  constexpr uint32_t kTmemCols = kAccCols <= 32 ? 32 : kAccCols <= 64 ? 64 : kAccCols <= 128 ? 128
                               : kAccCols <= 256 ? 256 : 512;
  static_assert(kAccCols <= 512 && P::ACC_COLS % 16 == 0 && P::PERSIST_COLS % 16 == 0, "TMEM budget");
  static_assert(P::EPI_SETS == 1 || P::EPI_SETS == 2 || P::EPI_SETS == 4, "EPI_SETS");

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 32 * WPS);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < NUM_ACC; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], 128);
    }
    if (P::PERSIST_COLS > 0) mbar_init(pfull, 1);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_base_slot, kTmemCols);
  if (P::RES_BYTES > 0 && warp >= kEpiWarps && warp < kMmaWarp) {
    P::load_resident(g, res, tid - kEpiWarps * 32, prod_threads<P>());
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;
  const int items = P::num_items(g);
  // Programmatic dependent launch: everything above (barriers, TMEM, the resident weight image --
  // written by arl_prepare_weights, never by the kernel just before this one: arl_prepare_weights
  // builds the conv images first and ends with the fc256 splits) overlaps the tail of
  // the previous kernel in the stream; its results are touched only after the wait.  The next
  // kernel may begin its own prologue as soon as SMs free up.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  if (warp >= kEpiWarps && warp < kMmaWarp) {
    // ===================== producers: warp group pg owns stage pg =====================
    const int pw = warp - kEpiWarps;
    const int pg = pw / WPS, glane = (pw % WPS) * 32 + lane;
    uint8_t* st = smem + pg * P::STAGE_BYTES;
    int i = 0;                                         // running stage index over all items
    typename P::Prod ps;
    if (P::PROD_PER_CTA) P::prod_begin(ps);
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const TileCoord tc = P::coord(g, item);
      const int ns = P::num_stages(g, tc);
      if (!P::PROD_PER_CTA) P::prod_begin(ps);
      bool first = true;
      for (int s = 0; s < ns; ++s, ++i) {
        if (i % STAGES != pg) continue;
        if (P::PREFETCH && first) P::prefetch_stage(g, tc, s, glane, 32 * WPS, ps);
        first = false;
        mbar_wait_backoff<128>(&empty[pg], ((i / STAGES) & 1) ^ 1);
        P::load_stage(g, tc, s, st, glane, 32 * WPS, ps);
        fence_proxy_async_smem();        // generic-proxy stores -> visible to the MMA (async proxy)
        if (!P::bulk_stage(g, tc, s, st, glane, 32 * WPS, &full[pg])) mbar_arrive(&full[pg]);
        if (P::PREFETCH && s + STAGES < ns) P::prefetch_stage(g, tc, s + STAGES, glane, 32 * WPS, ps);
      }
      if (!P::PROD_PER_CTA) P::prod_end(g, tc, ps, pw, lane);
    }
    if (P::PROD_PER_CTA) {
      TileCoord cta{};
      cta.ks = blockIdx.x;
      P::prod_end(g, cta, ps, pw, lane);
    }
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer (one thread) =====================
    {                                                    // the whole warp, converged (see elect_one)
      int i = 0, k = 0;                                  // k = this CTA's running tile count
      const uint32_t res_addr = smem_u32(res);
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++k) {
        const TileCoord tc = P::coord(g, item);
        const int ns = P::num_stages(g, tc);
        const uint32_t acc = k % NUM_ACC, acc_phase = (k / NUM_ACC) & 1;
        mbar_wait_sleep(&tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * P::ACC_COLS;
        for (int s = 0; s < ns; ++s, ++i) {
          const int stage = i % STAGES;
          mbar_wait_sleep(&full[stage], (i / STAGES) & 1);
          tc_fence_after();
          if (elect_one()) {
            if constexpr (P::PERSIST_COLS > 0)
              P::issue(g, tc, s, smem_u32(smem + stage * P::STAGE_BYTES), res_addr, d_tmem,
                       tmem_base + NUM_ACC * P::ACC_COLS);
            else
              P::issue(g, tc, s, smem_u32(smem + stage * P::STAGE_BYTES), res_addr, d_tmem);
            umma_commit(&empty[stage]);      // frees the smem stage when these MMAs retire
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(&tfull[acc]);       // accumulator ready for the epilogue
        __syncwarp();
      }
      if (P::PERSIST_COLS > 0) {
        if (elect_one()) umma_commit(pfull);             // after the CTA's last stage
        __syncwarp();
      }
    }
  } else {
    // ===================== epilogue =====================
    constexpr int SEG = P::SEG, NSEG = P::OUT_COLS / SEG, LPR = SEG / 4, RPI = 32 / LPR;
    static_assert((SEG == 16 || SEG == 32) && P::OUT_COLS % SEG == 0, "SEG");
    uint8_t* ep = smem + S::EPI_OFF + warp * S::EPI_WARP;
    float* stg = reinterpret_cast<float*>(ep);
    float** rowp = reinterpret_cast<float**>(ep + 32 * S::EPI_ROW);
    int64_t* rowa = reinterpret_cast<int64_t*>(ep + 32 * S::EPI_ROW + 32 * 8);
    constexpr int NI = 32 / RPI;
    const int c4 = lane % LPR, rsub = lane / LPR, quad = warp & 3, set = warp >> 2;
    int k = 0;
    typename P::EpiState est;
    P::epi_begin(est);
    for (int item = blockIdx.x; item < items; item += gridDim.x, ++k) {
      if (P::EPI_SETS > 1 && (k % P::EPI_SETS) != set) continue;
      const uint32_t acc = k % NUM_ACC, acc_phase = (k / NUM_ACC) & 1;
      const TileCoord tc = P::coord(g, item);
      if constexpr (P::CUSTOM_EPI) {
        // the policy reads its accumulator row (lane = row) and writes its output itself
        typename P::EpiPre pre;
        P::epi_prefetch(g, tc, quad * 32 + lane, pre);
        mbar_wait_backoff<64>(&tfull[acc], acc_phase);
        tc_fence_after();
        P::custom_epilogue(g, tc, res, tmem_base + ((uint32_t)(quad * 32) << 16) + acc * P::ACC_COLS,
                           quad * 32 + lane, pre, est);
        tc_fence_before();
        mbar_arrive(&tempty[acc]);
        continue;
      }
      __syncwarp();
      rowp[lane] = P::row_ptr(g, tc, quad * 32 + lane);
      if (P::HAS_AUX && !P::AUX_ROW_INVARIANT) rowa[lane] = P::row_aux(g, tc, quad * 32 + lane);
      int64_t prow = 0;
      if constexpr (P::HAS_PRE) prow = P::pre_row(g, tc, quad * 32 + lane);
      __syncwarp();
      bool waited = false;
      // HAS_PRE: the whole tile's mask vectors are requested before the accumulator is waited for
      // (per-segment requests left three exposed load latencies per tile); the segment loop is
      // then fully unrolled so that they stay in registers
      uint4 pmall[P::HAS_PRE ? NSEG : 1][SEG / 8];
      if constexpr (P::HAS_PRE) {
#pragma unroll
        for (int sg = 0; sg < NSEG; ++sg) {
#pragma unroll
          for (int h = 0; h < SEG / 8; ++h) pmall[sg][h] = P::pre_load(g, tc, prow, sg * SEG + h * 8);
        }
      }
#pragma unroll(P::HAS_PRE ? NSEG : 1)
      for (int sg = 0; sg < NSEG; ++sg) {
        if (!P::seg_valid(g, tc, sg)) continue;
        // (1) destination of every float4 this lane will write + the operand its finishing op
        //     needs from HBM (relu mask / bias): issued BEFORE the accumulator is waited for, so
        //     the load latency hides behind the MMAs (first segment) / the TMEM read-out
        const int64_t soff = P::seg_offset(g, tc, sg) + c4 * 4;
        const bool cok = P::col_valid(g, tc, sg * SEG + c4 * 4);
        float4 aux[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          const float* base = rowp[i * RPI + rsub];
          aux[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (P::HAS_AUX && !P::AUX_ROW_INVARIANT && cok && base != nullptr)
            aux[i] = P::aux_load(g, tc, base + soff, sg * SEG + c4 * 4, rowa[i * RPI + rsub]);
        }
        if (P::HAS_AUX && P::AUX_ROW_INVARIANT && cok) {         // e.g. a bias: one load serves all rows
          const float4 a = P::aux_load(g, tc, nullptr, sg * SEG + c4 * 4, 0);
#pragma unroll
          for (int i = 0; i < NI; ++i) aux[i] = a;
        }
        if (!waited) {
          mbar_wait_backoff<64>(&tfull[acc], acc_phase);
          tc_fence_after();
          waited = true;
        }
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * P::ACC_COLS;
        // (2) TMEM -> registers (lane = row) -> staging
#pragma unroll
        for (int h = 0; h < SEG / 8; ++h) {
          float v[8];
          const int c = sg * SEG + h * 8;
          const uint32_t ta = taddr + P::acc_col(c & ~15) + (c & 15);
          if (P::ACC_LIMBS3) {
            const float* sc = reinterpret_cast<const float*>(res + P::SCALE_OFF);
            tmem_ld8_limbs3(ta, ta + P::LO_DELTA, ta + 2 * P::LO_DELTA, sc[0], sc[1], sc[2], v);
          } else if (P::LO_DELTA > 0) tmem_ld8_sum(ta, ta + P::LO_DELTA, v);
          else tmem_ld8(ta, v);
          if constexpr (P::HAS_PRE) P::pre_apply(v, pmall[sg][h]);
          float4* d = reinterpret_cast<float4*>(stg + lane * (SEG + 4) + h * 8);
          d[0] = make_float4(v[0], v[1], v[2], v[3]);
          d[1] = make_float4(v[4], v[5], v[6], v[7]);
        }
        __syncwarp();
        // (3) coalesced finish: LPR lanes cover one row's SEG floats, RPI rows per instruction
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          const float4 val = *reinterpret_cast<const float4*>(stg + (i * RPI + rsub) * (SEG + 4) + c4 * 4);
          float* base = rowp[i * RPI + rsub];
          if (cok && base != nullptr)
            *reinterpret_cast<float4*>(base + soff) = P::finish(g, val, aux[i]);
        }
        __syncwarp();
      }
      if (!waited) {
        mbar_wait_backoff<64>(&tfull[acc], acc_phase);
        tc_fence_after();
      }
      tc_fence_before();
      mbar_arrive(&tempty[acc]);
    }
    if constexpr (P::PERSIST_COLS > 0) {
      mbar_wait_backoff<64>(pfull, 0);
      tc_fence_after();
      P::persist_epilogue(g, tmem_base + ((uint32_t)(quad * 32) << 16) + NUM_ACC * P::ACC_COLS,
                          quad * 32 + lane, set);
    }
    P::epi_end(g, est, warp, lane);
  }

  if constexpr (P::CLUSTER > 1) {
    __syncwarp();                                        // (the MMA warp ran its loop on one lane)
    cluster_sync_all();                                  // every CTA's partial is in its shared memory
    if (warp < kEpiWarps) P::cluster_reduce(g, smem, warp, lane);
    cluster_sync_all();                                  // nobody reads a peer's shared memory after this
    if constexpr (P::CLUSTER_PHASES > 1) {
      if (warp < kEpiWarps) P::cluster_reduce2(g, smem, warp, lane);
      cluster_sync_all();                                // ... (second phase)
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

template <class P>
int launch(const typename P::Args& g, int items, cudaStream_t stream) {
  using S = Smem<P>;
  static_assert(S::TOTAL <= 227 * 1024, "smem budget");
  auto kern = tc_kernel<P>;
  // function attributes are per device: one flag per device index (a process may drive several
  // GPUs through arl_init(device)); racing host threads at worst set the attribute twice
  static std::atomic<uint64_t> attr_set{0};
  int dev = 0;
  ARL_CUDA(cudaGetDevice(&dev));
  const uint64_t bit = 1ull << (dev & 63);
  if (!(attr_set.load(std::memory_order_acquire) & bit)) {
    ARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    attr_set.fetch_or(bit, std::memory_order_release);
  }
  if (items <= 0) return ARL_OK;
  const int grid = items < num_sms() || (P::CLUSTER > 1 && P::MULTI_WAVE) ? items : num_sms();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(cta_threads<P>());
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (P::CLUSTER > 1) {
    if (items > grid || grid % P::CLUSTER != 0) {
      set_error("tc::launch: a cluster policy needs one work item per CTA and whole clusters (%d items)", items);
      return ARL_ERR_INVALID;
    }
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = P::CLUSTER;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.numAttrs = 2;
  }
  ARL_CUDA(cudaLaunchKernelEx(&cfg, kern, g));
  ARL_LAUNCH_CHECK("tc_kernel");
  return ARL_OK;
}

// ====================== GEMM on split-bf16 operands kept in HBM (fc256) ========================
// Every operand of the fc256 contractions lives in HBM already split into bf16 hi and lo parts, in
// 16-byte vectors of 8 consecutive columns ("chunks") with the ROWS contiguous:
//     xs[block][part (hi, lo)][chunk][row in block][8 bf16]          (same bytes as fp32 [rows][8*chunks])
// written that way by the kernel that produces the tensor (conv2 forward: a2, heads backward:
// d_h, arl_fc_prepare: l4_w).  A run of consecutive rows of one (part, chunk) is then one
// contiguous byte range AND one contiguous range of the UMMA no-swizzle operand image:
//   rows = the operand's M/N index, chunks over k  -> K-major image  (vector (r, kc) at kc*PLANE + r*16)
//   rows = k, chunks over the M/N index            -> MN-major image (vector (k, c)  at c*PLANE  + k*16)
// so the producers are cp.async.bulk copies (one elected lane per run, mbarrier complete_tx) and no
// operand byte crosses the LSU: the L1 data pipe carries only the tensor-core operand reads.
// Blocks: a tensor written by several launches (a2: one launch per env step) is a sequence of
// blocks of block_rows rows, each a complete [part][chunk][row] array.
enum { EPI_PLAIN = 0, EPI_BIAS_RELU = 1, EPI_MASK = 2 };

struct SplitMat {
  const uint8_t* base;
  int rows;          // total rows (all blocks)
  int block_rows;    // rows per block
  int chunks;        // 8-column chunks per row
};
__host__ __device__ __forceinline__ int64_t split_part_bytes(const SplitMat& m) {
  return (int64_t)m.chunks * m.block_rows * 16;
}
// rows [row0, row0 + cnt) of (part, chunk) -> cnt*16 contiguous bytes at dst
__device__ __forceinline__ void split_bulk_rows(uint8_t* dst, const SplitMat& m, int part, int chunk,
                                                int row0, int cnt, uint64_t* full) {
  const int64_t pb = split_part_bytes(m);
  int blk = row0 / m.block_rows, off = row0 - blk * m.block_rows;
  while (cnt > 0) {
    const int c = min(cnt, m.block_rows - off);
    const uint8_t* src = m.base + (int64_t)blk * 2 * pb + part * pb + ((int64_t)chunk * m.block_rows + off) * 16;
    bulk_g2s(dst, src, (uint32_t)c * 16u, full);
    dst += c * 16; cnt -= c; off = 0; ++blk;
  }
}

struct BulkGemmArgs {
  SplitMat A, B;       // K-major operand: rows = M (N) index; MN-major operand: rows = k
  SplitMat mask;       // EPI_MASK: split matrix [M rows][N columns]; output kept where its hi part > 0
  float* D;            // D[m*ldd + n]; split-K slice z writes D + z*M*ldd
  const float* bias;   // EPI_BIAS_RELU: bias[n]
  int M, N, K;
  int64_t ldd;
  int k_chunk, k_splits;   // K range per split-K slice (multiple of KB); ceil(K / k_chunk)
  int m_tiles, n_tiles;
};

// D[128 x NT] += A . B^T with the three bf16 products of the split:  A_hi.[B_hi | B_lo] as ONE MMA
// of width 2*NT (the lo image of B sits right behind its hi image along N) and A_lo.B_hi of
// width NT; output column c = acc[c] + acc[c + NT].
// CONCAT = false (NT up to 256): three MMAs of width NT into the same NT accumulator columns.
template <int NT, int KB_, bool A_MN, bool B_MN, int EPI, int STAGES_, bool CONCAT = true>
struct BulkGemm : PolicyBase {
  using Args = BulkGemmArgs;
  static constexpr int N_TILE = NT, KB = KB_, STAGES = STAGES_, PROD_WARPS = STAGES_;   // one warp per stage
  static constexpr int ACC_COLS = CONCAT ? 2 * NT : NT, OUT_COLS = NT, LO_DELTA = CONCAT ? NT : 0, SEG = 32;
  static constexpr bool HAS_AUX = EPI == EPI_BIAS_RELU, AUX_ROW_INVARIANT = true;
  static constexpr bool HAS_PRE = EPI == EPI_MASK;
  static constexpr int EPI_SETS = EPI == EPI_MASK ? 2 : 1;
  static __device__ __forceinline__ int acc_col(int c) { return c; }
  // stage = [A hi | A lo | B hi,lo]
  static constexpr int A_PLANE = A_MN ? KB * 16 : kTileM * 16;       // K-major: 128 rows; MN-major: KB k
  static constexpr int A_PART = kTileM * KB * 2;
  static constexpr int B_PLANE = B_MN ? KB * 16 : 2 * NT * 16;       // K-major: rows [hi NT | lo NT]
  static constexpr int B_OFF = 2 * A_PART;
  static constexpr int STAGE_BYTES = 2 * A_PART + 4 * NT * KB;
  static constexpr int RES_BYTES = 0;
  static constexpr int RA = A_MN ? kTileM / 8 : KB / 8, RB = B_MN ? NT / 8 : KB / 8;   // runs per part
  static constexpr int NRUN = 2 * (RA + RB);

  static __device__ __forceinline__ int num_items(const Args& g) { return g.m_tiles * g.n_tiles * g.k_splits; }
  static __device__ __forceinline__ TileCoord coord(const Args& g, int item) {
    TileCoord t;
    t.ks = item % g.k_splits;
    t.nt = (item / g.k_splits) % g.n_tiles;
    t.mt = item / (g.k_splits * g.n_tiles);
    t.k_begin = t.ks * g.k_chunk;
    t.k_end = min(g.K, t.k_begin + g.k_chunk);
    return t;
  }
  static __device__ __forceinline__ int num_stages(const Args&, const TileCoord& t) {
    return (t.k_end - t.k_begin + KB - 1) / KB;
  }
  static __device__ __forceinline__ void load_resident(const Args&, uint8_t*, int, int) {}

  // the part of the stage no copy will fill and the MMA reduces over: k >= the end of the K range
  static __device__ __forceinline__ void load_stage(const Args&, const TileCoord& t, int s, uint8_t* st,
                                                    int glane, int gsize, Prod&) {
    const int kvalid = t.k_end - (t.k_begin + s * KB);
    if (kvalid >= KB) return;
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    if (A_MN) {
      const int nk = KB - kvalid;
      for (int i = glane; i < 2 * RA * nk; i += gsize)
        *reinterpret_cast<uint4*>(st + (i / nk) * A_PLANE + (kvalid + i % nk) * 16) = z;
    } else {
      const int c0 = (kvalid + 7) / 8, nc = KB / 8 - c0;          // a partly valid chunk is copied (its tail is zero in HBM)
      for (int i = glane; i < 2 * nc * kTileM; i += gsize) {
        const int part = i / (nc * kTileM), r = i % (nc * kTileM);
        *reinterpret_cast<uint4*>(st + part * A_PART + c0 * A_PLANE + r * 16) = z;
      }
    }
    if (B_MN) {
      const int nk = KB - kvalid;
      for (int i = glane; i < 2 * RB * nk; i += gsize)
        *reinterpret_cast<uint4*>(st + B_OFF + (i / nk) * B_PLANE + (kvalid + i % nk) * 16) = z;
    } else {
      const int c0 = (kvalid + 7) / 8, nc = KB / 8 - c0;
      for (int i = glane; i < nc * 2 * NT; i += gsize)
        *reinterpret_cast<uint4*>(st + B_OFF + c0 * B_PLANE + i * 16) = z;
    }
  }
  // run -> (matrix, part, chunk, first row, rows, byte offset in the stage); rows <= 0: nothing to copy
  struct Run { const SplitMat* m; int part, chunk, row0, cnt, dst; };
  static __device__ __forceinline__ Run run_of(const Args& g, const TileCoord& t, int k0, int kvalid, int run) {
    Run r;
    if (run < 2 * RA) {
      const int c = run % RA;
      r.m = &g.A; r.part = run / RA;
      if (A_MN) {
        r.chunk = t.mt * (kTileM / 8) + c; r.row0 = k0; r.cnt = r.chunk * 8 < g.M ? kvalid : 0;
      } else {
        r.chunk = k0 / 8 + c; r.row0 = t.mt * kTileM; r.cnt = c * 8 < kvalid ? min(kTileM, g.M - r.row0) : 0;
      }
      r.dst = r.part * A_PART + c * A_PLANE;
    } else {
      const int q = run - 2 * RA, c = q % RB;
      r.m = &g.B; r.part = q / RB;
      if (B_MN) {
        r.chunk = t.nt * (NT / 8) + c; r.row0 = k0; r.cnt = r.chunk * 8 < g.N ? kvalid : 0;
        r.dst = B_OFF + (r.part * (NT / 8) + c) * B_PLANE;
      } else {
        r.chunk = k0 / 8 + c; r.row0 = t.nt * NT; r.cnt = c * 8 < kvalid ? min(NT, g.N - r.row0) : 0;
        r.dst = B_OFF + c * B_PLANE + r.part * NT * 16;
      }
    }
    return r;
  }
  static __device__ __forceinline__ bool bulk_stage(const Args& g, const TileCoord& t, int s, uint8_t* st,
                                                    int glane, int gsize, uint64_t* full) {
    if (glane >= NRUN) return false;
    const int k0 = t.k_begin + s * KB, kvalid = min(KB, t.k_end - k0);
    uint32_t bytes = 0;
    for (int run = glane; run < NRUN; run += gsize) {
      const Run r = run_of(g, t, k0, kvalid, run);
      bytes += r.cnt > 0 ? (uint32_t)r.cnt * 16u : 0u;
    }
    mbar_expect_tx(full, bytes);
    for (int run = glane; run < NRUN; run += gsize) {
      const Run r = run_of(g, t, k0, kvalid, run);
      if (r.cnt > 0) split_bulk_rows(st + r.dst, *r.m, r.part, r.chunk, r.row0, r.cnt, full);
    }
    return true;
  }
  static __device__ __forceinline__ void issue(const Args&, const TileCoord&, int s, uint32_t st, uint32_t,
                                               uint32_t d_tmem) {
    constexpr uint32_t idesc2 = make_idesc(CONCAT ? 2 * NT : NT, A_MN, B_MN), idesc1 = make_idesc(NT, A_MN, B_MN);
    // one descriptor derivation per stage and operand image; every MMA advances them by constants
    const uint64_t da_hi0 = A_MN ? make_sdesc(st, 128, A_PLANE) : make_sdesc(st, A_PLANE);
    const uint64_t db0 = B_MN ? make_sdesc(st + B_OFF, 128, B_PLANE) : make_sdesc(st + B_OFF, B_PLANE);
#pragma unroll
    for (int k16 = 0; k16 < KB / 16; ++k16) {
      const uint32_t aoff = A_MN ? k16 * 256 : k16 * 2 * A_PLANE;
      const uint32_t boff = B_MN ? k16 * 256 : k16 * 2 * B_PLANE;
      const uint64_t da_hi = sdesc_advance(da_hi0, aoff);
      const uint64_t da_lo = sdesc_advance(da_hi0, aoff + A_PART);
      const uint64_t db = sdesc_advance(db0, boff);
      if (CONCAT) {
        umma_f16(d_tmem, da_hi, db, idesc2, (s | k16) != 0 ? 1u : 0u);   // a_hi . [b_hi | b_lo]
        umma_f16(d_tmem, da_lo, db, idesc1, 1u);                          // a_lo . b_hi
      } else {
        // the lo image follows the hi image
        const uint64_t db_lo = sdesc_advance(db0, boff + (B_MN ? (NT / 8) * B_PLANE : NT * 16));
        umma_f16(d_tmem, da_hi, db, idesc1, (s | k16) != 0 ? 1u : 0u);   // a_hi . b_hi
        umma_f16(d_tmem, da_hi, db_lo, idesc1, 1u);                       // a_hi . b_lo
        umma_f16(d_tmem, da_lo, db, idesc1, 1u);                          // a_lo . b_hi
      }
    }
  }
  // ---- epilogue: row m of the tile is NT contiguous floats of D
  static __device__ __forceinline__ float* row_ptr(const Args& g, const TileCoord& t, int row) {
    const int m = t.mt * kTileM + row;
    if (m >= g.M) return nullptr;
    return g.D + (int64_t)t.ks * g.M * g.ldd + (int64_t)m * g.ldd + t.nt * NT;
  }
  static __device__ __forceinline__ bool seg_valid(const Args& g, const TileCoord& t, int sg) {
    return t.nt * NT + sg * SEG < g.N;
  }
  static __device__ __forceinline__ int64_t seg_offset(const Args&, const TileCoord&, int sg) { return sg * SEG; }
  static __device__ __forceinline__ bool col_valid(const Args& g, const TileCoord& t, int col) {
    return t.nt * NT + col < g.N;
  }
  static __device__ __forceinline__ float4 aux_load(const Args& g, const TileCoord& t, const float*, int col,
                                                    int64_t) {
    return ldg4(g.bias + t.nt * NT + col);
  }
  static __device__ __forceinline__ float4 finish(const Args&, float4 o, float4 x) {
    if (EPI == EPI_BIAS_RELU) {
      o.x = fmaxf(o.x + x.x, 0.f); o.y = fmaxf(o.y + x.y, 0.f);
      o.z = fmaxf(o.z + x.z, 0.f); o.w = fmaxf(o.w + x.w, 0.f);
    }
    return o;
  }
  // relu mask, applied in the lane = row arrangement of the TMEM read-out: 8 consecutive columns
  // = one chunk = one 16-byte vector of the mask's hi part; a warp reads 512 contiguous bytes
  static __device__ __forceinline__ int64_t pre_row(const Args& g, const TileCoord& t, int row) {
    const int m = t.mt * kTileM + row;
    if (m >= g.M) return -1;
    const int blk = m / g.mask.block_rows, off = m - blk * g.mask.block_rows;
    return (int64_t)blk * 2 * split_part_bytes(g.mask) + (int64_t)off * 16;
  }
  static __device__ __forceinline__ uint4 pre_load(const Args& g, const TileCoord& t, int64_t prow, int col) {
    const int n = t.nt * NT + col;
    if (prow < 0 || n >= g.N) return make_uint4(0u, 0u, 0u, 0u);
    return __ldg(reinterpret_cast<const uint4*>(g.mask.base + prow + (int64_t)(n >> 3) * g.mask.block_rows * 16));
  }
  static __device__ __forceinline__ void pre_apply(float (&v)[8], const uint4& m) {
    const uint32_t w[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if ((int16_t)(w[i] & 0xFFFFu) <= 0) v[2 * i] = 0.f;          // bf16 > 0  <=>  its bits as int16 > 0
      if ((int32_t)w[i] < 0x10000) v[2 * i + 1] = 0.f;
    }
  }
};

}  // namespace tc

// Launch a BulkGemm instance on g (M, N, K, operands, D filled in): k_splits split-K slices over K,
// slice z writing D + z*M*ldd
template <class P>
int run_gemm(tc::BulkGemmArgs& g, int k_splits, cudaStream_t st) {
  if (k_splits < 1) k_splits = 1;
  g.k_chunk = ((g.K + k_splits - 1) / k_splits + P::KB - 1) / P::KB * P::KB;
  g.k_splits = (g.K + g.k_chunk - 1) / g.k_chunk;
  g.m_tiles = (g.M + tc::kTileM - 1) / tc::kTileM;
  g.n_tiles = (g.N + P::N_TILE - 1) / P::N_TILE;
  return tc::launch<P>(g, g.m_tiles * g.n_tiles * g.k_splits, st);
}

inline tc::SplitMat mat(const void* base, int rows, int block_rows, int chunks) {
  tc::SplitMat m;
  m.base = (const uint8_t*)base; m.rows = rows; m.block_rows = block_rows; m.chunks = chunks;
  return m;
}

}  // namespace arl
