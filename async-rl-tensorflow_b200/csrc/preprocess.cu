// K1: Environment.screen (src/environment.py:49-53) fused with History.add
// (src/history.py:13-15).  u8 [B,210,160,3] -> luma (the reference's float64
// expression, truncated) -> cv2 INTER_LINEAR 84x84 (fixed point) -> ring slot.
//
// Layout / data flow per frame (one persistent CTA per SM, every compute warp a 2-stage bulk-copy pipeline):
//   HBM --cp.async.bulk (43 copies: the 168 source rows cv2 actually reads; L2 evict_first up to 8192 frames)--> smem raw[stage]
//   raw --luma, 8 px / lane-iteration, dp2a--> smem Y [168][160] u8 (8 rows private to a warp)
//   Y   --dp2a x taps, packed vertical terms--> smem out[ob] [84*84] u8 --cp.async.bulk--> ring[b][slot]
// Algorithmic HBM bytes per frame: 80 640 read + 7 056 written (x replicate).
//
// Luma: the reference computes (0.2126*R + 0.7152*G) + 0.0722*B in float64 and truncates.
// That equals floor((2126R+7152G+722B)/10000) except on 774 of the 3384 triples whose
// exact value is an integer, where float64 rounding lands one ulp below (white -> 254).
// For a given (R,G) at most one B in 0..255 makes the sum a multiple of 10000
// (722B mod 10000 has period 5000), so a 65536-bit bitmap indexed by (G,R) says "subtract
// one when the remainder is 0".  arl_init derives that bitmap on the device with IEEE
// __dmul_rn/__dadd_rn (never contracted to FMA) -- i.e. from the reference's own expression.
#include "common.cuh"

namespace arl {

constexpr int kH = ARL_FRAME_H, kW = ARL_FRAME_W, kS = ARL_SCREEN;
constexpr int kRowBytes = kW * 3;                 // 480
constexpr int kPairBytes = 2 * kRowBytes;         // 960: source rows sy, sy+1
constexpr int kRawBytes = kS * kPairBytes;        // 80640 per frame
constexpr int kYBytes = 2 * kS * kW;              // 26880
constexpr int kFrameBytes = kH * kW * 3;          // 100800
constexpr int kBitmapWords = 65536 / 32;          // 2048

constexpr int kPer = 21, kSeg = 40;                // x taps repeat every 21 outputs <-> 40 source pixels
__host__ __device__ constexpr int tap_sx(int d) { return (80 * d + 19) / 42; }   // floor((d+.5)*160/84 - .5)
struct TapTables {
  uint32_t x[kS];      // sx | c0 << 8 | c1 << 20   (sx must be tap_sx(d), c periodic in 21: checked at init)
  uint32_t y[kS];      // sy | b0 << 8 | b1 << 20   (sy must be 0,3,5,8,...: checked at init)
  uint32_t xc[kPer];   // c0 | c1 << 16 of output column r (mod 21): the dp2a coefficient pair
};
__constant__ TapTables c_taps;
__device__ uint32_t g_luma_fix[kBitmapWords];
static bool g_ready[64] = {};

// ---- init: derive the luma correction bitmap from the reference's float64 expression ----
__global__ void luma_fix_init_kernel() {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // idx = G*256 + R
  if (idx >= 65536) return;
  const int R = idx & 255, G = idx >> 8;
  for (int B = 0; B < 256; ++B) {
    const int s = 2126 * R + 7152 * G + 722 * B;
    if (s % 10000 != 0) continue;
    const double y = __dadd_rn(__dadd_rn(__dmul_rn(0.2126, (double)R), __dmul_rn(0.7152, (double)G)),
                               __dmul_rn(0.0722, (double)B));
    const int yt = (int)y;                                   // truncation, as astype(uint8)
    if (yt != s / 10000) atomicOr(&g_luma_fix[idx >> 5], 1u << (idx & 31));
  }
}

// cv2 INTER_LINEAR tap table for one axis (same float32 arithmetic as cv2's resize()).
static void linear_taps(int src, int dst, uint32_t* packed) {
  const double scale = 1.0 / ((double)dst / (double)src);
  for (int d = 0; d < dst; ++d) {
    float fx = (float)((d + 0.5) * scale - 0.5);
    int sx = (int)floorf(fx);
    fx -= (float)sx;
    if (sx < 0) { fx = 0.f; sx = 0; }
    if (sx >= src - 1) { fx = 0.f; sx = src - 1; }
    const int c0 = (int)lrintf((1.f - fx) * 2048.f);   // cvRound: half to even
    const int c1 = (int)lrintf(fx * 2048.f);
    packed[d] = (uint32_t)sx | ((uint32_t)c0 << 8) | ((uint32_t)c1 << 20);
  }
}

// ---- the kernel --------------------------------------------------------------------------
// One persistent CTA per SM: 21 compute warps + a store warp, no block-wide barrier in the loop.
//   compute warp w owns 4 output rows and is its own load pipeline: 43 cp.async.bulk loads per
//                 frame in all (the 168 source rows cv2 reads: rows 5k+2 are never touched; rows
//                 5k+3 .. 5k+6 are contiguous, so one 1920-B copy feeds two output rows), each
//                 into the private slice of raw[stage] of the warp that consumes it, behind that
//                 warp's own mbarrier; luma of its 8 source rows (160 groups of 8 px = 5 full warp
//                 iterations) into its private Y slice, then its 4 x 84 outputs.
//   store warp  : the 7056-B plane store(s) out[ob] -> ring (out_full/out_empty mbarriers).
constexpr int kComputeWarps = kS / 4;                       // 21
// Up to this many frames per launch K1 loads them with an L2 evict_first policy.  The forward
// kernels before it leave ~100 MB of dirty lines in the 126 MB L2 whatever the batch; streaming the
// frames past them moves that write-back into the forward kernels, which have DRAM bandwidth to
// spare.  On a B200 at 1000 W: 82 -> 71 us per launch at 4096 frames, 137 -> 129 us at 8192.  At
// 16 384 frames the hint cost K1 1-4 us per launch at t_max 20 on a power-capped card (268 -> 271 us,
// cycle +0.4 %), so launches that long load as before.  DESIGN.md §3.1.
constexpr int kK1EvictFirstMaxEnvs = 8192;
constexpr int kK1Threads = (kComputeWarps + 1) * 32;        // 704

struct __align__(16) K1Smem {
  uint8_t raw[2][kRawBytes];
  uint8_t Y[kYBytes];
  uint8_t out[2][kPlane];
  uint32_t fix[kBitmapWords];
  uint64_t full[2][kComputeWarps], out_full[2], out_empty[2];
};

// luma of 8 pixels (24 bytes = words w[0..5]) -> two packed words.  Branch-free common path, ~6
// instructions per pixel: 8 s = 8 (2126 R + 7152 G + 722 B) with two dp2a (16-bit coefficient x
// byte, taken from whichever words hold the pixel's bytes -- no byte shuffling), then ONE
// multiply-high h = (8 s * ceil(2^48 / 80000)) >> 32 = floor(s * 2^16 / 10000) (checked for every
// s <= 2 550 000): byte 2 of h is s / 10000 and the low 16 bits are zero exactly when s is a
// multiple of 10000.  The 8 zero tests are OR-ed and branched on ONCE; only then (1 group in ~600)
// the correction bitmap is consulted (774 of the 3384 exact-multiple triples need the -1).  The
// quotient bytes are gathered with byte permutes.
// The four coefficient words (x 8): KA = (2126, 7152), KB = (722, 0), KC = (0, 2126), KD = (7152, 722)
// as (low half, high half); dp2a_lo pairs them with bytes (b0, b1) of a word, dp2a_hi with (b2, b3).
struct LumaCoef { uint32_t ka, kb, kc, kd; };
__device__ __forceinline__ LumaCoef luma_coef() {
  LumaCoef k;      // opaque to constant propagation: stays in registers instead of a UMOV per use
  asm volatile("mov.u32 %0, 0xDF804270;" : "=r"(k.ka));
  asm volatile("mov.u32 %0, 0x00001690;" : "=r"(k.kb));
  asm volatile("mov.u32 %0, 0x42700000;" : "=r"(k.kc));
  asm volatile("mov.u32 %0, 0x1690DF80;" : "=r"(k.kd));
  return k;
}
// 4 pixels = 12 bytes = words a, b, c -> their sums (x 8)
__device__ __forceinline__ void luma_sums4(uint32_t a, uint32_t b, uint32_t c, const LumaCoef& k,
                                           uint32_t (&s)[4]) {
  s[0] = __dp2a_hi(k.kb, a, __dp2a_lo(k.ka, a, 0u));          // bytes a0 a1 a2
  s[1] = __dp2a_lo(k.kd, b, __dp2a_hi(k.kc, a, 0u));          // bytes a3 b0 b1
  s[2] = __dp2a_lo(k.kb, c, __dp2a_hi(k.ka, b, 0u));          // bytes b2 b3 c0
  s[3] = __dp2a_hi(k.kd, c, __dp2a_lo(k.kc, c, 0u));          // bytes c1 c2 c3
}
__device__ __forceinline__ uint2 luma_8px(const uint32_t (&w)[6], const LumaCoef& k, const uint32_t* fix) {
  uint32_t h[8];
  {
    uint32_t lo4[4], hi4[4];
    luma_sums4(w[0], w[1], w[2], k, lo4);
    luma_sums4(w[3], w[4], w[5], k, hi4);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      h[i] = __umulhi(lo4[i], 3518437209u);                   // floor(s * 2^16 / 10000)
      h[4 + i] = __umulhi(hi4[i], 3518437209u);
    }
  }
  const uint32_t any0 = ((h[0] & 0xFFFFu) == 0) | ((h[1] & 0xFFFFu) == 0) | ((h[2] & 0xFFFFu) == 0) |
                        ((h[3] & 0xFFFFu) == 0) | ((h[4] & 0xFFFFu) == 0) | ((h[5] & 0xFFFFu) == 0) |
                        ((h[6] & 0xFFFFu) == 0) | ((h[7] & 0xFFFFu) == 0);
  if (__builtin_expect(any0 != 0, 0)) {
    // G*256 + R of the 8 pixels (R, G = the first two of a pixel's three bytes)
    const uint32_t rg[8] = {w[0] & 0xFFFFu, __byte_perm(w[0], w[1], 0x7743) & 0xFFFFu, w[1] >> 16,
                            (w[2] >> 8) & 0xFFFFu,
                            w[3] & 0xFFFFu, __byte_perm(w[3], w[4], 0x7743) & 0xFFFFu, w[4] >> 16,
                            (w[5] >> 8) & 0xFFFFu};
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((h[i] & 0xFFFFu) == 0) h[i] -= ((fix[rg[i] >> 5] >> (rg[i] & 31)) & 1u) << 16;
  }
  // byte 2 of each h
  return make_uint2(__byte_perm(__byte_perm(h[0], h[1], 0x0062), __byte_perm(h[2], h[3], 0x0062), 0x5410),
                    __byte_perm(__byte_perm(h[4], h[5], 0x0062), __byte_perm(h[6], h[7], 0x0062), 0x5410));
}

// kEvictFirst: the frame loads carry an L2 evict_first policy (arl_preprocess_push picks it by batch size)
template <bool kEvictFirst>
__global__ void __launch_bounds__(kK1Threads, 1)
preprocess_kernel(const uint8_t* __restrict__ frames, uint8_t* __restrict__ ring, int num_envs,
                  int ring_slots, int slot, int replicate) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  K1Smem& sm = *reinterpret_cast<K1Smem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  const int frames_here = num_envs > (int)blockIdx.x ? (num_envs - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  // A compute warp's load barriers are private to it: lane 0 initialises them and issues the
  // copies of its first two frames before anything else happens in the CTA (the 8-KB correction
  // bitmap and the output barriers are set up while those copies are in flight).
  // The frames are read once per step: evict_first lets their stream pass through L2 without
  // evicting the previous kernels' dirty lines (whose write-back would then fall into this kernel)
  // or the ring planes the next kernel reads.
  auto issue_loads = [&](int f) {                               // lane 0 of a compute warp only
    const int stage = f & 1;
    uint64_t* bar = &sm.full[stage][warp];
    mbar_expect_tx(bar, 4 * kPairBytes);
    const uint64_t once = kEvictFirst ? l2_policy_evict_first() : 0;
    auto load = [&](uint8_t* dst, const uint8_t* src, uint32_t bytes) {
      if (kEvictFirst) bulk_g2s_hint(dst, src, bytes, bar, once);
      else bulk_g2s(dst, src, bytes, bar);
    };
    const uint8_t* src = frames + (size_t)(blockIdx.x + (size_t)f * gridDim.x) * kFrameBytes;
    uint8_t* dst = sm.raw[stage] + warp * (4 * kPairBytes);
    load(dst, src + (10 * warp + 3) * kRowBytes, 2 * kPairBytes);
    if (warp < kComputeWarps - 1) {
      load(dst + 2 * kPairBytes, src + (10 * warp + 8) * kRowBytes, 2 * kPairBytes);
    } else {
      load(dst + 2 * kPairBytes, src + (kH - 2) * kRowBytes, kPairBytes);
      load(dst + 3 * kPairBytes, src, kPairBytes);
    }
  };
  if (warp < kComputeWarps && lane == 0) {
    mbar_init(&sm.full[0][warp], 1);
    mbar_init(&sm.full[1][warp], 1);
    fence_mbar_init();
  }
  if (tid == kK1Threads - 1) {
    for (int k = 0; k < 2; ++k) {
      mbar_init(&sm.out_full[k], kComputeWarps);
      mbar_init(&sm.out_empty[k], 1);
    }
    fence_mbar_init();
  }
  for (int i = tid; i < kBitmapWords; i += kK1Threads) sm.fix[i] = g_luma_fix[i];
  // launched programmatically: the barriers and the correction bitmap (static data) are set up
  // while the kernel before this one is still running; the frames (whoever produced them) and the
  // ring are touched only after it has completed
  pdl_wait();
  if (warp < kComputeWarps && lane == 0) {
    if (frames_here > 0) issue_loads(0);
    if (frames_here > 1) issue_loads(1);
  }
  __syncthreads();
  // the next kernel in the stream (conv1 forward, launched with programmatic stream serialization)
  // may run its prologue on SMs this kernel has left; it waits for this grid before reading the ring
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp == kComputeWarps) {
    // ===================== store warp =====================
    if (lane == 0) {
      for (int g = 0; g < frames_here; ++g) {
        const int ob = g & 1;
        mbar_wait_sleep(&sm.out_full[ob], (g >> 1) & 1);
        uint8_t* dst = ring + ((size_t)(blockIdx.x + (size_t)g * gridDim.x) * ring_slots) * kPlane;
        for (int r = 0; r < replicate; ++r) {
          int sl = slot + r;
          if (sl >= ring_slots) sl -= ring_slots;
          bulk_s2g(dst + (size_t)sl * kPlane, sm.out[ob], kPlane);
        }
        bulk_commit();
        bulk_wait_read<0>();                                 // smem has been read: buffer reusable
        mbar_arrive(&sm.out_empty[ob]);
      }
      bulk_wait<0>();
    }
    return;
  }

  // ===================== compute warps =====================
  // Warp w owns output rows dy = 4w+1 .. 4w+4 (warp 20: 81, 82, 83, 0).  Their source rows are its
  // private slice of a raw stage, fetched by the warp's own two copies (rows 10w+3 .. 10w+6 and
  // 10w+8 .. 10w+11, 1920 B each; warp 20: rows 203-206, 208-209 and 0-1) and refilled for frame
  // f+2 the moment its phase A of frame f is done -- no warp ever waits for another warp's data.
  // phase B lane roles: lane = ry*8 + s*4 + m handles source row 2*ry + s of the warp's Y slice and
  // output columns 21 m .. 21 m + 20, whose taps lie in the row's bytes 40 m .. 40 m + 39 at
  // compile-time offsets (the x taps repeat every 21 outputs <-> 40 source pixels).
  const int ry = lane >> 3, srow = (lane >> 2) & 1, m = lane & 3;
  int dy = 4 * warp + 1 + ry;
  if (dy >= kS) dy -= kS;
  uint32_t bw;                                                  // this lane's vertical weight
  {
    const uint32_t yt = c_taps.y[dy];
    bw = srow ? (yt >> 20) : ((yt >> 8) & 0xFFFu);
  }
  const uint32_t sh = srow ? 18u : 2u;                          // lane s stores outputs 2k + s
  // ring planes are stored in 4x4 blocks (space-to-depth): byte (y,x) of the screen sits at
  // ((y/4)*21 + x/4)*16 + (y%4)*4 + x%4, so conv1's 8x8-stride-4 windows are 16-B vectors.
  // x = 21 m + s + 2k = 20 m + q, q = q0 + 2k: offset(k) = base + 16*((q0 + 2k) / 4) + (q0 + 2k) % 4
  //   = addr[k & 1] + 16 * (k / 2)
  uint32_t oaddr[2];
  {
    const int q0 = m + srow, base = ((dy >> 2) * 21 + 5 * m) * 16 + (dy & 3) * 4;
    oaddr[0] = base + (q0 >> 2) * 16 + (q0 & 3);
    oaddr[1] = base + ((q0 + 2) >> 2) * 16 + ((q0 + 2) & 3);
  }
  uint8_t* Yw = sm.Y + warp * (8 * kW);
  const uint2* seg = reinterpret_cast<const uint2*>(Yw + lane * kSeg);   // (2 ry + s) * 160 + 40 m
  const LumaCoef coef = luma_coef();
  for (int f = 0; f < frames_here; ++f) {
    const int stage = f & 1, ob = f & 1;
    mbar_wait_sleep(&sm.full[stage][warp], (f >> 1) & 1);
    // phase A: luma of this warp's 8 source rows, 8 pixels (24 B) per lane-iteration
    const uint2* raw2 = reinterpret_cast<const uint2*>(sm.raw[stage] + warp * (4 * kPairBytes));
#pragma unroll
    for (int it = 0; it < 5; ++it) {
      const int u = it * 32 + lane;
      const uint2 a = raw2[3 * u], b = raw2[3 * u + 1], c = raw2[3 * u + 2];
      const uint32_t w[6] = {a.x, a.y, b.x, b.y, c.x, c.y};
      reinterpret_cast<uint2*>(Yw)[u] = luma_8px(w, coef, sm.fix);
    }
    __syncwarp();
    if (lane == 0 && f + 2 < frames_here) issue_loads(f + 2);   // the slice has been read: refill it
    // phase B: cv2 fixed-point bilinear.  Horizontal pass of one source row: 21 dp2a sums
    // h = c0 Y[sx] + c1 Y[sx+1]; vertical weight applied to pairs of them; the partner row's terms
    // arrive with one shuffle per pair; ((t0 + t1 + 2) >> 2) on both 16-bit halves at once.
    uint32_t yw[10];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const uint2 v = seg[i];
      yw[2 * i] = v.x;
      yw[2 * i + 1] = v.y;
    }
    uint32_t term[kPer + 1];
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
      const int sx = tap_sx(r), k = sx >> 2, o = sx & 3;        // compile-time after unrolling
      uint32_t h;
      if (o == 0) h = __dp2a_lo(c_taps.xc[r], yw[k], 0u);
      else if (o == 2) h = __dp2a_hi(c_taps.xc[r], yw[k], 0u);
      else if (o == 1) h = __dp2a_lo(c_taps.xc[r], yw[k] >> 8, 0u);
      else h = __dp2a_lo(c_taps.xc[r], __funnelshift_r(yw[k], yw[k + 1 < 10 ? k + 1 : 9], 24), 0u);
      term[r] = (h >> 4) * bw;                                  // < 2^26; its bits 16.. are the cv2 term
    }
    term[kPer] = 0;
    mbar_wait(&sm.out_empty[ob], ((f >> 1) & 1) ^ 1);
    uint8_t* out = sm.out[ob];
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const uint32_t mine = __byte_perm(term[2 * k], term[2 * k + 1], 0x7632);   // (t[2k] >> 16) | (t[2k+1] >> 16) << 16
      const uint32_t sum = mine + __shfl_xor_sync(0xFFFFFFFFu, mine, 4) + 0x00020002u;
      if (k < 10 || srow == 0) out[oaddr[k & 1] + 16 * (k >> 1)] = (uint8_t)(sum >> sh);
    }
    fence_proxy_async_smem();                                   // generic writes -> bulk store
    __syncwarp();
    if (lane == 0) mbar_arrive(&sm.out_full[ob]);
  }
}

// ---- the other branch of environment.py:5-12: scipy.misc.imresize = PIL BILINEAR ------------
// Pillow's 8-bit resize (ImagingResample): antialiased triangle filter with support = scale,
// coefficients int(0.5 + w * 2^22) of the double weights normalised to sum 1, accumulator seeded
// with 2^21, >> 22, clip; horizontal pass to u8 [210][84] first, then the vertical pass.
// This branch reads every source row.  One CTA per frame, phases separated by __syncthreads: it is
// the optional mode (resize='pil'); the executed reference takes the cv2 branch above.
constexpr int kPilMaxTaps = 8;
struct PilTaps {
  int xmin[kS], xn[kS], xk[kS][kPilMaxTaps];     // horizontal: 160 -> 84
  int ymin[kS], yn[kS], yk[kS][kPilMaxTaps];     // vertical:   210 -> 84
};
__device__ PilTaps g_pil;

static bool pil_coeffs(int src, int dst, int* mn, int* cnt, int (*k)[kPilMaxTaps]) {
  const double scale = (double)src / (double)dst;
  const double filterscale = scale < 1.0 ? 1.0 : scale;
  const double support = 1.0 * filterscale;
  for (int i = 0; i < dst; ++i) {
    const double center = (i + 0.5) * scale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > src) xmax = src;
    const int n = xmax - xmin;
    if (n > kPilMaxTaps) return false;
    double w[kPilMaxTaps], tot = 0.0;
    for (int j = 0; j < n; ++j) {
      double x = (j + xmin - center + 0.5) / filterscale;
      if (x < 0) x = -x;
      w[j] = x < 1.0 ? 1.0 - x : 0.0;
      tot += w[j];
    }
    for (int j = 0; j < kPilMaxTaps; ++j) k[i][j] = 0;
    for (int j = 0; j < n; ++j) {
      const double v = tot != 0.0 ? w[j] / tot : w[j];
      k[i][j] = v >= 0 ? (int)(0.5 + v * 4194304.0) : (int)(-0.5 + v * 4194304.0);
    }
    mn[i] = xmin;
    cnt[i] = n;
  }
  return true;
}

struct __align__(16) PilSmem {
  uint8_t raw[kFrameBytes];          // 100 800
  uint8_t Y[kH * kW];                // 33 600
  uint8_t tmp[kH * kS];              // 17 640 (+8 pad below keeps out 16-B aligned)
  uint8_t pad[8];
  uint8_t out[kPlane];
  uint32_t fix[kBitmapWords];
  uint64_t full;
};

__global__ void __launch_bounds__(512, 1)
preprocess_pil_kernel(const uint8_t* __restrict__ frames, uint8_t* __restrict__ ring, int num_envs,
                      int ring_slots, int slot, int replicate) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  PilSmem& sm = *reinterpret_cast<PilSmem*>(smem_raw);
  const int tid = threadIdx.x;
  for (int i = tid; i < kBitmapWords; i += 512) sm.fix[i] = g_luma_fix[i];
  if (tid == 0) {
    mbar_init(&sm.full, 1);
    fence_mbar_init();
  }
  __syncthreads();
  const LumaCoef coef = luma_coef();
  int it = 0;
  for (int env = blockIdx.x; env < num_envs; env += gridDim.x, ++it) {
    if (tid == 0) {
      bulk_wait_read<0>();                                    // previous plane store has read sm.out
      mbar_expect_tx(&sm.full, kFrameBytes);
      const uint8_t* src = frames + (size_t)env * kFrameBytes;
      const uint64_t once = l2_policy_evict_first();          // frames are read once (see issue_loads)
      for (int c = 0; c < 4; ++c)                             // 4 x 25 200 B
        bulk_g2s_hint(sm.raw + c * (kFrameBytes / 4), src + c * (kFrameBytes / 4), kFrameBytes / 4, &sm.full,
                      once);
    }
    mbar_wait(&sm.full, it & 1);
    // luma of all 210 x 160 pixels, 8 per thread-iteration
    const uint2* raw2 = reinterpret_cast<const uint2*>(sm.raw);
    for (int u = tid; u < kH * kW / 8; u += 512) {
      const uint2 a = raw2[3 * u], b = raw2[3 * u + 1], c = raw2[3 * u + 2];
      const uint32_t w[6] = {a.x, a.y, b.x, b.y, c.x, c.y};
      reinterpret_cast<uint2*>(sm.Y)[u] = luma_8px(w, coef, sm.fix);
    }
    __syncthreads();
    // horizontal pass -> u8 [210][84]
    for (int o = tid; o < kH * kS; o += 512) {
      const int row = o / kS, dx = o - row * kS;
      const uint8_t* p = sm.Y + row * kW + g_pil.xmin[dx];
      int acc = 1 << 21;
      const int n = g_pil.xn[dx];
      for (int j = 0; j < n; ++j) acc += (int)p[j] * g_pil.xk[dx][j];
      acc >>= 22;
      sm.tmp[o] = (uint8_t)min(max(acc, 0), 255);
    }
    __syncthreads();
    // vertical pass -> the ring's 4x4-blocked plane
    for (int o = tid; o < kPlane; o += 512) {
      const int dy = o / kS, dx = o - dy * kS;
      const uint8_t* p = sm.tmp + g_pil.ymin[dy] * kS + dx;
      int acc = 1 << 21;
      const int n = g_pil.yn[dy];
      for (int j = 0; j < n; ++j) acc += (int)p[j * kS] * g_pil.yk[dy][j];
      acc >>= 22;
      sm.out[((dy >> 2) * 21 + (dx >> 2)) * 16 + (dy & 3) * 4 + (dx & 3)] = (uint8_t)min(max(acc, 0), 255);
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      uint8_t* dst = ring + ((size_t)env * ring_slots) * kPlane;
      for (int r = 0; r < replicate; ++r) {
        int sl = slot + r;
        if (sl >= ring_slots) sl -= ring_slots;
        bulk_s2g(dst + (size_t)sl * kPlane, sm.out, kPlane);
      }
      bulk_commit();
    }
  }
  if (tid == 0) bulk_wait<0>();
}

// ---- History.get / reset -----------------------------------------------------------------
template <typename OutT>
__global__ void history_get_kernel(const uint8_t* __restrict__ ring, OutT* __restrict__ out,
                                   int num_envs, int ring_slots, int first_slot) {
  const int64_t total = (int64_t)num_envs * kPlane;            // one thread per (env, pixel)
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int env = (int)(i / kPlane);
    const int px = (int)(i - (int64_t)env * kPlane);
    const int y = px / kS, x = px - y * kS;                      // ring planes are 4x4-blocked
    const uint8_t* base = ring + (size_t)env * ring_slots * kPlane +
                          ((y >> 2) * 21 + (x >> 2)) * 16 + (y & 3) * 4 + (x & 3);
    OutT v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      int s = first_slot + k;
      if (s >= ring_slots) s -= ring_slots;
      v[k] = (OutT)base[(size_t)s * kPlane];
    }
    OutT* o = out + i * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) o[k] = v[k];
  }
}

int preprocess_init(int device) {
  if (device < 0 || device >= 64) {
    set_error("arl_init: device %d out of range", device);
    return ARL_ERR_INVALID;
  }
  if (g_ready[device]) return ARL_OK;
  TapTables t;
  linear_taps(kW, kS, t.x);
  linear_taps(kH, kS, t.y);
  for (int d = 0; d < kS; ++d) {
    // the staged-row scheme needs both taps in range and adjacent (true for 210x160 -> 84x84)
    if ((int)(t.y[d] & 0xFF) + 1 >= kH || (int)(t.x[d] & 0xFF) + 1 >= kW) {
      set_error("arl_init: tap table needs edge clamping, unsupported geometry");
      return ARL_ERR_UNSUPPORTED;
    }
  }
  for (int d = 0; d < kS; ++d) {
    // the copy warp relies on sy(d) = 5*(d/2) + 3*(d%2): rows 5k+2 unused, 5k+3..5k+6 contiguous
    if ((int)(t.y[d] & 0xFF) != 5 * (d / 2) + 3 * (d % 2)) {
      set_error("arl_init: unexpected vertical tap pattern at row %d", d);
      return ARL_ERR_UNSUPPORTED;
    }
  }
  for (int d = 0; d < kS; ++d) {
    // phase B of K1 relies on sx(d) = (80 d + 19) / 42 and on coefficients periodic in 21 outputs
    const uint32_t want = (uint32_t)tap_sx(d);
    if ((t.x[d] & 0xFF) != want || (d >= kPer && (t.x[d] >> 8) != (t.x[d - kPer] >> 8))) {
      set_error("arl_init: unexpected horizontal tap pattern at column %d", d);
      return ARL_ERR_UNSUPPORTED;
    }
  }
  for (int r = 0; r < kPer; ++r) t.xc[r] = ((t.x[r] >> 8) & 0xFFFu) | ((t.x[r] >> 20) << 16);
  ARL_CUDA(cudaMemcpyToSymbol(c_taps, &t, sizeof(t)));
  void* fix = nullptr;
  ARL_CUDA(cudaGetSymbolAddress(&fix, g_luma_fix));
  ARL_CUDA(cudaMemset(fix, 0, sizeof(uint32_t) * kBitmapWords));
  luma_fix_init_kernel<<<65536 / 256, 256>>>();
  ARL_LAUNCH_CHECK("luma_fix_init_kernel");
  ARL_CUDA(cudaFuncSetAttribute(preprocess_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)sizeof(K1Smem)));
  ARL_CUDA(cudaFuncSetAttribute(preprocess_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)sizeof(K1Smem)));
  {
    static PilTaps pt;
    if (!pil_coeffs(kW, kS, pt.xmin, pt.xn, pt.xk) || !pil_coeffs(kH, kS, pt.ymin, pt.yn, pt.yk)) {
      set_error("arl_init: PIL resize needs more than %d taps", kPilMaxTaps);
      return ARL_ERR_UNSUPPORTED;
    }
    ARL_CUDA(cudaMemcpyToSymbol(g_pil, &pt, sizeof(pt)));
    ARL_CUDA(cudaFuncSetAttribute(preprocess_pil_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)sizeof(PilSmem)));
  }
  ARL_CUDA(cudaDeviceSynchronize());
  g_ready[device] = true;
  return ARL_OK;
}

}  // namespace arl

using namespace arl;

extern "C" int arl_preprocess_push(const uint8_t* frames, uint8_t* ring, int num_envs,
                                   int ring_slots, int slot, int replicate, void* stream) {
  ARL_REQUIRE(frames && ring, "arl_preprocess_push: null pointer");
  ARL_REQUIRE(num_envs >= 0, "arl_preprocess_push: num_envs %d < 0", num_envs);
  ARL_REQUIRE(ring_slots >= ARL_HISTORY, "arl_preprocess_push: ring_slots %d < %d", ring_slots,
              ARL_HISTORY);
  ARL_REQUIRE(slot >= 0 && slot < ring_slots, "arl_preprocess_push: slot %d outside [0,%d)", slot,
              ring_slots);
  ARL_REQUIRE(replicate >= 1 && replicate <= ring_slots,
              "arl_preprocess_push: replicate %d outside [1,%d]", replicate, ring_slots);
  ARL_REQUIRE((reinterpret_cast<uintptr_t>(frames) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(ring) & 15) == 0,
              "arl_preprocess_push: frames and ring must be 16-byte aligned");
  if (num_envs == 0) return ARL_OK;
  const int grid = num_envs < num_sms() ? num_envs : num_sms();
  ARL_CUDA(launch_pdl(num_envs <= kK1EvictFirstMaxEnvs ? preprocess_kernel<true> : preprocess_kernel<false>,
                      dim3(grid), dim3(kK1Threads), sizeof(K1Smem), (cudaStream_t)stream,
                      frames, ring, num_envs, ring_slots, slot, replicate));
  ARL_LAUNCH_CHECK("preprocess_kernel");
  return ARL_OK;
}

extern "C" int arl_preprocess_push_pil(const uint8_t* frames, uint8_t* ring, int num_envs,
                                       int ring_slots, int slot, int replicate, void* stream) {
  ARL_REQUIRE(frames && ring, "arl_preprocess_push_pil: null pointer");
  ARL_REQUIRE(num_envs >= 0, "arl_preprocess_push_pil: num_envs %d < 0", num_envs);
  ARL_REQUIRE(ring_slots >= ARL_HISTORY && slot >= 0 && slot < ring_slots && replicate >= 1 &&
                  replicate <= ring_slots,
              "arl_preprocess_push_pil: bad ring geometry (slots %d, slot %d, replicate %d)",
              ring_slots, slot, replicate);
  ARL_REQUIRE((reinterpret_cast<uintptr_t>(frames) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(ring) & 15) == 0,
              "arl_preprocess_push_pil: frames and ring must be 16-byte aligned");
  if (num_envs == 0) return ARL_OK;
  const int grid = num_envs < num_sms() ? num_envs : num_sms();
  preprocess_pil_kernel<<<grid, 512, sizeof(PilSmem), (cudaStream_t)stream>>>(
      frames, ring, num_envs, ring_slots, slot, replicate);
  ARL_LAUNCH_CHECK("preprocess_pil_kernel");
  return ARL_OK;
}

extern "C" int arl_upload_frames(const uint8_t* host_frames, uint8_t* dev_frames, int num_envs,
                                 void* stream) {
  ARL_REQUIRE(host_frames && dev_frames, "arl_upload_frames: null pointer");
  ARL_REQUIRE(num_envs >= 0, "arl_upload_frames: num_envs %d < 0", num_envs);
  if (num_envs == 0) return ARL_OK;
  // a frame = 42 groups of 5 rows (2400 B); K1 reads rows 0,1 and 3,4 of every group.  Because
  // 210 = 0 (mod 5) those rows form ONE uniform pattern over the whole batch: 4-row runs (1920 B)
  // at a 5-row pitch starting at row 3 (rows 3..6, 8..11, ...; a run that starts at row 208 of a
  // frame ends with rows 0, 1 of the next) -- one 2-D copy with half the DMA segments of two
  // 960-B-run copies -- plus rows 0, 1 of the first frame and rows 208, 209 of the last.
  cudaStream_t st = (cudaStream_t)stream;
  const size_t pitch = 5 * kRowBytes, groups = (size_t)num_envs * (kH / 5);
  ARL_CUDA(cudaMemcpyAsync(dev_frames, host_frames, 2 * kRowBytes, cudaMemcpyHostToDevice, st));
  if (groups > 1)
    ARL_CUDA(cudaMemcpy2DAsync(dev_frames + 3 * kRowBytes, pitch, host_frames + 3 * kRowBytes, pitch,
                               4 * kRowBytes, groups - 1, cudaMemcpyHostToDevice, st));
  const size_t tail = (groups * 5 - 2) * kRowBytes;
  ARL_CUDA(cudaMemcpyAsync(dev_frames + tail, host_frames + tail, 2 * kRowBytes, cudaMemcpyHostToDevice, st));
  return ARL_OK;
}

extern "C" int arl_upload_frames_full(const uint8_t* host_frames, uint8_t* dev_frames, int num_envs,
                                      void* stream) {
  ARL_REQUIRE(host_frames && dev_frames, "arl_upload_frames_full: null pointer");
  ARL_REQUIRE(num_envs >= 0, "arl_upload_frames_full: num_envs %d < 0", num_envs);
  if (num_envs == 0) return ARL_OK;
  ARL_CUDA(cudaMemcpyAsync(dev_frames, host_frames, (size_t)num_envs * kH * kRowBytes,
                           cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return ARL_OK;
}

extern "C" int arl_history_get(const uint8_t* ring, void* out, int out_is_u8, int num_envs,
                               int ring_slots, int first_slot, void* stream) {
  ARL_REQUIRE(ring && out, "arl_history_get: null pointer");
  ARL_REQUIRE(num_envs >= 0 && ring_slots >= ARL_HISTORY && first_slot >= 0 &&
                  first_slot < ring_slots,
              "arl_history_get: bad geometry (envs %d, slots %d, first %d)", num_envs, ring_slots,
              first_slot);
  if (num_envs == 0) return ARL_OK;
  const int64_t total = (int64_t)num_envs * kPlane;
  const int block = 256;
  int64_t grid64 = (total + block - 1) / block;
  const int grid = (int)(grid64 < (int64_t)num_sms() * 16 ? grid64 : (int64_t)num_sms() * 16);
  if (out_is_u8)
    history_get_kernel<uint8_t><<<grid, block, 0, (cudaStream_t)stream>>>(
        ring, (uint8_t*)out, num_envs, ring_slots, first_slot);
  else
    history_get_kernel<float><<<grid, block, 0, (cudaStream_t)stream>>>(
        ring, (float*)out, num_envs, ring_slots, first_slot);
  ARL_LAUNCH_CHECK("history_get_kernel");
  return ARL_OK;
}

extern "C" int arl_history_reset(uint8_t* ring, int num_envs, int ring_slots, void* stream) {
  ARL_REQUIRE(ring, "arl_history_reset: null pointer");
  ARL_REQUIRE(num_envs >= 0 && ring_slots >= ARL_HISTORY, "arl_history_reset: bad geometry");
  ARL_CUDA(cudaMemsetAsync(ring, 0, (size_t)num_envs * ring_slots * kPlane, (cudaStream_t)stream));
  return ARL_OK;
}
