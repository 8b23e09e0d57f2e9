// Shared helpers for the asyncrl_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/asyncrl_b200.h"

namespace arl {

// thread-local error text behind arl_last_error()
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
int num_sms();
void count_launch();

#define ARL_REQUIRE(cond, ...)                       \
  do {                                               \
    if (!(cond)) {                                   \
      arl::set_error(__VA_ARGS__);                   \
      return ARL_ERR_INVALID;                        \
    }                                                \
  } while (0)

#define ARL_CUDA(expr)                                             \
  do {                                                             \
    cudaError_t e__ = (expr);                                      \
    if (e__ != cudaSuccess) return arl::cuda_fail(e__, #expr);     \
  } while (0)

#define ARL_LAUNCH_CHECK(name)                                     \
  do {                                                             \
    cudaError_t e__ = cudaGetLastError();                          \
    if (e__ != cudaSuccess) return arl::cuda_fail(e__, name);      \
    arl::count_launch();                                           \
  } while (0)

// flat parameter layout (floats)
struct ParamLayout {
  int64_t off[ARL_NUM_TENSORS + 1];
};
enum { T_L1W = 0, T_L1B, T_L2W, T_L2B, T_L4W, T_L4B, T_PW, T_PB, T_QW, T_QB };

inline ParamLayout param_layout(int A) {
  ParamLayout L;
  const int64_t sz[ARL_NUM_TENSORS] = {8 * 8 * 4 * 16, 16,  4 * 4 * 16 * 32, 32, 2592 * 256,
                                       256,            256 * (int64_t)A, A,  256, 1};
  L.off[0] = 0;
  for (int i = 0; i < ARL_NUM_TENSORS; ++i) L.off[i + 1] = L.off[i] + sz[i];
  return L;
}

constexpr int kPlane = ARL_SCREEN * ARL_SCREEN;  // 7056 bytes, 441 x 16 B

// The action draw of a heads launch (heads.cu heads_fwd_kernel's template argument): SampleDraw is
// the policy sample of network.py:72, or no draw at all when `actions` is NULL; EgreedyDraw is
// agent.py:141-151 on the logits (arl_forward_egreedy).  SampleDraw carries nothing and its branch
// is the only one compiled in, so the A3C path pays nothing for the second kind.
struct SampleDraw {
  static constexpr bool kEgreedy = false;
};
struct EgreedyDraw {
  static constexpr bool kEgreedy = true;
  float ep;                                          // used when step_dev == nullptr
  double ep_start, ep_end, ep_end_t, learn_start;    // used with step_dev (agent.py:142-144)
};

// "prepared" weights (arl_prepare_weights): the operand images the tensor-core kernels keep
// resident, built once per parameter change instead of in every kernel prologue.  Byte offsets:
constexpr int64_t kPrepFcW = 0;                                   // l4_w as a split block (fc.cu)
constexpr int64_t kPrepFcWBytes = (int64_t)ARL_A2_ELEMS * ARL_FC * 4;
constexpr int64_t kPrepW1 = kPrepFcW + kPrepFcWBytes;             // conv1 fwd: s8 limbs | scales | bias
constexpr int64_t kPrepW1Bytes = 12800;
constexpr int64_t kPrepW2F = kPrepW1 + kPrepW1Bytes;              // conv2 fwd: [hi | lo] image | bias
constexpr int64_t kPrepW2FBytes = 33408;
constexpr int64_t kPrepW2D = kPrepW2F + kPrepW2FBytes;            // conv2 bwd: transposed fp16 [hi | lo] image
constexpr int64_t kPrepW2DBytes = 33024;
constexpr int64_t kPrepFcWT = kPrepW2D + kPrepW2DBytes;           // l4_w TRANSPOSED as a split block [256 rows][2592]
constexpr int64_t kPrepBytes = kPrepFcWT + kPrepFcWBytes;

// Dueling streams (include/asyncrl_b200_dueling_streams.h): the advantage stream's hidden layer
// la_w [2592,256], la_b [256] follows q_b; the ten tensors before it keep their offsets.
enum { T_LAW = ARL_NUM_TENSORS, T_LAB };
constexpr int kStreamsTensors = ARL_NUM_TENSORS + 2;
struct StreamsLayout {
  int64_t off[kStreamsTensors + 1];
};
inline StreamsLayout streams_layout(int A) {
  const ParamLayout P = param_layout(A);
  StreamsLayout L;
  for (int i = 0; i <= ARL_NUM_TENSORS; ++i) L.off[i] = P.off[i];
  L.off[T_LAW + 1] = L.off[T_LAW] + (int64_t)ARL_A2_ELEMS * ARL_FC;
  L.off[T_LAB + 1] = L.off[T_LAB] + ARL_FC;
  return L;
}
// The streams' prepared images: the plain ones at the plain offsets (kPrepFcW is not written), then
constexpr int64_t kPrepLaWT = kPrepBytes;                         // la_w TRANSPOSED [256 rows][2592], right behind
                                                                  // l4_w^T: the two read as ONE operand of 512 rows
                                                                  // (a SplitMat of two blocks of 256 rows)
constexpr int64_t kPrepSW = kPrepLaWT + kPrepFcWBytes;            // [l4_w | la_w] as one split block [2592 rows][512]
constexpr int64_t kPrepSB = kPrepSW + 2 * kPrepFcWBytes;          // [l4_b | la_b], 512 floats
constexpr int64_t kPrepStreamsBytes = kPrepSB + 2 * ARL_FC * 4;

// Peer-memory exchange state (comm.cu): every rank's gradient slots and flag words mapped into this
// process (CUDA IPC over NVLink); see arl_comm_enable_p2p.
constexpr int kMaxRanks = 16;
struct P2PView {
  float* slot[kMaxRanks];              // rank r's buffer base: [slot 0 | slot 1], `count` floats each
  unsigned long long* flags[kMaxRanks];// rank r's flag words [kMaxRanks]: flags[r][q] = last cycle rank q published
  unsigned long long* cycle;           // this rank's cycle counter
  unsigned int* done;                  // this rank's "blocks finished" counter of the publish kernel
  int* error;                          // this rank's error word (1 = a peer's flag did not arrive in time)
  long long count;                     // floats of a gradient the buffer was sized for
  long long stride;                    // floats from slot 0 to slot 1 (count rounded up to 256 B)
  int rank, nranks;
};
const P2PView* p2p_view();             // nullptr unless arl_comm_enable_p2p succeeded

// ---- small device helpers ----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes or
// the hint expires.  Without the hint the default time limit is ~100 cycles and every retry is a
// shared-memory wavefront: in the warp-specialised tcgen05 kernels, whose 17-25 warps mostly
// wait, polling took up to ~15 % of the L1 data pipe (fc dgrad: 291 -> 180 us with the hint).
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
        : "memory");
  } while (ok == 0);
}
// the many warps that wait for long (producers for a free stage, epilogue warps for an
// accumulator) back off between polls: every poll is a shared-memory wavefront
template <int NS>
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) __nanosleep(NS);
}
// 1-D TMA bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP).
// dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// 1-D TMA bulk copy shared -> global (bulk async-group completion).
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
               "r"(smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
// L2 eviction priority of the lines a copy touches, as a 64-bit cache policy for bulk_g2s_hint.
// evict_first: data read once (K1's frames) goes first, so a stream of it does not push out the
// lines the next kernels re-read or the dirty lines of the previous ones.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// bulk_g2s with an L2 cache policy (SASS: UBLKCP with a desc[UR] policy operand)
__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                              uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// Philox4x32-10, first output word (oracle/philox.py; Random123 known answers in the tests)
__device__ __forceinline__ uint32_t philox_first(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c0;
}

// inverse CDF over the float32 running sum in index order, fallback A-1 (the sampler contract of
// DESIGN.md §4): u = float(x >> 8) * 2^-24
__device__ __forceinline__ int sample_index(const float* p, int A, uint32_t x) {
  const float u = (float)(x >> 8) * 5.9604644775390625e-08f;
  float c = 0.f;
  int a = A - 1;
  for (int j = 0; j < A; ++j) {
    c = __fadd_rn(c, p[j]);
    if (u < c) { a = j; break; }
  }
  return a;
}

// Programmatic dependent launch for the small kernels between the tensor-core kernels: the launch
// (and whatever the kernel does before pdl_wait(): staging parameters the update wrote long ago)
// overlaps the tail of its predecessor in the stream; pdl_wait() returns when the predecessor has
// completed and its writes are visible.  EVERY kernel launched this way must call pdl_wait() --
// a kernel that skipped it would let its successor run ahead of its predecessor.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace arl
