// C-ABI glue: error reporting, init, parameter layout and the composed forward/backward.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "../../include/asyncrl_b200_dueling.h"
#include "../../include/asyncrl_b200_dueling_streams.h"

namespace arl {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return ARL_ERR_CUDA;
}

static long long g_launches = 0;
void count_launch() { __atomic_fetch_add(&g_launches, 1, __ATOMIC_RELAXED); }

// SM count per device index (arl_init fills it); num_sms() answers for the CURRENT device
static int g_num_sms[64] = {0};
int num_sms() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  const int n = g_num_sms[dev & 63];
  return n > 0 ? n : 148;
}

int preprocess_init(int device);
int conv_init();
int heads_init();

}  // namespace arl

using namespace arl;

extern "C" const char* arl_last_error(void) { return g_err; }
extern "C" int arl_version(void) { return 100; }
extern "C" int64_t arl_launch_count(int reset) {
  const long long v = __atomic_load_n(&g_launches, __ATOMIC_RELAXED);
  if (reset) __atomic_store_n(&g_launches, 0, __ATOMIC_RELAXED);
  return (int64_t)v;
}

extern "C" int arl_init(int device) {
  int count = 0;
  ARL_CUDA(cudaGetDeviceCount(&count));
  ARL_REQUIRE(device >= 0 && device < count, "arl_init: device %d not in [0,%d)", device, count);
  int prev = 0;
  ARL_CUDA(cudaGetDevice(&prev));
  ARL_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  ARL_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("arl_init: device %d is sm_%d%d; this library is built for sm_100a (B200) only",
              device, prop.major, prop.minor);
    cudaSetDevice(prev);
    return ARL_ERR_UNSUPPORTED;
  }
  g_num_sms[device & 63] = prop.multiProcessorCount;
  int rc = preprocess_init(device);
  if (rc == ARL_OK) rc = conv_init();
  if (rc == ARL_OK) rc = heads_init();
  cudaSetDevice(prev);
  return rc;
}

extern "C" int arl_param_layout(int action_size, int64_t* offsets) {
  ARL_REQUIRE(offsets, "arl_param_layout: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_param_layout: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  const ParamLayout L = param_layout(action_size);
  memcpy(offsets, L.off, sizeof(L.off));
  return ARL_OK;
}

extern "C" int64_t arl_backward_workspace_bytes(int action_size) {
  // largest user: fc weight-gradient split-K partials (8 x 2592 x 256 floats)
  (void)action_size;
  return (int64_t)8 * ARL_A2_ELEMS * ARL_FC * sizeof(float) + (1 << 20);
}

// Rows of one a2 block (= envs one forward launch handles).  A single launch of conv2 forward for
// more than ~16K envs scatters its epilogue's 16-byte vectors over 324 chunk planes that are then
// more than 256 KB apart -- TLB reach, not bandwidth: 0.32 of the HBM rate at 64K envs against 0.56
// at 16K (profiles/r02_sweep_n1.json) -- so a rollout step of a very large batch runs as several
// launches over env ranges, each writing its own a2 block.
extern "C" int64_t arl_a2_block_rows(int num_envs) {
  if (num_envs <= 16384) return num_envs;
  for (int c = 16384; c >= 2048; c -= 128)
    if (num_envs % c == 0) return c;
  return num_envs;
}

namespace arl {
template <class Draw, bool Dueling>
int fc_heads_forward(const float* params, const float* prepared, int action_size, const float* a2, float* h,
                     float* logits, float* probs, float* value, int32_t* actions, int64_t env_id_base, int64_t step,
                     const int64_t* step_dev, uint64_t seed, int64_t num_samples, Draw draw, void* stream);
template <class Draw>
int fc_heads_forward_streams(const float* params, const float* prepared, int action_size, const float* a2, float* h,
                             float* logits, float* probs, float* value, int32_t* actions, int64_t env_id_base,
                             int64_t step, const int64_t* step_dev, uint64_t seed, int64_t num_samples, Draw draw,
                             void* stream);
}

// One env step of the forward, env range by env range; `draw` is the action draw of the heads launch
// (common.cuh: SampleDraw with actions == NULL draws nothing), Dueling the head kind (heads.cu),
// Streams the dueling streams' network (h rows of 512)
template <bool Dueling = false, class Draw, bool Streams = false>
static int forward_step(const float* params, float* prepared, int action_size, const uint8_t* ring,
                        int num_envs, int ring_slots, int first_slot, float* a1, float* a2, float* h,
                        float* logits, float* probs, float* value, int32_t* actions, int64_t env_id_base,
                        int64_t step, const int64_t* step_dev, uint64_t seed, Draw draw, void* stream) {
  const int chunk = (int)arl_a2_block_rows(num_envs);
  for (int off = 0; off < num_envs; off += chunk) {
    const int n = num_envs - off < chunk ? num_envs - off : chunk;
    float* a1c = a1 + (size_t)off * 3200;                       // 12 800 bytes of fp16 per sample
    float* a2c = a2 + (size_t)off * ARL_A2_ELEMS;
    float* hc = h + (size_t)off * (Streams ? 2 * ARL_FC : ARL_FC);
    int rc = arl_conv1_forward(prepared, ring + (size_t)off * ring_slots * kPlane, a1c, n, ring_slots,
                               first_slot, 1, stream);
    if (rc) return rc;
    rc = arl_conv2_forward(prepared, a1c, a2c, n, stream);
    if (rc) return rc;
    // fc256, then heads + softmax (+ the action draw) in one launch
    if constexpr (Streams)
      rc = fc_heads_forward_streams<Draw>(params, prepared, action_size, a2c, hc, logits + (size_t)off * action_size,
                                          probs + (size_t)off * action_size, value + off,
                                          actions ? actions + off : nullptr, env_id_base + off, step, step_dev, seed,
                                          n, draw, stream);
    else
      rc = fc_heads_forward<Draw, Dueling>(params, prepared, action_size, a2c, hc, logits + (size_t)off * action_size,
                                           probs + (size_t)off * action_size, value + off,
                                           actions ? actions + off : nullptr, env_id_base + off, step, step_dev, seed,
                                           n, draw, stream);
    if (rc) return rc;
  }
  return ARL_OK;
}

extern "C" int arl_forward(const float* params, float* prepared, int refresh_prepared, int action_size,
                           const uint8_t* ring, int num_envs, int ring_slots, int first_slot, int steps,
                           float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                           void* stream) {
  // refused before the first launch: a bad action count must leave a1, a2 and `prepared` as they were
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_forward: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  const int64_t N = (int64_t)num_envs * steps;
  int rc = ARL_OK;
  if (refresh_prepared) rc = arl_prepare_weights(params, prepared, stream);
  if (rc) return rc;
  if (steps == 1)
    return forward_step(params, prepared, action_size, ring, num_envs, ring_slots, first_slot, a1, a2, h,
                        logits, probs, value, nullptr, 0, 0, nullptr, 0, SampleDraw{}, stream);
  rc = arl_conv1_forward(prepared, ring, a1, num_envs, ring_slots, first_slot, steps, stream);
  if (rc) return rc;
  rc = arl_conv2_forward(prepared, a1, a2, N, stream);
  if (rc) return rc;
  return arl_fc_heads_forward(params, prepared, action_size, a2, h, logits, probs, value, nullptr, 0, 0,
                              nullptr, 0, N, stream);
}

extern "C" int arl_forward_sample(const float* params, float* prepared, int refresh_prepared, int action_size,
                                  const uint8_t* ring, int num_envs, int ring_slots, int first_slot,
                                  float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                                  int32_t* actions, int64_t env_id_base, int64_t step,
                                  const int64_t* step_dev, uint64_t seed, void* stream) {
  ARL_REQUIRE(actions, "arl_forward_sample: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_forward_sample: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  int rc = ARL_OK;
  if (refresh_prepared) rc = arl_prepare_weights(params, prepared, stream);
  if (rc) return rc;
  return forward_step(params, prepared, action_size, ring, num_envs, ring_slots, first_slot, a1, a2, h,
                      logits, probs, value, actions, env_id_base, step, step_dev, seed, SampleDraw{}, stream);
}

// the argument checks of the epsilon-greedy forward (fn = the C entry's name, for errors)
static int egreedy_args(const char* fn, const float* params, const float* prepared, int action_size,
                        const uint8_t* ring, const float* a1, const float* a2, const float* h, const float* logits,
                        const float* probs, const float* value, const int32_t* actions, int num_envs,
                        int64_t env_id_base, int64_t step, const int64_t* step_dev, float ep, double ep_start,
                        double ep_end, double ep_end_t) {
  ARL_REQUIRE(params && prepared && ring && a1 && a2 && h && logits && probs && value && actions,
              "%s: null pointer", fn);
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "%s: action_size %d outside [1,%d]", fn, action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_envs >= 0 && env_id_base >= 0 && step >= 0, "%s: negative argument", fn);
  ARL_REQUIRE(ep >= 0.f && ep <= 1.f, "%s: ep %f outside [0,1]", fn, (double)ep);
  ARL_REQUIRE(step_dev == nullptr || (ep_start >= 0.0 && ep_start <= 1.0 && ep_end >= 0.0 && ep_end <= 1.0),
              "%s: ep_start %f / ep_end %f outside [0,1]", fn, ep_start, ep_end);
  ARL_REQUIRE(step_dev == nullptr || ep_end_t > 0.0, "%s: ep_end_t must be > 0", fn);
  return ARL_OK;
}

extern "C" int arl_forward_egreedy(const float* params, float* prepared, int refresh_prepared, int action_size,
                                   const uint8_t* ring, int num_envs, int ring_slots, int first_slot,
                                   float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                                   int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                                   uint64_t seed, float ep, double ep_start, double ep_end, double ep_end_t,
                                   double learn_start, void* stream) {
  int rc = egreedy_args("arl_forward_egreedy", params, prepared, action_size, ring, a1, a2, h, logits, probs, value,
                         actions, num_envs, env_id_base, step, step_dev, ep, ep_start, ep_end, ep_end_t);
  if (rc || num_envs == 0) return rc;
  if (refresh_prepared) rc = arl_prepare_weights(params, prepared, stream);
  if (rc) return rc;
  return forward_step(params, prepared, action_size, ring, num_envs, ring_slots, first_slot, a1, a2, h,
                      logits, probs, value, actions, env_id_base, step, step_dev, seed,
                      EgreedyDraw{ep, ep_start, ep_end, ep_end_t, learn_start}, stream);
}

extern "C" int arl_forward_dueling(const float* params, float* prepared, int refresh_prepared, int action_size,
                                   const uint8_t* ring, int num_envs, int ring_slots, int first_slot, int steps,
                                   float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                                   int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                                   uint64_t seed, float ep, double ep_start, double ep_end, double ep_end_t,
                                   double learn_start, void* stream) {
  int rc = ARL_OK;
  if (actions != nullptr) {                       // one env step + the draw of arl_forward_egreedy
    ARL_REQUIRE(steps == 1, "arl_forward_dueling: the action draw needs steps == 1, got %d", steps);
    rc = egreedy_args("arl_forward_dueling", params, prepared, action_size, ring, a1, a2, h, logits, probs, value,
                      actions, num_envs, env_id_base, step, step_dev, ep, ep_start, ep_end, ep_end_t);
    if (rc || num_envs == 0) return rc;
    if (refresh_prepared) rc = arl_prepare_weights(params, prepared, stream);
    if (rc) return rc;
    return forward_step<true>(params, prepared, action_size, ring, num_envs, ring_slots, first_slot, a1, a2, h,
                              logits, probs, value, actions, env_id_base, step, step_dev, seed,
                              EgreedyDraw{ep, ep_start, ep_end, ep_end_t, learn_start}, stream);
  }
  ARL_REQUIRE(params && prepared && ring && a1 && a2 && h && logits && probs && value,
              "arl_forward_dueling: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_forward_dueling: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_envs >= 0 && steps >= 0, "arl_forward_dueling: negative size");
  if (num_envs == 0 || steps == 0) return ARL_OK;
  if (refresh_prepared) rc = arl_prepare_weights(params, prepared, stream);
  if (rc) return rc;
  if (steps == 1)                                 // arl_forward's paths, no draw
    return forward_step<true>(params, prepared, action_size, ring, num_envs, ring_slots, first_slot, a1, a2, h,
                              logits, probs, value, nullptr, 0, 0, nullptr, 0, SampleDraw{}, stream);
  const int64_t N = (int64_t)num_envs * steps;
  rc = arl_conv1_forward(prepared, ring, a1, num_envs, ring_slots, first_slot, steps, stream);
  if (rc) return rc;
  rc = arl_conv2_forward(prepared, a1, a2, N, stream);
  if (rc) return rc;
  return fc_heads_forward<SampleDraw, true>(params, prepared, action_size, a2, h, logits, probs, value, nullptr, 0,
                                            0, nullptr, 0, N, SampleDraw{}, stream);
}

extern "C" int arl_backward(const float* params, const float* prepared, int action_size,
                            const uint8_t* ring, int num_envs, int ring_slots, int first_slot,
                            int steps, const float* a1,
                            const float* a2, const float* h, const float* dlogits,
                            const float* dvalue, float* d_h, float* d_a2, float* d_a1, float* grads,
                            void* workspace, float tensor_scale, int allreduce, void* stream) {
  ARL_REQUIRE(tensor_scale > 0.f, "arl_backward: tensor_scale must be > 0");
  const int64_t N = (int64_t)num_envs * steps;
  const float unscale = 1.0f / tensor_scale;
  int rc = arl_heads_backward(params, action_size, h, dlogits, dvalue, d_h, grads, workspace, N,
                              tensor_scale, stream);
  if (rc) return rc;
  rc = arl_fc_backward(prepared, a2, arl_a2_block_rows(num_envs), d_h, d_a2, grads, workspace, N, unscale, stream);
  if (rc) return rc;
  // l4_w .. q_b are final now: 98 % of the gradient bytes travel while the conv kernels run
  const bool comm = allreduce && arl_comm_size() > 1;
  const ParamLayout L = param_layout(action_size);
  // Default: ONE all-reduce of the whole buffer after the last backward kernel.  ARL_ALLREDUCE_OVERLAP=1
  // sends the l4_w..q_b bucket (98 % of the bytes) on the side stream right after the fc256 weight
  // gradient instead.  Measured on 2 B200s (profiles/r02_allreduce_overlap.txt): 2.262 / 2.340 ms per
  // cycle overlapped vs 2.252 / 2.245 serial (2.227 on one GPU) -- the conv backward kernels are
  // persistent one-CTA-per-SM grids, so NCCL's CTAs only get SMs at a kernel boundary and then delay
  // the statically scheduled CTAs of the next kernel by their own run time: nothing is hidden.
  static const bool overlap = [] { const char* e = getenv("ARL_ALLREDUCE_OVERLAP"); return e && e[0] == '1'; }();
  if (comm && !overlap) {
    rc = arl_conv2_backward(prepared, a1, d_a2, d_a1, grads, workspace, N, unscale, stream);
    if (rc) return rc;
    rc = arl_conv1_backward(ring, d_a1, grads, workspace, num_envs, ring_slots, first_slot, steps, unscale, stream);
    if (rc) return rc;
    return arl_allreduce_grads(grads, L.off[ARL_NUM_TENSORS], stream);
  }
  if (comm) {
    rc = arl_allreduce_begin(grads, L.off[T_L4W], L.off[ARL_NUM_TENSORS] - L.off[T_L4W], stream);
    if (rc) return rc;
  }
  rc = arl_conv2_backward(prepared, a1, d_a2, d_a1, grads, workspace, N, unscale, stream);
  if (rc) return rc;
  rc = arl_conv1_backward(ring, d_a1, grads, workspace, num_envs, ring_slots, first_slot, steps,
                          unscale, stream);
  if (rc || !comm) return rc;
  rc = arl_allreduce_begin(grads, 0, L.off[T_L4W], stream);        // l1_w .. l2_b
  if (rc) return rc;
  return arl_allreduce_end(stream);
}

// ---- dueling streams (include/asyncrl_b200_dueling_streams.h) ---------------------------------
extern "C" int arl_streams_param_layout(int action_size, int64_t* offsets) {
  ARL_REQUIRE(offsets, "arl_streams_param_layout: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_streams_param_layout: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  const StreamsLayout L = streams_layout(action_size);
  memcpy(offsets, L.off, sizeof(L.off));
  return ARL_OK;
}

extern "C" int64_t arl_streams_workspace_bytes(int action_size) {
  // largest user: the fc weight-gradient split-K partials of both streams (8 x 2592 x 512 floats)
  (void)action_size;
  return (int64_t)8 * ARL_A2_ELEMS * 2 * ARL_FC * sizeof(float) + (1 << 20);
}

extern "C" int arl_forward_streams(const float* params, float* prepared, int refresh_prepared, int action_size,
                                   const uint8_t* ring, int num_envs, int ring_slots, int first_slot, int steps,
                                   float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                                   int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                                   uint64_t seed, float ep, double ep_start, double ep_end, double ep_end_t,
                                   double learn_start, void* stream) {
  int rc = ARL_OK;
  if (actions != nullptr) {                       // one env step + the draw of arl_forward_egreedy
    ARL_REQUIRE(steps == 1, "arl_forward_streams: the action draw needs steps == 1, got %d", steps);
    rc = egreedy_args("arl_forward_streams", params, prepared, action_size, ring, a1, a2, h, logits, probs, value,
                      actions, num_envs, env_id_base, step, step_dev, ep, ep_start, ep_end, ep_end_t);
    if (rc || num_envs == 0) return rc;
    if (refresh_prepared) rc = arl_prepare_weights_streams(params, prepared, action_size, stream);
    if (rc) return rc;
    return forward_step<true, EgreedyDraw, true>(params, prepared, action_size, ring, num_envs, ring_slots,
                                                 first_slot, a1, a2, h, logits, probs, value, actions, env_id_base,
                                                 step, step_dev, seed,
                                                 EgreedyDraw{ep, ep_start, ep_end, ep_end_t, learn_start}, stream);
  }
  ARL_REQUIRE(params && prepared && ring && a1 && a2 && h && logits && probs && value,
              "arl_forward_streams: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_forward_streams: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_envs >= 0 && steps >= 0, "arl_forward_streams: negative size");
  if (num_envs == 0 || steps == 0) return ARL_OK;
  if (refresh_prepared) rc = arl_prepare_weights_streams(params, prepared, action_size, stream);
  if (rc) return rc;
  if (steps == 1)
    return forward_step<true, SampleDraw, true>(params, prepared, action_size, ring, num_envs, ring_slots, first_slot,
                                                a1, a2, h, logits, probs, value, nullptr, 0, 0, nullptr, 0,
                                                SampleDraw{}, stream);
  const int64_t N = (int64_t)num_envs * steps;
  rc = arl_conv1_forward(prepared, ring, a1, num_envs, ring_slots, first_slot, steps, stream);
  if (rc) return rc;
  rc = arl_conv2_forward(prepared, a1, a2, N, stream);
  if (rc) return rc;
  return fc_heads_forward_streams<SampleDraw>(params, prepared, action_size, a2, h, logits, probs, value, nullptr, 0,
                                              0, nullptr, 0, N, SampleDraw{}, stream);
}

// arl_backward with the streams' heads and fc256 backward; the conv backward and the exchange are
// arl_backward's, over all 12 tensors
extern "C" int arl_backward_streams(const float* params, const float* prepared, int action_size,
                                    const uint8_t* ring, int num_envs, int ring_slots, int first_slot,
                                    int steps, const float* a1, const float* a2, const float* h,
                                    const float* dlogits, const float* dvalue, float* d_h, float* d_a2,
                                    float* d_a1, float* grads, void* workspace, float tensor_scale,
                                    int allreduce, void* stream) {
  ARL_REQUIRE(tensor_scale > 0.f, "arl_backward_streams: tensor_scale must be > 0");
  const int64_t N = (int64_t)num_envs * steps;
  const float unscale = 1.0f / tensor_scale;
  int rc = arl_heads_backward_streams(params, action_size, h, dlogits, dvalue, d_h, grads, workspace, N,
                                      tensor_scale, stream);
  if (rc) return rc;
  rc = arl_fc_backward_streams(prepared, a2, arl_a2_block_rows(num_envs), d_h, d_a2, grads, workspace, N, unscale,
                               action_size, stream);
  if (rc) return rc;
  rc = arl_conv2_backward(prepared, a1, d_a2, d_a1, grads, workspace, N, unscale, stream);
  if (rc) return rc;
  rc = arl_conv1_backward(ring, d_a1, grads, workspace, num_envs, ring_slots, first_slot, steps, unscale, stream);
  if (rc || !(allreduce && arl_comm_size() > 1)) return rc;
  return arl_allreduce_grads(grads, streams_layout(action_size).off[kStreamsTensors], stream);
}
