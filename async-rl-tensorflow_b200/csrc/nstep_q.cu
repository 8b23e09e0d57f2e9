// Asynchronous n-step Q-learning (Mnih et al. 2016, supplementary algorithm next to A3C's): the
// forward with the epsilon-greedy draw fused into the heads launch, and the loss kernel that
// bootstraps from max_a Q(s_T; theta^-) and emits dQ for the acted action.  Everything else of the
// cycle -- backward, exchange, clip + RMSProp -- is the A3C cycle's.
#include "common.cuh"
#include "../../include/asyncrl_b200_nstep_q.h"

namespace arl {

int heads_forward_egreedy(const float* params, int action_size, const float* h, float* logits, float* probs,
                          float* value, int32_t* actions, int64_t env_id_base, int64_t step,
                          const int64_t* step_dev, uint64_t seed, float ep, double ep_start, double ep_end,
                          double ep_end_t, double learn_start, int64_t num_samples, cudaStream_t st);

// One thread per SAMPLE (t, b), as returns_lossgrad_kernel: the return recurrence runs from T-1
// down to the thread's own t (the same operations in the same order as a serial walk: identical
// bits), starting from the max over the target network's Q values of s_T.
__global__ void nstep_q_lossgrad_kernel(const float* __restrict__ rewards,
                                        const uint8_t* __restrict__ terminals,
                                        const int32_t* __restrict__ actions, const float* __restrict__ q,
                                        const float* __restrict__ q_boot, float* __restrict__ returns,
                                        float* __restrict__ dq, float* __restrict__ loss_sums, int T, int B,
                                        int A, float gamma, float rmin, float rmax, float grad_scale) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float s_loss = 0.f, s_q = 0.f;
  pdl_wait();
  if (n < (int64_t)T * B) {
    const int t = (int)(n / B), b = (int)(n - (int64_t)t * B);
    const float* qb = q_boot + (size_t)b * A;
    float R = qb[0];
    for (int j = 1; j < A; ++j) R = fmaxf(R, qb[j]);                     // max_a Q(s_T; theta^-)
    for (int tt = T - 1; tt >= t; --tt) {
      const size_t m = (size_t)tt * B + b;
      const float r = fminf(fmaxf(rewards[m], rmin), rmax);               // agent.py:154
      R = fmaf(gamma * (1.0f - (terminals[m] ? 1.0f : 0.0f)), R, r);      // agent.py:188-190
    }
    returns[n] = R;
    const int a = actions[n];
    const float qa = q[n * A + a];
    const float delta = R - qa;
    for (int j = 0; j < A; ++j) dq[n * A + j] = j == a ? -2.0f * delta * grad_scale : 0.f;
    s_loss = delta * delta;
    s_q = qa;
  }
  if (loss_sums) {
    s_loss = warp_sum(s_loss);
    s_q = warp_sum(s_q);
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(loss_sums + 0, s_loss);
      atomicAdd(loss_sums + 1, s_q);
    }
  }
}

}  // namespace arl

using namespace arl;

extern "C" int arl_forward_egreedy(const float* params, float* prepared, int refresh_prepared, int action_size,
                                   const uint8_t* ring, int num_envs, int ring_slots, int first_slot,
                                   float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                                   int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                                   uint64_t seed, float ep, double ep_start, double ep_end, double ep_end_t,
                                   double learn_start, void* stream) {
  ARL_REQUIRE(params && prepared && ring && a1 && a2 && h && logits && probs && value && actions,
              "arl_forward_egreedy: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_forward_egreedy: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_envs >= 0 && env_id_base >= 0 && step >= 0, "arl_forward_egreedy: negative argument");
  ARL_REQUIRE(ep >= 0.f && ep <= 1.f, "arl_forward_egreedy: ep %f outside [0,1]", (double)ep);
  ARL_REQUIRE(step_dev == nullptr || (ep_start >= 0.0 && ep_start <= 1.0 && ep_end >= 0.0 && ep_end <= 1.0),
              "arl_forward_egreedy: ep_start %f / ep_end %f outside [0,1]", ep_start, ep_end);
  ARL_REQUIRE(step_dev == nullptr || ep_end_t > 0.0, "arl_forward_egreedy: ep_end_t must be > 0");
  if (num_envs == 0) return ARL_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = ARL_OK;
  if (refresh_prepared) rc = arl_prepare_weights(params, prepared, stream);
  if (rc) return rc;
  // env range by env range, as arl_forward_sample: each range writes its own a2 block
  const int chunk = (int)arl_a2_block_rows(num_envs);
  for (int off = 0; off < num_envs; off += chunk) {
    const int n = num_envs - off < chunk ? num_envs - off : chunk;
    float* a1c = a1 + (size_t)off * 3200;                       // 12 800 bytes of fp16 per sample
    float* a2c = a2 + (size_t)off * ARL_A2_ELEMS;
    float* hc = h + (size_t)off * ARL_FC;
    rc = arl_conv1_forward(prepared, ring + (size_t)off * ring_slots * kPlane, a1c, n, ring_slots, first_slot, 1,
                           stream);
    if (rc) return rc;
    rc = arl_conv2_forward(prepared, a1c, a2c, n, stream);
    if (rc) return rc;
    rc = arl_fc_forward(params, prepared, a2c, hc, n, stream);
    if (rc) return rc;
    rc = heads_forward_egreedy(params, action_size, hc, logits + (size_t)off * action_size,
                               probs + (size_t)off * action_size, value + off, actions + off, env_id_base + off,
                               step, step_dev, seed, ep, ep_start, ep_end, ep_end_t, learn_start, n, st);
    if (rc) return rc;
  }
  return ARL_OK;
}

extern "C" int arl_nstep_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                    const float* q, const float* q_boot, float* returns, float* dq,
                                    float* loss_sums, int t_max, int num_envs, int action_size, float gamma,
                                    float reward_min, float reward_max, float grad_scale, void* stream) {
  ARL_REQUIRE(rewards && terminals && actions && q && q_boot && returns && dq,
              "arl_nstep_q_lossgrad: null pointer");
  ARL_REQUIRE(t_max >= 0 && num_envs >= 0, "arl_nstep_q_lossgrad: negative size");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_nstep_q_lossgrad: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  if (t_max == 0 || num_envs == 0) return ARL_OK;
  const int64_t total = (int64_t)t_max * num_envs;
  ARL_CUDA(launch_pdl(nstep_q_lossgrad_kernel, dim3((unsigned)((total + 127) / 128)), dim3(128), 0,
                      (cudaStream_t)stream, rewards, terminals, actions, q, q_boot, returns, dq, loss_sums, t_max,
                      num_envs, action_size, gamma, reward_min, reward_max, grad_scale));
  ARL_LAUNCH_CHECK("nstep_q_lossgrad_kernel");
  return ARL_OK;
}
