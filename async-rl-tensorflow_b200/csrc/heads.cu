// K3 (heads) + K4: policy/value heads, softmax, action sampling, n-step returns and the
// loss gradients.
//   heads fwd : logits = h.p_w + p_b (network.py:62), value = h.q_w + q_b (network.py:79),
//               probs = softmax(logits) (network.py:65)
//   sampling  : network.py:72 batch_sample -> Philox4x32-10 + inverse CDF (oracle/philox.py)
//   returns   : Algorithm 3 + agent.py:154,188-190;  loss grads: network.py:81-94 (repaired)
//   heads bwd : d_h, d p_w/p_b/q_w/q_b
#include <cuda_bf16.h>

#include "common.cuh"
#include "../../include/asyncrl_b200_sarsa.h"
#include "../../include/asyncrl_b200_dueling.h"
#include "../../include/asyncrl_b200_double.h"
#include "../../include/asyncrl_b200_dueling_streams.h"
#include "../../include/asyncrl_b200_lstm.h"

namespace arl {

// two floats -> packed bf16 hi parts and packed bf16 lo parts (value = hi + lo to ~2^-17)
__device__ __forceinline__ void tc_split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  const float2 hf = __bfloat1622float2(h);
  const __nv_bfloat162 l = __floats2bfloat162_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

int reduce_partials(const float* partials, float* out, int num_partials, int n,
                    cudaStream_t stream);

// Philox4x32-10: second output word of the same block (used by the epsilon-greedy draw)
__device__ __forceinline__ void philox_two(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                           uint32_t k0, uint32_t k1, uint32_t& x0, uint32_t& x1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  x0 = c0; x1 = c1;
}

// ------------------------------- heads forward --------------------------------------------
// One warp per sample: lane l holds h[8l .. 8l+7] (the warp reads the 1-KB row as 32-byte pieces),
// the weights sit in shared memory as wt[(j*8 + e)*32 + l] = W[k = 8l + e][j] (conflict-free),
// every output is 8 FMAs per lane + a butterfly sum; lane j keeps logit j, the softmax runs
// across the lanes.  (First version: 16 samples per CTA staged in shared memory, one thread per
// (sample, output) walking 256 k serially: 10 us per 4096 samples, latency-bound.)
//
// The action draw after the heads is chosen by the last argument's type (common.cuh: SampleDraw or
// EgreedyDraw).  Dueling (Wang et al. 2016, "average" aggregator) makes the A-wide head the advantage
// stream and the 1-wide head the value stream: the row written to `logits` (and softmaxed into
// `probs`, and drawn from) is then Q_j = v + (adv_j - mean_k adv_k); `value` is v either way.
// Streams (dueling only): each stream has its own hidden layer, h is [N][512] = [h_v | h_a]; the
// advantage head reads h_a, the value head h_v, and the rest is the dueling kernel's.

// agent.py:142-144  ep_end + max(0., (ep_start - ep_end) * (ep_end_t - max(0., step - learn_start))
// / ep_end_t), in double, one correctly rounded operation at a time in Python's order (the _rn
// intrinsics keep the compiler from contracting a multiply and an add), then rounded to float once:
// the float the host computes as c_float(Agent.ep), bit for bit
__device__ __forceinline__ float egreedy_epsilon(const EgreedyDraw& d, int64_t step) {
  const double s = __dsub_rn((double)step, d.learn_start);
  const double m = s > 0.0 ? s : 0.0;
  const double f = __ddiv_rn(__dmul_rn(__dsub_rn(d.ep_start, d.ep_end), __dsub_rn(d.ep_end_t, m)), d.ep_end_t);
  return __double2float_rn(__dadd_rn(d.ep_end, f > 0.0 ? f : 0.0));
}

constexpr int kHfThreads = 256;
template <class Draw, bool Dueling, bool Streams = false>
__global__ void __launch_bounds__(kHfThreads)
heads_fwd_kernel(const float* __restrict__ pw, const float* __restrict__ pb,
                 const float* __restrict__ qw, const float* __restrict__ qb,
                 const float* __restrict__ h, float* __restrict__ logits,
                 float* __restrict__ probs, float* __restrict__ value, int64_t num_samples, int A,
                 int32_t* __restrict__ actions, uint64_t env_id_base, uint64_t step, uint64_t seed,
                 const int64_t* __restrict__ step_dev, int wait_first, Draw draw) {
  extern __shared__ __align__(16) float sm[];   // [A+1][8][32]
  // wait_first: the kernel before this one in the stream may have written the parameters (a
  // stand-alone arl_heads_forward right after an update): nothing is read before the wait
  if (wait_first) pdl_wait();
  const int J = A + 1;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 256 * J; i += kHfThreads) {
    const int j = i >> 8, e = (i >> 5) & 7, l = i & 31, k = l * 8 + e;
    sm[i] = j < A ? pw[k * A + j] : qw[k];
  }
  const float bias = lane < A ? pb[lane] : 0.f, qb0 = qb[0];
  __syncthreads();
  // launched with programmatic stream serialization behind the fc256 kernel (arl_fc_heads_forward):
  // everything above (the parameters -- not written by fc256, and whatever ran before fc256 had
  // completed when fc256 passed its own wait) overlaps fc256's tail; h and the step counter are
  // touched only after it has completed
  if (!wait_first) pdl_wait();
  if (actions != nullptr && step_dev != nullptr) step += (uint64_t)*step_dev;
  float ep = 0.f;
  if constexpr (Draw::kEgreedy) ep = step_dev != nullptr ? egreedy_epsilon(draw, (int64_t)step) : draw.ep;
  const int64_t stride = (int64_t)gridDim.x * (kHfThreads / 32);
  for (int64_t n = (int64_t)blockIdx.x * (kHfThreads / 32) + warp; n < num_samples; n += stride) {
    const float4* hp = reinterpret_cast<const float4*>(h + n * (Streams ? 512 : 256) + (Streams ? 256 : 0)) + lane * 2;
    const float4 x0 = hp[0], x1 = hp[1];
    float4 v0 = x0, v1 = x1;                       // the value head's input: h_v with Streams
    if constexpr (Streams) {
      const float4* vp = reinterpret_cast<const float4*>(h + n * 512) + lane * 2;
      v0 = vp[0]; v1 = vp[1];
    }
    float z = 0.f, zv = 0.f;
    for (int j = 0; j < J; ++j) {
      const float* w = sm + j * 256 + lane;
      const float4 y0 = Streams && j == A ? v0 : x0, y1 = Streams && j == A ? v1 : x1;
      float a0 = y0.x * w[0], a1 = y0.y * w[32];
      a0 = fmaf(y0.z, w[64], a0);  a1 = fmaf(y0.w, w[96], a1);
      a0 = fmaf(y1.x, w[128], a0); a1 = fmaf(y1.y, w[160], a1);
      a0 = fmaf(y1.z, w[192], a0); a1 = fmaf(y1.w, w[224], a1);
      const float t = warp_sum(a0 + a1);           // every lane gets the total
      if (j == lane) z = t;
      if (j == A) zv = t;
    }
    z += bias;
    if constexpr (Dueling) {
      // lane A holds the value head's sum: the mean runs over the lanes < A, one division by A
      const float m = warp_sum(lane < A ? z : 0.f) / (float)A;
      z = (zv + qb0) + (z - m);                       // TF: value + (advantage - reduce_mean(advantage))
    }
    float mx = lane < A ? z : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float ex = lane < A ? expf(z - mx) : 0.f;
    const float inv = 1.0f / warp_sum(ex);
    const float pj = ex * inv;
    if (lane < A) {
      logits[n * A + lane] = z;
      probs[n * A + lane] = pj;
    }
    if (lane == 0) value[n] = zv + qb0;
    if constexpr (Draw::kEgreedy) {
      // the draw of egreedy_actions_kernel on the logits just written: Philox block (env, step_lo,
      // step_hi, 1), word 0 -> u < ep, word 1 -> uniform action, else argmax (ties -> lowest index)
      uint32_t x0, x1;
      philox_two((uint32_t)(env_id_base + (uint64_t)n), (uint32_t)step, (uint32_t)(step >> 32), 1u,
                 (uint32_t)seed, (uint32_t)(seed >> 32), x0, x1);
      const float u = (float)(x0 >> 8) * 5.9604644775390625e-08f;     // 2^-24
      int a = 0;
      float best = __shfl_sync(0xffffffffu, z, 0);
      for (int j = 1; j < A; ++j) {
        const float q = __shfl_sync(0xffffffffu, z, j);
        if (q > best) { best = q; a = j; }
      }
      if (u < ep) a = (int)(((uint64_t)x1 * (uint64_t)A) >> 32);
      if (lane == 0) actions[n] = a;
    } else if (actions != nullptr) {
      // network.py:72 in the same launch: the draw of sample_actions_kernel (Philox4x32-10 keyed by
      // the global env id and the step; inverse CDF over the float32 running sum in index order)
      const uint32_t x = philox_first((uint32_t)(env_id_base + (uint64_t)n), (uint32_t)step,
                                      (uint32_t)(step >> 32), 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
      const float u = (float)(x >> 8) * 5.9604644775390625e-08f;       // 2^-24
      float c = 0.f;
      int a = A - 1;
      bool done = false;
      for (int j = 0; j < A; ++j) {
        const float p = __shfl_sync(0xffffffffu, pj, j);
        if (!done) {
          c = __fadd_rn(c, p);
          if (u < c) { a = j; done = true; }
        }
      }
      if (lane == 0) actions[n] = a;
    }
  }
}

// ------------------------------- action selection -----------------------------------------
// step_dev (optional): the step counter lives in device memory (a captured CUDA graph cannot carry
// a host value that changes on every launch); the Philox step is then *step_dev + step
__global__ void sample_actions_kernel(const float* __restrict__ probs, int32_t* __restrict__ actions,
                                      int num_envs, int A, uint64_t env_id_base, uint64_t step,
                                      uint64_t seed, const int64_t* __restrict__ step_dev) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= num_envs) return;
  if (step_dev != nullptr) step += (uint64_t)*step_dev;
  const uint32_t env = (uint32_t)(env_id_base + (uint64_t)b);
  const uint32_t x = philox_first(env, (uint32_t)step, (uint32_t)(step >> 32), 0u, (uint32_t)seed,
                                  (uint32_t)(seed >> 32));
  const float u = (float)(x >> 8) * 5.9604644775390625e-08f;       // 2^-24
  const float* p = probs + (size_t)b * A;
  float c = 0.f;
  int a = A - 1;
  for (int j = 0; j < A; ++j) {
    c = __fadd_rn(c, p[j]);
    if (u < c) { a = j; break; }
  }
  actions[b] = a;
}

__global__ void greedy_actions_kernel(const float* __restrict__ scores, int32_t* __restrict__ actions,
                                      int num_envs, int A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= num_envs) return;
  const float* p = scores + (size_t)b * A;
  int a = 0;
  float best = p[0];
  for (int j = 1; j < A; ++j)
    if (p[j] > best) { best = p[j]; a = j; }        // ties -> lowest index (tf.argmax)
  actions[b] = a;
}

// agent.py:141-151: with probability ep a uniformly random action, else argmax_a Q (ties -> lowest
// index).  The reference draws from Python's `random` (main.py:41); here the draw is the Philox
// block (env, step_lo, step_hi, 1): word 0 -> u < ep, word 1 -> action = floor(x1 * A / 2^32).
__global__ void egreedy_actions_kernel(const float* __restrict__ q, int32_t* __restrict__ actions,
                                       int num_envs, int A, float ep, uint64_t env_id_base,
                                       uint64_t step, uint64_t seed) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= num_envs) return;
  uint32_t x0, x1;
  philox_two((uint32_t)(env_id_base + (uint64_t)b), (uint32_t)step, (uint32_t)(step >> 32), 1u,
             (uint32_t)seed, (uint32_t)(seed >> 32), x0, x1);
  const float u = (float)(x0 >> 8) * 5.9604644775390625e-08f;      // 2^-24
  int a;
  if (u < ep) {
    a = (int)(((uint64_t)x1 * (uint64_t)A) >> 32);
  } else {
    const float* p = q + (size_t)b * A;
    a = 0;
    float best = p[0];
    for (int j = 1; j < A; ++j)
      if (p[j] > best) { best = p[j]; a = j; }
  }
  actions[b] = a;
}

// ------------------------------- loss-kernel pieces ---------------------------------------
// Shared by the three loss kernels below: the n-step return (A3C and n-step Q, so that their R is
// bit-identical by construction), and the max over a Q row, the dQ row and the loss sums (async-Q
// and n-step Q).

// Algorithm 3 + agent.py:154,188-190: R_t of sample (t, b) from the bootstrap R_T, the recurrence
// run from T-1 down to t -- the same operations in the same order as a walk over the whole rollout
// (identical bits), T - t fused multiply-adds
__device__ __forceinline__ float nstep_return(const float* rewards, const uint8_t* terminals, float R, int t,
                                              int T, int B, int b, float gamma, float rmin, float rmax) {
  for (int tt = T - 1; tt >= t; --tt) {
    const size_t m = (size_t)tt * B + b;
    const float r = fminf(fmaxf(rewards[m], rmin), rmax);               // agent.py:154
    R = fmaf(gamma * (1.0f - (terminals[m] ? 1.0f : 0.0f)), R, r);      // agent.py:190
  }
  return R;
}

// max_a q[a], fmaxf in index order
__device__ __forceinline__ float q_row_max(const float* q, int A) {
  float mx = q[0];
  for (int j = 1; j < A; ++j) mx = fmaxf(mx, q[j]);
  return mx;
}

// argmax_a q[a], ties -> lowest index (greedy_actions_kernel's rule, tf.argmax)
__device__ __forceinline__ int q_row_argmax(const float* q, int A) {
  int a = 0;
  float best = q[0];
  for (int j = 1; j < A; ++j)
    if (q[j] > best) { best = q[j]; a = j; }
  return a;
}

// the gradient of grad_scale * delta^2 w.r.t. the Q row: -2 * delta * grad_scale at the acted action
__device__ __forceinline__ void acted_dq_row(float* dq, int A, int a, float delta, float grad_scale) {
  for (int j = 0; j < A; ++j) dq[j] = j == a ? -2.0f * delta * grad_scale : 0.f;
}

// the same gradient through the dueling combine Q_j = v + adv_j - mean_k adv_k (heads_fwd_kernel):
// g = -2 * delta * grad_scale, d adv_j = g * ([j == a] - 1/A), d v = g
__device__ __forceinline__ void acted_dq_row(float* dadv, float* dv, int A, int a, float delta, float grad_scale) {
  const float g = -2.0f * delta * grad_scale;
  for (int j = 0; j < A; ++j) dadv[j] = g * ((j == a ? 1.f : 0.f) - 1.f / A);
  *dv = g;
}

// the loss kernels' gradient store: the dQ row, or with Dueling the advantage row and d value
template <bool Dueling>
__device__ __forceinline__ void store_dq(float* dq, float* dvalue, int64_t n, int A, int a, float delta,
                                         float grad_scale) {
  if constexpr (Dueling) acted_dq_row(dq + n * A, dvalue + n, A, a, delta, grad_scale);
  else acted_dq_row(dq + n * A, A, a, delta, grad_scale);
}

// loss_sums (optional) += {sum delta^2, sum Q(s)[a]}: a warp sum, then one atomic per warp
__device__ __forceinline__ void add_q_loss_sums(float* loss_sums, float s_loss, float s_q) {
  if (loss_sums) {
    s_loss = warp_sum(s_loss);
    s_q = warp_sum(s_q);
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(loss_sums + 0, s_loss);
      atomicAdd(loss_sums + 1, s_q);
    }
  }
}

// ------------------------------- async-Q loss gradients -----------------------------------
// agent.py:186-190, 310-314: target = clip(r) + (1 - terminal) * discount * max_a Q_target(s'),
// delta = target - Q(s)[a], loss = mean(delta^2)  ->  dQ[a] = -2 * delta * grad_scale.
// The three Q loss kernels take the head kind as a template argument and dvalue (Dueling only) last.
// Double (van Hasselt et al. 2016, Double DQN): the bootstrap is Q(s', a*; theta^-) with
// a* = argmax_a Q(s', a; theta) in place of max_a Q(s'; theta^-).  The online rows of s' are the
// rollout's own Q rows (q row n + B) for t < T-1 and q_online_T (row b) for t = T-1; these
// arguments come after dvalue, so the plain instantiations keep their parameter offsets.
template <bool Dueling, bool Double>
__global__ void q_lossgrad_kernel(const float* __restrict__ rewards,
                                  const uint8_t* __restrict__ terminals,
                                  const int32_t* __restrict__ actions, const float* __restrict__ q,
                                  const float* __restrict__ q_next, float* __restrict__ target,
                                  float* __restrict__ dq, float* __restrict__ loss_sums,
                                  int64_t num_samples, int A, float discount, float rmin, float rmax,
                                  float grad_scale, float* __restrict__ dvalue,
                                  const float* __restrict__ q_online_T, int B) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float s_loss = 0.f, s_q = 0.f;
  if (n < num_samples) {
    float mx;
    if constexpr (Double) {
      const int64_t m = n + B;                                           // sample (t + 1, b)
      const float* online = m < num_samples ? q + m * A : q_online_T + (m - num_samples) * A;
      mx = q_next[n * A + q_row_argmax(online, A)];
    } else {
      mx = q_row_max(q_next + n * A, A);
    }
    const float r = fminf(fmaxf(rewards[n], rmin), rmax);                 // agent.py:154
    const float tgt = fmaf((1.0f - (terminals[n] ? 1.0f : 0.0f)) * discount, mx, r);   // agent.py:190
    const int a = actions[n];
    const float delta = tgt - q[n * A + a];
    target[n] = tgt;
    store_dq<Dueling>(dq, dvalue, n, A, a, delta, grad_scale);
    s_loss = delta * delta;
    s_q = q[n * A + a];
  }
  add_q_loss_sums(loss_sums, s_loss, s_q);
}

// ------------------------------- returns + loss gradients ---------------------------------
// One thread per SAMPLE (t, b): the return recurrence is the only serial part, and it is T - t
// fused multiply-adds, so every thread just runs it from T-1 down to its own t (nstep_return) and
// then does the softmax / gradient work of its one sample.  (One thread per env walking all T
// samples: 32 CTAs for 4096 envs, 14.4 us.)
__global__ void returns_lossgrad_kernel(const float* __restrict__ rewards,
                                        const uint8_t* __restrict__ terminals,
                                        const int32_t* __restrict__ actions,
                                        const float* __restrict__ logits,
                                        const float* __restrict__ value,
                                        const float* __restrict__ v_boot, float* __restrict__ returns,
                                        float* __restrict__ dlogits, float* __restrict__ dvalue,
                                        float* __restrict__ loss_sums, int T, int B, int A,
                                        float gamma, float beta, float rmin, float rmax,
                                        float grad_scale) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float s_pol = 0.f, s_val = 0.f, s_ent = 0.f;
  pdl_wait();
  if (n < (int64_t)T * B) {
    const int t = (int)(n / B), b = (int)(n - (int64_t)t * B);
    const float R = nstep_return(rewards, terminals, v_boot[b], t, T, B, b, gamma, rmin, rmax);
    returns[n] = R;
    const float* z = logits + n * A;
    float zz[ARL_MAX_ACTIONS];
    float mx = z[0];
#pragma unroll 1
    for (int j = 0; j < A; ++j) { zz[j] = z[j]; mx = fmaxf(mx, zz[j]); }
    float den = 0.f;
    for (int j = 0; j < A; ++j) den += expf(zz[j] - mx);
    const float lse = mx + logf(den);
    float ent = 0.f;
    for (int j = 0; j < A; ++j) {
      const float lp = zz[j] - lse;
      ent -= expf(lp) * lp;                                             // network.py:69
    }
    const float v = value[n];
    const float adv = R - v;
    const int a = actions[n];
    float* dz = dlogits + n * A;
    for (int j = 0; j < A; ++j) {
      const float lp = zz[j] - lse, p = expf(lp);
      const float g = -adv * ((j == a ? 1.0f : 0.0f) - p) + beta * p * (lp + ent);
      dz[j] = g * grad_scale;
    }
    dvalue[n] = -adv * grad_scale;                                      // d/dV (R-V)^2/2
    s_pol = -(zz[a] - lse) * adv - beta * ent;                          // network.py:87-88
    s_val = 0.5f * adv * adv;                                           // network.py:91
    s_ent = ent;
  }
  if (loss_sums) {
    s_pol = warp_sum(s_pol); s_val = warp_sum(s_val); s_ent = warp_sum(s_ent);
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(loss_sums + 0, s_pol);
      atomicAdd(loss_sums + 1, s_val);
      atomicAdd(loss_sums + 2, s_ent);
    }
  }
}

// ------------------------------- n-step Q loss gradients ----------------------------------
// Asynchronous n-step Q-learning (Mnih et al. 2016): one thread per SAMPLE (t, b) as in
// returns_lossgrad_kernel, the same return recurrence started from max_a Q(s_T; theta^-), then the
// async-Q gradient of the acted action.  Double: started from Q(s_T, a*; theta^-) with
// a* = argmax_a Q(s_T, a; theta), the online row b of q_online_T (an argument after dvalue, as in
// q_lossgrad_kernel).
template <bool Dueling, bool Double>
__global__ void nstep_q_lossgrad_kernel(const float* __restrict__ rewards,
                                        const uint8_t* __restrict__ terminals,
                                        const int32_t* __restrict__ actions, const float* __restrict__ q,
                                        const float* __restrict__ q_boot, float* __restrict__ returns,
                                        float* __restrict__ dq, float* __restrict__ loss_sums, int T, int B,
                                        int A, float gamma, float rmin, float rmax, float grad_scale,
                                        float* __restrict__ dvalue, const float* __restrict__ q_online_T) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float s_loss = 0.f, s_q = 0.f;
  pdl_wait();
  if (n < (int64_t)T * B) {
    const int t = (int)(n / B), b = (int)(n - (int64_t)t * B);
    float boot;
    if constexpr (Double) boot = q_boot[(size_t)b * A + q_row_argmax(q_online_T + (size_t)b * A, A)];
    else boot = q_row_max(q_boot + (size_t)b * A, A);
    const float R = nstep_return(rewards, terminals, boot, t, T, B, b, gamma, rmin, rmax);
    returns[n] = R;
    const int a = actions[n];
    const float qa = q[n * A + a];
    const float delta = R - qa;
    store_dq<Dueling>(dq, dvalue, n, A, a, delta, grad_scale);
    s_loss = delta * delta;
    s_q = qa;
  }
  add_q_loss_sums(loss_sums, s_loss, s_q);
}

// ------------------------------- one-step Sarsa loss gradients ----------------------------
// Asynchronous one-step Sarsa (Mnih et al. 2016): q_lossgrad_kernel's target expression with
// Q(s', a'; theta^-) of the action a' taken in s' in place of max_a.  actions holds a_0 .. a_T, so
// the next action of sample n is actions[n + B] for every t, the last step included.
template <bool Dueling>
__global__ void sarsa_lossgrad_kernel(const float* __restrict__ rewards,
                                      const uint8_t* __restrict__ terminals,
                                      const int32_t* __restrict__ actions, const float* __restrict__ q,
                                      const float* __restrict__ q_next, float* __restrict__ target,
                                      float* __restrict__ dq, float* __restrict__ loss_sums, int T, int B,
                                      int A, float gamma, float rmin, float rmax, float grad_scale,
                                      float* __restrict__ dvalue) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float s_loss = 0.f, s_q = 0.f;
  pdl_wait();
  if (n < (int64_t)T * B) {
    const float qn = q_next[n * A + actions[n + B]];
    const float r = fminf(fmaxf(rewards[n], rmin), rmax);                 // agent.py:154
    const float tgt = fmaf((1.0f - (terminals[n] ? 1.0f : 0.0f)) * gamma, qn, r);      // agent.py:190
    const int a = actions[n];
    const float qa = q[n * A + a];
    const float delta = tgt - qa;
    target[n] = tgt;
    store_dq<Dueling>(dq, dvalue, n, A, a, delta, grad_scale);
    s_loss = delta * delta;
    s_q = qa;
  }
  add_q_loss_sums(loss_sums, s_loss, s_q);
}

// ------------------------------- heads backward -------------------------------------------
// CTA = 256 threads (thread k owns hidden unit k).  Per sample: d_h[n][k] = (h>0) * sum_j
// dz[n][j]*Wcat[k][j];  dWcat[k][j] += h[n][k]*dz[n][j];  dbcat[j] += dz[n][j].
// Partials per CTA -> workspace [grid][256*J + J], reduced deterministically afterwards.
// d_h leaves as split bf16 in 16-byte chunk vectors (gemm_tc.cuh SplitMat), TWICE, because its two
// consumers reduce over different axes and a bulk copy wants long contiguous runs:
//   dhs  [hi|lo][32 column chunks][num_samples rows][8 columns]   fc dgrad's A operand (K-major)
//   dhsT [hi|lo][ceil(N/8) sample chunks][256 column rows][8 samples]   fc wgrad's B operand
//        (K-major over samples: one run = all 256 columns of 8 samples = 4 KB; samples >= N zero)
// 32 samples are staged in shared memory so that a warp writes 512 contiguous bytes either way.
// Relu = false (the LSTM network, include/asyncrl_b200_lstm.h: h = sigmoid(o) tanh(c) can be negative):
// no mask, and d_h leaves as plain f32 [num_samples][256] in dhs (times tensor_scale), the form the
// LSTM cell backward reads; dhsT is not written.
constexpr int kHbChunk = 64, kHbSub = 32;
template <int JMAX, bool Relu = true>
__global__ void __launch_bounds__(256)
heads_bwd_kernel(const float* __restrict__ pw, const float* __restrict__ qw,
                 const float* __restrict__ h, const float* __restrict__ dlogits,
                 const float* __restrict__ dvalue, uint8_t* __restrict__ dhs,
                 uint8_t* __restrict__ dhsT, float* __restrict__ partials, int64_t num_samples,
                 int64_t per, int A, float tensor_scale) {
  __shared__ float dzs[kHbChunk][JMAX];
  __shared__ float dt[kHbSub][257];
  const int J = A + 1;
  const int k = threadIdx.x;
  pdl_wait();      // before the weights too: the kernel before this one may be the update
  float w[JMAX], acc[JMAX];
#pragma unroll
  for (int j = 0; j < JMAX; ++j) {
    w[j] = j < A ? pw[k * A + j] : (j == A ? qw[k] : 0.f);
    acc[j] = 0.f;
  }
  float bacc = 0.f;                                   // thread j < J: sum of dz[:, j]
  const int64_t beg = per * blockIdx.x;                // per is a multiple of 8: sample chunks are not split
  const int64_t end = beg + per < num_samples ? beg + per : num_samples;
  const int64_t lo_part = (int64_t)32 * num_samples * 16;
  const int64_t lo_partT = ((num_samples + 7) / 8) * 256 * 16;
  for (int64_t c0 = beg; c0 < end; c0 += kHbChunk) {
    const int nc = (int)(end - c0 < kHbChunk ? end - c0 : kHbChunk);
    __syncthreads();
    for (int i = k; i < nc * J; i += 256) {
      const int s = i / J, j = i - s * J;
      dzs[s][j] = j < A ? dlogits[(c0 + s) * A + j] : dvalue[c0 + s];
    }
    __syncthreads();
    for (int s0 = 0; s0 < nc; s0 += kHbSub) {
      const int ns = nc - s0 < kHbSub ? nc - s0 : kHbSub;
      // all h values of the sub-chunk are requested before the first is used (one load per sample
      // in a serial loop left this kernel latency-bound: 32 us for 63 MB of traffic)
      float hvs[kHbSub];
#pragma unroll
      for (int s = 0; s < kHbSub; ++s) hvs[s] = s < ns ? h[(c0 + s0 + s) * 256 + k] : 0.f;
#pragma unroll
      for (int s = 0; s < kHbSub; ++s) {
        if (s < ns) {
          const float hv = hvs[s];
          float d = 0.f;
#pragma unroll
          for (int j = 0; j < JMAX; ++j) {
            if (j < J) {
              const float g = dzs[s0 + s][j];
              d = fmaf(g, w[j], d);
              acc[j] = fmaf(hv, g, acc[j]);
            }
          }
          dt[s][k] = !Relu || hv > 0.f ? d * tensor_scale : 0.f;       // d_h leaves scaled (arl_backward)
        }
      }
      if constexpr (!Relu) {                          // column k of the staging tile is this thread's own
        __syncthreads();
        for (int s = 0; s < ns; ++s) reinterpret_cast<float*>(dhs)[(c0 + s0 + s) * 256 + k] = dt[s][k];
        continue;
      }
      __syncthreads();
      for (int v = k; v < 32 * kHbSub; v += 256) {
        const int s = v % kHbSub, kc = v / kHbSub;
        if (s < ns) {
          const float* x = &dt[s][kc * 8];
          uint4 hi, lo;
          tc_split2(x[0], x[1], hi.x, lo.x);
          tc_split2(x[2], x[3], hi.y, lo.y);
          tc_split2(x[4], x[5], hi.z, lo.z);
          tc_split2(x[6], x[7], hi.w, lo.w);
          uint8_t* d = dhs + ((int64_t)kc * num_samples + c0 + s0 + s) * 16;
          *reinterpret_cast<uint4*>(d) = hi;
          *reinterpret_cast<uint4*>(d + lo_part) = lo;
        }
      }
      // transposed copy: thread k = column k of each of the (up to 4) sample chunks
      for (int sc = 0; sc * 8 < ns; ++sc) {
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = sc * 8 + e < ns ? dt[sc * 8 + e][k] : 0.f;
        uint4 hi, lo;
        tc_split2(x[0], x[1], hi.x, lo.x);
        tc_split2(x[2], x[3], hi.y, lo.y);
        tc_split2(x[4], x[5], hi.z, lo.z);
        tc_split2(x[6], x[7], hi.w, lo.w);
        uint8_t* d = dhsT + (((c0 + s0) / 8 + sc) * 256 + k) * 16;
        *reinterpret_cast<uint4*>(d) = hi;
        *reinterpret_cast<uint4*>(d + lo_partT) = lo;
      }
      __syncthreads();
    }
    if (k < J)
      for (int s = 0; s < nc; ++s) bacc += dzs[s][k];
  }
  float* out = partials + (size_t)blockIdx.x * (256 * J + J);
  // layout of a partial: p_w [256][A] | p_b [A] | q_w [256] | q_b [1]  (flat-buffer order)
#pragma unroll
  for (int j = 0; j < JMAX; ++j) {
    if (j < A) out[k * A + j] = acc[j];
    else if (j == A) out[256 * A + A + k] = acc[j];
  }
  if (k < A) out[256 * A + k] = bacc;
  else if (k == A) out[256 * A + A + 256] = bacc;
}

// heads_bwd_kernel for the dueling streams: h [N][512] = [h_v | h_a]; the advantage head (p_w, j < A)
// reads and feeds h_a, the value head (q_w, j = A) h_v.  d_h = [d_h_v | d_h_a] leaves as ONE split
// block of 512 columns, twice, as there:
//   dhs  [hi|lo][64 column chunks: 32 of d_h_v, then 32 of d_h_a][num_samples rows][8 columns]
//   dhsT [hi|lo][ceil(N/8) sample chunks][512 column rows][8 samples]
// 16 samples are staged per stream (two staging tiles of kHbSub rows would not fit 48 KB).
constexpr int kHbSubS = 16;
template <int JMAX>
__global__ void __launch_bounds__(256, 1)
heads_bwd_streams_kernel(const float* __restrict__ pw, const float* __restrict__ qw,
                         const float* __restrict__ h, const float* __restrict__ dlogits,
                         const float* __restrict__ dvalue, uint8_t* __restrict__ dhs,
                         uint8_t* __restrict__ dhsT, float* __restrict__ partials, int64_t num_samples,
                         int64_t per, int A, float tensor_scale) {
  __shared__ float dzs[kHbChunk][JMAX];
  __shared__ float dt[2][kHbSubS][257];               // [stream: 0 = v, 1 = a][sample][column]
  const int J = A + 1;
  const int k = threadIdx.x;
  pdl_wait();
  float w[JMAX], acc[JMAX];                          // the advantage head's columns (j < A)
#pragma unroll
  for (int j = 0; j < JMAX; ++j) {
    w[j] = j < A ? pw[k * A + j] : 0.f;
    acc[j] = 0.f;
  }
  const float wv = qw[k];                            // the value head's column
  float accv = 0.f, bacc = 0.f;
  const int64_t beg = per * blockIdx.x;
  const int64_t end = beg + per < num_samples ? beg + per : num_samples;
  const int64_t lo_part = (int64_t)64 * num_samples * 16;
  const int64_t lo_partT = ((num_samples + 7) / 8) * 512 * 16;
  for (int64_t c0 = beg; c0 < end; c0 += kHbChunk) {
    const int nc = (int)(end - c0 < kHbChunk ? end - c0 : kHbChunk);
    __syncthreads();
    for (int i = k; i < nc * J; i += 256) {
      const int s = i / J, j = i - s * J;
      dzs[s][j] = j < A ? dlogits[(c0 + s) * A + j] : dvalue[c0 + s];
    }
    __syncthreads();
    for (int s0 = 0; s0 < nc; s0 += kHbSubS) {
      const int ns = nc - s0 < kHbSubS ? nc - s0 : kHbSubS;
      float hvs[kHbSubS], has[kHbSubS];
#pragma unroll
      for (int s = 0; s < kHbSubS; ++s) {
        hvs[s] = s < ns ? h[(c0 + s0 + s) * 512 + k] : 0.f;
        has[s] = s < ns ? h[(c0 + s0 + s) * 512 + 256 + k] : 0.f;
      }
#pragma unroll
      for (int s = 0; s < kHbSubS; ++s) {
        if (s < ns) {
          const float hv = hvs[s], ha = has[s];
          float da = 0.f;
#pragma unroll
          for (int j = 0; j < JMAX; ++j) {
            if (j < A) {
              const float g = dzs[s0 + s][j];
              da = fmaf(g, w[j], da);
              acc[j] = fmaf(ha, g, acc[j]);
            }
          }
          const float gv = dzs[s0 + s][A], dv = gv * wv;
          accv = fmaf(hv, gv, accv);
          dt[0][s][k] = hv > 0.f ? dv * tensor_scale : 0.f;     // d_h leaves scaled (arl_backward)
          dt[1][s][k] = ha > 0.f ? da * tensor_scale : 0.f;
        }
      }
      __syncthreads();
      for (int v = k; v < 64 * kHbSubS; v += 256) {
        const int s = v % kHbSubS, kc = v / kHbSubS;           // kc: chunk of [d_h_v | d_h_a]
        if (s < ns) {
          const float* x = &dt[kc >> 5][s][(kc & 31) * 8];
          uint4 hi, lo;
          tc_split2(x[0], x[1], hi.x, lo.x);
          tc_split2(x[2], x[3], hi.y, lo.y);
          tc_split2(x[4], x[5], hi.z, lo.z);
          tc_split2(x[6], x[7], hi.w, lo.w);
          uint8_t* d = dhs + ((int64_t)kc * num_samples + c0 + s0 + s) * 16;
          *reinterpret_cast<uint4*>(d) = hi;
          *reinterpret_cast<uint4*>(d + lo_part) = lo;
        }
      }
      // transposed copy: thread k = column k of each stream and each of the (up to 2) sample chunks
      for (int sc = 0; sc * 8 < ns; ++sc) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float x[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] = sc * 8 + e < ns ? dt[q][sc * 8 + e][k] : 0.f;
          uint4 hi, lo;
          tc_split2(x[0], x[1], hi.x, lo.x);
          tc_split2(x[2], x[3], hi.y, lo.y);
          tc_split2(x[4], x[5], hi.z, lo.z);
          tc_split2(x[6], x[7], hi.w, lo.w);
          uint8_t* d = dhsT + (((c0 + s0) / 8 + sc) * 512 + q * 256 + k) * 16;
          *reinterpret_cast<uint4*>(d) = hi;
          *reinterpret_cast<uint4*>(d + lo_partT) = lo;
        }
      }
      __syncthreads();
    }
    if (k < J)
      for (int s = 0; s < nc; ++s) bacc += dzs[s][k];
  }
  float* out = partials + (size_t)blockIdx.x * (256 * J + J);
  // layout of a partial: p_w [256][A] | p_b [A] | q_w [256] | q_b [1]  (flat-buffer order)
#pragma unroll
  for (int j = 0; j < JMAX; ++j)
    if (j < A) out[k * A + j] = acc[j];
  out[256 * A + A + k] = accv;
  if (k < A) out[256 * A + k] = bacc;
  else if (k == A) out[256 * A + A + 256] = bacc;
}

// ------------------------------- env-step bookkeeping --------------------------------------
// GymEnvironment.act for action_repeat == 1 (environment.py:78-96): a life lost in training costs
// one reward point and ends the episode.  One launch instead of five elementwise ones.
__global__ void act_update_kernel(const float* __restrict__ step_reward,
                                  const uint8_t* __restrict__ step_terminal,
                                  const int32_t* __restrict__ lives_before,
                                  const int32_t* __restrict__ lives_after, int is_training,
                                  float* __restrict__ reward, uint8_t* __restrict__ terminal, int n) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  if (b >= n) return;
  const bool lost = is_training && lives_before[b] > lives_after[b];
  reward[b] = step_reward[b] - (lost ? 1.0f : 0.0f);
  terminal[b] = (step_terminal[b] != 0 || lost) ? 1 : 0;
}
// Agent.observe's rollout append (agent.py:158-160): reward and terminal of this step -> slot t
__global__ void observe_store_kernel(const float* __restrict__ reward, const uint8_t* __restrict__ terminal,
                                     float* __restrict__ reward_slot, uint8_t* __restrict__ terminal_slot,
                                     int n, int64_t* step_counter, int64_t inc) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  if (b == 0 && step_counter != nullptr) *step_counter += inc;      // agent.py:55: the loop's step
  if (b >= n) return;
  reward_slot[b] = reward[b];
  terminal_slot[b] = terminal[b] != 0 ? 1 : 0;
}

int heads_init() {
  const int smem = (int)((ARL_MAX_ACTIONS + 1) * 256 * sizeof(float));
  ARL_CUDA(cudaFuncSetAttribute(heads_fwd_kernel<SampleDraw, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  ARL_CUDA(cudaFuncSetAttribute(heads_fwd_kernel<EgreedyDraw, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  ARL_CUDA(cudaFuncSetAttribute(heads_fwd_kernel<SampleDraw, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  ARL_CUDA(cudaFuncSetAttribute(heads_fwd_kernel<EgreedyDraw, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  ARL_CUDA(cudaFuncSetAttribute(heads_fwd_kernel<SampleDraw, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                smem));
  ARL_CUDA(cudaFuncSetAttribute(heads_fwd_kernel<EgreedyDraw, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                smem));
  return ARL_OK;
}

}  // namespace arl

using namespace arl;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

namespace arl {
// heads + softmax + the draw; wait_first = 0 behind the fc256 kernel (fc_heads_forward), 1 stand-alone;
// Dueling: the Q row of the dueling combine (heads_fwd_kernel); Streams: h is [N][512] = [h_v | h_a]
template <class Draw, bool Dueling, bool Streams = false>
int heads_forward(const float* params, int action_size, const float* h, float* logits, float* probs, float* value,
                  int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev, uint64_t seed,
                  int64_t num_samples, int wait_first, Draw draw, cudaStream_t st) {
  const ParamLayout L = param_layout(action_size);
  const size_t smem = (size_t)(action_size + 1) * 256 * sizeof(float);
  const int64_t ctas = (num_samples + kHfThreads / 32 - 1) / (kHfThreads / 32);   // one warp per sample
  // up to 4 CTAs per SM: one env step of 4096 samples is ONE round of warps (two rounds cost a second
  // exposed load latency)
  const int grid = (int)(ctas < 4LL * num_sms() ? ctas : 4LL * num_sms());
  ARL_CUDA(launch_pdl(heads_fwd_kernel<Draw, Dueling, Streams>, dim3(grid), dim3(kHfThreads), smem, st, params + L.off[T_PW],
                      params + L.off[T_PB], params + L.off[T_QW], params + L.off[T_QB], h, logits, probs, value,
                      num_samples, action_size, actions, (uint64_t)env_id_base, (uint64_t)step, seed, step_dev,
                      wait_first, draw));
  ARL_LAUNCH_CHECK("heads_fwd_kernel");
  return ARL_OK;
}
template int heads_forward<SampleDraw, false>(const float*, int, const float*, float*, float*, float*, int32_t*,
                                             int64_t, int64_t, const int64_t*, uint64_t, int64_t, int, SampleDraw,
                                             cudaStream_t);
template int heads_forward<EgreedyDraw, false>(const float*, int, const float*, float*, float*, float*, int32_t*,
                                              int64_t, int64_t, const int64_t*, uint64_t, int64_t, int, EgreedyDraw,
                                              cudaStream_t);
template int heads_forward<SampleDraw, true>(const float*, int, const float*, float*, float*, float*, int32_t*,
                                            int64_t, int64_t, const int64_t*, uint64_t, int64_t, int, SampleDraw,
                                            cudaStream_t);
template int heads_forward<EgreedyDraw, true>(const float*, int, const float*, float*, float*, float*, int32_t*,
                                             int64_t, int64_t, const int64_t*, uint64_t, int64_t, int, EgreedyDraw,
                                             cudaStream_t);
template int heads_forward<SampleDraw, true, true>(const float*, int, const float*, float*, float*, float*, int32_t*,
                                                  int64_t, int64_t, const int64_t*, uint64_t, int64_t, int,
                                                  SampleDraw, cudaStream_t);
template int heads_forward<EgreedyDraw, true, true>(const float*, int, const float*, float*, float*, float*,
                                                   int32_t*, int64_t, int64_t, const int64_t*, uint64_t, int64_t, int,
                                                   EgreedyDraw, cudaStream_t);
}  // namespace arl

extern "C" int arl_heads_forward(const float* params, int action_size, const float* h,
                                 float* logits, float* probs, float* value, int64_t num_samples,
                                 void* stream) {
  ARL_REQUIRE(params && h && logits && probs && value, "arl_heads_forward: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_heads_forward: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_samples >= 0, "arl_heads_forward: negative size");
  ARL_REQUIRE(aligned16(h), "arl_heads_forward: h must be 16-byte aligned");
  if (num_samples == 0) return ARL_OK;
  return heads_forward<SampleDraw, false>(params, action_size, h, logits, probs, value, nullptr, 0, 0, nullptr, 0,
                                          num_samples, /*wait_first=*/1, SampleDraw{}, (cudaStream_t)stream);
}

extern "C" int arl_sample_actions(const float* probs, int32_t* actions, int num_envs,
                                  int action_size, int64_t env_id_base, int64_t step, uint64_t seed,
                                  void* stream) {
  ARL_REQUIRE(probs && actions, "arl_sample_actions: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_sample_actions: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_envs >= 0 && env_id_base >= 0 && step >= 0, "arl_sample_actions: negative argument");
  if (num_envs == 0) return ARL_OK;
  sample_actions_kernel<<<(num_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      probs, actions, num_envs, action_size, (uint64_t)env_id_base, (uint64_t)step, seed, nullptr);
  ARL_LAUNCH_CHECK("sample_actions_kernel");
  return ARL_OK;
}

extern "C" int arl_sample_actions_dev(const float* probs, int32_t* actions, int num_envs,
                                      int action_size, int64_t env_id_base, const int64_t* step_dev,
                                      uint64_t seed, void* stream) {
  ARL_REQUIRE(probs && actions && step_dev, "arl_sample_actions_dev: null pointer");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_sample_actions_dev: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_envs >= 0 && env_id_base >= 0, "arl_sample_actions_dev: negative argument");
  if (num_envs == 0) return ARL_OK;
  sample_actions_kernel<<<(num_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      probs, actions, num_envs, action_size, (uint64_t)env_id_base, 0ull, seed, step_dev);
  ARL_LAUNCH_CHECK("sample_actions_kernel");
  return ARL_OK;
}

namespace arl {
__global__ void step_advance_kernel(int64_t* counter, int64_t inc) { *counter += inc; }
}  // namespace arl

extern "C" int arl_step_advance(int64_t* counter, int64_t inc, void* stream) {
  ARL_REQUIRE(counter, "arl_step_advance: null pointer");
  step_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter, inc);
  ARL_LAUNCH_CHECK("step_advance_kernel");
  return ARL_OK;
}

extern "C" int arl_greedy_actions(const float* scores, int32_t* actions, int num_envs,
                                  int action_size, void* stream) {
  ARL_REQUIRE(scores && actions, "arl_greedy_actions: null pointer");
  ARL_REQUIRE(action_size >= 1 && num_envs >= 0, "arl_greedy_actions: bad size");
  if (num_envs == 0) return ARL_OK;
  greedy_actions_kernel<<<(num_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      scores, actions, num_envs, action_size);
  ARL_LAUNCH_CHECK("greedy_actions_kernel");
  return ARL_OK;
}

extern "C" int arl_egreedy_actions(const float* q, int32_t* actions, int num_envs, int action_size,
                                   float ep, int64_t env_id_base, int64_t step, uint64_t seed,
                                   void* stream) {
  ARL_REQUIRE(q && actions, "arl_egreedy_actions: null pointer");
  ARL_REQUIRE(num_envs >= 0, "arl_egreedy_actions: negative size");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_egreedy_actions: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(ep >= 0.f && ep <= 1.f, "arl_egreedy_actions: ep %f outside [0,1]", (double)ep);
  if (num_envs == 0) return ARL_OK;
  egreedy_actions_kernel<<<(num_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      q, actions, num_envs, action_size, ep, (uint64_t)env_id_base, (uint64_t)step, seed);
  ARL_LAUNCH_CHECK("egreedy_actions_kernel");
  return ARL_OK;
}

// The Q loss entries: one launcher per learner for both head kinds and both targets (fn = the C
// entry's name, for errors; q_online_T and num_envs: Double only)
template <bool Dueling, bool Double = false>
static int q_lossgrad(const char* fn, const float* rewards, const uint8_t* terminals, const int32_t* actions,
                      const float* q, const float* q_next, float* target, float* dq, float* dvalue,
                      float* loss_sums, int64_t num_samples, int action_size, float discount, float reward_min,
                      float reward_max, float grad_scale, void* stream, const float* q_online_T = nullptr,
                      int num_envs = 0) {
  ARL_REQUIRE(rewards && terminals && actions && q && q_next && target && dq && (dvalue || !Dueling) &&
                  (q_online_T || !Double),
              "%s: null pointer", fn);
  ARL_REQUIRE(num_samples >= 0, "%s: negative size", fn);
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "%s: action_size %d outside [1,%d]", fn, action_size, ARL_MAX_ACTIONS);
  if (num_samples == 0) return ARL_OK;
  q_lossgrad_kernel<Dueling, Double><<<(unsigned)((num_samples + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      rewards, terminals, actions, q, q_next, target, dq, loss_sums, num_samples, action_size,
      discount, reward_min, reward_max, grad_scale, dvalue, q_online_T, num_envs);
  ARL_LAUNCH_CHECK("q_lossgrad_kernel");
  return ARL_OK;
}

extern "C" int arl_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                              const float* q, const float* q_next, float* target, float* dq,
                              float* loss_sums, int64_t num_samples, int action_size, float discount,
                              float reward_min, float reward_max, float grad_scale, void* stream) {
  return q_lossgrad<false>("arl_q_lossgrad", rewards, terminals, actions, q, q_next, target, dq, nullptr,
                           loss_sums, num_samples, action_size, discount, reward_min, reward_max, grad_scale,
                           stream);
}

extern "C" int arl_q_lossgrad_dueling(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                      const float* q, const float* q_next, float* target, float* dq,
                                      float* dvalue, float* loss_sums, int64_t num_samples, int action_size,
                                      float discount, float reward_min, float reward_max, float grad_scale,
                                      void* stream) {
  return q_lossgrad<true>("arl_q_lossgrad_dueling", rewards, terminals, actions, q, q_next, target, dq, dvalue,
                          loss_sums, num_samples, action_size, discount, reward_min, reward_max, grad_scale,
                          stream);
}

// Double DQN targets (include/asyncrl_b200_double.h): t_max x num_envs samples, so that the kernel
// knows which rows are the last step
template <bool Dueling>
static int double_q_lossgrad(const char* fn, const float* rewards, const uint8_t* terminals, const int32_t* actions,
                             const float* q, const float* q_next, const float* q_online_T, float* target, float* dq,
                             float* dvalue, float* loss_sums, int t_max, int num_envs, int action_size,
                             float discount, float reward_min, float reward_max, float grad_scale, void* stream) {
  ARL_REQUIRE(t_max >= 0 && num_envs >= 0, "%s: negative size", fn);
  return q_lossgrad<Dueling, true>(fn, rewards, terminals, actions, q, q_next, target, dq, dvalue, loss_sums,
                                   (int64_t)t_max * num_envs, action_size, discount, reward_min, reward_max,
                                   grad_scale, stream, q_online_T, num_envs);
}

extern "C" int arl_double_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                     const float* q, const float* q_next, const float* q_online_T, float* target,
                                     float* dq, float* loss_sums, int t_max, int num_envs, int action_size,
                                     float discount, float reward_min, float reward_max, float grad_scale,
                                     void* stream) {
  return double_q_lossgrad<false>("arl_double_q_lossgrad", rewards, terminals, actions, q, q_next, q_online_T,
                                  target, dq, nullptr, loss_sums, t_max, num_envs, action_size, discount,
                                  reward_min, reward_max, grad_scale, stream);
}

extern "C" int arl_double_q_lossgrad_dueling(const float* rewards, const uint8_t* terminals,
                                             const int32_t* actions, const float* q, const float* q_next,
                                             const float* q_online_T, float* target, float* dq, float* dvalue,
                                             float* loss_sums, int t_max, int num_envs, int action_size,
                                             float discount, float reward_min, float reward_max, float grad_scale,
                                             void* stream) {
  return double_q_lossgrad<true>("arl_double_q_lossgrad_dueling", rewards, terminals, actions, q, q_next,
                                 q_online_T, target, dq, dvalue, loss_sums, t_max, num_envs, action_size, discount,
                                 reward_min, reward_max, grad_scale, stream);
}

extern "C" int arl_returns_lossgrad(const float* rewards, const uint8_t* terminals,
                                    const int32_t* actions, const float* logits, const float* value,
                                    const float* v_boot, float* returns, float* dlogits,
                                    float* dvalue, float* loss_sums, int t_max, int num_envs,
                                    int action_size, float gamma, float beta, float reward_min,
                                    float reward_max, float grad_scale, void* stream) {
  ARL_REQUIRE(rewards && terminals && actions && logits && value && v_boot && returns && dlogits &&
                  dvalue,
              "arl_returns_lossgrad: null pointer");
  ARL_REQUIRE(t_max >= 0 && num_envs >= 0, "arl_returns_lossgrad: negative size");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_returns_lossgrad: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  if (t_max == 0 || num_envs == 0) return ARL_OK;
  const int64_t total = (int64_t)t_max * num_envs;
  ARL_CUDA(launch_pdl(returns_lossgrad_kernel, dim3((unsigned)((total + 127) / 128)), dim3(128), 0,
                      (cudaStream_t)stream, rewards, terminals, actions, logits, value, v_boot, returns, dlogits,
                      dvalue, loss_sums, t_max, num_envs, action_size, gamma, beta, reward_min, reward_max,
                      grad_scale));
  ARL_LAUNCH_CHECK("returns_lossgrad_kernel");
  return ARL_OK;
}

template <bool Dueling, bool Double = false>
static int nstep_q_lossgrad(const char* fn, const float* rewards, const uint8_t* terminals, const int32_t* actions,
                            const float* q, const float* q_boot, float* returns, float* dq, float* dvalue,
                            float* loss_sums, int t_max, int num_envs, int action_size, float gamma,
                            float reward_min, float reward_max, float grad_scale, void* stream,
                            const float* q_online_T = nullptr) {
  ARL_REQUIRE(rewards && terminals && actions && q && q_boot && returns && dq && (dvalue || !Dueling) &&
                  (q_online_T || !Double),
              "%s: null pointer", fn);
  ARL_REQUIRE(t_max >= 0 && num_envs >= 0, "%s: negative size", fn);
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "%s: action_size %d outside [1,%d]", fn, action_size, ARL_MAX_ACTIONS);
  if (t_max == 0 || num_envs == 0) return ARL_OK;
  const int64_t total = (int64_t)t_max * num_envs;
  ARL_CUDA(launch_pdl(nstep_q_lossgrad_kernel<Dueling, Double>, dim3((unsigned)((total + 127) / 128)), dim3(128),
                      0, (cudaStream_t)stream, rewards, terminals, actions, q, q_boot, returns, dq, loss_sums, t_max,
                      num_envs, action_size, gamma, reward_min, reward_max, grad_scale, dvalue, q_online_T));
  ARL_LAUNCH_CHECK("nstep_q_lossgrad_kernel");
  return ARL_OK;
}

extern "C" int arl_nstep_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                    const float* q, const float* q_boot, float* returns, float* dq,
                                    float* loss_sums, int t_max, int num_envs, int action_size, float gamma,
                                    float reward_min, float reward_max, float grad_scale, void* stream) {
  return nstep_q_lossgrad<false>("arl_nstep_q_lossgrad", rewards, terminals, actions, q, q_boot, returns, dq,
                                 nullptr, loss_sums, t_max, num_envs, action_size, gamma, reward_min, reward_max,
                                 grad_scale, stream);
}

extern "C" int arl_nstep_q_lossgrad_dueling(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                            const float* q, const float* q_boot, float* returns, float* dq,
                                            float* dvalue, float* loss_sums, int t_max, int num_envs,
                                            int action_size, float gamma, float reward_min, float reward_max,
                                            float grad_scale, void* stream) {
  return nstep_q_lossgrad<true>("arl_nstep_q_lossgrad_dueling", rewards, terminals, actions, q, q_boot, returns,
                                dq, dvalue, loss_sums, t_max, num_envs, action_size, gamma, reward_min,
                                reward_max, grad_scale, stream);
}

extern "C" int arl_double_nstep_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                           const float* q, const float* q_boot, const float* q_online_T,
                                           float* returns, float* dq, float* loss_sums, int t_max, int num_envs,
                                           int action_size, float gamma, float reward_min, float reward_max,
                                           float grad_scale, void* stream) {
  return nstep_q_lossgrad<false, true>("arl_double_nstep_q_lossgrad", rewards, terminals, actions, q, q_boot,
                                       returns, dq, nullptr, loss_sums, t_max, num_envs, action_size, gamma,
                                       reward_min, reward_max, grad_scale, stream, q_online_T);
}

extern "C" int arl_double_nstep_q_lossgrad_dueling(const float* rewards, const uint8_t* terminals,
                                                   const int32_t* actions, const float* q, const float* q_boot,
                                                   const float* q_online_T, float* returns, float* dq,
                                                   float* dvalue, float* loss_sums, int t_max, int num_envs,
                                                   int action_size, float gamma, float reward_min, float reward_max,
                                                   float grad_scale, void* stream) {
  return nstep_q_lossgrad<true, true>("arl_double_nstep_q_lossgrad_dueling", rewards, terminals, actions, q,
                                      q_boot, returns, dq, dvalue, loss_sums, t_max, num_envs, action_size, gamma,
                                      reward_min, reward_max, grad_scale, stream, q_online_T);
}

template <bool Dueling>
static int sarsa_lossgrad(const char* fn, const float* rewards, const uint8_t* terminals, const int32_t* actions,
                          const float* q, const float* q_next, float* target, float* dq, float* dvalue,
                          float* loss_sums, int t_max, int num_envs, int action_size, float gamma,
                          float reward_min, float reward_max, float grad_scale, void* stream) {
  ARL_REQUIRE(rewards && terminals && actions && q && q_next && target && dq && (dvalue || !Dueling),
              "%s: null pointer", fn);
  ARL_REQUIRE(t_max >= 0 && num_envs >= 0, "%s: negative size", fn);
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "%s: action_size %d outside [1,%d]", fn, action_size, ARL_MAX_ACTIONS);
  if (t_max == 0 || num_envs == 0) return ARL_OK;
  const int64_t total = (int64_t)t_max * num_envs;
  ARL_CUDA(launch_pdl(sarsa_lossgrad_kernel<Dueling>, dim3((unsigned)((total + 127) / 128)), dim3(128), 0,
                      (cudaStream_t)stream, rewards, terminals, actions, q, q_next, target, dq, loss_sums, t_max,
                      num_envs, action_size, gamma, reward_min, reward_max, grad_scale, dvalue));
  ARL_LAUNCH_CHECK("sarsa_lossgrad_kernel");
  return ARL_OK;
}

extern "C" int arl_sarsa_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                  const float* q, const float* q_next, float* target, float* dq,
                                  float* loss_sums, int t_max, int num_envs, int action_size, float gamma,
                                  float reward_min, float reward_max, float grad_scale, void* stream) {
  return sarsa_lossgrad<false>("arl_sarsa_lossgrad", rewards, terminals, actions, q, q_next, target, dq, nullptr,
                               loss_sums, t_max, num_envs, action_size, gamma, reward_min, reward_max, grad_scale,
                               stream);
}

extern "C" int arl_sarsa_lossgrad_dueling(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                          const float* q, const float* q_next, float* target, float* dq,
                                          float* dvalue, float* loss_sums, int t_max, int num_envs,
                                          int action_size, float gamma, float reward_min, float reward_max,
                                          float grad_scale, void* stream) {
  return sarsa_lossgrad<true>("arl_sarsa_lossgrad_dueling", rewards, terminals, actions, q, q_next, target, dq,
                              dvalue, loss_sums, t_max, num_envs, action_size, gamma, reward_min, reward_max,
                              grad_scale, stream);
}

extern "C" int arl_act_update(const float* step_reward, const uint8_t* step_terminal,
                              const int32_t* lives_before, const int32_t* lives_after, int is_training,
                              float* reward, uint8_t* terminal, int num_envs, void* stream) {
  ARL_REQUIRE(step_reward && step_terminal && lives_before && lives_after && reward && terminal,
              "arl_act_update: null pointer");
  ARL_REQUIRE(num_envs >= 0, "arl_act_update: negative size");
  if (num_envs == 0) return ARL_OK;
  ARL_CUDA(launch_pdl(act_update_kernel, dim3((num_envs + 255) / 256), dim3(256), 0, (cudaStream_t)stream,
                      step_reward, step_terminal, lives_before, lives_after, is_training, reward, terminal,
                      num_envs));
  ARL_LAUNCH_CHECK("act_update_kernel");
  return ARL_OK;
}

extern "C" int arl_observe_store(const float* reward, const uint8_t* terminal, float* reward_slot,
                                 uint8_t* terminal_slot, int num_envs, void* stream) {
  ARL_REQUIRE(reward && terminal && reward_slot && terminal_slot, "arl_observe_store: null pointer");
  ARL_REQUIRE(num_envs >= 0, "arl_observe_store: negative size");
  if (num_envs == 0) return ARL_OK;
  ARL_CUDA(launch_pdl(observe_store_kernel, dim3((num_envs + 255) / 256), dim3(256), 0, (cudaStream_t)stream,
                      reward, terminal, reward_slot, terminal_slot, num_envs, (int64_t*)nullptr, (int64_t)0));
  ARL_LAUNCH_CHECK("observe_store_kernel");
  return ARL_OK;
}

extern "C" int arl_observe_store_advance(const float* reward, const uint8_t* terminal, float* reward_slot,
                                         uint8_t* terminal_slot, int num_envs, int64_t* step_counter,
                                         int64_t inc, void* stream) {
  ARL_REQUIRE(reward && terminal && reward_slot && terminal_slot && step_counter,
              "arl_observe_store_advance: null pointer");
  ARL_REQUIRE(num_envs >= 1, "arl_observe_store_advance: num_envs must be >= 1");
  ARL_CUDA(launch_pdl(observe_store_kernel, dim3((num_envs + 255) / 256), dim3(256), 0, (cudaStream_t)stream,
                      reward, terminal, reward_slot, terminal_slot, num_envs, step_counter, inc));
  ARL_LAUNCH_CHECK("observe_store_kernel");
  return ARL_OK;
}

// arl_heads_backward (Relu) and arl_heads_backward_lstm (fn: the entry's name, for errors)
template <bool Relu>
static int heads_backward(const char* fn, const float* params, int action_size, const float* h,
                          const float* dlogits, const float* dvalue, float* d_h, float* grads, void* workspace,
                          int64_t num_samples, float tensor_scale, void* stream) {
  ARL_REQUIRE(params && h && dlogits && dvalue && d_h && grads && workspace, "%s: null pointer", fn);
  ARL_REQUIRE(tensor_scale > 0.f, "%s: tensor_scale must be > 0", fn);
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "%s: action_size %d outside [1,%d]", fn, action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_samples >= 0, "%s: negative size", fn);
  cudaStream_t st = (cudaStream_t)stream;
  const ParamLayout L = param_layout(action_size);
  const int A = action_size, J = A + 1;
  float* g = grads + L.off[T_PW];
  if (num_samples == 0) {
    ARL_CUDA(cudaMemsetAsync(g, 0, (size_t)(256 * J + J) * sizeof(float), st));
    return ARL_OK;
  }
  int grid = 2 * num_sms();
  if ((int64_t)grid > (num_samples + kHbChunk - 1) / kHbChunk)
    grid = (int)((num_samples + kHbChunk - 1) / kHbChunk);
  // empty trailing CTAs would write zero partials, which is fine; keep every CTA non-empty anyway.
  // Whole sample chunks (8) per CTA: the transposed copy of d_h is written chunk by chunk.
  const int64_t per = ((num_samples + grid - 1) / grid + 7) / 8 * 8;
  grid = (int)((num_samples + per - 1) / per);
  float* part = (float*)workspace;
  uint8_t* dhs = (uint8_t*)d_h;
  uint8_t* dhsT = dhs + (size_t)num_samples * 256 * sizeof(float);
  auto kern = J <= 8 ? heads_bwd_kernel<8, Relu> : J <= 20 ? heads_bwd_kernel<20, Relu>
                                                   : heads_bwd_kernel<ARL_MAX_ACTIONS + 1, Relu>;
  ARL_CUDA(launch_pdl(kern, dim3(grid), dim3(256), 0, st, params + L.off[T_PW], params + L.off[T_QW], h, dlogits,
                      dvalue, dhs, dhsT, part, num_samples, per, A, tensor_scale));
  ARL_LAUNCH_CHECK("heads_bwd_kernel");
  return reduce_partials(part, g, grid, 256 * J + J, st);
}

extern "C" int arl_heads_backward(const float* params, int action_size, const float* h,
                                  const float* dlogits, const float* dvalue, float* d_h,
                                  float* grads, void* workspace, int64_t num_samples,
                                  float tensor_scale, void* stream) {
  return heads_backward<true>("arl_heads_backward", params, action_size, h, dlogits, dvalue, d_h, grads, workspace,
                              num_samples, tensor_scale, stream);
}

extern "C" int arl_heads_backward_lstm(const float* params, int action_size, const float* h_lstm,
                                       const float* dlogits, const float* dvalue, float* d_h_lstm, float* grads,
                                       void* workspace, int64_t num_samples, float tensor_scale, void* stream) {
  return heads_backward<false>("arl_heads_backward_lstm", params, action_size, h_lstm, dlogits, dvalue, d_h_lstm,
                               grads, workspace, num_samples, tensor_scale, stream);
}

extern "C" int arl_heads_backward_streams(const float* params, int action_size, const float* h,
                                          const float* dlogits, const float* dvalue, float* d_h,
                                          float* grads, void* workspace, int64_t num_samples,
                                          float tensor_scale, void* stream) {
  ARL_REQUIRE(params && h && dlogits && dvalue && d_h && grads && workspace,
              "arl_heads_backward_streams: null pointer");
  ARL_REQUIRE(tensor_scale > 0.f, "arl_heads_backward_streams: tensor_scale must be > 0");
  ARL_REQUIRE(action_size >= 1 && action_size <= ARL_MAX_ACTIONS,
              "arl_heads_backward_streams: action_size %d outside [1,%d]", action_size, ARL_MAX_ACTIONS);
  ARL_REQUIRE(num_samples >= 0, "arl_heads_backward_streams: negative size");
  cudaStream_t st = (cudaStream_t)stream;
  const ParamLayout L = param_layout(action_size);
  const int A = action_size, J = A + 1;
  float* g = grads + L.off[T_PW];
  if (num_samples == 0) {
    ARL_CUDA(cudaMemsetAsync(g, 0, (size_t)(256 * J + J) * sizeof(float), st));
    return ARL_OK;
  }
  // arl_heads_backward's grid: whole sample chunks (8) per CTA, every CTA non-empty
  int grid = 2 * num_sms();
  if ((int64_t)grid > (num_samples + kHbChunk - 1) / kHbChunk)
    grid = (int)((num_samples + kHbChunk - 1) / kHbChunk);
  const int64_t per = ((num_samples + grid - 1) / grid + 7) / 8 * 8;
  grid = (int)((num_samples + per - 1) / per);
  float* part = (float*)workspace;
  uint8_t* dhs = (uint8_t*)d_h;
  uint8_t* dhsT = dhs + (size_t)num_samples * 512 * sizeof(float);
  auto kern = J <= 8 ? heads_bwd_streams_kernel<8>
                     : J <= 20 ? heads_bwd_streams_kernel<20> : heads_bwd_streams_kernel<ARL_MAX_ACTIONS + 1>;
  ARL_CUDA(launch_pdl(kern, dim3(grid), dim3(256), 0, st, params + L.off[T_PW], params + L.off[T_QW], h, dlogits,
                      dvalue, dhs, dhsT, part, num_samples, per, A, tensor_scale));
  ARL_LAUNCH_CHECK("heads_bwd_streams_kernel");
  return reduce_partials(part, g, grid, 256 * J + J, st);
}
