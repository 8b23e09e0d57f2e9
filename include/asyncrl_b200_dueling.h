/*
 * asyncrl_b200 -- dueling Q heads (Wang et al. 2016, "Dueling Network Architectures for Deep
 * Reinforcement Learning", the "average" aggregator) for the async-Q, n-step Q and Sarsa learners.
 *
 * A companion of asyncrl_b200.h with the same conventions: int status (0 = ok, negative =
 * arl_status, message in arl_last_error()), device pointers owned by the caller, samples indexed
 * n = t * num_envs + b, launches asynchronous on `stream` (last argument).
 *
 * No parameter is added: the A-wide p_w/p_b head is the advantage stream and the 1-wide q_w/q_b
 * head the value stream, both on the shared fc256 output h (one sample, A actions):
 *   adv_j = h . p_w[:, j] + p_b[j]      (arl_forward's logit j, the same bits)
 *   v     = h . q_w + q_b               (arl_forward's value, the same bits)
 *   m     = (sum_j adv_j) / A           (a float32 warp sum over the A lanes, one division by A)
 *   Q_j   = v + (adv_j - m)
 * `logits` receives Q, `value` receives v, `probs` the softmax of Q.  The backward is arl_backward
 * unchanged, fed with d_logits = dL/d adv and d_value = dL/dv from the loss entries below.
 */
#ifndef ASYNCRL_B200_DUELING_H_
#define ASYNCRL_B200_DUELING_H_

#include "asyncrl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* arl_forward with the dueling Q row, plus the draw arguments of arl_forward_egreedy.
 *   actions == NULL: no draw; `steps` env steps from first_slot as in arl_forward (the target
 *     forwards over s_T or s_1..s_T, evaluation).  The draw arguments are ignored.
 *   actions != NULL: steps must be 1; the epsilon-greedy draw of arl_forward_egreedy (same Philox
 *     block, same epsilon rules, same argument checks, ties -> lowest index) on the Q row written
 *     to `logits`, inside the heads launch.
 * Batches above one a2 block (arl_a2_block_rows) run env range by env range, as arl_forward does. */
ARL_API int arl_forward_dueling(const float* params, float* prepared, int refresh_prepared, int action_size,
                                const uint8_t* ring, int num_envs, int ring_slots, int first_slot, int steps,
                                float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                                int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                                uint64_t seed, float ep, double ep_start, double ep_end, double ep_end_t,
                                double learn_start, void* stream);

/* The loss entries of the three Q learners through the dueling combine.  Each takes its plain
 * entry's arguments (asyncrl_b200.h, asyncrl_b200_sarsa.h) with `dvalue` f32 [N] after `dq`;
 * targets / returns and loss_sums are computed exactly as there.  With
 * g_n = -2 * delta_n * grad_scale (the plain entry's dq[n][a_n]):
 *   dq[n][j]  = g_n * ((j == a_n ? 1 : 0) - 1.f / A)   -- dL/d adv_j: dQ_j - mean_k dQ_k
 *   dvalue[n] = g_n                                    -- dL/dv: sum_j dQ_j
 * in float32, in this order. */
ARL_API int arl_q_lossgrad_dueling(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                   const float* q, const float* q_next, float* target, float* dq, float* dvalue,
                                   float* loss_sums, int64_t num_samples, int action_size, float discount,
                                   float reward_min, float reward_max, float grad_scale, void* stream);

ARL_API int arl_nstep_q_lossgrad_dueling(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                         const float* q, const float* q_boot, float* returns, float* dq,
                                         float* dvalue, float* loss_sums, int t_max, int num_envs,
                                         int action_size, float gamma, float reward_min, float reward_max,
                                         float grad_scale, void* stream);

ARL_API int arl_sarsa_lossgrad_dueling(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                       const float* q, const float* q_next, float* target, float* dq,
                                       float* dvalue, float* loss_sums, int t_max, int num_envs, int action_size,
                                       float gamma, float reward_min, float reward_max, float grad_scale,
                                       void* stream);

#ifdef __cplusplus
}
#endif

#endif  // ASYNCRL_B200_DUELING_H_
