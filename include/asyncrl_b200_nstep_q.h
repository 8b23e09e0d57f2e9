/*
 * asyncrl_b200 -- n-step Q-learning entries (Mnih et al. 2016, "Asynchronous Methods for Deep
 * Reinforcement Learning", supplementary Algorithm "asynchronous n-step Q-learning").
 *
 * A companion of asyncrl_b200.h with the same conventions: int status (0 = ok, negative =
 * arl_status, message in arl_last_error()), device pointers owned by the caller, samples indexed
 * n = t * num_envs + b, launches asynchronous on `stream` (last argument).  The Q values are the
 * p_w/p_b head ("logits"), as in the async-Q entries of asyncrl_b200.h; the value head q_w/q_b is
 * computed but unused by this learner.
 */
#ifndef ASYNCRL_B200_NSTEP_Q_H_
#define ASYNCRL_B200_NSTEP_Q_H_

#include "asyncrl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* arl_forward_sample with the epsilon-greedy draw of agent.py:141-151 in place of the policy
 * sample: conv1, conv2, fc256, then heads + softmax + the draw in one launch (env range by env
 * range above arl_a2_block_rows envs), after arl_prepare_weights when refresh_prepared != 0.
 * The draw is arl_egreedy_actions' on the logits this call writes: Philox4x32-10 block
 * (env_id_base + b, step_lo, step_hi, 1) keyed by seed; word 0 -> u = (x0 >> 8) * 2^-24, u < ep
 * draws floor(x1 * A / 2^32), otherwise argmax (ties -> lowest index).
 *   step_dev == NULL: the step is `step` and epsilon is `ep`.
 *   step_dev != NULL: the step is step + *step_dev and epsilon is agent.py:142-144 evaluated on
 *     the device from it -- ep_end + max(0, (ep_start - ep_end) * (ep_end_t - max(0, step -
 *     learn_start)) / ep_end_t) in double, operation by operation, rounded to float once (the
 *     value a host computing the same expression in double passes as `ep`).  `ep` is ignored.
 * ep, ep_start, ep_end in [0,1]; ep_end_t > 0 (checked when step_dev != NULL). */
ARL_API int arl_forward_egreedy(const float* params, float* prepared, int refresh_prepared, int action_size,
                                const uint8_t* ring, int num_envs, int ring_slots, int first_slot,
                                float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                                int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                                uint64_t seed, float ep, double ep_start, double ep_end, double ep_end_t,
                                double learn_start, void* stream);

/* n-step Q targets and the loss gradient of one rollout (T = t_max steps of num_envs envs):
 *   R_T = max_a q_boot[b][a]  (Q(s_T) under the target parameters, fmaxf in index order)
 *   R_t = fmaf(gamma * (1 - term_t), R_{t+1}, clip(r_t))  -- the operation sequence of
 *         arl_returns_lossgrad, so `returns` equals its output for v_boot = max_a q_boot
 *   delta_n = R_n - q[n][a_n];  dq[n][a_n] = -2 * delta_n * grad_scale, dq[n][j != a_n] = 0
 *   loss_sums[0] += sum delta^2, loss_sums[1] += sum q[n][a_n]  (the pair of arl_q_lossgrad;
 *   loss_sums may be NULL).
 * rewards f32 [T][B] (clipped to [reward_min, reward_max] here), terminals u8 [T][B], actions
 * i32 [T*B], q f32 [T*B][A], q_boot f32 [B][A], returns f32 [T*B], dq f32 [T*B][A]. */
ARL_API int arl_nstep_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                 const float* q, const float* q_boot, float* returns, float* dq,
                                 float* loss_sums, int t_max, int num_envs, int action_size, float gamma,
                                 float reward_min, float reward_max, float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif

#endif  // ASYNCRL_B200_NSTEP_Q_H_
