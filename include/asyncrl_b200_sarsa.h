/*
 * asyncrl_b200 -- one-step Sarsa entry (Mnih et al. 2016, "Asynchronous Methods for Deep
 * Reinforcement Learning", supplementary Algorithm "asynchronous one-step Sarsa").
 *
 * A companion of asyncrl_b200.h with the same conventions: int status (0 = ok, negative =
 * arl_status, message in arl_last_error()), device pointers owned by the caller, samples indexed
 * n = t * num_envs + b, launches asynchronous on `stream` (last argument).  The Q values are the
 * p_w/p_b head ("logits"), as in the async-Q and n-step Q entries of asyncrl_b200.h; the value head
 * q_w/q_b is computed but unused by this learner (asyncrl_b200_dueling.h: with dueling heads it is
 * the value stream).  The rest of the Sarsa cycle runs on entries of
 * asyncrl_b200.h: arl_forward on the target parameters over s_1..s_T (q_next), arl_forward_egreedy
 * on s_T for the action a_T the next rollout starts with, arl_backward.
 */
#ifndef ASYNCRL_B200_SARSA_H_
#define ASYNCRL_B200_SARSA_H_

#include "asyncrl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* One-step Sarsa targets and the loss gradient of one rollout (T = t_max steps of num_envs envs):
 *   y_n     = fmaf((1 - term_n) * gamma, q_next[n][actions[n + B]], clip(r_n))  -- the expression
 *             of arl_q_lossgrad with the next action's Q in place of max_a, so for
 *             actions[n + B] = argmax_a q_next[n][a] `target` and `dq` equal its output
 *   delta_n = y_n - q[n][a_n];  dq[n][a_n] = -2 * delta_n * grad_scale, dq[n][j != a_n] = 0
 *   loss_sums[0] += sum delta^2, loss_sums[1] += sum q[n][a_n]  (loss_sums may be NULL).
 * rewards f32 [T][B] (clipped to [reward_min, reward_max] here), terminals u8 [T][B], actions
 * i32 [(T+1)*B] = a_0 .. a_T (row T: the action taken in s_T, the first of the next rollout),
 * q f32 [T*B][A] = Q(s_t; theta), q_next f32 [T*B][A] = Q(s_{t+1}; theta^-), target f32 [T*B],
 * dq f32 [T*B][A].  Every action must lie in [0, action_size). */
ARL_API int arl_sarsa_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                               const float* q, const float* q_next, float* target, float* dq,
                               float* loss_sums, int t_max, int num_envs, int action_size, float gamma,
                               float reward_min, float reward_max, float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif

#endif  // ASYNCRL_B200_SARSA_H_
