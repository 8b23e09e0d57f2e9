/*
 * asyncrl_b200 -- double Q-learning targets (van Hasselt, Guez & Silver 2016, "Deep Reinforcement
 * Learning with Double Q-learning") for the async-Q and n-step Q learners.
 *
 * A companion of asyncrl_b200.h with the same conventions: int status (0 = ok, negative =
 * arl_status, message in arl_last_error()), device pointers owned by the caller, samples indexed
 * n = t * num_envs + b, launches asynchronous on `stream` (last argument).
 *
 * The online network theta (the parameters the rollout was collected with) chooses the bootstrap
 * action, the target network theta^- evaluates it:
 *   a*    = argmax_a Q(s', a; theta)        (ties -> lowest index, as arl_greedy_actions)
 *   boot  = Q(s', a*; theta^-)              in place of max_a Q(s'; theta^-)
 * Everything else -- the target / return expression, dq (and dvalue), loss_sums -- is the plain
 * entry's, in the same order.  With dueling heads every Q is the dueling Q row (the `logits` of
 * arl_forward_dueling), with no other change.
 */
#ifndef ASYNCRL_B200_DOUBLE_H_
#define ASYNCRL_B200_DOUBLE_H_

#include "asyncrl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* arl_q_lossgrad with double targets, over t_max * num_envs samples (the kernel needs to know
 * which rows are the last step):
 *   q          f32 [t_max*num_envs, A]  Q(s_t; theta), the rollout's own Q rows; rows 1..t_max-1
 *                                       (row n + num_envs for sample n) are the online rows of s'
 *   q_next     f32 [t_max*num_envs, A]  Q(s_{t+1}; theta^-)
 *   q_online_T f32 [num_envs, A]        Q(s_T; theta), the online rows of s' for t = t_max - 1
 *   target[n]  = fmaf((1 - term_n) * discount, q_next[n][a*_n], clip(r_n)) */
ARL_API int arl_double_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                  const float* q, const float* q_next, const float* q_online_T, float* target,
                                  float* dq, float* loss_sums, int t_max, int num_envs, int action_size,
                                  float discount, float reward_min, float reward_max, float grad_scale,
                                  void* stream);

/* the same through the dueling combine: `dvalue` f32 [N] after `dq`, as arl_q_lossgrad_dueling */
ARL_API int arl_double_q_lossgrad_dueling(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                          const float* q, const float* q_next, const float* q_online_T,
                                          float* target, float* dq, float* dvalue, float* loss_sums, int t_max,
                                          int num_envs, int action_size, float discount, float reward_min,
                                          float reward_max, float grad_scale, void* stream);

/* arl_nstep_q_lossgrad with the return recurrence started from R_T = q_boot[b][a*_b],
 * a*_b = argmax_a q_online_T[b][a]:
 *   q_boot     f32 [num_envs, A]  Q(s_T; theta^-)
 *   q_online_T f32 [num_envs, A]  Q(s_T; theta) */
ARL_API int arl_double_nstep_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                                        const float* q, const float* q_boot, const float* q_online_T,
                                        float* returns, float* dq, float* loss_sums, int t_max, int num_envs,
                                        int action_size, float gamma, float reward_min, float reward_max,
                                        float grad_scale, void* stream);

/* the same through the dueling combine: `dvalue` f32 [N] after `dq`, as arl_nstep_q_lossgrad_dueling */
ARL_API int arl_double_nstep_q_lossgrad_dueling(const float* rewards, const uint8_t* terminals,
                                                const int32_t* actions, const float* q, const float* q_boot,
                                                const float* q_online_T, float* returns, float* dq, float* dvalue,
                                                float* loss_sums, int t_max, int num_envs, int action_size,
                                                float gamma, float reward_min, float reward_max, float grad_scale,
                                                void* stream);

#ifdef __cplusplus
}
#endif

#endif  // ASYNCRL_B200_DOUBLE_H_
