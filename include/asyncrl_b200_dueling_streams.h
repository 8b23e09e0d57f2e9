/*
 * asyncrl_b200 -- the dueling architecture of Wang et al. 2016 ("Dueling Network Architectures for
 * Deep Reinforcement Learning") with a hidden layer per stream, for the async-Q, n-step Q and Sarsa
 * learners on the nips trunk.
 *
 * A companion of asyncrl_b200.h with the same conventions: int status (0 = ok, negative =
 * arl_status, message in arl_last_error()), device pointers owned by the caller, samples indexed
 * n = t * num_envs + b, launches asynchronous on `stream` (last argument).
 *
 * Network (one sample, A actions; a2 = conv2's output, 2592 values):
 *   h_v = relu(a2 . l4_w + l4_b)        the value stream's hidden layer, 256 wide
 *   h_a = relu(a2 . la_w + la_b)        the advantage stream's hidden layer, 256 wide
 *   v     = h_v . q_w + q_b
 *   adv_j = h_a . p_w[:, j] + p_b[j]
 *   Q_j   = v + (adv_j - (sum_k adv_k) / A)   (asyncrl_b200_dueling.h's aggregator, the same operations)
 * `logits` receives Q, `value` receives v, `probs` the softmax of Q.  The loss entries of
 * asyncrl_b200_dueling.h and asyncrl_b200_double.h (the `_dueling` forms) write d_logits = dL/d adv
 * and d_value = dL/dv for the backward below.
 *
 * Parameters: the 10 tensors of arl_param_layout at their offsets, then la_w [2592,256] and
 * la_b [256] (arl_streams_param_layout, 13 offsets).
 *
 * Buffers (N samples):
 *   h          f32 [N][512]: a row is [h_v | h_a]
 *   d_h        f32 [N + ceil(N/8)*8][512]: [d_h_v | d_h_a] as a split block of 512 columns
 *              (asyncrl_b200.h), then its transposed copy ([hi|lo][ceil(N/8)][512][8 samples]);
 *              multiplied by tensor_scale
 *   prepared   arl_streams_prepared_floats() floats (arl_prepare_weights_streams)
 *   workspace  arl_streams_workspace_bytes(A) bytes
 */
#ifndef ASYNCRL_B200_DUELING_STREAMS_H_
#define ASYNCRL_B200_DUELING_STREAMS_H_

#include "asyncrl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* offsets[13]: the 12 tensors l1_w .. q_b, la_w, la_b and the total */
ARL_API int arl_streams_param_layout(int action_size, int64_t* offsets);
ARL_API int64_t arl_streams_prepared_floats(void);
ARL_API int64_t arl_streams_workspace_bytes(int action_size);

/* arl_prepare_weights for the streams' network: the conv images, l4_w^T and la_w^T (the clustered
 * fc forward), [l4_w | la_w] as one split block (the streaming fc forward and the fc input
 * gradient) and [l4_b | la_b]. */
ARL_API int arl_prepare_weights_streams(const float* params, float* prepared, int action_size, void* stream);

/* [h_v | h_a] = relu(a2 . [l4_w | la_w] + [l4_b | la_b]) from the prepared images, h f32 [N][512], in one
 * launch (the stream is an N tile of the fc kernel). */
ARL_API int arl_fc_forward_streams(const float* prepared, const float* a2, float* h, int64_t num_samples,
                                   void* stream);

/* arl_forward_dueling (asyncrl_b200_dueling.h) on the streams' network: the same arguments, checks,
 * draws and env-range chunking; h is [num_envs * steps][512] and `prepared` the streams' image. */
ARL_API int arl_forward_streams(const float* params, float* prepared, int refresh_prepared, int action_size,
                                const uint8_t* ring, int num_envs, int ring_slots, int first_slot, int steps,
                                float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                                int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                                uint64_t seed, float ep, double ep_start, double ep_end, double ep_end_t,
                                double learn_start, void* stream);

/* The heads backward: d_h_v = d_value q_w^T masked by h_v > 0, d_h_a = d_logits p_w^T masked by
 * h_a > 0 (both times tensor_scale, into d_h as above); p_w, p_b from h_a and d_logits, q_w, q_b from
 * h_v and d_value. */
ARL_API int arl_heads_backward_streams(const float* params, int action_size, const float* h, const float* dlogits,
                                       const float* dvalue, float* d_h, float* grads, void* workspace,
                                       int64_t num_samples, float tensor_scale, void* stream);

/* The fc backward of both streams: [dl4_w | dla_w] = a2^T . [d_h_v | d_h_a], l4_b / la_b = column
 * sums, d_a2 = ([d_h_v | d_h_a] . [l4_w | la_w]^T) masked by a2 > 0 (K = 512); gradients times
 * grad_unscale. */
ARL_API int arl_fc_backward_streams(const float* prepared, const float* a2, int64_t a2_block_rows, const float* d_h,
                                    float* d_a2, float* grads, void* workspace, int64_t num_samples,
                                    float grad_unscale, int action_size, void* stream);

/* arl_backward on the streams' network: heads, fc, conv2 and conv1 backward, then (allreduce != 0
 * and a communicator of more than one rank) one all-reduce of all 12 tensors. */
ARL_API int arl_backward_streams(const float* params, const float* prepared, int action_size, const uint8_t* ring,
                                 int num_envs, int ring_slots, int first_slot, int steps, const float* a1,
                                 const float* a2, const float* h, const float* dlogits, const float* dvalue,
                                 float* d_h, float* d_a2, float* d_a1, float* grads, void* workspace,
                                 float tensor_scale, int allreduce, void* stream);

#ifdef __cplusplus
}
#endif

#endif  // ASYNCRL_B200_DUELING_STREAMS_H_
