/*
 * asyncrl_b200 -- the A3C LSTM agent of Mnih et al. 2016: a recurrent layer of 256 LSTM cells between
 * fc256 and the policy / value heads, for the a3c learner on the nips trunk.
 *
 * A companion of asyncrl_b200.h with the same conventions: int status (0 = ok, negative =
 * arl_status, message in arl_last_error()), device pointers owned by the caller, samples indexed
 * n = t * num_envs + b, launches asynchronous on `stream` (last argument).
 *
 * Network (one sample; x = h_fc = relu(a2 . l4_w + l4_b), fc256's output):
 *   keep  = 0 if the env's previous step was terminal (the `reset` row), else 1
 *   z     = [x | keep * h_prev] . lstm_w + lstm_b        lstm_w [512,1024], lstm_b [1024]
 *   i, j, f, o = z[0:256], z[256:512], z[512:768], z[768:1024]   (TF BasicLSTMCell order)
 *   c     = sigmoid(f + 1) * keep * c_prev + sigmoid(i) * tanh(j)
 *   h     = sigmoid(o) * tanh(c)
 * The heads read h in place of h_fc.  forget_bias = 1 is a constant; no peepholes, no clipping.
 *
 * Parameters: the 10 tensors of arl_param_layout at their offsets, then lstm_w [512,1024] and
 * lstm_b [1024] (arl_lstm_param_layout, 13 offsets).
 *
 * Buffers (B envs, T steps, N = T * B samples; f32 unless stated):
 *   state_h, state_c   [B][256]   the recurrent state the next step reads (and, with advance, writes)
 *   h_fc               [N][256]   fc256's output (the plain path's `h`)
 *   xh                 [T][B * 512] one split block ([hi|lo][64 chunks][B rows][8] bf16, asyncrl_b200.h)
 *                      per step: [x | keep * h_prev], the LSTM operand of the forward and of the
 *                      weight gradient
 *   z                  [B][1024]  scratch: the pre-activations of one step
 *   gates              [N][1024]  sigmoid(i), tanh(j), sigmoid(f + 1), sigmoid(o)
 *   c_prev             [N][256]   keep * c_prev, the cell state the step read
 *   c                  [N][256]   the step's cell state
 *   h_lstm             [N][256]   the step's h, the heads' input
 *   d_h_lstm           [N][256]   dL/dh from the heads (unmasked), times tensor_scale
 *   dz                 [T][B * 1024] one split block per step: dL/dz times tensor_scale
 *   dxh                [N][512]   [dL/dx | dL/d(keep * h_prev)] times tensor_scale
 *   dc                 [B][256]   the cell-state gradient carried from step t to step t - 1
 *   d_h                as in arl_backward: dL/dh_fc masked by h_fc > 0, split block + transposed copy
 *   prepared           arl_lstm_prepared_floats() floats (arl_prepare_weights_lstm)
 *   workspace          arl_lstm_workspace_bytes(A) bytes
 */
#ifndef ASYNCRL_B200_LSTM_H_
#define ASYNCRL_B200_LSTM_H_

#include "asyncrl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* offsets[13]: the 12 tensors l1_w .. q_b, lstm_w, lstm_b and the total */
ARL_API int arl_lstm_param_layout(int action_size, int64_t* offsets);
ARL_API int64_t arl_lstm_prepared_floats(void);
ARL_API int64_t arl_lstm_workspace_bytes(int action_size);

/* arl_prepare_weights, then lstm_w^T [1024 rows][512] (the forward's operand) and lstm_w [512 rows][1024]
 * (the input gradient's operand) as split blocks. */
ARL_API int arl_prepare_weights_lstm(const float* params, float* prepared, int action_size, void* stream);

/* One LSTM step of num_envs samples from x = h_fc: packs [x | keep * state_h] into the split block xh,
 * z = xh . lstm_w (one tcgen05 GEMM), then the cell.  Writes h_out, c_out and (when not NULL) gates and
 * c_prev_out; with advance != 0 also state_h = h_out, state_c = c_out.  reset (u8 [num_envs], NULL =
 * no reset): nonzero = the env's previous step was terminal. */
ARL_API int arl_lstm_step(const float* params, const float* prepared, int action_size, const float* h_fc,
                          float* state_h, float* state_c, const uint8_t* reset, int advance, float* xh, float* z,
                          float* gates, float* c_prev_out, float* c_out, float* h_out, int num_envs, void* stream);

/* The rollout step / the bootstrap forward: conv1 -> conv2 -> fc256 (env range by env range above
 * arl_a2_block_rows), then arl_lstm_step over all envs and the heads (+ the policy draw of
 * arl_forward_sample when `actions` is not NULL) on h_out.  The bootstrap passes advance = 0 and
 * actions = NULL: V(s_T) from the state, which stays as it is. */
ARL_API int arl_forward_lstm(const float* params, float* prepared, int refresh_prepared, int action_size,
                             const uint8_t* ring, int num_envs, int ring_slots, int first_slot, float* a1,
                             float* a2, float* h_fc, float* state_h, float* state_c, const uint8_t* reset,
                             int advance, float* xh, float* z, float* gates, float* c_prev_out, float* c_out,
                             float* h_out, float* logits, float* probs, float* value, int32_t* actions,
                             int64_t env_id_base, int64_t step, const int64_t* step_dev, uint64_t seed,
                             void* stream);

/* arl_heads_backward without the relu mask: d_h_lstm = (d_logits p_w^T + d_value q_w^T) * tensor_scale as
 * f32 [N][256]; p_w, p_b, q_w, q_b as there. */
ARL_API int arl_heads_backward_lstm(const float* params, int action_size, const float* h_lstm, const float* dlogits,
                                    const float* dvalue, float* d_h_lstm, float* grads, void* workspace,
                                    int64_t num_samples, float tensor_scale, void* stream);

/* Truncated BPTT over the `steps` steps of the rollout (the state the rollout started from is a
 * constant) and the LSTM weight gradient: for t = steps-1 .. 0 the cell backward (dz_t from d_h_lstm_t +
 * the recurrent gradient of step t+1, masked by keep of step t+1 = 1 - terminals[t]) and
 * dxh_t = dz_t . lstm_w^T (one tcgen05 GEMM per step); then d lstm_w = xh^T . dz over all N samples
 * (split-K, partials summed in a fixed order), d lstm_b = column sums of dz, both times 1/tensor_scale,
 * and d_h = dx masked by h_fc > 0 in arl_fc_backward's form.  terminals: u8 [steps][num_envs]. */
ARL_API int arl_lstm_backward(const float* params, const float* prepared, int action_size, int num_envs, int steps,
                              const uint8_t* terminals, const float* h_fc, const float* xh, const float* gates,
                              const float* c_prev, const float* c, const float* d_h_lstm, float* dz, float* dxh,
                              float* dc, float* d_h, float* grads, void* workspace, float tensor_scale,
                              void* stream);

/* arl_backward on the LSTM network: heads (unmasked), BPTT + LSTM weight gradient, then the fc, conv2
 * and conv1 backward, then (allreduce != 0 and a communicator of more than one rank) one all-reduce
 * of all 12 tensors. */
ARL_API int arl_backward_lstm(const float* params, const float* prepared, int action_size, const uint8_t* ring,
                              int num_envs, int ring_slots, int first_slot, int steps, const uint8_t* terminals,
                              const float* a1, const float* a2, const float* h_fc, const float* xh,
                              const float* gates, const float* c_prev, const float* c, const float* h_lstm,
                              const float* dlogits, const float* dvalue, float* d_h_lstm, float* dz, float* dxh,
                              float* dc, float* d_h, float* d_a2, float* d_a1, float* grads, void* workspace,
                              float tensor_scale, int allreduce, void* stream);

#ifdef __cplusplus
}
#endif

#endif  // ASYNCRL_B200_LSTM_H_
