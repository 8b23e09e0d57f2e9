/*
 * asyncrl_b200 -- C-ABI of the B200-native A3C worker hot path.
 *
 * Drop-in boundary for datavizweb/async-rl-tensorflow.  The reference has no
 * FFI of its own: its seams are Python classes plus tf.Session.run(feed_dict)
 * (SURVEY.md §8b).  Each entry point below replaces the TensorFlow / cv2 work
 * behind one of those seams and cites it (paths relative to the reference).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  All tensor pointers are DEVICE
 *     pointers owned by the caller; the library allocates nothing per call.
 *   - every function returns 0 on success, a negative arl_status otherwise; the
 *     message is in arl_last_error() (thread-local).
 *   - launches are asynchronous on `stream` (a cudaStream_t passed as void*);
 *     no hidden synchronisation.
 *   - samples are indexed n = t * num_envs + b  (t-major).  The frame ring is
 *     u8 [num_envs][ring_slots][84*84]; sample (t,b) reads the 4 planes
 *     ring[b][(first_slot + t + k) % ring_slots], k = 0 (oldest) .. 3 (newest),
 *     i.e. History.get() channel order (src/history.py:20-24).  Inside a plane the
 *     bytes are stored in 4x4 blocks (space-to-depth): screen byte (y,x) sits at
 *     ((y/4)*21 + x/4)*16 + (y%4)*4 + x%4 -- arl_preprocess_push writes that order,
 *     arl_conv1_* read it, arl_history_get returns the reference's row-major stack.
 *   - conv1's output a1 (12 800 bytes per sample) holds ONE fp16 per value in space-to-depth
 *     blocks: [n][kc = (i*2+j)*2 + chalf][q = yp*10 + xp][8 channels] with pixel
 *     (y,x) = (2yp+i, 2xp+j).  Only arl_conv1_forward writes it and only
 *     arl_conv2_forward / arl_conv2_backward read it (as tensor-core operand and relu mask);
 *     src/network.py:decode_a1 turns it back into f32 NHWC.  (DESIGN.md section 5.1: the measured
 *     precision behind the 16-bit format; round 1 kept a bf16 hi + lo pair.)
 *   - the fc256 layer's tensors are kept as "split blocks": a logical f32 matrix [rows][8*chunks]
 *     stored as [part (hi, lo)][chunk][row][8 bf16] (16-byte vectors, value = hi + lo, same bytes
 *     as the f32 matrix), which the tcgen05 kernels fetch with cp.async.bulk and never convert:
 *       a2  (the f32 [N,2592]-sized buffer): one block per arl_conv2_forward call, rows = the
 *           call's num_samples, 324 chunks in NHWC-flatten order (agent.py:231-232);
 *       d_h ((N + roundup8(N)) * 256 floats): one block of N rows, 32 chunks, followed by its
 *           transposed copy -- a block of 256 rows (the columns of d_h) with one chunk per 8
 *           samples, samples >= N zero -- both written by arl_heads_backward: fc dgrad reduces
 *           over the columns, fc wgrad over the samples, and each gets contiguous KB-sized runs;
 *       l4_w: one block of 2592 rows, 32 chunks, at the start of the `prepared` buffer.
 *   - `prepared` (arl_prepared_floats() floats, written by arl_prepare_weights) holds the weights in
 *     the form the tensor-core kernels keep resident: l4_w as a split block, l1_w as three s8
 *     limbs + scales + l1_b, l2_w as [hi | lo] bf16 images (forward and transposed) + l2_b.  It
 *     must be refreshed whenever the parameters change (arl_clip_rmsprop, a checkpoint load, ...).
 *     src/network.py:decode_split turns a block back into f32 [rows][cols].
 *   - d_a1, the gradient w.r.t. conv1's output, is the reduction operand of the conv1 weight
 *     gradient: ONE fp16 per value (x tensor_scale) on conv1's 21x21 space-to-depth grid,
 *     [channel group (2)][row n*441 + y*21 + x][8 channels], rows y = 20 / x = 20 zero:
 *     ARL_DA1_BYTES = 14 112 bytes per sample.  arl_conv2_backward writes it (and, since it
 *     has the values in registers, the conv1 bias gradient l1_b); arl_conv1_backward reads it.
 *     src/network.py:decode_da1 turns it into f32 [N,20,20,16].
 *   - parameters / gradients / RMSProp slots are flat f32 buffers in the
 *     reference's own variable order and layouts (see arl_param_layout).
 */
#ifndef ASYNCRL_B200_H_
#define ASYNCRL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ARL_FRAME_H 210
#define ARL_FRAME_W 160
#define ARL_FRAME_C 3
#define ARL_SCREEN 84            /* config.py:38-39 screen_width/height          */
#define ARL_HISTORY 4            /* config.py:22 history_length                  */
#define ARL_A1_ELEMS 6400        /* 20*20*16  conv1 output per sample            */
#define ARL_A2_ELEMS 2592        /* 9*9*32    conv2 output per sample (flatten)  */
#define ARL_DA1_ELEMS 7056       /* 21*21*16  values of d_a1 per sample (grid)   */
#define ARL_DA1_BYTES 14112      /* ... stored as fp16                          */
#define ARL_FC 256               /* agent.py:251 / network.py:51                 */
#define ARL_NUM_TENSORS 10       /* l1_w l1_b l2_w l2_b l4_w l4_b p_w p_b q_w q_b */
#define ARL_MAX_ACTIONS 32
#define ARL_NATURE_TENSORS 12    /* l1_w l1_b l2_w l2_b l3_w l3_b l4_w l4_b p_w p_b q_w q_b (network.py:34-42,62,79) */
#define ARL_NATURE_FC 512        /* network.py:41-42                              */

#if defined(__GNUC__)
#define ARL_API __attribute__((visibility("default")))
#else
#define ARL_API
#endif

typedef enum {
  ARL_OK = 0,
  ARL_ERR_INVALID = -1,          /* bad argument (message says which)            */
  ARL_ERR_CUDA = -2,             /* CUDA runtime error                           */
  ARL_ERR_UNSUPPORTED = -3       /* valid request this build does not implement  */
} arl_status;

/* Thread-local message of the last failing call on this thread. */
ARL_API const char* arl_last_error(void);
ARL_API int arl_version(void);
/* Number of kernels this library has launched in this process (optionally reset to 0). */
ARL_API int64_t arl_launch_count(int reset);

/* One-time per-process set-up on `device`: derives the luma correction bitmap
 * (the 774 RGB triples where the reference's float64 luma truncates one below the
 * exact quotient) with IEEE f64 on the device and raises the shared-memory limits
 * of the big kernels.  Must precede every other call. */
ARL_API int arl_init(int device);

/* Offsets (in floats) of the 10 tensors inside the flat buffers and the total.
 * Order/layout: l1_w[8,8,4,16] l1_b[16] l2_w[4,4,16,32] l2_b[32] l4_w[2592,256]
 * l4_b[256] p_w[256,A] p_b[A] q_w[256,1] q_b[1]  -- ops.py:19-24,36-39;
 * agent.py:226-229,251; network.py:62,79.  offsets has ARL_NUM_TENSORS+1 entries. */
ARL_API int arl_param_layout(int action_size, int64_t* offsets);

/* ---- K1: Environment.screen + History.add ------------------------------------------
 * src/environment.py:49-53 (float64 luma, truncate, cv2.resize INTER_LINEAR 84x84) fused
 * with src/history.py:13-15 (push newest).  frames u8 [num_envs,210,160,3] ->
 * ring[b][(slot + r) % ring_slots] for r in [0, replicate)   (replicate = 4 reproduces
 * agent.py:37-38, which seeds the stack with 4 copies of the first screen).
 * Bit-exact against the reference's executed expression. */
ARL_API int arl_preprocess_push(const uint8_t* frames, uint8_t* ring, int num_envs, int ring_slots,
                        int slot, int replicate, void* stream);

/* The other resize branch of environment.py:5-12: scipy.misc.imresize(y, (84,84)) = PIL
 * Image.resize(BILINEAR) on the truncated luma (antialiased triangle filter, 22-bit fixed point,
 * horizontal pass to u8 then vertical).  Same arguments and ring layout as arl_preprocess_push;
 * bit-exact against Pillow.  Reads every source row. */
ARL_API int arl_preprocess_push_pil(const uint8_t* frames, uint8_t* ring, int num_envs, int ring_slots,
                            int slot, int replicate, void* stream);

/* Host -> device upload of exactly the frame rows K1 reads (environment.py:53 -> cv2.resize
 * 210x160 -> 84x84 never touches source rows == 2 mod 5): 80 640 of the 100 800 B of a frame, as
 * ONE strided async copy of 1920-B runs (4 rows) at a 2400-B pitch over the whole batch plus the
 * two 960-B ends.  host_frames should be pinned; dev_frames keeps the full [num_envs,210,160,3]
 * layout (the skipped rows are left as they are: NOT valid input for arl_preprocess_push_pil). */
ARL_API int arl_upload_frames(const uint8_t* host_frames, uint8_t* dev_frames, int num_envs,
                      void* stream);

/* The whole frames (one plain async copy of num_envs * 100 800 B): the upload to use with the
 * scipy/PIL resize branch (arl_preprocess_push_pil reads every source row). */
ARL_API int arl_upload_frames_full(const uint8_t* host_frames, uint8_t* dev_frames, int num_envs,
                           void* stream);

/* History.get()/copy() (src/history.py:20-27): materialise the NHWC stack
 * f32 [num_envs,84,84,4] (or u8 when out_is_u8) whose oldest plane is `first_slot`. */
ARL_API int arl_history_get(const uint8_t* ring, void* out, int out_is_u8, int num_envs,
                    int ring_slots, int first_slot, void* stream);
/* History.reset() (src/history.py:17-18): zero every slot. */
ARL_API int arl_history_reset(uint8_t* ring, int num_envs, int ring_slots, void* stream);

/* ---- K2/K3: trunk + heads forward ---------------------------------------------------
 * agent.py:226-232,251 (s_t/255 -> conv 8x8s4 relu -> conv 4x4s2 relu -> NHWC flatten ->
 * fc256 relu), network.py:62 (policy logits), network.py:79 (value), network.py:65
 * (softmax).  steps*num_envs samples.  a1 [N,20,20,16], a2 [N,2592], h [N,256] are
 * written for the backward pass (a1 and a2 in the device layouts described at the top of this
 * file); logits/probs [N,A], value [N]. */
/* params -> prepared (see the top of this file): 2 small kernels.  Call after every change of
 * the parameters. */
ARL_API int64_t arl_prepared_floats(void);
ARL_API int arl_prepare_weights(const float* params, float* prepared, void* stream);
ARL_API int arl_conv1_forward(const float* prepared, const uint8_t* ring, float* a1, int num_envs,
                      int ring_slots, int first_slot, int steps, void* stream);
/* a2 = ONE split block of num_samples rows. */
ARL_API int arl_conv2_forward(const float* prepared, const float* a1, float* a2, int64_t num_samples,
                      void* stream);
/* a2 = one split block of num_samples rows (as arl_conv2_forward wrote it); h f32 [N,256]. */
ARL_API int arl_fc_forward(const float* params, const float* prepared, const float* a2, float* h,
                   int64_t num_samples, void* stream);
ARL_API int arl_heads_forward(const float* params, int action_size, const float* h, float* logits,
                      float* probs, float* value, int64_t num_samples, void* stream);
/* fc256, then heads + softmax and -- when `actions` is not NULL -- the action draw of
 * arl_sample_actions in the SAME launch as the heads (Philox step = step + *step_dev when step_dev
 * is not NULL): two launches for agent.py:251-254 / network.py:62-79 instead of three.  (Fusing the
 * heads into the fc256 kernel's cluster reduction was built, measured slower and dropped: fc.cu.) */
ARL_API int arl_fc_heads_forward(const float* params, const float* prepared, int action_size,
                         const float* a2, float* h, float* logits, float* probs, float* value,
                         int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                         uint64_t seed, int64_t num_samples, void* stream);

/* The four above back to back, after arl_prepare_weights when refresh_prepared != 0 (pass 1
 * unless `prepared` was made from these very parameters by an earlier call). */
/* Rows of one a2 block = the envs one forward launch handles: num_envs up to 16 384, else the
 * largest divisor of num_envs that is <= 16 384 (arl_forward with steps == 1, arl_forward_sample
 * and arl_forward_egreedy then run several launches over env ranges, arl_backward hands this to
 * arl_fc_backward). */
ARL_API int64_t arl_a2_block_rows(int num_envs);
ARL_API int arl_forward(const float* params, float* prepared, int refresh_prepared, int action_size,
                const uint8_t* ring, int num_envs, int ring_slots, int first_slot, int steps,
                float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                void* stream);
/* arl_forward for ONE env step (steps = 1) that also draws the actions (network.py:72):
 * conv1, conv2, then arl_fc_heads_forward. */
ARL_API int arl_forward_sample(const float* params, float* prepared, int refresh_prepared, int action_size,
                       const uint8_t* ring, int num_envs, int ring_slots, int first_slot,
                       float* a1, float* a2, float* h, float* logits, float* probs, float* value,
                       int32_t* actions, int64_t env_id_base, int64_t step, const int64_t* step_dev,
                       uint64_t seed, void* stream);
/* arl_forward_sample with the epsilon-greedy draw of agent.py:141-151 in place of the policy
 * sample (the n-step Q learner, Mnih et al. 2016): conv1, conv2, fc256, then heads + softmax + the
 * draw in one launch.  The Q values are the p_w/p_b head ("logits"), as in arl_q_lossgrad.
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

/* Test hook for the tcgen05 GEMM behind arl_fc_forward/backward (fp32 inputs are split into
 * scratch blocks first; bf16x3 products, fp32 accumulation in TMEM), on caller-chosen shapes.
 * N % 16 == 0, K % 8 == 0.  Synchronises the stream.
 *   variant 0/1: D[M,N] = relu(A[M,K] . B[K,N] + extra[N])            (forward instantiation)
 *   variant 2  : D[M,N] = (A[M,K] . B[N,K]^T) where extra[M,N] > 0, else 0        (dgrad)
 *   variant 3/4: D[z][M,N] = A[K,M]^T . B[K,N] over split-K slice z  (M % 8 == 0)  (wgrad) */
ARL_API int arl_debug_gemm(int variant, const float* A, const float* B, float* D, const float* extra,
                           int M, int N, int K, int k_splits, void* stream);

/* ---- K4: action sampling, returns, loss gradients -----------------------------------
 * network.py:72 batch_sample(policy) (undefined in the reference): Philox4x32-10 keyed
 * (seed; env_id_base + b, step), inverse CDF over the f32 running sum.  actions i32. */
ARL_API int arl_sample_actions(const float* probs, int32_t* actions, int num_envs, int action_size,
                       int64_t env_id_base, int64_t step, uint64_t seed, void* stream);
/* agent.py:146-149 epsilon-greedy over argmax (ties -> lowest index, agent.py:254). */
ARL_API int arl_greedy_actions(const float* scores, int32_t* actions, int num_envs, int action_size,
                       void* stream);

/* agent.py:141-151 (the as-running async-Q learner): with probability ep a uniform random action,
 * else argmax_a q (ties -> lowest index).  The reference draws from Python's `random`
 * (main.py:41); here: Philox4x32-10 block (env_id_base + b, step, 1) keyed by seed, word 0 ->
 * u < ep, word 1 -> floor(x * A / 2^32).  q f32 [num_envs, A]. */
ARL_API int arl_egreedy_actions(const float* q, int32_t* actions, int num_envs, int action_size, float ep,
                        int64_t env_id_base, int64_t step, uint64_t seed, void* stream);

/* GymEnvironment.act for action_repeat == 1 (environment.py:78-96), batched: with is_training, an
 * env whose lives dropped during the step loses one reward point and its episode ends
 * (environment.py:86-88).  step_terminal / terminal are bytes (0/1; torch.bool storage). */
ARL_API int arl_act_update(const float* step_reward, const uint8_t* step_terminal,
                   const int32_t* lives_before, const int32_t* lives_after, int is_training,
                   float* reward, uint8_t* terminal, int num_envs, void* stream);
/* Agent.observe's rollout append (agent.py:158-160): this step's reward / terminal -> slot t of
 * the [T,B] rollout buffers (the reward clip of agent.py:154 happens in arl_returns_lossgrad). */
ARL_API int arl_observe_store(const float* reward, const uint8_t* terminal, float* reward_slot,
                      uint8_t* terminal_slot, int num_envs, void* stream);

/* agent.py:186-190 + 310-314 (async 1-step Q learning with a target network):
 *   target = clip(r) + (1-terminal) * discount * max_a q_next[n][a]
 *   delta  = target - q[n][actions[n]];   dq[n][a] = -2 * delta * grad_scale  (0 elsewhere)
 * i.e. the gradient of grad_scale * sum(delta^2)  (grad_scale = 1/N gives the reference's
 * mean(delta^2)).  loss_sums (optional) f32 [2] += {sum delta^2, sum q[n][a]}. */
ARL_API int arl_q_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                   const float* q, const float* q_next, float* target, float* dq, float* loss_sums,
                   int64_t num_samples, int action_size, float discount, float reward_min,
                   float reward_max, float grad_scale, void* stream);

/* n-step Q targets and the loss gradient of one rollout (asynchronous n-step Q-learning, Mnih et
 * al. 2016; T = t_max steps of num_envs envs):
 *   R_T = max_a q_boot[b][a]  (Q(s_T) under the target parameters, fmaxf in index order)
 *   R_t = fmaf(gamma * (1 - term_t), R_{t+1}, clip(r_t))  -- the recurrence of
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

/* Algorithm 3 (assets/a3c.png) returns with the terminal mask of agent.py:188-190 and the
 * reward clip of agent.py:154, then d(total_loss)/d(logits,value) per network.py:81-94:
 *   R_t = clip(r_t) + gamma*(1-term_t)*R_{t+1},  R_T = v_boot
 *   dlogits = grad_scale*(-(R-V)*(onehot(a)-p) + beta*p*(logp+H)),  dvalue = grad_scale*(V-R)
 * rewards f32 [T,B], terminals u8 [T,B], actions i32 [T,B], logits [T,B,A], value [T,B].
 * loss_sums (optional, may be NULL) f32 [3] += {sum policy_loss, sum value_loss, sum entropy}
 * unscaled. */
ARL_API int arl_returns_lossgrad(const float* rewards, const uint8_t* terminals, const int32_t* actions,
                         const float* logits, const float* value, const float* v_boot,
                         float* returns, float* dlogits, float* dvalue, float* loss_sums,
                         int t_max, int num_envs, int action_size, float gamma, float beta,
                         float reward_min, float reward_max, float grad_scale, void* stream);

/* ---- backward: agent.py:317 compute_gradients ---------------------------------------
 * Accumulation over the T steps of Algorithm 3 is the reduction over samples inside the
 * weight-gradient kernels.  grads is the flat buffer (overwritten).  Scratch buffers are
 * caller-owned: d_h [(N + roundup8(N)),256] (two split blocks, see the top of this file), d_a2 [N,2592],
 * d_a1 [N * ARL_DA1_BYTES bytes] (fp16 grid layout, see the top of this file),
 * workspace >= arl_backward_workspace_bytes.  a2 = the rollout's conv2 outputs as a sequence of
 * split blocks of a2_block_rows rows each (one per forward call: a2_block_rows = num_envs);
 * prepared must hold arl_prepare_weights of the parameters the forward used. */
ARL_API int64_t arl_backward_workspace_bytes(int action_size);
/* tensor_scale / grad_unscale: the gradients handed from layer to layer (d_h, d_a2, d_a1) are
 * stored multiplied by tensor_scale, a power of two chosen by the host so that they sit in the
 * middle of the range of the 16-bit operand formats whatever the batch size is (the loss gradient
 * is divided by the number of envs, agent.py's mean); arl_heads_backward applies it when it writes
 * d_h, the three weight-gradient entries divide it out again (grad_unscale = 1 / tensor_scale:
 * exact), so `grads` always holds the true gradient.  arl_backward takes tensor_scale. */
ARL_API int arl_heads_backward(const float* params, int action_size, const float* h,
                       const float* dlogits, const float* dvalue, float* d_h, float* grads,
                       void* workspace, int64_t num_samples, float tensor_scale, void* stream);
ARL_API int arl_fc_backward(const float* prepared, const float* a2, int64_t a2_block_rows,
                    const float* d_h, float* d_a2, float* grads, void* workspace,
                    int64_t num_samples, float grad_unscale, void* stream);
/* l2_w, l2_b, d_a1 and l1_b (the column sums of d_a1). */
ARL_API int arl_conv2_backward(const float* prepared, const float* a1, const float* d_a2, float* d_a1,
                       float* grads, void* workspace, int64_t num_samples, float grad_unscale,
                       void* stream);
/* l1_w only (l1_b comes from arl_conv2_backward). */
ARL_API int arl_conv1_backward(const uint8_t* ring, const float* d_a1, float* grads, void* workspace,
                       int num_envs, int ring_slots, int first_slot, int steps, float grad_unscale,
                       void* stream);
ARL_API int arl_backward(const float* params, const float* prepared, int action_size,
                 const uint8_t* ring, int num_envs, int ring_slots, int first_slot, int steps,
                 const float* a1, const float* a2,
                 const float* h, const float* dlogits, const float* dvalue, float* d_h,
                 float* d_a2, float* d_a1, float* grads, void* workspace, float tensor_scale,
                 int allreduce, void* stream);

/* ---- the 'nature' trunk (network.py:30-42): conv32 8x8 s4 -> conv64 4x4 s2 -> conv64 3x3 s1 ->
 * fc512 -> heads.  A second shape set with plain float32 NHWC tensors on both sides:
 *   x  f32 [N,84,84,4]  the stacks (History.get(), values 0..255; the /255 of network.py:33 is folded in)
 *   a1 [N,20,20,32]  a2 [N,9,9,64]  a3 [N,7,7,64] (flatten (h*7+w)*64+c)  h [N,512]
 * Parameters / gradients: flat f32 in the order l1_w [8,8,4,32] l1_b l2_w [4,4,32,64] l2_b
 * l3_w [3,3,64,64] l3_b l4_w [3136,512] l4_b p_w [512,A] p_b q_w [512,1] q_b (TF layouts;
 * arl_nature_param_layout: ARL_NATURE_TENSORS+1 offsets).  Every contraction is one generic
 * tcgen05 kernel whose producers gather the operands (im2col, its transpose, the transposed
 * convolution per stride-parity class) -- csrc/nature.cu.  d_* are the gradients w.r.t. the
 * layer outputs before their relu, kept for inspection.  Update: arl_clip_rmsprop_layout. */
ARL_API int arl_nature_param_layout(int action_size, int64_t* offsets);
ARL_API int64_t arl_nature_workspace_bytes(int action_size);
ARL_API int arl_nature_forward(const float* params, int action_size, const float* x, float* a1, float* a2,
                       float* a3, float* h, float* logits, float* probs, float* value,
                       int64_t num_samples, void* stream);
ARL_API int arl_nature_backward(const float* params, int action_size, const float* x, const float* a1,
                        const float* a2, const float* a3, const float* h, const float* dlogits,
                        const float* dvalue, float* d_h, float* d_a3, float* d_a2, float* d_a1,
                        float* grads, void* workspace, int64_t num_samples, void* stream);
/* arl_clip_rmsprop for any flat layout: num_tensors segments given by offsets[num_tensors+1]
 * (host array).  step_dev == NULL: use lr; else the schedule of arl_clip_rmsprop_sched. */
ARL_API int arl_clip_rmsprop_layout(float* params, float* rms, const float* grads, const int64_t* offsets,
                            int num_tensors, float lr, const int64_t* step_dev, int64_t step_offset,
                            double base_lr, int64_t max_step, float decay, float eps, float clip_norm,
                            float* norms_out, void* workspace, void* stream);

/* ---- device-resident step counter (CUDA-graph capture of the loop, SURVEY a16) -------------
 * A captured graph replays fixed kernel arguments, so the two host values that change on every
 * launch -- the Philox step of the sampler and the step the learning rate is annealed on
 * (agent.py:393-395) -- can also be read from an int64 counter in device memory:
 *   arl_sample_actions_dev   like arl_sample_actions with step = *step_dev
 *   arl_step_advance         *counter += inc (one thread)
 *   arl_clip_rmsprop_sched   like arl_clip_rmsprop with
 *                            lr = (max_step - (*step_dev + step_offset) + 1) / max_step * base_lr
 *                            evaluated in double on the device and rounded to float once. */
ARL_API int arl_sample_actions_dev(const float* probs, int32_t* actions, int num_envs, int action_size,
                           int64_t env_id_base, const int64_t* step_dev, uint64_t seed, void* stream);
ARL_API int arl_step_advance(int64_t* counter, int64_t inc, void* stream);
/* arl_observe_store + arl_step_advance as one launch (the per-step rollout append of agent.py:158-160
 * and the loop's step increment of agent.py:55). */
ARL_API int arl_observe_store_advance(const float* reward, const uint8_t* terminal, float* reward_slot,
                              uint8_t* terminal_slot, int num_envs, int64_t* step_counter, int64_t inc,
                              void* stream);
ARL_API int arl_clip_rmsprop_sched(float* params, float* rms, const float* grads, int action_size,
                           const int64_t* step_dev, int64_t step_offset, double base_lr,
                           int64_t max_step, float decay, float eps, float clip_norm,
                           float* norms_out, void* workspace, void* stream);

/* ---- the exchange step: gradient all-reduce across the GPUs of a box ---------------------
 * Replaces the reference's parameter-server push (main.py:60-62 places the variables on the ps,
 * agent.py:321 applies every worker's gradients there): one process per GPU, replicas of the
 * parameters, and ONE all-reduce(sum) of the flat gradient buffer per t_max cycle (NCCL over
 * NVLink, bound at run time from libnccl.so.2).  Rank 0 makes an id (arl_comm_unique_id,
 * ARL_COMM_ID_BYTES bytes), the host distributes it by any means, every rank calls
 * arl_comm_init on its own device; one communicator per process.
 *   arl_allreduce_grads   in-place sum over ranks of grads[0, count) on `stream`.
 *   arl_allreduce_begin / arl_allreduce_end   the same for a slice, on the library's side stream,
 *     ordered after what is already queued on `stream`; `end` makes `stream` wait for all slices
 *     begun.  arl_backward(allreduce = 1) sums the whole buffer with ONE arl_allreduce_grads after
 *     its last kernel; with ARL_ALLREDUCE_OVERLAP=1 in the environment it sends the l4_w..q_b slice
 *     (98 % of the bytes, final after the fc256 weight gradient) through begin / end while the conv
 *     backward kernels run instead -- measured: nothing is hidden (the persistent conv kernels leave
 *     NCCL no SMs), profiles/r02_allreduce_overlap.txt. */
#define ARL_COMM_ID_BYTES 128
ARL_API int arl_comm_unique_id(uint8_t* id_out);
ARL_API int arl_comm_init(const uint8_t* id_bytes, int rank, int nranks);
ARL_API int arl_comm_size(void);                 /* ranks of the communicator, 0 = none */
ARL_API int arl_comm_nccl_version(void);         /* e.g. 22809; 0 = NCCL not loadable */
ARL_API int arl_comm_destroy(void);
ARL_API int arl_allreduce_grads(float* grads, int64_t count, void* stream);
ARL_API int arl_allreduce_begin(float* grads, int64_t offset, int64_t count, void* stream);
ARL_API int arl_allreduce_end(void* stream);
/* The same exchange WITHOUT a collective kernel, over NVLink peer memory (CUDA IPC), fused into the
 * update: arl_comm_enable_p2p(count) gives every rank a buffer of two gradient slots + flag words
 * mapped into every other rank.  arl_exchange_clip_rmsprop is arl_clip_rmsprop_layout whose norm
 * pass first publishes this rank's `grads` (copy into a slot, flag word raised in every peer's
 * memory), waits for every rank's flag and then READS all ranks' slots, adding them in rank order
 * (bit-identical on every rank) into `grads` while it accumulates the per-tensor sums of squares:
 * no NCCL kernel, no extra pass over the gradient.  Call it INSTEAD of arl_allreduce_grads +
 * arl_clip_rmsprop*, on every rank, once per cycle.  arl_comm_p2p_error() != 0: a peer's flag did
 * not arrive within ~3 s (the reduction gives up instead of hanging the GPU). */
ARL_API int arl_comm_enable_p2p(int64_t count);
ARL_API int arl_comm_p2p_enabled(void);
ARL_API int arl_comm_p2p_error(void);
ARL_API int arl_exchange_clip_rmsprop(float* params, float* rms, float* grads, const int64_t* offsets,
                              int num_tensors, float lr, const int64_t* step_dev, int64_t step_offset,
                              double base_lr, int64_t max_step, float decay, float eps,
                              float clip_norm, float* norms_out, void* workspace, void* stream);

/* ---- K5: per-tensor clip + shared RMSProp -------------------------------------------
 * agent.py:316-319 clip_by_norm(g, clip) per tensor, then TF ApplyRMSProp as configured at
 * main.py:63-65:  ms += (g^2-ms)(1-decay);  w -= lr*g/sqrt(ms+eps).  `lr` per agent.py:393-395
 * is computed by the caller.  norms_out (optional) f32 [ARL_NUM_TENSORS] = pre-clip norms. */
ARL_API int arl_clip_rmsprop(float* params, float* rms, const float* grads, int action_size, float lr,
                     float decay, float eps, float clip_norm, float* norms_out, void* workspace,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* ASYNCRL_B200_H_ */
