"""Network: the A3C policy/value net (reference src/network.py:6-127, 'nips' trunk as wired in
agent.py:226-252), with the reference's attribute names: ``w`` {l1_w..q_b}, ``policy_logits``,
``policy``, ``log_policy``, ``policy_entropy``, ``sampled_action``, ``value``, ``R``,
``total_loss``, ``copy_from_global``, ``save_model``, ``load_model``.

The reference builds a TF graph; this class owns flat f32 device buffers (parameters,
gradients, RMSProp slot) plus the rollout activations, and launches the sm_100a kernels
through the C-ABI.  Repairs of the reference's dead/broken graph (SURVEY.md D2-D3) follow
the paper's Algorithm 3 and are listed in DESIGN.md.
"""
import os
from collections import OrderedDict

import numpy as np
import torch

from .. import _cabi

PARAM_NAMES = ("l1_w", "l1_b", "l2_w", "l2_b", "l4_w", "l4_b", "p_w", "p_b", "q_w", "q_b")
# dueling streams (include/asyncrl_b200_dueling_streams.h): the advantage stream's hidden layer follows q_b
STREAMS_PARAM_NAMES = PARAM_NAMES + ("la_w", "la_b")
# the A3C LSTM agent (include/asyncrl_b200_lstm.h): the LSTM layer's kernel and bias follow q_b
LSTM_PARAM_NAMES = PARAM_NAMES + ("lstm_w", "lstm_b")
LSTM_CELLS = 256
A1_ELEMS, A2_ELEMS, FC, DA1_ELEMS = 6400, 2592, 256, 7056
A1_STORE = 3200                                               # float32 words of storage per sample of a1 (fp16)
DA1_STORE = 3528                                              # ... of d_a1 (fp16 on the 21x21 grid)


def decode_a1(raw, n=None):
    """conv1's output lives in HBM as fp16 in space-to-depth blocks (csrc/convs_tc.cu "a1s":
    [n][kc = (i*2+j)*2 + chalf][q = yp*10 + xp][8 ch], pixel (y,x) = (2yp+i, 2xp+j), 12 800 bytes
    per sample) -- the layout the conv2 tensor-core kernels consume without conversion.  ``raw`` is
    the storage the C-ABI filled (any shape whose first dimension is the sample count, or pass
    ``n``); returns the float32 [N,20,20,16] activations (network.py:47-48 l1)."""
    n = raw.shape[0] if n is None else n
    b = raw.reshape(-1)[:n * A1_STORE].view(torch.float16).reshape(n, 2, 2, 2, 10, 10, 8)
    return b.float().permute(0, 4, 1, 5, 2, 3, 6).reshape(n, 20, 20, 16)   # [n, yp, i, xp, j, chalf, 8]


def decode_split(raw, rows, cols):
    """A "split block" (include/asyncrl_b200.h: [hi|lo][cols/8 chunks][rows][8] bf16, the operand
    layout of the fc256 tensor-core kernels) -> float32 [rows, cols].  ``raw`` is the float32
    storage of rows*cols elements the C-ABI filled."""
    b = raw.reshape(-1).view(torch.bfloat16).reshape(2, cols // 8, rows, 8)
    return (b[0].float() + b[1].float()).permute(1, 0, 2).reshape(rows, cols)


def encode_split(x):
    """float32 [rows, cols] -> the split block decode_split reads (same element count, float32
    storage): hi = bf16(x), lo = bf16(x - hi).  Host-side helper for feeding a plain activation
    matrix to a kernel that expects a block (ops.linear(..., input_is_split=False)) and for tests;
    the kernels write blocks themselves."""
    rows, cols = x.shape
    hi = x.float().to(torch.bfloat16)
    lo = (x.float() - hi.float()).to(torch.bfloat16)
    b = torch.stack([hi, lo]).reshape(2, rows, cols // 8, 8).permute(0, 2, 1, 3).contiguous()
    return b.view(torch.float32).reshape(rows, cols)


def decode_da1(raw, n):
    """The gradient w.r.t. conv1's output (include/asyncrl_b200.h: one fp16 per value on the 21x21
    grid, [2 channel groups][n*441 + y*21 + x][8], 14 112 bytes per sample, still multiplied by
    tensor_scale) -> float32 [n,20,20,16]."""
    b = raw.reshape(-1)[:n * DA1_STORE].view(torch.float16).reshape(2, n, 21, 21, 8)
    return b.float().permute(1, 2, 3, 0, 4).reshape(n, 21, 21, 16)[:, :20, :20]


def param_shapes(action_size, streams=False, lstm=False):
    shapes = OrderedDict([
        ("l1_w", (8, 8, 4, 16)), ("l1_b", (16,)), ("l2_w", (4, 4, 16, 32)), ("l2_b", (32,)),
        ("l4_w", (A2_ELEMS, FC)), ("l4_b", (FC,)), ("p_w", (FC, action_size)),
        ("p_b", (action_size,)), ("q_w", (FC, 1)), ("q_b", (1,))])
    if streams:
        shapes["la_w"], shapes["la_b"] = (A2_ELEMS, FC), (FC,)
    if lstm:
        shapes["lstm_w"], shapes["lstm_b"] = (FC + LSTM_CELLS, 4 * LSTM_CELLS), (4 * LSTM_CELLS,)
    return shapes


def initial_weights(action_size, seed=123, stddev=0.02, streams=False, lstm=False):
    """network.py:10 truncated_normal(0,.02) for convs, ops.py:36-39 normal(.02) for ``linear``
    matrices, zero biases (ops.py:24,38-39).  Returns an OrderedDict of CPU float32 tensors.
    ``streams``: la_w / la_b too, drawn after the others (a plain network's weights do not change);
    ``lstm``: lstm_w (like the ``linear`` matrices) / lstm_b the same way."""
    g = torch.Generator().manual_seed(int(seed))
    out = OrderedDict()
    for name, shape in param_shapes(action_size, streams, lstm).items():
        if name.endswith("_b"):
            out[name] = torch.zeros(shape)
        elif name in ("l1_w", "l2_w"):
            w = torch.empty(shape)
            torch.nn.init.trunc_normal_(w, 0.0, stddev, -2 * stddev, 2 * stddev, generator=g)
            out[name] = w
        else:
            out[name] = torch.randn(shape, generator=g) * stddev
    return out


class Network(object):
    # dueling Q heads (Wang et al. 2016, include/asyncrl_b200_dueling.h): the Q row every Q forward
    # writes to ``policy_logits`` is v + (adv - mean adv), with p_w/p_b the advantage stream and q_w/q_b
    # the value stream; the Q losses then train both heads.  Fixed for the network's life.
    dueling = False
    # double Q-learning targets (van Hasselt et al. 2016, include/asyncrl_b200_double.h): the async_q and
    # nstep_q losses bootstrap from Q(s', a*; theta^-), a* = argmax_a Q(s'; theta); one more forward per
    # update gives Q(s_T; theta) (``q_online_T``).  No parameter or stored state: fixed for the network's life.
    double_q = False
    # dueling streams (Wang et al. 2016's architecture, include/asyncrl_b200_dueling_streams.h): with
    # ``dueling``, each stream on its own fc256 layer on a2 -- l4_w/l4_b the value stream's, la_w/la_b
    # (appended to the parameters) the advantage stream's; h (``l4``) is [N, 512] = [h_v | h_a].
    dueling_streams = False
    # the A3C LSTM agent (Mnih et al. 2016, include/asyncrl_b200_lstm.h): 256 LSTM cells between fc256 and
    # the heads, lstm_w/lstm_b appended to the parameters; each env carries (h, c) (``lstm_state``) from
    # step to step, reset where the previous step was terminal.  a3c only; fixed for the network's life.
    lstm = False

    def __init__(self, sess=None, data_format='NHWC', history_length=4, screen_height=84,
                 screen_width=84, action_size=6, activation_fn='relu', initializer=None,
                 gamma=0.99, beta=0.01, global_network=None, global_optim=None, DQN_type='nips',
                 num_envs=256, t_max=5, device='cuda', seed=123, decay=0.99, epsilon=0.1,
                 clip_norm=40.0, min_reward=-1.0, max_reward=1.0, dueling=False, double_q=False,
                 dueling_streams=False, lstm=False):
        if DQN_type.lower() != 'nips':
            raise ValueError("Network is the 'nips' trunk (network.py:43-52); DQN_type='nature' "
                             "(network.py:30-42) is network_nature.NatureNetwork -- use "
                             "make_network(DQN_type=...); got %r" % (DQN_type,))
        if data_format != 'NHWC':
            raise ValueError("main.py:45 forces NHWC; NCHW is not built")
        if (history_length, screen_height, screen_width) != (4, 84, 84):
            raise ValueError("kernels are built for 84x84x4 stacks")
        if activation_fn not in ('relu', None) and getattr(activation_fn, '__name__', '') != 'relu':
            raise ValueError("only relu is built")
        self.sess = sess
        self.device = torch.device(device)
        _cabi.init(self.device)
        self.action_size, self.num_envs, self.t_max = int(action_size), int(num_envs), int(t_max)
        self.gamma, self.beta = float(gamma), float(beta)
        self.decay, self.epsilon, self.clip_norm = float(decay), float(epsilon), float(clip_norm)
        self.min_reward, self.max_reward = float(min_reward), float(max_reward)
        self.global_network = global_network
        self.dueling = bool(dueling)
        self.double_q = bool(double_q)
        self.dueling_streams = bool(dueling_streams)
        if self.dueling_streams and not self.dueling:
            raise ValueError("dueling_streams=True gives the dueling heads a hidden layer per stream; it needs "
                             "dueling=True")
        self.lstm = bool(lstm)
        if self.lstm and (self.dueling or self.dueling_streams or self.double_q):
            raise ValueError("lstm=True is the A3C LSTM agent (a policy/value network); it has no dueling or "
                             "double-Q form")
        S, L = self.dueling_streams, self.lstm
        self.param_names = STREAMS_PARAM_NAMES if S else LSTM_PARAM_NAMES if L else PARAM_NAMES

        A, B, T = self.action_size, self.num_envs, self.t_max
        self.offsets = (_cabi.streams_param_layout(A) if S else _cabi.lstm_param_layout(A) if L
                        else _cabi.param_layout(A))
        n_params = self.offsets[-1]
        dev = self.device
        self.params = torch.zeros(n_params, device=dev)
        self.grads = torch.zeros(n_params, device=dev)
        self.rms = torch.ones(n_params, device=dev)           # TF RMSProp slot starts at 1.0
        self.w, self.g = OrderedDict(), OrderedDict()
        for i, (name, shape) in enumerate(param_shapes(A, S, L).items()):
            self.w[name] = self.params[self.offsets[i]:self.offsets[i + 1]].view(shape)
            self.g[name] = self.grads[self.offsets[i]:self.offsets[i + 1]].view(shape)
        # the weights as the tensor-core kernels keep them resident (arl_prepare_weights); refreshed
        # lazily: the key is (tensor version, number of C-ABI writes) of the parameters it was made from
        self.fc_w = torch.empty(_cabi.prepared_floats(S, L), device=dev)
        self._fc_w_key = None
        self._param_writes = 0
        self.set_weights(initial_weights(A, seed, streams=S, lstm=L))
        H = 2 * FC if S else FC                               # width of h (streams: [h_v | h_a])

        N = B * T
        f32 = dict(device=dev, dtype=torch.float32)
        # rollout activations, t-major: sample n = t*B + b
        self.l1 = torch.empty(N, A1_STORE, **f32)             # network.py:47-48, stored as blocked fp16: see a1()
        self.l2 = torch.empty(N, A2_ELEMS, **f32)             # network.py:49-50 (flattened NHWC), one split block per step: see a2()
        self.l4 = torch.empty(N, H, **f32)                    # network.py:51-52
        self.policy_logits = torch.empty(N, A, **f32)         # network.py:62
        self.policy = torch.empty(N, A, **f32)                # network.py:65
        self.value = torch.empty(N, **f32)                    # network.py:79
        self.sampled_action = torch.zeros(N, dtype=torch.int32, device=dev)   # network.py:72
        self.R = torch.empty(N, **f32)                        # network.py:82
        # bootstrap-state scratch (not kept for backward)
        self._b = dict(l1=torch.empty(B, A1_STORE, **f32), l2=torch.empty(B, A2_ELEMS, **f32),
                       l4=torch.empty(B, H, **f32), logits=torch.empty(B, A, **f32),
                       probs=torch.empty(B, A, **f32), value=torch.empty(B, **f32))
        # backward scratch
        self.d_logits = torch.empty(N, A, **f32)
        self.d_value = torch.empty(N, **f32)
        # d_h twice (include/asyncrl_b200.h): a split block of N rows, then its transposed copy
        # (groups of 8 samples x 256 columns) for the fc256 weight gradient: see d_h()
        self.d_l4 = torch.empty(N + (N + 7) // 8 * 8, H, **f32)
        self.d_l2 = torch.empty(N, A2_ELEMS, **f32)
        self.d_l1 = torch.empty(N, DA1_STORE, **f32)          # fp16 on the 21x21 grid: see decode_da1
        self.workspace = torch.empty(_cabi.workspace_bytes(A, S, L), dtype=torch.uint8, device=dev)
        self.loss_sums = torch.zeros(3, **f32)                # sum policy / value loss, entropy
        self.grad_norms = torch.zeros(len(self.param_names), **f32)
        self.events = {}
        self.tensor_scale = 1.0                               # set by compute_gradients
        if L:
            C = LSTM_CELLS
            # the recurrent state the next rollout step reads (fixed addresses: CUDA-graph replay), and
            # play's own, which Agent.play resets per episode
            self.state_h, self.state_c = torch.zeros(B, C, **f32), torch.zeros(B, C, **f32)
            self.play_h, self.play_c = torch.zeros(B, C, **f32), torch.zeros(B, C, **f32)
            # per rollout step (include/asyncrl_b200_lstm.h): x = h_fc is ``l4``; xh one split block per step
            self.xh = torch.empty(N, 2 * C, **f32)
            self.lstm_z = torch.empty(B, 4 * C, **f32)
            self.gates = torch.empty(N, 4 * C, **f32)
            self.c_prev = torch.empty(N, C, **f32)
            self.c_seq = torch.empty(N, C, **f32)
            self.h_lstm = torch.empty(N, C, **f32)            # the heads' input
            self._b.update(xh=torch.empty(B, 2 * C, **f32), h=torch.empty(B, C, **f32), c=torch.empty(B, C, **f32))
            # BPTT scratch
            self.d_h_lstm = torch.empty(N, C, **f32)
            self.dz = torch.empty(N, 4 * C, **f32)
            self.dxh = torch.empty(N, 2 * C, **f32)
            self.dc = torch.empty(B, C, **f32)

    # -- the LSTM state ---------------------------------------------------------------------
    def lstm_state(self, play=False):
        """(h, c) of every env, float32 [B, 256] each (copies): the state the next step reads; ``play``:
        Agent.play's."""
        if play:
            return self.play_h.clone(), self.play_c.clone()
        return self.state_h.clone(), self.state_c.clone()

    def reset_lstm_state(self, play=False):
        """Zero the recurrent state (a new game for every env)."""
        if self.lstm:
            for t in ((self.play_h, self.play_c) if play else (self.state_h, self.state_c)):
                t.zero_()

    def _forward_lstm(self, history, refresh, l1, l2, h_fc, state, reset, advance, xh, gates, c_prev, c, h, logits,
                      probs, value, actions=None, env_id_base=0, step=0, step_dev=None, seed=0):
        """arl_forward_lstm: one env step of the trunk, the LSTM step from ``state`` = (h, c) (``reset``: u8 [B],
        nonzero = the env's previous step was terminal; advanced when ``advance``) and the heads on h."""
        P = _cabi.ptr
        self._timed_call("arl_forward_lstm", P(self.params), P(self.fc_w), int(bool(refresh)), self.action_size,
                         P(history.ring), self.num_envs, history.ring_slots, history.first_slot(0), P(l1), P(l2),
                         P(h_fc), P(state[0]), P(state[1]),
                         P(reset), int(bool(advance)), P(xh), P(self.lstm_z), P(gates), P(c_prev), P(c), P(h),
                         P(logits), P(probs), P(value), P(actions), int(env_id_base), int(step), P(step_dev),
                         int(seed), _cabi.stream_ptr())

    # -- parameters -----------------------------------------------------------------------
    def set_weights(self, weights):
        for name in self.param_names:
            self.w[name].copy_(torch.as_tensor(np.asarray(weights[name]), dtype=torch.float32))

    def get_weights(self):
        return OrderedDict((k, v.detach().cpu().numpy().copy()) for k, v in self.w.items())

    def copy_from_global(self):
        """network.py:96-107: theta' <- theta.  Replicas are updated synchronously with the same
        all-reduced gradient, so this is the identity unless a global_network was given."""
        if self.global_network is not None and self.global_network is not self:
            self.params.copy_(self.global_network.params)

    # -- forward ----------------------------------------------------------------------------
    def _rows(self, t):
        B = self.num_envs
        return slice(t * B, (t + 1) * B)

    # Optional per-entry timing (bench.py): ``timed`` is a set of C-ABI entry names (or {'*'});
    # the composed arl_forward/arl_backward are then issued as their per-layer entries -- the
    # same kernels in the same order -- with a CUDA-event pair around each selected entry.
    timed = None

    def _timed_call(self, name, *args):
        if self.timed is not None and (name in self.timed or '*' in self.timed):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _cabi.call(name, *args)
            e1.record()
            self.events.setdefault(name, []).append((e0, e1))
        else:
            _cabi.call(name, *args)

    def _fc_w_stale(self):
        """True (once) when l4_w has changed since fc_w was made: torch bumps ``_version`` on every
        in-place write to params or to a view of it, C-ABI writes are counted by hand."""
        key = (self.params._version, self._param_writes)
        stale = key != self._fc_w_key
        self._fc_w_key = key
        return stale

    def _prepare(self, params, fc_w):
        """Rebuild the prepared weight images ``fc_w`` from ``params``."""
        P, st = _cabi.ptr, _cabi.stream_ptr()
        if self.dueling_streams:
            _cabi.call("arl_prepare_weights_streams", P(params), P(fc_w), self.action_size, st)
        elif self.lstm:
            _cabi.call("arl_prepare_weights_lstm", P(params), P(fc_w), self.action_size, st)
        else:
            _cabi.call("arl_prepare_weights", P(params), P(fc_w), st)

    def _refresh(self, refresh):
        """A ``refresh`` argument as the C-ABI's int, None decided from the parameter version."""
        return (1 if self._fc_w_stale() else 0) if refresh is None else int(bool(refresh))

    def _forward_into(self, history, l1, l2, l4, logits, probs, value, refresh=None):
        """``refresh``: rebuild the prepared weight images first; None = decide here from the
        parameter version (host state).  A captured region passes the decision in."""
        P, st = _cabi.ptr, _cabi.stream_ptr()
        B, A = self.num_envs, self.action_size
        refresh = self._refresh(refresh)
        if self.dueling:
            self._forward_dueling(self.params, self.fc_w, refresh, history, history.first_slot(0), 1, l1, l2, l4,
                                  logits, probs, value)
            return
        if self.timed is None:
            _cabi.call("arl_forward", P(self.params), P(self.fc_w), refresh, A, P(history.ring), B,
                       history.ring_slots, history.first_slot(0), 1, P(l1), P(l2), P(l4),
                       P(logits), P(probs), P(value), st)
            return
        if refresh:
            self._prepare(self.params, self.fc_w)
        self._timed_layers(history, l1, l2, l4, logits, probs, value, None, 0, 0, None, 0)

    def _forward_dueling(self, params, fc_w, refresh, history, first_slot, steps, l1, l2, l4, logits, probs, value,
                         actions=None, env_id_base=0, step=0, step_dev=None, seed=0, ep=0.0, ep_sched=None):
        """arl_forward_dueling (arl_forward_streams with ``dueling_streams``): ``steps`` env steps from
        ``first_slot`` under ``params`` with the dueling Q row into ``logits``; with ``actions`` (one step)
        also the epsilon-greedy draw of ``forward_egreedy``.  One entry under ``timed``."""
        P = _cabi.ptr
        e0, e1, et, ls = (float(x) for x in (ep_sched if ep_sched is not None else (0.0, 0.0, 1.0, 0.0)))
        entry = "arl_forward_streams" if self.dueling_streams else "arl_forward_dueling"
        self._timed_call(entry, P(params), P(fc_w), int(bool(refresh)), self.action_size,
                         P(history.ring), self.num_envs, history.ring_slots, first_slot, steps, P(l1), P(l2), P(l4),
                         P(logits), P(probs), P(value), P(actions), int(env_id_base), int(step), P(step_dev),
                         int(seed), float(ep), e0, e1, et, ls, _cabi.stream_ptr())

    def _timed_layers(self, history, l1, l2, l4, logits, probs, value, actions, env_id_base, step, sd, seed):
        """The per-layer entries arl_forward / arl_forward_sample are made of, one event pair each
        (bench.py): the same launches in the same order, env range by env range when the batch is
        larger than one a2 block (arl_a2_block_rows)."""
        P, st = _cabi.ptr, _cabi.stream_ptr()
        B, A = self.num_envs, self.action_size
        c = _cabi.a2_block_rows(B)
        for o in range(0, B, c):
            r = slice(o, o + c)
            self._timed_call("arl_conv1_forward", P(self.fc_w), P(history.ring[r]), P(l1[r]), c,
                             history.ring_slots, history.first_slot(0), 1, st)
            self._timed_call("arl_conv2_forward", P(self.fc_w), P(l1[r]), P(l2[r]), c, st)
            # fc256, then heads + softmax (+ the action draw) as one launch
            self._timed_call("arl_fc_heads_forward", P(self.params), P(self.fc_w), A, P(l2[r]), P(l4[r]),
                             P(logits[r]), P(probs[r]), P(value[r]),
                             P(actions[r]) if actions is not None else None, int(env_id_base) + o,
                             int(step), sd, int(seed), c, st)

    def forward(self, history, t, refresh=None):
        """Forward of the current stack into rollout slot ``t``; returns (logits, policy, value)."""
        self._not_lstm("forward")
        r = self._rows(t)
        self._forward_into(history, self.l1[r], self.l2[r], self.l4[r], self.policy_logits[r],
                           self.policy[r], self.value[r], refresh)
        return self.policy_logits[r], self.policy[r], self.value[r]

    def forward_sample(self, history, t, step, seed, env_id_base=0, step_dev=None, refresh=None, reset=None):
        """``forward`` into rollout slot t + ``sample`` (network.py:72) as one composed call: the
        heads and the Philox draw run inside the fc256 kernel (arl_forward_sample).  The Philox step
        is ``step`` (+ the int64 device counter ``step_dev`` when given).  ``lstm``: the LSTM step runs
        between fc256 and the heads and advances the state; ``reset`` (u8 [B], None = none) marks the envs
        whose previous step was terminal (arl_forward_lstm)."""
        self._policy_value_only("forward_sample")
        r = self._rows(t)
        P, st = _cabi.ptr, _cabi.stream_ptr()
        B, A = self.num_envs, self.action_size
        refresh = self._refresh(refresh)
        if self.lstm:
            self._forward_lstm(history, refresh, self.l1[r], self.l2[r], self.l4[r], (self.state_h, self.state_c),
                               reset, True, self.xh[r], self.gates[r], self.c_prev[r], self.c_seq[r], self.h_lstm[r],
                               self.policy_logits[r], self.policy[r], self.value[r], self.sampled_action[r],
                               env_id_base, step, step_dev, seed)
            return self.sampled_action[r]
        sd = P(step_dev) if step_dev is not None else None
        if self.timed is None:
            _cabi.call("arl_forward_sample", P(self.params), P(self.fc_w), refresh, A, P(history.ring), B,
                       history.ring_slots, history.first_slot(0), P(self.l1[r]), P(self.l2[r]),
                       P(self.l4[r]), P(self.policy_logits[r]), P(self.policy[r]), P(self.value[r]),
                       P(self.sampled_action[r]), int(env_id_base), int(step), sd, int(seed), st)
            return self.sampled_action[r]
        if refresh:
            _cabi.call("arl_prepare_weights", P(self.params), P(self.fc_w), st)
        self._timed_layers(history, self.l1[r], self.l2[r], self.l4[r], self.policy_logits[r], self.policy[r],
                           self.value[r], self.sampled_action[r], env_id_base, step, sd, seed)
        return self.sampled_action[r]

    def a1(self):
        """conv1 activations of the rollout as float32 [N,20,20,16] (decoded from the device layout)."""
        return decode_a1(self.l1)

    def a2(self):
        """conv2 activations of the rollout as float32 [N,2592] (NHWC flatten, agent.py:231-232),
        decoded from the per-step split blocks."""
        B, c = self.num_envs, _cabi.a2_block_rows(self.num_envs)
        return torch.cat([decode_split(self.l2[t * B + o:t * B + o + c], c, A2_ELEMS)
                          for t in range(self.t_max) for o in range(0, B, c)])

    @staticmethod
    def pick_tensor_scale(grad_scale):
        """The power of two the layer-to-layer gradients are stored multiplied by
        (include/asyncrl_b200.h, arl_backward): 64 / grad_scale rounded to a power of two, i.e. the
        loss gradient as if it were multiplied by ~64 instead of divided by the env count."""
        import math
        e = int(round(math.log2(64.0 / max(float(grad_scale), 1e-30))))
        return float(2.0 ** max(-20, min(40, e)))

    def d_h(self):
        """Gradient w.r.t. the fc256 output of the last backward as float32 [N,256] ([N,512] =
        [d_h_v | d_h_a] with ``dueling_streams``)."""
        N = self.num_envs * self.t_max
        return decode_split(self.d_l4[:N], N, self.l4.shape[1]) / self.tensor_scale

    def d_a2(self):
        """Gradient w.r.t. the conv2 output (pre-relu) of the last backward, float32 [N,2592]."""
        return self.d_l2 / self.tensor_scale

    def d_a1(self):
        """Gradient w.r.t. the conv1 output (pre-relu) of the last backward, float32 [N,20,20,16]."""
        return decode_da1(self.d_l1, self.num_envs * self.t_max) / self.tensor_scale

    def d_h_transposed(self):
        """The same gradient decoded from its second, transposed copy (what fc wgrad reads)."""
        N = self.num_envs * self.t_max
        n8, H = (N + 7) // 8 * 8, self.l4.shape[1]
        b = self.d_l4[N:].reshape(-1).view(torch.bfloat16).reshape(2, n8 // 8, H, 8)
        return (b[0].float() + b[1].float()).permute(0, 2, 1).reshape(n8, H)[:N] / self.tensor_scale

    def sample(self, t, step, seed, env_id_base=0):
        """network.py:72-73 sampled_action for rollout slot t."""
        r = self._rows(t)
        self._timed_call("arl_sample_actions", _cabi.ptr(self.policy[r]),
                         _cabi.ptr(self.sampled_action[r]), self.num_envs, self.action_size,
                         int(env_id_base), int(step), int(seed), _cabi.stream_ptr())
        return self.sampled_action[r]

    def bootstrap_value(self, history, refresh=None, reset=None):
        """V(s_T) under the same theta (Algorithm 3: R = V(s_t, theta'_v)).  ``lstm``: from the state after
        the rollout's last step (with ``reset`` applied as in forward_sample), which is not advanced."""
        self._policy_value_only("bootstrap_value")
        b = self._b
        if self.lstm:
            self._forward_lstm(history, self._refresh(refresh), b['l1'], b['l2'], b['l4'],
                               (self.state_h, self.state_c), reset, False, b['xh'], None, None, b['c'], b['h'],
                               b['logits'], b['probs'], b['value'])
            return b['value']
        self._forward_into(history, b['l1'], b['l2'], b['l4'], b['logits'], b['probs'], b['value'],
                           refresh)
        return b['value']

    def sample_dev(self, t, step_dev, seed, env_id_base=0):
        """``sample`` with the Philox step read from the int64 device counter ``step_dev`` (the
        form a captured CUDA graph can replay)."""
        r = self._rows(t)
        _cabi.call("arl_sample_actions_dev", _cabi.ptr(self.policy[r]),
                   _cabi.ptr(self.sampled_action[r]), self.num_envs, self.action_size,
                   int(env_id_base), _cabi.ptr(step_dev), int(seed), _cabi.stream_ptr())
        return self.sampled_action[r]

    def evaluate(self, history, step, seed, ep=None, env_id_base=0):
        """Forward of ``history``'s current stack into the scratch buffers (no rollout slot is
        touched) and one action per env: epsilon-greedy over the Q values when ``ep`` is given
        (agent.py:141-151), else a sample from the policy (network.py:72).  Used by Agent.play."""
        b = self._b
        if self.lstm:                                          # play's own state (reset_lstm_state(play=True))
            self._forward_lstm(history, self._refresh(None), b['l1'], b['l2'], b['l4'], (self.play_h, self.play_c),
                               None, True, b['xh'], None, None, b['c'], b['h'], b['logits'], b['probs'], b['value'])
        else:
            self._forward_into(history, b['l1'], b['l2'], b['l4'], b['logits'], b['probs'], b['value'])
        if 'action' not in b:
            b['action'] = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        if ep is not None:
            _cabi.call("arl_egreedy_actions", _cabi.ptr(b['logits']), _cabi.ptr(b['action']),
                       self.num_envs, self.action_size, float(ep), int(env_id_base), int(step),
                       int(seed), _cabi.stream_ptr())
        else:
            _cabi.call("arl_sample_actions", _cabi.ptr(b['probs']), _cabi.ptr(b['action']),
                       self.num_envs, self.action_size, int(env_id_base), int(step), int(seed),
                       _cabi.stream_ptr())
        return b['action']

    @property
    def log_policy(self):                                   # network.py:67 (log OF the softmax)
        return torch.log(self.policy)

    @property
    def policy_entropy(self):                               # network.py:69
        return -(self.policy * self.log_policy).sum(1)

    @property
    def total_loss(self):
        """network.py:94 summed over the last rollout (policy + value), as a host float."""
        s = self.loss_sums.tolist()
        return s[0] + s[1]

    # -- backward ---------------------------------------------------------------------------
    def compute_gradients(self, history, rewards, terminals, v_boot, actions=None,
                          grad_scale=1.0, allreduce=False, refresh=None):
        """Returns + loss grads (K4) then the full backward (agent.py:317) over the T*B samples
        of the rollout.  ``history`` must have had exactly t_max pushes since s_0."""
        self._policy_value_only("compute_gradients")
        T, B, A = self.t_max, self.num_envs, self.action_size
        acts = self.sampled_action if actions is None else actions
        self.loss_sums.zero_()
        st = _cabi.stream_ptr()
        self._timed_call("arl_returns_lossgrad", _cabi.ptr(rewards), _cabi.ptr(terminals),
                         _cabi.ptr(acts), _cabi.ptr(self.policy_logits), _cabi.ptr(self.value),
                         _cabi.ptr(v_boot), _cabi.ptr(self.R), _cabi.ptr(self.d_logits),
                         _cabi.ptr(self.d_value), _cabi.ptr(self.loss_sums), T, B, A, self.gamma,
                         self.beta, self.min_reward, self.max_reward, float(grad_scale), st)
        if self.lstm:
            return self._backward_lstm(history, terminals, grad_scale, allreduce, refresh)
        return self._backward(history, grad_scale, allreduce, refresh)

    def _backward_lstm(self, history, terminals, grad_scale, allreduce, refresh):
        """arl_backward_lstm: heads (unmasked), truncated BPTT over the rollout (``terminals`` u8 [T, B] reset
        the state between steps) and the LSTM weight gradient, then the trunk's backward; one entry."""
        T, B, A = self.t_max, self.num_envs, self.action_size
        P = _cabi.ptr
        if self._refresh(refresh):
            self._prepare(self.params, self.fc_w)
        S = self.tensor_scale = self.pick_tensor_scale(grad_scale)
        self._timed_call("arl_backward_lstm", P(self.params), P(self.fc_w), A, P(history.ring), B, history.ring_slots,
                         history.first_slot(T), T, P(terminals), P(self.l1), P(self.l2), P(self.l4), P(self.xh),
                         P(self.gates), P(self.c_prev), P(self.c_seq), P(self.h_lstm), P(self.d_logits),
                         P(self.d_value), P(self.d_h_lstm), P(self.dz), P(self.dxh), P(self.dc), P(self.d_l4),
                         P(self.d_l2), P(self.d_l1), P(self.grads), P(self.workspace), S, 1 if allreduce else 0,
                         _cabi.stream_ptr())
        return self.grads

    def _not_lstm(self, entry):
        """The Q-learner entry points and the plain forward run the heads on fc256's output; an LSTM network's
        heads read the LSTM's h, which only the A3C entries (forward_sample, bootstrap_value, evaluate,
        compute_gradients) compute."""
        if self.lstm:
            raise ValueError("Network.%s has no LSTM form; an LSTM network (lstm=True) serves the A3C learner "
                             "only" % entry)

    def _policy_value_only(self, entry):
        """The A3C entry points (policy sample, V(s_T) bootstrap, policy/value loss) have no dueling
        form: with dueling heads the A-wide head is an advantage stream, not policy logits."""
        if self.dueling:
            raise ValueError("Network.%s is the A3C policy/value path; a dueling network (dueling=True) "
                             "serves the Q learners only" % entry)

    def _backward(self, history, grad_scale, allreduce, refresh):
        """The backward (agent.py:317) of every learner from d_logits / d_value over the T*B samples
        of the rollout, after rebuilding fc_w when ``refresh`` (None = decide from the parameter
        version; a forward normally did this already).  Under ``timed`` it runs as its per-layer
        entries."""
        T, B, A = self.t_max, self.num_envs, self.action_size
        P, st = _cabi.ptr, _cabi.stream_ptr()
        if self._refresh(refresh):
            self._prepare(self.params, self.fc_w)
        S = self.tensor_scale = self.pick_tensor_scale(grad_scale)
        if self.dueling_streams:                               # one entry, the exchange inside
            self._timed_call("arl_backward_streams", P(self.params), P(self.fc_w), A, P(history.ring), B,
                             history.ring_slots, history.first_slot(T), T, P(self.l1), P(self.l2), P(self.l4),
                             P(self.d_logits), P(self.d_value), P(self.d_l4), P(self.d_l2), P(self.d_l1),
                             P(self.grads), P(self.workspace), S, 1 if allreduce else 0, st)
            return self.grads
        if self.timed is None:
            _cabi.call("arl_backward", P(self.params), P(self.fc_w), A, P(history.ring), B,
                       history.ring_slots, history.first_slot(T), T, P(self.l1), P(self.l2),
                       P(self.l4), P(self.d_logits), P(self.d_value), P(self.d_l4), P(self.d_l2),
                       P(self.d_l1), P(self.grads), P(self.workspace), S, 1 if allreduce else 0, st)
            return self.grads
        N = T * B
        self._timed_call("arl_heads_backward", P(self.params), A, P(self.l4), P(self.d_logits),
                         P(self.d_value), P(self.d_l4), P(self.grads), P(self.workspace), N, S, st)
        self._timed_call("arl_fc_backward", P(self.fc_w), P(self.l2), _cabi.a2_block_rows(B), P(self.d_l4),
                         P(self.d_l2), P(self.grads), P(self.workspace), N, 1.0 / S, st)
        # the exchange as arl_backward does it: ONE all-reduce after the last backward kernel, or
        # (ARL_ALLREDUCE_OVERLAP=1) the l4_w..q_b bucket on the side stream from here on
        overlap = allreduce and os.environ.get("ARL_ALLREDUCE_OVERLAP", "")[:1] == "1"
        if overlap:
            lo = self.offsets[4]
            _cabi.call("arl_allreduce_begin", P(self.grads), lo, self.offsets[-1] - lo, st)
        self._timed_call("arl_conv2_backward", P(self.fc_w), P(self.l1), P(self.d_l2),
                         P(self.d_l1), P(self.grads), P(self.workspace), N, 1.0 / S, st)
        self._timed_call("arl_conv1_backward", P(history.ring), P(self.d_l1), P(self.grads),
                         P(self.workspace), B, history.ring_slots, history.first_slot(T), T, 1.0 / S, st)
        if overlap:
            _cabi.call("arl_allreduce_begin", P(self.grads), 0, self.offsets[4], st)
            _cabi.call("arl_allreduce_end", st)
        elif allreduce:
            self._timed_call("arl_allreduce_grads", P(self.grads), self.offsets[-1], st)
        return self.grads

    # -- async-Q mode (agent.py:169-207, 298-314): the Q head lives in the p_w/p_b slot ---------
    def make_target(self, one_step=True, next_actions=False):
        """agent.py:257-296: a second parameter set, the target network.  ``one_step``: also the
        [T*B] target buffers of the 1-step learners (async_q, sarsa); the n-step learner (nstep_q)
        evaluates the target network on the B states s_T only (``q_boot``).  ``next_actions``
        (sarsa): the rollout's actions get one more row, a_T, the action taken in s_T
        (``sarsa_actions`` [(T+1)*B]; ``sampled_action`` becomes a view of its first T rows)."""
        self._not_lstm("make_target")
        self.target_params = self.params.clone()
        B, A = self.num_envs, self.action_size
        N = B * self.t_max
        f32 = dict(device=self.device, dtype=torch.float32)
        if one_step:
            self.target_q = torch.empty(N, A, **f32)          # agent.py:186 q_t_plus_1
            self.target_q_t = torch.empty(N, **f32)           # agent.py:190
            self._tq_scratch = (torch.empty(N, A, **f32), torch.empty(N, **f32))
            if next_actions:
                self.sarsa_actions = torch.zeros(N + B, dtype=torch.int32, device=self.device)
                self.sampled_action = self.sarsa_actions[:N]
                self._target_fc_w_key = None
        else:
            self.q_boot = torch.empty(B, A, **f32)            # Q(s_T; theta^-)
            self._target_fc_w_key = None
        if self.double_q:                                     # Q(s_T; theta) + its probs / value scratch
            self.q_online_T = torch.empty(B, A, **f32)
            self._online_scratch = (torch.empty(B, A, **f32), torch.empty(B, **f32))
        self.target_fc_w = torch.empty(_cabi.prepared_floats(self.dueling_streams), device=self.device)
        return self.target_params

    def update_target(self):
        """agent.py:298-303, 342-344: target <- prediction network."""
        self.target_params.copy_(self.params)

    def egreedy(self, t, step, seed, ep, env_id_base=0):
        """agent.py:141-151 on the Q values of rollout slot t."""
        r = self._rows(t)
        _cabi.call("arl_egreedy_actions", _cabi.ptr(self.policy_logits[r]),
                   _cabi.ptr(self.sampled_action[r]), self.num_envs, self.action_size, float(ep),
                   int(env_id_base), int(step), int(seed), _cabi.stream_ptr())
        return self.sampled_action[r]

    def _forward_online_T(self, history, refresh):
        """Double Q: Q(s_T; theta) of the B current stacks into ``q_online_T`` under ``params`` / ``fc_w``
        (rebuilt first when ``refresh``; None = decide from the parameter version), through the forward
        every Q learner uses."""
        P, b = _cabi.ptr, self._b
        probs, value = self._online_scratch
        refresh = self._refresh(refresh)
        if self.dueling:
            self._forward_dueling(self.params, self.fc_w, refresh, history, history.first_slot(0), 1, b['l1'],
                                  b['l2'], b['l4'], self.q_online_T, probs, value)
        else:
            self._timed_call("arl_forward", P(self.params), P(self.fc_w), refresh, self.action_size,
                             P(history.ring), self.num_envs, history.ring_slots, history.first_slot(0), 1,
                             P(b['l1']), P(b['l2']), P(b['l4']), P(self.q_online_T), P(probs), P(value),
                             _cabi.stream_ptr())

    def compute_q_gradients(self, history, rewards, terminals, grad_scale, allreduce=False):
        """agent.py:186-197: target-network forward over s_1..s_T, 1-step targets, MSE gradient,
        backward.  The backward scratch buffers hold the target activations meanwhile.  Double Q: the
        online rows of s_1..s_{T-1} are the rollout's own Q rows, Q(s_T; theta) one more forward."""
        self._not_lstm("compute_q_gradients")
        T, B, A = self.t_max, self.num_envs, self.action_size
        P, st = _cabi.ptr, _cabi.stream_ptr()
        probs, value = self._tq_scratch
        if self.dueling:
            self._forward_dueling(self.target_params, self.target_fc_w, 1, history, history.first_slot(T - 1), T,
                                  self.d_l1, self.d_l2, self.d_l4, self.target_q, probs, value)
        else:
            _cabi.call("arl_forward", P(self.target_params), P(self.target_fc_w), 1, A, P(history.ring),
                       B, history.ring_slots, history.first_slot(T - 1), T, P(self.d_l1), P(self.d_l2),
                       P(self.d_l4), P(self.target_q), P(probs), P(value), st)
        refresh = None
        if self.double_q:
            self._forward_online_T(history, None)
            refresh = False                                    # fc_w: refreshed by the online forward
        self.loss_sums.zero_()
        if self.double_q:
            self._q_lossgrad("arl_double_q_lossgrad", (P(rewards), P(terminals), P(self.sampled_action),
                                                       P(self.policy_logits), P(self.target_q), P(self.q_online_T),
                                                       P(self.target_q_t)),
                             (P(self.loss_sums), T, B, A, self.gamma, self.min_reward, self.max_reward,
                              float(grad_scale), st), timed=False)
        else:
            self._q_lossgrad("arl_q_lossgrad", (P(rewards), P(terminals), P(self.sampled_action),
                                                P(self.policy_logits), P(self.target_q), P(self.target_q_t)),
                             (P(self.loss_sums), T * B, A, self.gamma, self.min_reward, self.max_reward,
                              float(grad_scale), st), timed=False)
        return self._backward(history, grad_scale, allreduce, refresh)

    def _q_lossgrad(self, name, head, tail, timed=True):
        """A Q learner's loss entry ``name``: its arguments are ``head``, the dQ row (d_logits), ``tail``.
        Dueling: the entry's dueling form, which also writes d_value (dL/dv); else the value head is
        unused and d_value is zeroed.  ``timed``: an event pair around it under ``timed``."""
        P = _cabi.ptr
        call = self._timed_call if timed else _cabi.call
        if self.dueling:
            call(name + "_dueling", *head, P(self.d_logits), P(self.d_value), *tail)
        else:
            call(name, *head, P(self.d_logits), *tail)
            self.d_value.zero_()                               # the value head is unused

    # -- n-step Q mode (Mnih et al. 2016, asynchronous n-step Q-learning): the Q head is the p_w/p_b
    # slot as in async_q; the cycle is the A3C cycle with the bootstrap taken from the target network
    def _target_fc_w_stale(self):
        """True (once) when target_params has changed since target_fc_w was made from it (a target
        sync, a checkpoint load): torch bumps ``_version`` on every in-place write."""
        key = self.target_params._version
        stale = key != self._target_fc_w_key
        self._target_fc_w_key = key
        return stale

    def forward_egreedy(self, history, t, seed, env_id_base=0, step_dev=None, ep_sched=None, refresh=None,
                        step=0, ep=0.0):
        """``forward`` into rollout slot t + the epsilon-greedy draw of agent.py:141-151 on the Q values
        as one composed call (arl_forward_egreedy: the draw runs inside the heads launch).  With the
        int64 device counter ``step_dev`` the step is ``step`` + *step_dev and epsilon is agent.py:142-144
        evaluated on the device from it with ``ep_sched`` = (ep_start, ep_end, ep_end_t, learn_start);
        without it the step is ``step`` and epsilon is ``ep``."""
        self._not_lstm("forward_egreedy")
        r = self._rows(t)
        P, st = _cabi.ptr, _cabi.stream_ptr()
        refresh = self._refresh(refresh)
        if step_dev is not None and ep_sched is None:
            raise ValueError("forward_egreedy: step_dev needs ep_sched = (ep_start, ep_end, ep_end_t, learn_start)")
        if self.dueling:
            self._forward_dueling(self.params, self.fc_w, refresh, history, history.first_slot(0), 1, self.l1[r],
                                  self.l2[r], self.l4[r], self.policy_logits[r], self.policy[r], self.value[r],
                                  self.sampled_action[r], env_id_base, step, step_dev, seed, ep, ep_sched)
            return self.sampled_action[r]
        e0, e1, et, ls = (float(x) for x in (ep_sched if ep_sched is not None else (0.0, 0.0, 1.0, 0.0)))
        self._timed_call("arl_forward_egreedy", P(self.params), P(self.fc_w), refresh, self.action_size,
                         P(history.ring), self.num_envs, history.ring_slots, history.first_slot(0), P(self.l1[r]),
                         P(self.l2[r]), P(self.l4[r]), P(self.policy_logits[r]), P(self.policy[r]),
                         P(self.value[r]), P(self.sampled_action[r]), int(env_id_base), int(step),
                         P(step_dev) if step_dev is not None else None, int(seed), float(ep), e0, e1, et, ls, st)
        return self.sampled_action[r]

    def compute_nstep_q_gradients(self, history, rewards, terminals, grad_scale, allreduce=False,
                                  target_refresh=None, refresh=None):
        """The n-step Q learner's gradient over the rollout: target-network forward over the B
        states s_T (into ``q_boot``, after rebuilding target_fc_w when ``target_refresh``; None =
        decide from the target's version), R_T = max_a q_boot, the n-step returns and dQ of the acted
        actions (arl_nstep_q_lossgrad), then the backward (agent.py:317).  ``history`` must have had
        exactly t_max pushes since s_0.  Double Q: first the online forward of s_T (``q_online_T``,
        with ``refresh``), and R_T = q_boot[a*], a* = argmax_a q_online_T (arl_double_nstep_q_lossgrad)."""
        self._not_lstm("compute_nstep_q_gradients")
        T, B, A = self.t_max, self.num_envs, self.action_size
        P, st = _cabi.ptr, _cabi.stream_ptr()
        b = self._b
        if target_refresh is None:
            target_refresh = self._target_fc_w_stale()
        if self.double_q:
            self._forward_online_T(history, refresh)
            refresh = False                                    # fc_w: refreshed by the online forward
        if self.dueling:
            self._forward_dueling(self.target_params, self.target_fc_w, target_refresh, history,
                                  history.first_slot(0), 1, b['l1'], b['l2'], b['l4'], self.q_boot, b['probs'],
                                  b['value'])
        else:
            self._timed_call("arl_forward", P(self.target_params), P(self.target_fc_w), int(bool(target_refresh)),
                             A, P(history.ring), B, history.ring_slots, history.first_slot(0), 1, P(b['l1']),
                             P(b['l2']), P(b['l4']), P(self.q_boot), P(b['probs']), P(b['value']), st)
        self.loss_sums.zero_()
        if self.double_q:
            self._q_lossgrad("arl_double_nstep_q_lossgrad", (P(rewards), P(terminals), P(self.sampled_action),
                                                         P(self.policy_logits), P(self.q_boot), P(self.q_online_T),
                                                         P(self.R)),
                             (P(self.loss_sums), T, B, A, self.gamma, self.min_reward, self.max_reward,
                              float(grad_scale), st))
            return self._backward(history, grad_scale, allreduce, refresh)
        self._q_lossgrad("arl_nstep_q_lossgrad", (P(rewards), P(terminals), P(self.sampled_action),
                                                  P(self.policy_logits), P(self.q_boot), P(self.R)),
                         (P(self.loss_sums), T, B, A, self.gamma, self.min_reward, self.max_reward,
                          float(grad_scale), st))
        return self._backward(history, grad_scale, allreduce, refresh)

    # -- one-step Sarsa mode (Mnih et al. 2016, asynchronous one-step Sarsa): async_q's Q head,
    # target forward and 1-step targets, bootstrapped from the action taken in s' instead of max_a
    def compute_sarsa_gradients(self, history, rewards, terminals, grad_scale, step_dev, seed, ep_sched,
                                env_id_base=0, allreduce=False, target_refresh=None, refresh=None):
        """The one-step Sarsa learner's gradient over the rollout:
          1. target-network forward over s_1..s_T into ``target_q`` (async_q's call; target_fc_w is
             rebuilt only when ``target_refresh``, None = decide from the target's version);
          2. the action a_T taken in s_T, drawn now: the epsilon-greedy draw of ``forward_egreedy`` on
             Q(s_T; theta) under the parameters before this update, with the step and epsilon of the
             int64 device counter ``step_dev`` (the next rollout's first step), into row T of
             ``sarsa_actions`` -- the next rollout's step 0 takes it;
          3. targets y = clip(r) + gamma (1 - term) Q(s', a'; theta^-) and dQ of the acted actions
             (arl_sarsa_lossgrad);
          4. the backward (agent.py:317).
        ``history`` must have had exactly t_max pushes since s_0."""
        self._not_lstm("compute_sarsa_gradients")
        T, B, A = self.t_max, self.num_envs, self.action_size
        P, st = _cabi.ptr, _cabi.stream_ptr()
        b = self._b
        probs, value = self._tq_scratch
        if target_refresh is None:
            target_refresh = self._target_fc_w_stale()
        if self.dueling:
            self._forward_dueling(self.target_params, self.target_fc_w, target_refresh, history,
                                  history.first_slot(T - 1), T, self.d_l1, self.d_l2, self.d_l4, self.target_q, probs,
                                  value)
            self._forward_dueling(self.params, self.fc_w, self._refresh(refresh), history, history.first_slot(0), 1,
                                  b['l1'], b['l2'], b['l4'], b['logits'], b['probs'], b['value'],
                                  self.sarsa_actions[T * B:], env_id_base, 0, step_dev, seed, 0.0, ep_sched)
        else:
            self._timed_call("arl_forward", P(self.target_params), P(self.target_fc_w), int(bool(target_refresh)),
                             A, P(history.ring), B, history.ring_slots, history.first_slot(T - 1), T, P(self.d_l1),
                             P(self.d_l2), P(self.d_l4), P(self.target_q), P(probs), P(value), st)
            e0, e1, et, ls = (float(x) for x in ep_sched)
            self._timed_call("arl_forward_egreedy", P(self.params), P(self.fc_w), self._refresh(refresh), A,
                             P(history.ring), B, history.ring_slots, history.first_slot(0), P(b['l1']), P(b['l2']),
                             P(b['l4']), P(b['logits']), P(b['probs']), P(b['value']),
                             P(self.sarsa_actions[T * B:]), int(env_id_base), 0, P(step_dev), int(seed), 0.0, e0, e1,
                             et, ls, st)
        self.loss_sums.zero_()
        self._q_lossgrad("arl_sarsa_lossgrad", (P(rewards), P(terminals), P(self.sarsa_actions),
                                                P(self.policy_logits), P(self.target_q), P(self.target_q_t)),
                         (P(self.loss_sums), T, B, A, self.gamma, self.min_reward, self.max_reward,
                          float(grad_scale), st))
        return self._backward(history, grad_scale, allreduce, False)   # fc_w: refreshed by step 2

    @property
    def q(self):                                               # agent.py:252
        return self.policy_logits

    def _exchange_update(self, lr, step_dev, step_offset, base_lr, max_step):
        """K5 with the gradient exchange inside (arl_exchange_clip_rmsprop: every rank's gradient
        is read over NVLink peer memory in the norm pass; no separate all-reduce)."""
        import ctypes
        if not hasattr(self, '_offsets_c'):
            self._offsets_c = (ctypes.c_int64 * len(self.offsets))(*self.offsets)
        self._timed_call("arl_exchange_clip_rmsprop", _cabi.ptr(self.params), _cabi.ptr(self.rms),
                         _cabi.ptr(self.grads), self._offsets_c, len(self.offsets) - 1, float(lr),
                         _cabi.ptr(step_dev) if step_dev is not None else None, int(step_offset),
                         float(base_lr), int(max_step), self.decay, self.epsilon, self.clip_norm,
                         _cabi.ptr(self.grad_norms), _cabi.ptr(self.workspace), _cabi.stream_ptr())

    def _layout_update(self, lr, step_dev, step_offset, base_lr, max_step):
        """K5 over the tensors of ``offsets`` (arl_clip_rmsprop_layout): the dueling streams' or the LSTM
        network's 12 tensors."""
        import ctypes
        if not hasattr(self, '_offsets_c'):
            self._offsets_c = (ctypes.c_int64 * len(self.offsets))(*self.offsets)
        self._timed_call("arl_clip_rmsprop_layout", _cabi.ptr(self.params), _cabi.ptr(self.rms),
                         _cabi.ptr(self.grads), self._offsets_c, len(self.offsets) - 1, float(lr),
                         _cabi.ptr(step_dev) if step_dev is not None else None, int(step_offset),
                         float(base_lr), int(max_step), self.decay, self.epsilon, self.clip_norm,
                         _cabi.ptr(self.grad_norms), _cabi.ptr(self.workspace), _cabi.stream_ptr())

    def apply_gradients(self, lr, exchange=False):
        """agent.py:316-321: per-tensor clip_by_norm(40) + shared RMSProp (K5).  ``exchange``: sum
        the gradient over the ranks first, inside the same kernels (NVLink peer memory)."""
        if exchange:
            self._exchange_update(lr, None, 0, 0.0, 1)
        elif self.dueling_streams or self.lstm:
            self._layout_update(lr, None, 0, 0.0, 1)
        else:
            self._timed_call("arl_clip_rmsprop", _cabi.ptr(self.params), _cabi.ptr(self.rms),
                             _cabi.ptr(self.grads), self.action_size, float(lr), self.decay, self.epsilon,
                             self.clip_norm, _cabi.ptr(self.grad_norms), _cabi.ptr(self.workspace),
                             _cabi.stream_ptr())
        self._param_writes += 1                                # the kernel wrote params: fc_w is stale

    def apply_gradients_sched(self, step_dev, step_offset, base_lr, max_step, count_write=True,
                              exchange=False):
        """``apply_gradients`` with the learning rate of agent.py:393-395 evaluated on the device
        from the int64 step counter ``step_dev`` (+ ``step_offset``): replayable by a CUDA graph."""
        if exchange:
            self._exchange_update(0.0, step_dev, step_offset, base_lr, max_step)
        elif self.dueling_streams or self.lstm:
            self._layout_update(0.0, step_dev, step_offset, base_lr, max_step)
        else:
            self._timed_call("arl_clip_rmsprop_sched", _cabi.ptr(self.params), _cabi.ptr(self.rms),
                             _cabi.ptr(self.grads), self.action_size, _cabi.ptr(step_dev), int(step_offset),
                             float(base_lr), int(max_step), self.decay, self.epsilon, self.clip_norm,
                             _cabi.ptr(self.grad_norms), _cabi.ptr(self.workspace), _cabi.stream_ptr())
        if count_write:
            self._param_writes += 1

    # -- checkpoints (network.py:109-127), reference variable names + the rms slot ----------
    def save_model(self, saver=None, checkpoint_dir='checkpoints', step=None):
        os.makedirs(checkpoint_dir, exist_ok=True)
        path = os.path.join(checkpoint_dir, "Network-%s.npz" % (step if step is not None else 0))
        blobs = {k: v.detach().cpu().numpy() for k, v in self.w.items()}
        blobs["rms"] = self.rms.detach().cpu().numpy()
        blobs["step"] = np.int64(step if step is not None else 0)
        if self.dueling:                                       # absent = not dueling: older files load as such
            blobs["dueling"] = np.bool_(True)
        if self.dueling_streams:                               # absent = no hidden layer per stream
            blobs["dueling_streams"] = np.bool_(True)
        if self.lstm:                                          # absent = no LSTM; the (h, c) state is not saved
            blobs["lstm"] = np.bool_(True)
        np.savez(path, **blobs)
        return path

    def load_model(self, saver=None, checkpoint_dir='checkpoints'):
        if not os.path.isdir(checkpoint_dir):
            return False
        files = sorted((f for f in os.listdir(checkpoint_dir) if f.startswith("Network-")),
                       key=lambda f: int(f[8:-4]))
        if not files:
            return False
        z = np.load(os.path.join(checkpoint_dir, files[-1]))
        saved = bool(z["dueling"]) if "dueling" in z.files else False
        if saved != self.dueling:                              # same weights, another function: refuse
            raise ValueError("checkpoint %s was written by a %s network; this network is %s"
                             % (files[-1], "dueling" if saved else "non-dueling",
                                "dueling" if self.dueling else "non-dueling"))
        saved = bool(z["dueling_streams"]) if "dueling_streams" in z.files else False
        if saved != self.dueling_streams:                      # other parameters: refuse
            raise ValueError("checkpoint %s was written by a %s network; this network is %s"
                             % (files[-1], "dueling_streams" if saved else "non-dueling_streams",
                                "dueling_streams" if self.dueling_streams else "non-dueling_streams"))
        saved = bool(z["lstm"]) if "lstm" in z.files else False
        if saved != self.lstm:                                 # other parameters: refuse
            raise ValueError("checkpoint %s was written by a %s network; this network is %s"
                             % (files[-1], "lstm" if saved else "non-lstm", "lstm" if self.lstm else "non-lstm"))
        self.set_weights({k: z[k] for k in self.param_names})
        self.rms.copy_(torch.as_tensor(z["rms"]))
        self.loaded_step = int(z["step"])
        return True


def make_network(DQN_type='nips', **kw):
    """network.py:30-55: the trunk is chosen by ``DQN_type`` ('nature' | 'nips'); anything else is
    the reference's ValueError('Wrong DQN type')."""
    kind = str(DQN_type).lower()
    if kind == 'nips':
        return Network(DQN_type='nips', **kw)
    if kind == 'nature':
        if kw.pop('dueling', False):
            raise NotImplementedError("dueling Q heads are built on the nips trunk (agent.py:226-252); the "
                                      "nature trunk is A3C-only")
        if kw.pop('dueling_streams', False):
            raise NotImplementedError("dueling streams are built on the nips trunk (agent.py:226-252); the "
                                      "nature trunk is A3C-only")
        if kw.pop('lstm', False):
            raise NotImplementedError("the A3C LSTM agent is built on the nips trunk (agent.py:226-252); the nature "
                                      "trunk has no LSTM")
        if kw.pop('double_q', False):
            raise NotImplementedError("double Q-learning targets are built on the nips trunk (agent.py:226-252); "
                                      "the nature trunk is A3C-only")
        from .network_nature import NatureNetwork
        return NatureNetwork(DQN_type='nature', **kw)
    raise ValueError('Wrong DQN type: %s' % DQN_type)
