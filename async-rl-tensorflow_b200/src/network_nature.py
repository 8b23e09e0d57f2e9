"""NatureNetwork: the 'nature' trunk of the reference's Network (src/network.py:30-42:
conv32 8x8 s4 -> conv64 4x4 s2 -> conv64 3x3 s1 -> fc512) with the same heads, loss and update as
the 'nips' Network and the same Python surface (``w``, ``policy_logits``, ``policy``, ``value``,
``forward`` / ``sample`` / ``bootstrap_value`` / ``compute_gradients`` / ``apply_gradients``,
``save_model`` / ``load_model``), so that Agent runs either trunk.

Second shape set (SURVEY §8 f4): every contraction is the generic gathering tcgen05 kernel of
csrc/nature.cu on plain float32 NHWC tensors -- correct to the same 1e-3 bar as the nips path,
not laid out for the HBM roofline the way the nips kernels are.  network.py:41-42 passes the 4-D
conv output to ``linear`` (which cannot run); as in agent.py:231-232 the fc reads the NHWC flatten.
"""
import ctypes
from collections import OrderedDict

import numpy as np
import torch

from .. import _cabi
from .network import Network

PARAM_NAMES = ("l1_w", "l1_b", "l2_w", "l2_b", "l3_w", "l3_b", "l4_w", "l4_b", "p_w", "p_b", "q_w", "q_b")
FC = 512


def param_shapes(action_size):
    return OrderedDict([
        ("l1_w", (8, 8, 4, 32)), ("l1_b", (32,)), ("l2_w", (4, 4, 32, 64)), ("l2_b", (64,)),
        ("l3_w", (3, 3, 64, 64)), ("l3_b", (64,)), ("l4_w", (3136, FC)), ("l4_b", (FC,)),
        ("p_w", (FC, action_size)), ("p_b", (action_size,)), ("q_w", (FC, 1)), ("q_b", (1,))])


def initial_weights(action_size, seed=123, stddev=0.02):
    """network.py:10 truncated_normal(0,.02) for the convs, ops.py:36-39 normal(.02) for ``linear``
    matrices, zero biases."""
    g = torch.Generator().manual_seed(int(seed))
    out = OrderedDict()
    for name, shape in param_shapes(action_size).items():
        if name.endswith("_b"):
            out[name] = torch.zeros(shape)
        elif len(shape) == 4:
            w = torch.empty(shape)
            torch.nn.init.trunc_normal_(w, 0.0, stddev, -2 * stddev, 2 * stddev, generator=g)
            out[name] = w
        else:
            out[name] = torch.randn(shape, generator=g) * stddev
    return out


class NatureNetwork(Network):
    PARAM_NAMES = PARAM_NAMES

    def __init__(self, sess=None, data_format='NHWC', history_length=4, screen_height=84,
                 screen_width=84, action_size=6, activation_fn='relu', initializer=None,
                 gamma=0.99, beta=0.01, global_network=None, global_optim=None, DQN_type='nature',
                 num_envs=256, t_max=5, device='cuda', seed=123, decay=0.99, epsilon=0.1,
                 clip_norm=40.0, min_reward=-1.0, max_reward=1.0):
        if data_format != 'NHWC':
            raise ValueError("main.py:45 forces NHWC; NCHW is not built")
        if (history_length, screen_height, screen_width) != (4, 84, 84):
            raise ValueError("kernels are built for 84x84x4 stacks")
        self.sess = sess
        self.device = torch.device(device)
        _cabi.init(self.device)
        self.action_size, self.num_envs, self.t_max = int(action_size), int(num_envs), int(t_max)
        self.gamma, self.beta = float(gamma), float(beta)
        self.decay, self.epsilon, self.clip_norm = float(decay), float(epsilon), float(clip_norm)
        self.min_reward, self.max_reward = float(min_reward), float(max_reward)
        self.global_network = global_network
        A, B, T = self.action_size, self.num_envs, self.t_max
        self.offsets = _cabi.nature_param_layout(A)
        self._offsets_c = (ctypes.c_int64 * len(self.offsets))(*self.offsets)
        n_params = self.offsets[-1]
        dev = self.device
        f32 = dict(device=dev, dtype=torch.float32)
        self.params = torch.zeros(n_params, **f32)
        self.grads = torch.zeros(n_params, **f32)
        self.rms = torch.ones(n_params, **f32)                # TF RMSProp slot starts at 1.0
        self.w, self.g = OrderedDict(), OrderedDict()
        for i, (name, shape) in enumerate(param_shapes(A).items()):
            self.w[name] = self.params[self.offsets[i]:self.offsets[i + 1]].view(shape)
            self.g[name] = self.grads[self.offsets[i]:self.offsets[i + 1]].view(shape)
        self._param_writes = 0
        self.set_weights(initial_weights(A, seed))
        N = B * T
        # rollout tensors, t-major (sample n = t*B + b): the stacks (History.get) and activations
        self.x = torch.empty(N, 84, 84, 4, **f32)             # network.py:13-15 s_t (0..255)
        self.l1 = torch.empty(N, 20, 20, 32, **f32)           # network.py:34-35
        self.l2 = torch.empty(N, 9, 9, 64, **f32)             # network.py:36-37
        self.l3 = torch.empty(N, 7 * 7 * 64, **f32)           # network.py:38-39, NHWC flatten
        self.l4 = torch.empty(N, FC, **f32)                   # network.py:40-42
        self.policy_logits = torch.empty(N, A, **f32)
        self.policy = torch.empty(N, A, **f32)
        self.value = torch.empty(N, **f32)
        self.sampled_action = torch.zeros(N, dtype=torch.int32, device=dev)
        self.R = torch.empty(N, **f32)
        self._b = dict(x=torch.empty(B, 84, 84, 4, **f32), l1=torch.empty(B, 20, 20, 32, **f32),
                       l2=torch.empty(B, 9, 9, 64, **f32), l3=torch.empty(B, 3136, **f32),
                       l4=torch.empty(B, FC, **f32), logits=torch.empty(B, A, **f32),
                       probs=torch.empty(B, A, **f32), value=torch.empty(B, **f32))
        self.d_logits = torch.empty(N, A, **f32)
        self.d_value = torch.empty(N, **f32)
        self.d_l4 = torch.empty(N, FC, **f32)
        self.d_l3 = torch.empty(N, 3136, **f32)
        self.d_l2 = torch.empty(N, 9, 9, 64, **f32)
        self.d_l1 = torch.empty(N, 20, 20, 32, **f32)
        self.workspace = torch.empty(int(_cabi.load().arl_nature_workspace_bytes(A)), dtype=torch.uint8,
                                     device=dev)
        self.loss_sums = torch.zeros(3, **f32)
        self.grad_norms = torch.zeros(len(PARAM_NAMES), **f32)
        self.events = {}

    def set_weights(self, weights):
        for name in PARAM_NAMES:
            self.w[name].copy_(torch.as_tensor(np.asarray(weights[name]), dtype=torch.float32))

    def _fc_w_stale(self):
        return False                                           # no prepared weight images on this path

    # -- forward ----------------------------------------------------------------------------
    def _stacks_into(self, history, x):
        """History.get() (history.py:20-24) of the current stack into ``x`` f32 [B,84,84,4]."""
        _cabi.call("arl_history_get", _cabi.ptr(history.ring), _cabi.ptr(x), 0, self.num_envs,
                   history.ring_slots, history.first_slot(0), _cabi.stream_ptr())

    def _forward_into(self, history, x, l1, l2, l3, l4, logits, probs, value):
        P = _cabi.ptr
        self._stacks_into(history, x)
        self._timed_call("arl_nature_forward", P(self.params), self.action_size, P(x), P(l1), P(l2), P(l3),
                         P(l4), P(logits), P(probs), P(value), self.num_envs, _cabi.stream_ptr())

    def forward(self, history, t, refresh=None):
        r = self._rows(t)
        self._forward_into(history, self.x[r], self.l1[r], self.l2[r], self.l3[r], self.l4[r],
                           self.policy_logits[r], self.policy[r], self.value[r])
        return self.policy_logits[r], self.policy[r], self.value[r]

    def forward_sample(self, history, t, step, seed, env_id_base=0, step_dev=None, refresh=None):
        self.forward(history, t)
        if step_dev is not None:
            return self.sample_dev(t, step_dev, seed, env_id_base)
        return self.sample(t, step, seed, env_id_base)

    def bootstrap_value(self, history, refresh=None):
        b = self._b
        self._forward_into(history, b['x'], b['l1'], b['l2'], b['l3'], b['l4'], b['logits'], b['probs'],
                           b['value'])
        return b['value']

    def evaluate(self, history, step, seed, ep=None, env_id_base=0):
        b = self._b
        self._forward_into(history, b['x'], b['l1'], b['l2'], b['l3'], b['l4'], b['logits'], b['probs'],
                           b['value'])
        if 'action' not in b:
            b['action'] = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        name, src = ("arl_egreedy_actions", b['logits']) if ep is not None else ("arl_sample_actions", b['probs'])
        args = [_cabi.ptr(src), _cabi.ptr(b['action']), self.num_envs, self.action_size]
        if ep is not None:
            args.append(float(ep))
        _cabi.call(name, *args, int(env_id_base), int(step), int(seed), _cabi.stream_ptr())
        return b['action']

    def a1(self):
        return self.l1

    def a2(self):
        return self.l2

    def a3(self):
        return self.l3

    # -- backward ---------------------------------------------------------------------------
    def compute_gradients(self, history, rewards, terminals, v_boot, actions=None, grad_scale=1.0,
                          allreduce=False, refresh=None):
        """K4 (returns + loss gradients, shared with the nips path) then the nature backward."""
        T, B, A = self.t_max, self.num_envs, self.action_size
        acts = self.sampled_action if actions is None else actions
        self.loss_sums.zero_()
        P, st = _cabi.ptr, _cabi.stream_ptr()
        self._timed_call("arl_returns_lossgrad", P(rewards), P(terminals), P(acts), P(self.policy_logits),
                         P(self.value), P(v_boot), P(self.R), P(self.d_logits), P(self.d_value),
                         P(self.loss_sums), T, B, A, self.gamma, self.beta, self.min_reward,
                         self.max_reward, float(grad_scale), st)
        self._timed_call("arl_nature_backward", P(self.params), A, P(self.x), P(self.l1), P(self.l2),
                         P(self.l3), P(self.l4), P(self.d_logits), P(self.d_value), P(self.d_l4),
                         P(self.d_l3), P(self.d_l2), P(self.d_l1), P(self.grads), P(self.workspace),
                         T * B, st)
        if allreduce:
            _cabi.call("arl_allreduce_grads", P(self.grads), int(self.grads.numel()), st)
        return self.grads

    def make_target(self, one_step=True, next_actions=False):
        if next_actions:
            raise NotImplementedError("loss_mode='sarsa' is built on the nips trunk (agent.py:226-252); "
                                      "the nature trunk is A3C-only")
        raise NotImplementedError("loss_mode='async_q' runs the reference's agent.py net, which is the "
                                  "nips trunk (agent.py:226-252); the nature trunk is A3C-only"
                                  if one_step else
                                  "loss_mode='nstep_q' is built on the nips trunk (agent.py:226-252); "
                                  "the nature trunk is A3C-only")

    def _update(self, lr, step_dev, step_offset, base_lr, max_step, exchange=False):
        _cabi.call("arl_exchange_clip_rmsprop" if exchange else "arl_clip_rmsprop_layout",
                   _cabi.ptr(self.params), _cabi.ptr(self.rms),
                   _cabi.ptr(self.grads), self._offsets_c, len(PARAM_NAMES), float(lr),
                   _cabi.ptr(step_dev) if step_dev is not None else None, int(step_offset),
                   float(base_lr), int(max_step), self.decay, self.epsilon, self.clip_norm,
                   _cabi.ptr(self.grad_norms), _cabi.ptr(self.workspace), _cabi.stream_ptr())

    def apply_gradients(self, lr, exchange=False):
        self._update(lr, None, 0, 0.0, 1, exchange)
        self._param_writes += 1

    def apply_gradients_sched(self, step_dev, step_offset, base_lr, max_step, count_write=True,
                              exchange=False):
        self._update(0.0, step_dev, step_offset, base_lr, max_step, exchange)
        if count_write:
            self._param_writes += 1

    def load_model(self, saver=None, checkpoint_dir='checkpoints'):
        import os
        if not os.path.isdir(checkpoint_dir):
            return False
        files = sorted((f for f in os.listdir(checkpoint_dir) if f.startswith("Network-")),
                       key=lambda f: int(f[8:-4]))
        if not files:
            return False
        z = np.load(os.path.join(checkpoint_dir, files[-1]))
        self.set_weights({k: z[k] for k in PARAM_NAMES})
        self.rms.copy_(torch.as_tensor(z["rms"]))
        self.loaded_step = int(z["step"])
        return True
