"""Float64 reference of the dueling streams (Wang et al. 2016's dueling architecture: a hidden layer per
stream) on the three Q learners, built from the oracle's trunk, targets and loss (oracle/a3c.py):
    h_v = relu(a2 . l4_w + l4_b),  h_a = relu(a2 . la_w + la_b)
    v = h_v . q_w + q_b,  adv = h_a . p_w + p_b,  Q = v + (adv - mean(adv))
each learner's targets and loss are its plain ones on that Q (tests/dueling_oracle.py), optionally with
double Q-learning targets, differentiated by autograd."""
from collections import OrderedDict

import numpy as np
import torch

from dueling_oracle import combine
from oracle import a3c
from sarsa_oracle import sarsa_targets

STREAMS_PARAM_NAMES = a3c.PARAM_NAMES + ("la_w", "la_b")


def init_streams_params(A, seed=0, bias_std=0.01, scale=1.0):
    """Random parameters of the streams network (float32 numpy): the nips set, then la_w / la_b."""
    p = a3c.init_params(A, seed)
    rng = np.random.default_rng(seed + 1)
    p["la_w"] = rng.normal(0, 0.02, (2592, 256)).astype(np.float32)
    p["la_b"] = np.zeros(256, np.float32)
    for k in p:
        if k.endswith("_b"):
            p[k] = rng.normal(0, bias_std, p[k].shape).astype(np.float32)
        else:
            p[k] = (p[k] * scale).astype(np.float32)
    return p


def flatten(p):
    return np.concatenate([np.asarray(p[k], np.float32).reshape(-1) for k in STREAMS_PARAM_NAMES])


def forward(p, stacks, masks=None):
    """Returns q, v, adv, h_v, h_a.  ``masks``: a1, a2 as oracle.a3c.forward, h [N, 512] = the relu pattern
    of [h_v | h_a]."""
    m = dict(masks or {})
    mh = m.pop("h", None)
    trunk = OrderedDict((k, v) for k, v in p.items() if k not in ("la_w", "la_b"))
    _, _, kept = a3c.forward(trunk, stacks, keep=True, masks=m)
    a2 = kept["a2"]
    hv = a3c._relu(a2 @ p["l4_w"] + p["l4_b"], None if mh is None else mh[:, :256])
    ha = a3c._relu(a2 @ p["la_w"] + p["la_b"], None if mh is None else mh[:, 256:])
    v = (hv @ p["q_w"] + p["q_b"]).reshape(-1)
    adv = ha @ p["p_w"] + p["p_b"]
    return combine(adv, v), v, adv, hv, ha


def q_forward(p, stacks, masks=None):
    return forward(p, stacks, masks)[0]


def heads_backward(h, p_w, q_w, d_logits, d_value):
    """The closed form of arl_heads_backward_streams (float64 numpy): h [N, 512] = [h_v | h_a]."""
    hv, ha = h[:, :256], h[:, 256:]
    d_hv = np.outer(d_value, q_w.reshape(-1)) * (hv > 0)
    d_ha = (d_logits @ p_w.T) * (ha > 0)
    return dict(d_h=np.concatenate([d_hv, d_ha], axis=1), p_w=ha.T @ d_logits, p_b=d_logits.sum(0),
                q_w=(hv.T @ d_value).reshape(-1, 1), q_b=np.array([d_value.sum()]))


def streams_gradients(mode, params, target_params, stacks, actions, rewards, terminals, gamma=0.99, scale=1.0,
                      masks=None, double_q=False, dtype=torch.float64):
    """tests/dueling_oracle.dueling_gradients on the streams network; ``double_q`` (async_q, nstep_q): the
    bootstrap is Q(s', a*; theta^-) with a* = argmax_a Q(s'; theta)."""
    stacks = np.asarray(stacks)
    actions = np.asarray(actions)
    T, B = np.asarray(rewards).shape
    shape = (T * B,) + stacks.shape[2:]
    tp = a3c.to_torch(target_params, dtype)
    p0 = a3c.to_torch(params, dtype)
    with torch.no_grad():
        nxt = stacks[T] if mode == 'nstep_q' else stacks[1:T + 1].reshape(shape)
        q_next = q_forward(tp, nxt).numpy()
        if double_q:
            a_star = q_forward(p0, nxt).numpy().argmax(axis=1)
            boot = q_next[np.arange(len(q_next)), a_star]
        else:
            boot = q_next.max(axis=1)
        if mode == 'nstep_q':
            y = a3c.nstep_returns(a3c.clip_rewards(rewards), np.asarray(terminals), boot, gamma).reshape(-1)
        elif mode == 'sarsa':
            y = sarsa_targets(q_next, actions[1:], rewards, terminals, gamma)
        else:
            y = a3c.clip_rewards(np.asarray(rewards).reshape(-1)) + \
                gamma * (1.0 - np.asarray(terminals, np.float64).reshape(-1)) * boot
    p = a3c.to_torch(params, dtype, requires_grad=True)
    q = q_forward(p, stacks[:T].reshape(shape), masks=masks)
    at = torch.as_tensor(actions[:T].reshape(-1)).long()
    loss, delta = a3c.async_q_loss(q, at, torch.as_tensor(y, dtype=dtype), scale)
    loss.backward()
    grads = OrderedDict((k, (v.grad if v.grad is not None else torch.zeros_like(v)).detach().numpy().copy())
                        for k, v in p.items())
    aux = dict(q=q.detach().numpy(), q_next=q_next, target=np.asarray(y), delta=delta.detach().numpy(),
               loss=float(loss.detach()))
    return grads, aux
