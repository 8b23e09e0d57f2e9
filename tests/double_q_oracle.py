"""Float64 reference of double Q-learning targets (van Hasselt, Guez & Silver 2016, Double DQN) on the
async-Q and n-step Q learners, built from the oracle's forward / targets / returns / loss
(oracle/a3c.py) and, with dueling heads, on dueling_oracle.q_forward: the online parameters theta
choose the bootstrap action, the target parameters theta^- evaluate it,
    a*   = argmax_a Q(s', a; theta)          (ties -> lowest index, np.argmax)
    boot = Q(s', a*; theta^-)                in place of max_a Q(s'; theta^-)."""
from collections import OrderedDict

import numpy as np
import torch

from dueling_oracle import q_forward
from oracle import a3c


def double_boot(q_online, q_next, a_star=None):
    """(a*, Q(s', a*; theta^-)) per row: a* the first index of each online row's max unless given."""
    q_next = np.asarray(q_next)
    a = np.argmax(np.asarray(q_online), axis=1) if a_star is None else np.asarray(a_star).reshape(-1)
    return a, q_next[np.arange(q_next.shape[0]), a]


def double_q_gradients(mode, params, target_params, stacks, actions, rewards, terminals, gamma=0.99, scale=1.0,
                       masks=None, dueling=False, a_star=None, dtype=torch.float64):
    """``mode`` 'async_q' | 'nstep_q'.  stacks [T+1, B, 84, 84, 4] (s_0..s_T,
    oracle.a3c.stacks_from_screens), actions / rewards / terminals [T, B].  ``a_star`` overrides the
    online argmax ([T*B] for async_q, [B] for nstep_q).  Targets (no gradient):
        async_q  y = clip(r) + gamma (1 - term) Q(s_{t+1}, a*; theta^-)      (a3c.q_targets)
        nstep_q  R = nstep_returns(clip(r), term, Q(s_T, a*; theta^-))
    loss = scale * sum_n (y_n - Q(s_n, a_n; theta))^2.  Returns (grads, aux) with aux = q, q_online
    (Q(s'; theta)), q_next (Q(s'; theta^-)), a_star, target, delta, loss."""
    stacks = np.asarray(stacks)
    T, B = np.asarray(rewards).shape
    shape = (T * B,) + stacks.shape[2:]
    fwd = q_forward if dueling else (lambda p, s, masks=None: a3c.forward(p, s, masks=masks)[0])
    with torch.no_grad():
        s_next = stacks[T] if mode == 'nstep_q' else stacks[1:T + 1].reshape(shape)
        q_online = fwd(a3c.to_torch(params, dtype), s_next).numpy()
        q_next = fwd(a3c.to_torch(target_params, dtype), s_next).numpy()
    a, boot = double_boot(q_online, q_next, a_star)
    if mode == 'nstep_q':
        y = a3c.nstep_returns(a3c.clip_rewards(rewards), np.asarray(terminals), boot, gamma).reshape(-1)
    else:
        y = a3c.q_targets(boot[:, None], np.asarray(rewards).reshape(-1), np.asarray(terminals).reshape(-1), gamma)
    p = a3c.to_torch(params, dtype, requires_grad=True)
    q = fwd(p, stacks[:T].reshape(shape), masks=masks)
    at = torch.as_tensor(np.asarray(actions)[:T].reshape(-1)).long()
    loss, delta = a3c.async_q_loss(q, at, torch.as_tensor(y, dtype=dtype), scale)
    loss.backward()
    grads = OrderedDict((k, (v.grad if v.grad is not None else torch.zeros_like(v)).detach().numpy().copy())
                        for k, v in p.items())
    aux = dict(q=q.detach().numpy(), q_online=q_online, q_next=q_next, a_star=a, target=np.asarray(y),
               delta=delta.detach().numpy(), loss=float(loss.detach()))
    return grads, aux
