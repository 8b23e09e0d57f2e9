"""Float64 reference of the one-step Sarsa learner (Mnih et al. 2016, asynchronous one-step Sarsa),
built from the oracle's forward / loss (oracle/a3c.py) and tied to the reference's executed formula
through ``q_targets`` (agent.py:188-190) evaluated on the single column of the action taken in s':
with a' = argmax_a Q(s'; theta^-) it is ``async_q_gradients``."""
from collections import OrderedDict

import numpy as np
import torch

from oracle import a3c


def sarsa_targets(q_next, next_actions, rewards, terminals, gamma=0.99):
    """y_n = clip(r_n) + gamma (1 - term_n) Q(s'_n, a'_n; theta^-): ``a3c.q_targets`` on the one
    column of the next action (its max over one column is that column)."""
    q_next = np.asarray(q_next, np.float64)
    a = np.asarray(next_actions).reshape(-1)
    acted = q_next[np.arange(q_next.shape[0]), a][:, None]
    return a3c.q_targets(acted, np.asarray(rewards).reshape(-1), np.asarray(terminals).reshape(-1), gamma)


def sarsa_gradients(params, target_params, stacks, actions, rewards, terminals, gamma=0.99, scale=1.0,
                    masks=None, dtype=torch.float64):
    """stacks [T+1, B, 84, 84, 4] (s_0..s_T, oracle.a3c.stacks_from_screens), actions [T+1, B]
    (a_0..a_T: row T is the action taken in s_T), rewards / terminals [T, B].  Q = the p_w/p_b head:
        q_next = Q(s_{t+1}; theta^-)                                    (no gradient)
        y      = clip(r) + gamma (1 - term) q_next[a_{t+1}]             (agent.py:154, 188-190)
        loss   = scale * sum_n (y_n - Q(s_n, a_n; theta))^2            (autograd)
    Returns (grads, aux) with aux = q, q_next, target, delta, loss."""
    stacks = np.asarray(stacks)
    actions = np.asarray(actions)
    T, B = np.asarray(rewards).shape
    assert actions.shape == (T + 1, B), actions.shape
    shape = (T * B,) + stacks.shape[2:]
    with torch.no_grad():
        q_next, _ = a3c.forward(a3c.to_torch(target_params, dtype), stacks[1:T + 1].reshape(shape))
    y = sarsa_targets(q_next.numpy(), actions[1:], rewards, terminals, gamma)
    p = a3c.to_torch(params, dtype, requires_grad=True)
    q, _ = a3c.forward(p, stacks[:T].reshape(shape), masks=masks)
    at = torch.as_tensor(actions[:T].reshape(-1)).long()
    loss, delta = a3c.async_q_loss(q, at, torch.as_tensor(y, dtype=dtype), scale)
    loss.backward()
    grads = OrderedDict((k, (v.grad if v.grad is not None else torch.zeros_like(v)).detach().numpy().copy())
                        for k, v in p.items())
    aux = dict(q=q.detach().numpy(), q_next=q_next.numpy(), target=y, delta=delta.detach().numpy(),
               loss=float(loss.detach()))
    return grads, aux
