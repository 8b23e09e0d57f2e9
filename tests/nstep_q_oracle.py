"""Float64 reference of the n-step Q learner (Mnih et al. 2016, asynchronous n-step Q-learning),
built from the oracle's forward / returns / clip (oracle/a3c.py) and tied to the reference's
executed formula through ``q_targets`` (agent.py:188-190): with T = 1 it is ``async_q_gradients``."""
from collections import OrderedDict

import numpy as np
import torch

from oracle import a3c


def nstep_q_gradients(params, target_params, stacks, actions, rewards, terminals, gamma=0.99, scale=1.0,
                      masks=None, dtype=torch.float64):
    """stacks [T+1, B, 84, 84, 4] (s_0..s_T, oracle.a3c.stacks_from_screens), actions / rewards /
    terminals [T, B].  Q = the p_w/p_b head:
        q_boot = Q(s_T; theta^-)                                   (no gradient)
        R      = nstep_returns(clip(r), term, max_a q_boot)        (agent.py:154, 188-190)
        loss   = scale * sum_n (R_n - Q(s_n, a_n; theta))^2       (autograd)
    Returns (grads, aux) with aux = q, q_boot, R [T, B], delta, loss."""
    stacks = np.asarray(stacks)
    T, B = np.asarray(actions).shape
    with torch.no_grad():
        q_boot, _ = a3c.forward(a3c.to_torch(target_params, dtype), stacks[T])
    R = a3c.nstep_returns(a3c.clip_rewards(rewards), np.asarray(terminals), q_boot.numpy().max(axis=1), gamma)
    p = a3c.to_torch(params, dtype, requires_grad=True)
    q, _ = a3c.forward(p, stacks[:T].reshape((T * B,) + stacks.shape[2:]), masks=masks)
    at = torch.as_tensor(np.asarray(actions).reshape(-1)).long()
    loss, delta = a3c.async_q_loss(q, at, torch.as_tensor(R.reshape(-1), dtype=dtype), scale)
    loss.backward()
    grads = OrderedDict((k, (v.grad if v.grad is not None else torch.zeros_like(v)).detach().numpy().copy())
                        for k, v in p.items())
    aux = dict(q=q.detach().numpy(), q_boot=q_boot.numpy(), R=R, delta=delta.detach().numpy(),
               loss=float(loss.detach()))
    return grads, aux
