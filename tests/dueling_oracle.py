"""Float64 reference of the dueling Q heads (Wang et al. 2016, "average" aggregator) on the three Q
learners, built from the oracle's forward / targets / loss (oracle/a3c.py): the p_w/p_b head is the
advantage stream, the q_w/q_b head the value stream, both on the shared fc256 output,
    Q = value + (logits - mean(logits)),
and each learner's targets and loss are its plain ones (tests/nstep_q_oracle.py,
tests/sarsa_oracle.py) on that Q, differentiated by autograd."""
from collections import OrderedDict

import numpy as np
import torch

from oracle import a3c
from sarsa_oracle import sarsa_targets


def combine(logits, value):
    """Q = value + (advantage - mean(advantage)), advantage = the A-wide head."""
    return value.reshape(-1, 1) + (logits - logits.mean(dim=1, keepdim=True))


def q_forward(p, stacks, masks=None):
    logits, value = a3c.forward(p, stacks, masks=masks)
    return combine(logits, value)


def dueling_gradients(mode, params, target_params, stacks, actions, rewards, terminals, gamma=0.99, scale=1.0,
                      masks=None, dtype=torch.float64):
    """``mode`` 'async_q' | 'nstep_q' | 'sarsa'.  stacks [T+1, B, 84, 84, 4] (s_0..s_T,
    oracle.a3c.stacks_from_screens), rewards / terminals [T, B], actions [T, B] ([T+1, B] for sarsa:
    row T is the action taken in s_T).  Targets from the dueling Q of theta^- (no gradient):
        async_q  y = clip(r) + gamma (1 - term) max_a Q(s_{t+1})          (agent.py:186-190)
        nstep_q  R = nstep_returns(clip(r), term, max_a Q(s_T))
        sarsa    y = clip(r) + gamma (1 - term) Q(s_{t+1}, a_{t+1})
    loss = scale * sum_n (y_n - Q(s_n, a_n; theta))^2.  Returns (grads, aux) with aux = q, q_next
    (q_boot for nstep_q), target, delta, loss."""
    stacks = np.asarray(stacks)
    actions = np.asarray(actions)
    T, B = np.asarray(rewards).shape
    shape = (T * B,) + stacks.shape[2:]
    tp = a3c.to_torch(target_params, dtype)
    with torch.no_grad():
        if mode == 'nstep_q':
            q_next = q_forward(tp, stacks[T]).numpy()
            y = a3c.nstep_returns(a3c.clip_rewards(rewards), np.asarray(terminals), q_next.max(axis=1), gamma)
            y = y.reshape(-1)
        else:
            q_next = q_forward(tp, stacks[1:T + 1].reshape(shape)).numpy()
            if mode == 'sarsa':
                y = sarsa_targets(q_next, actions[1:], rewards, terminals, gamma)
            else:
                y = a3c.q_targets(q_next, np.asarray(rewards).reshape(-1), np.asarray(terminals).reshape(-1), gamma)
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


def head_gradients(actions, delta, A, scale):
    """The closed form the loss kernels write (include/asyncrl_b200_dueling.h), float64:
    g = -2 delta scale, d logits[n][j] = g ([j == a_n] - 1/A), d value[n] = g."""
    g = -2.0 * np.asarray(delta, np.float64) * scale
    onehot = np.eye(A)[np.asarray(actions).reshape(-1)]
    return g[:, None] * (onehot - 1.0 / A), g
