"""Float64 reference of the A3C LSTM agent (include/asyncrl_b200_lstm.h) on oracle/a3c.py's nips trunk:
the rollout with carried (h, c) and terminal resets, the bootstrap from the unadvanced state, returns
and loss (a3c's), gradients by autograd (truncated BPTT: the rollout-start state is a constant), and an
explicit BPTT recurrence of the LSTM layer alone.  Pure torch/numpy: imports on a machine without a GPU."""
import os
import sys
from collections import OrderedDict

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import a3c  # noqa: E402

C = 256
LSTM_NAMES = a3c.PARAM_NAMES + ("lstm_w", "lstm_b")


def init_params(action_size, seed=3, stddev=0.02):
    """oracle/a3c.py's weights, then lstm_w ~ N(0, stddev) and a small nonzero lstm_b (a zero bias would
    leave the bias paths untested)."""
    p = a3c.init_params(action_size, seed=seed)
    rng = np.random.RandomState(seed + 1)
    p["lstm_w"] = (rng.randn(2 * C, 4 * C) * stddev).astype(np.float32)
    p["lstm_b"] = (rng.randn(4 * C) * 0.1).astype(np.float32)
    return p


def cell(x, h, c, w, b, keep):
    """One BasicLSTMCell step; keep [B] (0 = reset the incoming state)."""
    k = keep.to(x.dtype)[:, None]
    z = torch.cat([x, h * k], 1) @ w + b
    i, j, f, o = z.split(C, 1)
    c2 = torch.sigmoid(f + 1.0) * (c * k) + torch.sigmoid(i) * torch.tanh(j)
    return torch.sigmoid(o) * torch.tanh(c2), c2


def keeps(terminals, reset0):
    """keep[t] for t = 0..T-1: 1 - (terminal of the step before), step 0 from ``reset0``."""
    term = np.asarray(terminals).astype(bool)
    prev = np.concatenate([np.asarray(reset0, bool)[None], term[:-1]], 0)
    return torch.as_tensor(~prev)


def forward_rollout(p, stacks, state, keep, masks=None):
    """stacks [T, B, 84, 84, 4]; state (h0, c0) [B, 256]; keep [T, B].  Returns per-step logits, value,
    h_fc, h_lstm, c [T, B, ...] and the final state."""
    T, B = stacks.shape[:2]
    m = None if masks is None else {k: np.asarray(v).reshape((T, B) + np.asarray(v).shape[1:]) for k, v in masks.items()}
    h, c = state
    out = dict(logits=[], value=[], h_fc=[], h=[], c=[])
    for t in range(T):
        mt = None if m is None else {k: v[t] for k, v in m.items()}
        _, _, kp = a3c.forward(p, stacks[t], keep=True, masks=mt)
        x = kp["h"]
        h, c = cell(x, h, c, p["lstm_w"], p["lstm_b"], keep[t])
        if h.requires_grad:                  # d loss / d h_fc and d loss / d h per step
            x.retain_grad()
            h.retain_grad()
        out["logits"].append(h @ p["p_w"] + p["p_b"])
        out["value"].append((h @ p["q_w"] + p["q_b"]).reshape(-1))
        out["h_fc"].append(x)
        out["h"].append(h)
        out["c"].append(c)
    steps = dict(h_fc=out["h_fc"], h=out["h"])
    out = {k: torch.stack(v) for k, v in out.items()}
    out["steps"] = steps
    return out, (h, c)


def bootstrap(p, stack_T, state, keep_T):
    """V(s_T) from the state after step T-1 (reset by the last terminal); the state is not advanced."""
    _, _, kp = a3c.forward(p, stack_T, keep=True)
    h, _ = cell(kp["h"], state[0], state[1], p["lstm_w"], p["lstm_b"], keep_T)
    return (h @ p["q_w"] + p["q_b"]).reshape(-1)


def lstm_cycle(params, rms, screens, actions, rewards, terminals, step, state0, reset0, *, beta=0.01, gamma=0.99,
               num_envs=None, max_step=80000000, base_lr=0.0007, masks=None):
    """One A3C LSTM cycle: screens [T+4, B, 84, 84] u8, actions/rewards/terminals [T, B], state0 = (h0, c0)
    float [B, 256] the rollout started from, reset0 [B] the terminal row before step 0.  Returns new
    params / rms and aux (grads, R, v_boot, the state after the rollout, per-step outputs)."""
    T, B = np.asarray(actions).shape
    stacks = a3c.stacks_from_screens(np.asarray(screens), T)
    keep = keeps(terminals, reset0)
    p = a3c.to_torch(params, torch.float64, requires_grad=True)
    s0 = tuple(torch.as_tensor(np.asarray(s), dtype=torch.float64) for s in state0)
    out, state = forward_rollout(p, stacks[:T], s0, keep, masks)
    with torch.no_grad():
        keep_T = torch.as_tensor(~np.asarray(terminals, bool)[T - 1])
        v_boot = bootstrap(p, stacks[T], tuple(s.detach() for s in state), keep_T)
    R = a3c.nstep_returns(a3c.clip_rewards(rewards), np.asarray(terminals), v_boot.numpy(), gamma)
    total, _, _ = a3c.loss_per_sample(out["logits"].reshape(T * B, -1), out["value"].reshape(-1),
                                      torch.as_tensor(np.asarray(actions).reshape(-1)),
                                      torch.as_tensor(R.reshape(-1)), beta)
    loss = total.sum() / float(num_envs if num_envs is not None else B)
    loss.backward()
    grads = OrderedDict((k, v.grad.detach().numpy().copy()) for k, v in p.items())
    lr = a3c.learning_rate(step, max_step, base_lr)
    new_p, new_r = OrderedDict(), OrderedDict()
    for k in LSTM_NAMES:                     # a3c.update over all 12 tensors
        g = a3c.clip_by_norm(np.asarray(grads[k], np.float64))
        new_p[k], new_r[k] = a3c.rmsprop_apply(np.asarray(params[k], np.float64), np.asarray(rms[k], np.float64), g, lr)
    h_fc = out["h_fc"].detach()
    grad = lambda k: torch.stack([v.grad for v in out["steps"][k]])
    # a forced activation pattern is the relu derivative (oracle/a3c.py gradients)
    on = h_fc > 0 if masks is None else torch.as_tensor(np.asarray(masks["h"]).reshape(h_fc.shape))
    d_h_fc = (grad("h_fc") * on).numpy()
    aux = dict(grads=grads, R=R, v_boot=v_boot.numpy(), state=tuple(s.detach().numpy() for s in state),
               logits=out["logits"].detach().numpy(), value=out["value"].detach().numpy(),
               h=out["h"].detach().numpy(), c=out["c"].detach().numpy(), h_fc=h_fc.numpy(), d_h_fc=d_h_fc,
               d_h=grad("h").numpy())
    return new_p, new_r, aux


def bptt(x, d_h, w, b, h0, c0, keep):
    """The LSTM layer's explicit truncated BPTT in float64 (torch tensors on any device, or numpy arrays):
    x [T,B,256] inputs, d_h [T,B,256] the loss gradient w.r.t. each step's h from outside the recurrence,
    keep [T,B].  Returns (dW, db, dx) as the input's kind."""
    is_np = isinstance(x, np.ndarray)
    f64 = lambda v: torch.as_tensor(v).to(torch.float64)
    x, d_h, w, b, h0, c0 = (f64(v) for v in (x, d_h, w, b, h0, c0))
    keep = torch.as_tensor(keep).to(device=x.device, dtype=torch.float64)
    T, B, _ = x.shape
    cs, cps, xh, gs = [], [], [], []
    h, c = h0, c0
    for t in range(T):
        k = keep[t][:, None]
        inp = torch.cat([x[t], h * k], 1)
        z = inp @ w + b
        i, j = torch.sigmoid(z[:, :C]), torch.tanh(z[:, C:2 * C])
        f, o = torch.sigmoid(z[:, 2 * C:3 * C] + 1.0), torch.sigmoid(z[:, 3 * C:])
        cp = c * k
        c = f * cp + i * j
        h = o * torch.tanh(c)
        xh.append(inp); gs.append((i, j, f, o)); cps.append(cp); cs.append(c)
    dW, db, dx = bptt_given(torch.stack(xh), torch.stack([torch.cat(g, 1) for g in gs]), torch.stack(cps),
                            torch.stack(cs), d_h, w, keep)
    return tuple(v.cpu().numpy() for v in (dW, db, dx)) if is_np else (dW, db, dx)


def bptt_given(xh, gates, c_prev, c, d_h, w, keep):
    """The backward half of ``bptt`` from a forward's stored quantities (float64 torch): xh [T,B,512] =
    [x | keep*h_prev], gates [T,B,1024] = sigmoid(i), tanh(j), sigmoid(f+1), sigmoid(o), c_prev [T,B,256] =
    keep*c_prev, c [T,B,256].  Returns (dW, db, dx)."""
    T = xh.shape[0]
    dW, db, dx = torch.zeros_like(w), torch.zeros(w.shape[1], dtype=w.dtype, device=w.device), torch.zeros_like(d_h)
    dh_rec, dc_next = torch.zeros_like(d_h[0]), torch.zeros_like(d_h[0])
    for t in range(T - 1, -1, -1):
        i, j, f, o = gates[t].split(C, 1)
        tc = torch.tanh(c[t])
        dh = d_h[t] + dh_rec
        dc = dc_next + dh * o * (1 - tc ** 2)
        dz = torch.cat([dc * j * i * (1 - i), dc * i * (1 - j ** 2), dc * c_prev[t] * f * (1 - f),
                        dh * tc * o * (1 - o)], 1)
        dW += xh[t].T @ dz
        db += dz.sum(0)
        dinp = dz @ w.T
        dx[t] = dinp[:, :C]
        k = keep[t][:, None]
        dh_rec, dc_next = dinp[:, C:] * k, dc * f * k
    return dW, db, dx
