"""CPU: the n-step Q reference against the reference's executed 1-step formula and an explicit
discounted sum."""
import numpy as np

from oracle import a3c
from nstep_q_oracle import nstep_q_gradients


def _inputs(T, B, A, seed):
    rng = np.random.default_rng(seed)
    params, tparams = a3c.init_params(A, seed), a3c.init_params(A, seed + 1)
    for p in (params, tparams):
        for k in p:
            p[k] = (p[k] * 3.0 + (rng.normal(0, 0.02, p[k].shape) if k.endswith("_b") else 0)).astype(np.float32)
    screens = rng.integers(0, 256, (T + 4, B, 84, 84), dtype=np.uint8)
    stacks = a3c.stacks_from_screens(screens, T)
    acts = rng.integers(0, A, (T, B))
    rews = rng.choice([-2.5, -1.0, 0.0, 0.3, 1.0, 4.0], (T, B)).astype(np.float32)
    terms = rng.random((T, B)) < 0.3
    return params, tparams, stacks, acts, rews, terms


def test_one_step_equals_async_q():
    """T = 1: R_0 = clip(r) + gamma (1 - term) max_a Q(s_1; theta^-), the target of agent.py:188-190."""
    A, B = 6, 5
    params, tparams, stacks, acts, rews, terms = _inputs(1, B, A, 3)
    scale = 1.0 / B
    g, aux = nstep_q_gradients(params, tparams, stacks, acts, rews, terms, 0.99, scale)
    g_ref, aux_ref = a3c.async_q_gradients(params, tparams, stacks[0], stacks[1], acts, rews, terms, 0.99,
                                           scale=scale)
    assert np.abs(aux["R"].reshape(-1) - aux_ref["target"]).max() <= 1e-12
    assert abs(aux["loss"] - aux_ref["loss"]) <= 1e-12 * max(1.0, abs(aux_ref["loss"]))
    for k in a3c.PARAM_NAMES:
        s = max(float(np.abs(g_ref[k]).max()), 1e-30)
        assert float(np.abs(g[k] - g_ref[k]).max()) / s <= 1e-12, k
    assert not g["q_w"].any() and not g["q_b"].any()                  # the value head is unused


def test_returns_are_the_masked_discounted_sum():
    """R_t = sum_{k=t}^{T-1} gamma^{k-t} prod_{j=t}^{k-1}(1 - term_j) clip(r_k)
             + gamma^{T-t} prod_{j=t}^{T-1}(1 - term_j) max_a q_boot."""
    T, B, A, gamma = 4, 3, 4, 0.9
    params, tparams, stacks, acts, rews, terms = _inputs(T, B, A, 7)
    _, aux = nstep_q_gradients(params, tparams, stacks, acts, rews, terms, gamma)
    r = np.clip(rews.astype(np.float64), -1, 1)
    boot = aux["q_boot"].max(axis=1)
    ref = np.zeros((T, B))
    for t in range(T):
        disc = np.ones(B)
        for k in range(t, T):
            ref[t] += disc * r[k]
            disc = disc * gamma * (1.0 - terms[k])
        ref[t] += disc * boot
    assert np.abs(aux["R"] - ref).max() <= 1e-12
    assert np.abs(aux["delta"] - (ref.reshape(-1) - aux["q"][np.arange(T * B), acts.reshape(-1)])).max() <= 1e-12
