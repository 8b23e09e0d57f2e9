"""CPU: the one-step Sarsa reference against the reference's executed 1-step formula and an explicit
per-transition loop, and the C-ABI surface of include/asyncrl_b200_sarsa.h (ctypes table == header,
every declared symbol exported)."""
import ctypes
import os
import re

import numpy as np
import torch

from oracle import a3c
from sarsa_oracle import sarsa_gradients

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "asyncrl_b200_sarsa.h")


def _inputs(T, B, A, seed):
    rng = np.random.default_rng(seed)
    params, tparams = a3c.init_params(A, seed), a3c.init_params(A, seed + 1)
    for p in (params, tparams):
        for k in p:
            p[k] = (p[k] * 3.0 + (rng.normal(0, 0.02, p[k].shape) if k.endswith("_b") else 0)).astype(np.float32)
    screens = rng.integers(0, 256, (T + 4, B, 84, 84), dtype=np.uint8)
    stacks = a3c.stacks_from_screens(screens, T)
    acts = rng.integers(0, A, (T + 1, B))
    rews = rng.choice([-2.5, -1.0, 0.0, 0.3, 1.0, 4.0], (T, B)).astype(np.float32)
    terms = rng.random((T, B)) < 0.3
    return params, tparams, stacks, acts, rews, terms


def test_greedy_next_actions_equal_async_q():
    """a_{t+1} = argmax_a Q(s_{t+1}; theta^-): the Sarsa target is the target of agent.py:188-190."""
    T, B, A = 3, 4, 6
    params, tparams, stacks, acts, rews, terms = _inputs(T, B, A, 3)
    scale = 1.0 / B
    shape = (T * B,) + stacks.shape[2:]
    with torch.no_grad():
        q_next, _ = a3c.forward(a3c.to_torch(tparams), stacks[1:].reshape(shape))
    acts[1:] = q_next.numpy().argmax(axis=1).reshape(T, B)
    g, aux = sarsa_gradients(params, tparams, stacks, acts, rews, terms, 0.99, scale)
    g_ref, aux_ref = a3c.async_q_gradients(params, tparams, stacks[:T].reshape(shape), stacks[1:].reshape(shape),
                                           acts[:T], rews, terms, 0.99, scale=scale)
    assert np.abs(aux["target"] - aux_ref["target"]).max() <= 1e-12
    assert abs(aux["loss"] - aux_ref["loss"]) <= 1e-12 * max(1.0, abs(aux_ref["loss"]))
    for k in a3c.PARAM_NAMES:
        s = max(float(np.abs(g_ref[k]).max()), 1e-30)
        assert float(np.abs(g[k] - g_ref[k]).max()) / s <= 1e-12, k
    assert not g["q_w"].any() and not g["q_b"].any()                  # the value head is unused


def test_targets_are_the_per_transition_formula():
    """y(t, b) = clip(r) + gamma (1 - term) Q(s_{t+1}, a_{t+1}; theta^-), the last step bootstrapping
    from a_T, written as a loop over transitions."""
    T, B, A, gamma = 4, 3, 4, 0.9
    params, tparams, stacks, acts, rews, terms = _inputs(T, B, A, 7)
    _, aux = sarsa_gradients(params, tparams, stacks, acts, rews, terms, gamma)
    assert not np.array_equal(acts[1:].reshape(-1), aux["q_next"].argmax(axis=1))   # not the greedy target
    ref = np.zeros(T * B)
    for t in range(T):
        for b in range(B):
            n = t * B + b
            r = min(max(float(rews[t, b]), -1.0), 1.0)
            ref[n] = r + (0.0 if terms[t, b] else gamma * aux["q_next"][n, acts[t + 1, b]])
    assert np.abs(aux["target"] - ref).max() <= 1e-12
    assert np.abs(aux["delta"] - (ref - aux["q"][np.arange(T * B), acts[:T].reshape(-1)])).max() <= 1e-12


def _decls():
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    return dict((m.group(1), m.group(2)) for m in
                re.finditer(r"ARL_API\s+int\s+(arl_\w+)\s*\(([^;]*?)\)\s*;", src, re.S))


def test_ctypes_prototypes_match_the_companion_header(pkg):
    """The check of test_ctypes_prototypes_match_the_header for the Sarsa table."""
    decls = _decls()
    table = pkg._cabi.SARSA_SIGNATURES
    assert sorted(decls) == sorted(table) == ["arl_sarsa_lossgrad"]
    assert not set(table) & set(pkg._cabi.EXPORTS)                    # kept out of the main table
    kind = {ctypes.c_void_p: "ptr", ctypes.c_int: "int", ctypes.c_int64: "i64",
            ctypes.c_uint64: "u64", ctypes.c_float: "f32", ctypes.c_double: "f64"}

    def ckind(param):
        p = " ".join(param.split())
        if "*" in p:
            return "ptr"
        for prefix, k in (("float", "f32"), ("double", "f64"), ("int64_t", "i64"), ("uint64_t", "u64")):
            if p.startswith(prefix):
                return k
        assert p.startswith("int "), p
        return "int"

    for name, argtypes in table.items():
        params = [p for p in decls[name].split(",") if p.strip() and p.strip() != "void"]
        got = ["ptr" if isinstance(a, type) and issubclass(a, ctypes._Pointer) else kind[a] for a in argtypes]
        assert got == [ckind(p) for p in params], (name, got, params)


def test_library_exports_the_companion_header(pkg):
    lib = pkg._cabi.load()
    for name in _decls():
        fn = getattr(lib, name)
        assert fn.argtypes == pkg._cabi.SARSA_SIGNATURES[name]         # bound by load()
