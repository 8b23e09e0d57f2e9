"""CPU: the dueling Q reference (closed-form head gradients against autograd, invariance of Q to a
constant added to the advantage stream) and the C-ABI surface of include/asyncrl_b200_dueling.h
(ctypes table == header, every declared symbol exported, the main header untouched)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from dueling_oracle import combine, dueling_gradients, head_gradients, q_forward
from oracle import a3c

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "asyncrl_b200_dueling.h")


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


@pytest.mark.parametrize("A", [3, 6, 18])
def test_closed_form_head_gradients_equal_autograd(A):
    """d loss / d logits = g ([j == a] - 1/A) and d loss / d value = g, g = -2 delta scale."""
    rng = np.random.default_rng(A)
    N, scale = 40, 0.125
    logits = torch.tensor(rng.normal(0, 1, (N, A)), requires_grad=True)
    value = torch.tensor(rng.normal(0, 1, N), requires_grad=True)
    acts = rng.integers(0, A, N)
    y = torch.tensor(rng.normal(0, 1, N))
    loss, delta = a3c.async_q_loss(combine(logits, value), torch.as_tensor(acts), y, scale)
    loss.backward()
    dl, dv = head_gradients(acts, delta.detach().numpy(), A, scale)
    assert np.abs(logits.grad.numpy() - dl).max() <= 1e-12
    assert np.abs(value.grad.numpy() - dv).max() <= 1e-12
    assert np.abs(dl.sum(axis=1)).max() <= 1e-12                       # the advantage gradient has zero mean


def test_q_is_unchanged_by_a_constant_on_the_advantage_bias():
    T, B, A = 1, 3, 6
    params, _, stacks, _, _, _ = _inputs(T, B, A, 5)
    p = a3c.to_torch(params)
    shifted = dict(p, p_b=p["p_b"] + 2.5)                                # in float64: exact
    s = stacks[0]
    q0, q1 = q_forward(p, s).numpy(), q_forward(shifted, s).numpy()
    logits0, _ = a3c.forward(p, s)
    logits1, _ = a3c.forward(shifted, s)
    assert np.abs(q0 - q1).max() <= 1e-12
    assert np.abs((logits1 - logits0).numpy() - 2.5).max() <= 1e-12      # the plain head does move


@pytest.mark.parametrize("mode", ["async_q", "nstep_q", "sarsa"])
def test_reference_trains_both_streams(mode):
    """Every learner's dueling loss reaches the value head, and its head gradients are the closed
    form through the shared h."""
    T, B, A = 3, 4, 6
    params, tparams, stacks, acts, rews, terms = _inputs(T, B, A, 11)
    a = acts if mode == "sarsa" else acts[:T]
    g, aux = dueling_gradients(mode, params, tparams, stacks, a, rews, terms, 0.99, scale=0.25)
    assert np.abs(g["q_w"]).max() > 0 and np.abs(g["q_b"]).max() > 0
    dl, dv = head_gradients(acts[:T], aux["delta"], A, 0.25)
    assert abs(g["q_b"][0] - dv.sum()) <= 1e-12 * max(1.0, np.abs(dv).sum())
    assert np.abs(g["p_b"] - dl.sum(axis=0)).max() <= 1e-12
    assert np.abs(g["p_b"].sum()) <= 1e-12                              # the mean is taken out


def _decls(path):
    src = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
    return dict((m.group(1), m.group(2)) for m in
                re.finditer(r"ARL_API\s+int\s+(arl_\w+)\s*\(([^;]*?)\)\s*;", src, re.S))


def test_ctypes_prototypes_match_the_companion_header(pkg):
    decls = _decls(HEADER)
    table = pkg._cabi.DUELING_SIGNATURES
    assert sorted(decls) == sorted(table) == ["arl_forward_dueling", "arl_nstep_q_lossgrad_dueling",
                                              "arl_q_lossgrad_dueling", "arl_sarsa_lossgrad_dueling"]
    assert not set(table) & set(pkg._cabi.EXPORTS) and not set(table) & set(pkg._cabi.SARSA_SIGNATURES)
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
        got = [kind[a] for a in argtypes]
        assert got == [ckind(p) for p in params], (name, got, params)


def test_main_header_keeps_its_59_symbols():
    src = open(os.path.join(ROOT, "include", "asyncrl_b200.h")).read()
    syms = set(re.findall(r"ARL_API[^;(]*?\b(arl_\w+)\s*\(", src))
    assert len(syms) == 59
    assert not syms & set(_decls(HEADER))


def test_library_exports_the_companion_header(pkg):
    lib = pkg._cabi.load()
    for name in _decls(HEADER):
        fn = getattr(lib, name)
        assert fn.argtypes == pkg._cabi.DUELING_SIGNATURES[name]       # bound by load()
