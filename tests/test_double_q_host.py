"""CPU: the double Q-learning reference (equal to the plain targets when theta^- = theta, never above
them, ties to the lowest index) and the C-ABI surface of include/asyncrl_b200_double.h (ctypes table ==
header, every declared symbol exported, the main header untouched)."""
import ctypes
import os
import re

import numpy as np
import pytest

from double_q_oracle import double_boot, double_q_gradients
from dueling_oracle import dueling_gradients
from nstep_q_oracle import nstep_q_gradients
from oracle import a3c

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "asyncrl_b200_double.h")


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


def _plain(mode, dueling, params, tparams, stacks, acts, rews, terms):
    """The plain learner's targets / returns (max_a Q(s'; theta^-)) as a flat [T*B] array."""
    if dueling:
        return dueling_gradients(mode, params, tparams, stacks, acts, rews, terms)[1]["target"].reshape(-1)
    if mode == "nstep_q":
        return nstep_q_gradients(params, tparams, stacks, acts, rews, terms)[1]["R"].reshape(-1)
    return a3c.async_q_gradients(params, tparams, stacks[:-1].reshape((-1,) + stacks.shape[2:]),
                                 stacks[1:].reshape((-1,) + stacks.shape[2:]), acts.reshape(-1),
                                 rews.reshape(-1), terms.reshape(-1))[1]["target"].reshape(-1)


@pytest.mark.parametrize("dueling", [False, True])
@pytest.mark.parametrize("mode", ["async_q", "nstep_q"])
def test_equal_to_plain_when_target_is_online(mode, dueling):
    T, B, A = 3, 4, 6
    params, _, stacks, acts, rews, terms = _inputs(T, B, A, 3)
    _, aux = double_q_gradients(mode, params, params, stacks, acts, rews, terms, dueling=dueling)
    assert np.array_equal(aux["q_online"], aux["q_next"])
    assert np.abs(aux["target"] - _plain(mode, dueling, params, params, stacks, acts, rews, terms)).max() == 0.0


@pytest.mark.parametrize("dueling", [False, True])
@pytest.mark.parametrize("mode", ["async_q", "nstep_q"])
def test_never_above_plain_and_below_on_some_rows(mode, dueling):
    """Q(s', a*; theta^-) <= max_a Q(s'; theta^-), and the targets / the return recurrence are monotone
    in the bootstrap for gamma >= 0."""
    T, B, A = 3, 6, 6
    params, tparams, stacks, acts, rews, terms = _inputs(T, B, A, 7)
    _, aux = double_q_gradients(mode, params, tparams, stacks, acts, rews, terms, dueling=dueling)
    plain = _plain(mode, dueling, params, tparams, stacks, acts, rews, terms)
    y = aux["target"]
    assert bool((y <= plain + 1e-12).all())
    assert bool((y < plain - 1e-9).any())
    assert bool((aux["a_star"] != aux["q_next"].argmax(axis=1)).any())


def test_ties_pick_the_lowest_index():
    q_online = np.array([[1.0, 3.0, 3.0, 0.0], [2.0, 2.0, 2.0, 2.0], [0.0, -1.0, 5.0, 5.0]])
    q_next = np.array([[0.0, 1.0, 9.0, 2.0], [4.0, 8.0, 7.0, 6.0], [1.0, 2.0, 3.0, 4.0]])
    a, boot = double_boot(q_online, q_next)
    assert a.tolist() == [1, 0, 2] and boot.tolist() == [1.0, 4.0, 3.0]
    a, boot = double_boot(q_online, q_next, a_star=[2, 1, 3])               # the override
    assert boot.tolist() == [9.0, 8.0, 4.0]


def _decls(path):
    src = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
    return dict((m.group(1), m.group(2)) for m in
                re.finditer(r"ARL_API\s+int\s+(arl_\w+)\s*\(([^;]*?)\)\s*;", src, re.S))


def test_ctypes_prototypes_match_the_companion_header(pkg):
    decls = _decls(HEADER)
    table = pkg._cabi.DOUBLE_SIGNATURES
    assert sorted(decls) == sorted(table) == ["arl_double_nstep_q_lossgrad", "arl_double_nstep_q_lossgrad_dueling",
                                              "arl_double_q_lossgrad", "arl_double_q_lossgrad_dueling"]
    for other in (pkg._cabi.EXPORTS, pkg._cabi.SARSA_SIGNATURES, pkg._cabi.DUELING_SIGNATURES):
        assert not set(table) & set(other)
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
    # each entry is its plain entry's signature with q_online_T after q_next / q_boot (and t_max,
    # num_envs in place of num_samples for the 1-step entry)
    for name, plain in (("arl_double_nstep_q_lossgrad", pkg._cabi.SIGNATURES["arl_nstep_q_lossgrad"]),
                        ("arl_double_nstep_q_lossgrad_dueling",
                         pkg._cabi.DUELING_SIGNATURES["arl_nstep_q_lossgrad_dueling"])):
        assert table[name] == plain[:5] + [ctypes.c_void_p] + plain[5:]
    names = [p.split()[-1].lstrip("*") for p in decls["arl_double_q_lossgrad"].split(",")]
    assert names[4:6] == ["q_next", "q_online_T"] and names[9:11] == ["t_max", "num_envs"]


def test_main_header_keeps_its_59_symbols():
    src = open(os.path.join(ROOT, "include", "asyncrl_b200.h")).read()
    syms = set(re.findall(r"ARL_API[^;(]*?\b(arl_\w+)\s*\(", src))
    assert len(syms) == 59
    assert not syms & set(_decls(HEADER))


def test_library_exports_the_companion_header(pkg):
    lib = pkg._cabi.load()
    for name in _decls(HEADER):
        fn = getattr(lib, name)
        assert fn.argtypes == pkg._cabi.DOUBLE_SIGNATURES[name]       # bound by load()
