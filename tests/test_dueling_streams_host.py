"""CPU: the dueling streams (a hidden layer per stream) -- the float64 reference's closed-form head and
stream gradients against autograd, the aggregator's invariance, the reduction to the shared-fc dueling
reference, the companion header against its ctypes table, the main header's size and the refusals."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import dueling_oracle
import dueling_streams_oracle as so
from oracle import a3c

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "asyncrl_b200_dueling_streams.h")


def _stacks(n, seed):
    return np.random.default_rng(seed).integers(0, 256, (n, 84, 84, 4)).astype(np.float64)


def test_closed_form_head_and_stream_gradients_equal_autograd():
    A, N = 6, 7
    p = a3c.to_torch(so.init_streams_params(A, seed=3, scale=2.0, bias_std=0.1))
    rng = np.random.default_rng(0)
    h = torch.tensor(rng.normal(0, 1, (N, 512)), dtype=torch.float64).relu().requires_grad_(True)
    pw, qw = p["p_w"].clone().requires_grad_(True), p["q_w"].clone().requires_grad_(True)
    pb, qb = p["p_b"].clone().requires_grad_(True), p["q_b"].clone().requires_grad_(True)
    v = (h[:, :256] @ qw + qb).reshape(-1)
    adv = h[:, 256:] @ pw + pb
    q = dueling_oracle.combine(adv, v)
    acts = rng.integers(0, A, N)
    delta = rng.normal(0, 1, N)
    # the loss gradient the dueling loss entries write, pushed through the network by hand ...
    d_logits, d_value = dueling_oracle.head_gradients(acts, delta, A, 0.5)
    ref = so.heads_backward(h.detach().numpy(), pw.detach().numpy(), qw.detach().numpy(), d_logits, d_value)
    # ... and by autograd from dL/dQ = g [j == a]
    dq = np.zeros((N, A))
    dq[np.arange(N), acts] = -2.0 * delta * 0.5
    q.backward(torch.tensor(dq))
    mask = (h.detach() > 0).numpy()
    np.testing.assert_allclose(ref["d_h"], h.grad.numpy() * mask, rtol=1e-12, atol=1e-12)
    for k, t in (("p_w", pw), ("p_b", pb), ("q_w", qw), ("q_b", qb)):
        np.testing.assert_allclose(ref[k], t.grad.numpy(), rtol=1e-12, atol=1e-12)


def test_q_is_invariant_to_a_constant_added_to_p_b():
    A = 5
    p = a3c.to_torch(so.init_streams_params(A, seed=4, scale=2.0, bias_std=0.1))
    s = _stacks(3, 1)
    q0 = so.q_forward(p, s)
    p["p_b"] = p["p_b"] + 3.25
    assert torch.allclose(so.q_forward(p, s), q0, rtol=0, atol=1e-12)


def test_with_la_equal_to_l4_the_reference_is_the_shared_fc_dueling_reference():
    A = 6
    p = a3c.to_torch(so.init_streams_params(A, seed=5, scale=2.0, bias_std=0.1))
    p["la_w"], p["la_b"] = p["l4_w"].clone(), p["l4_b"].clone()
    s = _stacks(4, 2)
    plain = {k: v for k, v in p.items() if k not in ("la_w", "la_b")}
    assert torch.allclose(so.q_forward(p, s), dueling_oracle.q_forward(plain, s), rtol=0, atol=1e-12)


def test_stream_gradients_reach_both_hidden_layers():
    A, T, B = 4, 2, 3
    rng = np.random.default_rng(9)
    params = so.init_streams_params(A, seed=6, scale=2.0, bias_std=0.1)
    tparams = so.init_streams_params(A, seed=7, scale=2.0, bias_std=0.1)
    stacks = rng.integers(0, 256, (T + 1, B, 84, 84, 4)).astype(np.float64)
    for mode in ("async_q", "nstep_q", "sarsa"):
        acts = rng.integers(0, A, (T + 1 if mode == "sarsa" else T, B))
        g, aux = so.streams_gradients(mode, params, tparams, stacks, acts, rng.normal(0, 1, (T, B)),
                                      np.zeros((T, B), np.uint8))
        assert np.abs(g["la_w"]).max() > 0 and np.abs(g["l4_w"]).max() > 0 and np.abs(g["q_w"]).max() > 0


def _decls(path):
    src = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
    return dict((m.group(2), (m.group(1), m.group(3))) for m in
                re.finditer(r"ARL_API\s+(int64_t|int)\s+(arl_\w+)\s*\(([^;]*?)\)\s*;", src, re.S))


def test_companion_header_matches_its_ctypes_table(pkg):
    decls = _decls(HEADER)
    cabi = pkg._cabi
    assert set(decls) == set(cabi.STREAMS_SIGNATURES) | set(cabi.STREAMS_OTHER)
    kind = {ctypes.c_void_p: "ptr", ctypes.c_int: "int", ctypes.c_int64: "i64", ctypes.c_uint64: "u64",
            ctypes.c_float: "f32", ctypes.c_double: "f64"}

    def ckind(param):
        p = " ".join(param.split())
        if "*" in p:
            return "ptr"
        for pre, k in (("float", "f32"), ("double", "f64"), ("int64_t", "i64"), ("uint64_t", "u64"), ("int ", "int")):
            if p.startswith(pre):
                return k
        raise AssertionError(p)

    table = dict((n, (a, ctypes.c_int)) for n, a in cabi.STREAMS_SIGNATURES.items())
    table.update(cabi.STREAMS_OTHER)
    for name, (ret, params) in decls.items():
        argtypes, restype = table[name]
        ps = [p for p in params.split(",") if p.strip() and p.strip() != "void"]
        got = ["ptr" if isinstance(a, type) and issubclass(a, ctypes._Pointer) else kind[a] for a in argtypes]
        assert got == [ckind(p) for p in ps], (name, got, ps)
        assert restype == (ctypes.c_int64 if ret == "int64_t" else ctypes.c_int), name
    lib = cabi.load()
    for name in decls:
        assert getattr(lib, name) is not None


def test_main_header_keeps_its_59_symbols():
    src = open(os.path.join(ROOT, "include", "asyncrl_b200.h")).read()
    assert len(set(re.findall(r"ARL_API[^;(]*?\b(arl_\w+)\s*\(", src))) == 59


def test_streams_layout_appends_la_after_q_b(pkg):
    for A in (1, 6, 18, 32):
        plain, streams = pkg._cabi.param_layout(A), pkg._cabi.streams_param_layout(A)
        assert streams[:11] == plain
        assert streams[11] - streams[10] == 2592 * 256 and streams[12] - streams[11] == 256
    # about 5.4 MB of gradient with the flag on (2.71 MB without)
    assert abs(pkg._cabi.streams_param_layout(6)[-1] * 4 / 1e6 - 5.38) < 0.05
    assert pkg._cabi.prepared_floats(True) > pkg._cabi.prepared_floats()
    assert pkg._cabi.workspace_bytes(6, True) > pkg._cabi.workspace_bytes(6)


def test_initial_weights_of_a_plain_network_do_not_change(pkg):
    from importlib import import_module
    net = import_module(pkg.__name__ + ".src.network")
    plain, streams = net.initial_weights(6, 123), net.initial_weights(6, 123, streams=True)
    assert list(streams)[-2:] == ["la_w", "la_b"] and list(streams)[:10] == list(plain)
    for k in plain:
        assert torch.equal(plain[k], streams[k])
    assert float(streams["la_w"].std()) == pytest.approx(0.02, rel=0.02)
    assert not torch.equal(streams["la_w"], streams["l4_w"]) and not bool(streams["la_b"].any())


def test_refusals_without_a_device(pkg):
    """The trunk rule, checked before anything touches a device (Agent's rules: test_gpu_dueling_streams)."""
    assert pkg.config.AgentConfig.dueling_streams is False
    from importlib import import_module
    net = import_module(pkg.__name__ + ".src.network")
    with pytest.raises(NotImplementedError, match="nips"):
        net.make_network(DQN_type="nature", dueling_streams=True)
