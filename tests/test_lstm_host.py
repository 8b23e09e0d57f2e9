"""CPU: the A3C LSTM agent -- the float64 reference's explicit BPTT recurrence against autograd, the reset
semantics across a rollout boundary, the parameter layout, the plain network's initial weights, the
companion header against its ctypes table, the main header's size and the refusals."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import lstm_oracle as lo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "asyncrl_b200_lstm.h")


def _layer(T, B, seed):
    rng = np.random.default_rng(seed)
    x = np.abs(rng.normal(size=(T, B, 256)))
    d_h = rng.normal(size=(T, B, 256))
    w = rng.normal(size=(512, 1024)) * 0.05
    b = rng.normal(size=1024) * 0.1
    h0, c0 = rng.normal(size=(B, 256)) * 0.5, rng.normal(size=(B, 256))
    return x, d_h, w, b, h0, c0


def _autograd(x, d_h, w, b, h0, c0, keep):
    X = torch.tensor(x, requires_grad=True)
    W, Bb = torch.tensor(w, requires_grad=True), torch.tensor(b, requires_grad=True)
    h, c = torch.tensor(h0), torch.tensor(c0)
    loss = 0
    for t in range(x.shape[0]):
        h, c = lo.cell(X[t], h, c, W, Bb, torch.as_tensor(keep[t]))
        loss = loss + (h * torch.tensor(d_h[t])).sum()
    loss.backward()
    return W.grad.numpy(), Bb.grad.numpy(), X.grad.numpy()


@pytest.mark.parametrize("T", [1, 5])
def test_explicit_bptt_equals_autograd(T):
    x, d_h, w, b, h0, c0 = _layer(T, 7, T)
    keep = np.ones((T, 7), bool)
    keep[:, 2] = False                       # an env reset at every step
    if T > 1:
        keep[2, 4] = False                   # ... and one reset inside the rollout
    ref = _autograd(x, d_h, w, b, h0, c0, keep)
    got = lo.bptt(x, d_h, w, b, h0, c0, keep)
    for g, r in zip(got, ref):
        assert np.abs(g - r).max() <= 1e-12 * max(1.0, np.abs(r).max())


def test_reset_semantics_across_a_rollout_boundary():
    """keep[0] comes from the previous rollout's last terminal; a reset env's step equals a fresh start,
    a live env's depends on the carried state."""
    T, B = 3, 4
    term = np.zeros((T, B), bool)
    term[0, 1] = True                        # env 1 ends at step 0: step 1 starts from zero
    term[2, 3] = True                        # env 3 ends at the last step: the next rollout's step 0 resets
    keep = lo.keeps(term, np.array([True, False, False, False]))   # env 0's previous rollout ended
    assert keep.numpy().tolist() == [[False, True, True, True], [True, False, True, True], [True, True, True, True]]
    assert lo.keeps(np.zeros((T, B), bool), term[-1])[0].numpy().tolist() == [True, True, True, False]
    x, _, w, b, h0, c0 = _layer(1, B, 11)
    X, W, Bb = (torch.tensor(v) for v in (x[0], w, b))
    h_reset, c_reset = lo.cell(X, torch.tensor(h0), torch.tensor(c0), W, Bb, torch.zeros(B, dtype=torch.bool))
    h_zero, c_zero = lo.cell(X, torch.zeros(B, 256, dtype=torch.float64), torch.zeros(B, 256, dtype=torch.float64),
                             W, Bb, torch.ones(B, dtype=torch.bool))
    assert torch.equal(h_reset, h_zero) and torch.equal(c_reset, c_zero)
    h_live, _ = lo.cell(X, torch.tensor(h0), torch.tensor(c0), W, Bb, torch.ones(B, dtype=torch.bool))
    assert not torch.allclose(h_live, h_zero)


def test_zero_weights_keep_sigmoid_one_of_the_cell_state():
    x, _, w, b, h0, c0 = _layer(1, 3, 5)
    _, c = lo.cell(torch.tensor(x[0]), torch.tensor(h0), torch.tensor(c0), torch.zeros(512, 1024, dtype=torch.float64),
                   torch.zeros(1024, dtype=torch.float64), torch.ones(3, dtype=torch.bool))
    # i = j = 0 -> sigmoid(0) tanh(0) = 0; f = sigmoid(0 + forget_bias 1)
    assert torch.allclose(c, torch.sigmoid(torch.tensor(1.0, dtype=torch.float64)) * torch.tensor(c0), rtol=0, atol=1e-15)


def test_lstm_layout_appends_lstm_after_q_b(pkg):
    for A in (1, 6, 18, 32):
        plain, lstm = pkg._cabi.param_layout(A), pkg._cabi.lstm_param_layout(A)
        assert lstm[:11] == plain
        assert lstm[11] - lstm[10] == 512 * 1024 and lstm[12] - lstm[11] == 1024
    assert pkg._cabi.lstm_param_layout(6)[-1] == 1203255          # 4.81 MB at A = 6
    assert pkg._cabi.prepared_floats(lstm=True) > pkg._cabi.prepared_floats()
    assert pkg._cabi.workspace_bytes(6, lstm=True) > pkg._cabi.workspace_bytes(6)


def test_initial_weights_of_a_plain_network_do_not_change(pkg):
    from importlib import import_module
    net = import_module(pkg.__name__ + ".src.network")
    plain, lstm = net.initial_weights(6, 123), net.initial_weights(6, 123, lstm=True)
    assert list(lstm)[-2:] == ["lstm_w", "lstm_b"] and list(lstm)[:10] == list(plain)
    for k in plain:
        assert torch.equal(plain[k], lstm[k])
    assert tuple(lstm["lstm_w"].shape) == (512, 1024)
    assert float(lstm["lstm_w"].std()) == pytest.approx(0.02, rel=0.02)
    assert not bool(lstm["lstm_b"].any())


def _decls(path):
    src = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
    return dict((m.group(2), (m.group(1), m.group(3))) for m in
                re.finditer(r"ARL_API\s+(int64_t|int)\s+(arl_\w+)\s*\(([^;]*?)\)\s*;", src, re.S))


def test_companion_header_matches_its_ctypes_table(pkg):
    decls = _decls(HEADER)
    cabi = pkg._cabi
    assert set(decls) == set(cabi.LSTM_SIGNATURES) | set(cabi.LSTM_OTHER)
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

    table = dict((n, (a, ctypes.c_int)) for n, a in cabi.LSTM_SIGNATURES.items())
    table.update(cabi.LSTM_OTHER)
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


def test_refusals_without_a_device(pkg):
    """The trunk rule, checked before anything touches a device (Agent's rules: test_gpu_lstm)."""
    assert pkg.config.AgentConfig.lstm is False
    from importlib import import_module
    net = import_module(pkg.__name__ + ".src.network")
    with pytest.raises(NotImplementedError, match="nips"):
        net.make_network(DQN_type="nature", lstm=True)
