"""GPU: the A3C LSTM agent (lstm=True) -- the LSTM step against float64 (tile edges, a reset env next to a
live one, zero weights), the unmasked heads backward, one cycle and a carried-state second cycle against
the float64 reference (terminals inside and at the end of the rollout), graph replay against the eager
loop, full-size determinism, the chunked forward at 18 432 envs, checkpoints, play and the refusals."""
import random

import numpy as np
import pytest
import torch

import kernel_ref as kr
import lstm_oracle as lo
from oracle import a3c
from test_gpu_network import gpu_masks
from util import REL_TOL, rel_err

pytestmark = pytest.mark.gpu


def _flat(pkg, cuda, p, A):
    off = pkg._cabi.lstm_param_layout(A)
    flat = torch.zeros(off[-1], device=cuda)
    for i, k in enumerate(lo.LSTM_NAMES):
        flat[off[i]:off[i + 1]] = torch.as_tensor(np.asarray(p[k]).reshape(-1), device=cuda)
    return flat, off


def _prepare(pkg, cuda, flat, A):
    prep = torch.empty(pkg._cabi.prepared_floats(lstm=True), device=cuda)
    pkg._cabi.call("arl_prepare_weights_lstm", pkg._cabi.ptr(flat), pkg._cabi.ptr(prep), A, pkg._cabi.stream_ptr())
    return prep


# ---- 1. the LSTM step ----------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 37, 200, 4096, 4097])
def test_lstm_step_against_float64(pkg, cuda, B):
    A = 6
    p = lo.init_params(A, seed=B)
    p["lstm_w"] = p["lstm_w"] * 5.0                                  # gates well away from 1/2
    flat, off = _flat(pkg, cuda, p, A)
    prep = _prepare(pkg, cuda, flat, A)
    g = torch.Generator(device=cuda).manual_seed(B)
    x = torch.relu(torch.randn(B, 256, device=cuda, generator=g))
    h0 = torch.randn(B, 256, device=cuda, generator=g) * 0.5
    c0 = torch.randn(B, 256, device=cuda, generator=g)
    reset = (torch.arange(B, device=cuda) % 3 == 1).to(torch.uint8)   # a reset env next to live ones
    P, st = pkg._cabi.ptr, pkg._cabi.stream_ptr()
    f32 = dict(device=cuda, dtype=torch.float32)
    outs = []
    for _ in range(2):
        sh, sc = h0.clone(), c0.clone()
        xh, z = torch.empty(B, 512, **f32), torch.empty(B, 1024, **f32)
        gates, cp = torch.empty(B, 1024, **f32), torch.empty(B, 256, **f32)
        cbuf, c = kr.canary(B * 256 * 4, cuda)
        hbuf, h = kr.canary(B * 256 * 4, cuda)
        pkg._cabi.call("arl_lstm_step", P(flat), P(prep), A, P(x), P(sh), P(sc), P(reset), 1, P(xh), P(z), P(gates),
                       P(cp), P(cbuf), P(hbuf), B, st)
        torch.cuda.synchronize()
        kr.check_canary(hbuf, B * 256 * 4, torch.float32, "lstm h")
        kr.check_canary(cbuf, B * 256 * 4, torch.float32, "lstm c")
        outs.append((h.reshape(B, 256).clone(), c.reshape(B, 256).clone(), sh, sc))
    assert all(kr.same_bits(a, b) for a, b in zip(outs[0], outs[1]))   # bit-identical repeat
    h, c, sh, sc = outs[0]
    assert torch.equal(sh, h) and torch.equal(sc, c)                    # advance: the state is the step's output
    d = lambda k: torch.as_tensor(p[k], device=cuda).double()
    hr, cr = lo.cell(x.double(), h0.double(), c0.double(), d("lstm_w"), d("lstm_b"), reset == 0)
    report = {}
    kr.check("h", h, hr, (0,), REL_TOL, report)
    kr.check("c", c, cr, (0,), REL_TOL, report)
    kr.show("lstm step B=%d" % B, report)


def test_lstm_step_zero_weights_and_no_advance(pkg, cuda):
    A, B = 6, 300
    p = lo.init_params(A, seed=1)
    p["lstm_w"][:] = 0.0
    p["lstm_b"][:] = 0.0
    flat, _ = _flat(pkg, cuda, p, A)
    prep = _prepare(pkg, cuda, flat, A)
    x = torch.rand(B, 256, device=cuda)
    h0, c0 = torch.randn(B, 256, device=cuda), torch.randn(B, 256, device=cuda)
    sh, sc = h0.clone(), c0.clone()
    f32 = dict(device=cuda, dtype=torch.float32)
    h, c = torch.empty(B, 256, **f32), torch.empty(B, 256, **f32)
    P = pkg._cabi.ptr
    pkg._cabi.call("arl_lstm_step", P(flat), P(prep), A, P(x), P(sh), P(sc), None, 0, P(torch.empty(B, 512, **f32)),
                   P(torch.empty(B, 1024, **f32)), None, None, P(c), P(h), B, pkg._cabi.stream_ptr())
    torch.cuda.synchronize()
    ref = torch.sigmoid(torch.tensor(1.0, dtype=torch.float64)) * c0.double()     # c = sigmoid(1) c_prev
    assert kr.rel_err(c, ref) <= 1e-6
    assert torch.equal(sh, h0) and torch.equal(sc, c0)                             # not advanced


# ---- 2. the unmasked heads backward --------------------------------------------------------------
@pytest.mark.parametrize("A", [1, 6, 18, 32])
def test_unmasked_heads_backward(pkg, cuda, A):
    N = 4096 * 5 + 3
    p = lo.init_params(A, seed=A)
    flat, off = _flat(pkg, cuda, p, A)
    g = torch.Generator(device=cuda).manual_seed(A)
    h = torch.tanh(torch.randn(N, 256, device=cuda, generator=g))                # negative values too
    dl, dv = torch.randn(N, A, device=cuda, generator=g), torch.randn(N, device=cuda, generator=g)
    grads = torch.zeros_like(flat)
    ws = torch.empty(pkg._cabi.workspace_bytes(A, lstm=True), dtype=torch.uint8, device=cuda)
    S = 64.0
    outs = []
    for _ in range(2):
        buf, dh = kr.canary(N * 256 * 4, cuda)
        pkg._cabi.call("arl_heads_backward_lstm", pkg._cabi.ptr(flat), A, pkg._cabi.ptr(h), pkg._cabi.ptr(dl),
                       pkg._cabi.ptr(dv), pkg._cabi.ptr(buf), pkg._cabi.ptr(grads), pkg._cabi.ptr(ws), N, S,
                       pkg._cabi.stream_ptr())
        torch.cuda.synchronize()
        kr.check_canary(buf, N * 256 * 4, torch.float32, "d_h_lstm")
        outs.append((dh.reshape(N, 256).clone(), grads.clone()))
    assert kr.same_bits(outs[0][0], outs[1][0]) and kr.same_bits(outs[0][1], outs[1][1])
    d = lambda k: torch.as_tensor(p[k], device=cuda).double()
    hd, dld, dvd = h.double(), dl.double(), dv.double()
    report = {}
    kr.check("d_h", outs[0][0] / S, dld @ d("p_w").T + dvd[:, None] @ d("q_w").T, (0,), REL_TOL, report)
    gr = outs[0][1]
    kr.check("p_w", gr[off[6]:off[7]].reshape(256, A), hd.T @ dld, (1,), REL_TOL, report)
    kr.check("p_b", gr[off[7]:off[8]], dld.sum(0), (0,), REL_TOL, report)
    kr.check("q_w", gr[off[8]:off[9]], hd.T @ dvd, (0,), REL_TOL, report)
    kr.show("unmasked heads backward A=%d" % A, report)


# ---- 3. BPTT + LSTM weight gradient at full size ------------------------------------------------
@pytest.mark.parametrize("B,T", [(4096, 5), (4096, 20)])
@pytest.mark.parametrize("A", [6, 18])
def test_bptt_and_wgrad_against_float64(pkg, cuda, B, T, A):
    """arl_lstm_backward on the forward the device ran (arl_lstm_step per step, terminals inside the rollout
    and before it), against the explicit float64 recurrence from that forward's stored values: d lstm_w,
    d lstm_b and d_h_fc (both copies, relu pattern of x), bit-identical on repeat, nothing written outside
    its buffers."""
    N, S = B * T, 64.0
    p = lo.init_params(A, seed=100 + T)
    p["lstm_w"] = p["lstm_w"] * 4.0
    flat, off = _flat(pkg, cuda, p, A)
    prep = _prepare(pkg, cuda, flat, A)
    g = torch.Generator(device=cuda).manual_seed(T * 7 + A)
    x = torch.relu(torch.randn(N, 256, device=cuda, generator=g))                  # h_fc, exact zeros included
    h0 = torch.randn(B, 256, device=cuda, generator=g) * 0.5
    c0 = torch.randn(B, 256, device=cuda, generator=g)
    terms = (torch.rand(T, B, device=cuda, generator=g) < 0.1).to(torch.uint8)
    reset0 = (torch.rand(B, device=cuda, generator=g) < 0.1).to(torch.uint8)
    d_h_lstm = torch.randn(N, 256, device=cuda, generator=g) * S                   # leaves the heads scaled
    P, st = pkg._cabi.ptr, pkg._cabi.stream_ptr()
    f32 = dict(device=cuda, dtype=torch.float32)
    xh, z = torch.empty(N, 512, **f32), torch.empty(B, 1024, **f32)
    gates, cp, c, h = torch.empty(N, 1024, **f32), torch.empty(N, 256, **f32), torch.empty(N, 256, **f32), \
        torch.empty(N, 256, **f32)
    sh, sc = h0.clone(), c0.clone()
    for t in range(T):
        r = slice(t * B, (t + 1) * B)
        pkg._cabi.call("arl_lstm_step", P(flat), P(prep), A, P(x[r]), P(sh), P(sc), P(reset0 if t == 0 else terms[t - 1]),
                       1, P(xh[r]), P(z), P(gates[r]), P(cp[r]), P(c[r]), P(h[r]), B, st)
    ws = torch.empty(pkg._cabi.workspace_bytes(A, lstm=True), dtype=torch.uint8, device=cuda)
    n8 = (N + 7) // 8 * 8
    dh_bytes = (N + n8) * 256 * 4
    outs = []
    for _ in range(2):
        dz_buf, dz = kr.canary(N * 1024 * 4, cuda)
        dxh_buf, dxh = kr.canary(N * 512 * 4, cuda)
        dh_buf, dh = kr.canary(dh_bytes, cuda)
        dc = torch.full((B, 256), float("nan"), **f32)
        grads = torch.zeros_like(flat)
        pkg._cabi.call("arl_lstm_backward", P(flat), P(prep), A, B, T, P(terms), P(x), P(xh), P(gates), P(cp), P(c),
                       P(d_h_lstm), P(dz_buf), P(dxh_buf), P(dc), P(dh_buf), P(grads), P(ws), S, st)
        torch.cuda.synchronize()
        kr.check_canary(dz_buf, N * 1024 * 4, torch.float32, "dz")
        kr.check_canary(dxh_buf, N * 512 * 4, torch.float32, "dxh")
        kr.check_canary(dh_buf, dh_bytes, torch.float32, "d_h")
        outs.append((grads.clone(), dh_buf.clone(), dxh_buf.clone()))
    assert all(kr.same_bits(a, b) for a, b in zip(outs[0], outs[1]))               # bit-identical repeat
    grads, dh_raw = outs[0][0], outs[0][1][:dh_bytes].view(torch.float32)
    d = lambda k: torch.as_tensor(p[k], device=cuda).double()
    keep = lo.keeps(terms.cpu().numpy(), reset0.cpu().numpy()).to(cuda).double()
    net = _net_mod(pkg)
    # the backward on the forward's stored values as the kernels read them (xh: its split blocks); the
    # forward itself is checked against float64 above
    xh_d = torch.stack([net.decode_split(xh[t * B:(t + 1) * B], B, 512) for t in range(T)]).double()
    v = lambda a, w: a.double().reshape(T, B, w)
    dW, db, dx = lo.bptt_given(xh_d, v(gates, 1024), v(cp, 256), v(c, 256), v(d_h_lstm, 256) / S, d("lstm_w"), keep)
    dx = (dx.reshape(N, 256) * (x > 0)).double()
    bT = dh_raw[N * 256:].view(torch.bfloat16).reshape(2, n8 // 8, 256, 8)
    dh_T = (bT[0].float() + bT[1].float()).permute(0, 2, 1).reshape(n8, 256)[:N] / S
    report = {}
    kr.check("lstm_w", grads[off[10]:off[11]].reshape(512, 1024), dW, (1,), REL_TOL, report)
    kr.check("lstm_b", grads[off[11]:off[12]], db, (0,), REL_TOL, report)
    kr.check("d_h_fc", net.decode_split(dh_raw[:N * 256], N, 256) / S, dx, (0,), REL_TOL, report)
    kr.check("d_h_fc^T", dh_T, dx, (0,), REL_TOL, report)
    kr.show("bptt + wgrad B=%d T=%d A=%d" % (B, T, A), report)


def _net_mod(pkg):
    from importlib import import_module
    return import_module(pkg.__name__ + ".src.network")


# ---- 4. cycles against the reference -------------------------------------------------------------
def _agent(pkg, cuda, B, T, A, over=None, pool=None, p_terminal=0.25, seed=3):
    cfg = pkg.config.get_config(dict({"model": "m1", "num_envs": B, "t_max": T, "lstm": True}, **(over or {})))
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=seed, pool=pool or T + 3, device=cuda,
                                                         p_terminal=p_terminal), device=cuda)
    return pkg.Agent(cfg, env, device=cuda), env


def _rollout(agent, env):
    """One rollout by hand (Agent.observe without the update trigger); returns screens, rewards, terminals."""
    hist, T = agent.history, agent.t_max
    first = hist.first_slot(0)
    snap = hist.planes().cpu().numpy()
    screens = [snap[:, (first + k) % hist.ring_slots] for k in range(4)]
    rews, terms = [], []
    for t in range(T):
        action = agent.predict()
        scr, rew, term = env.act(action, is_training=True, fused=True)
        hist.add(scr)
        agent.batch_reward[t].copy_(rew)
        agent.batch_terminal[t].copy_(term)
        rews.append(rew.cpu().numpy()); terms.append(term.cpu().numpy())
        screens.append(hist.planes(hist.head).cpu().numpy())
        agent.t += 1
        agent.step += 1
    return screens, np.stack(rews), np.stack(terms)


@pytest.mark.parametrize("A,B,T", [(6, 64, 5), (18, 64, 20), (6, 9, 4)])
def test_two_cycles_vs_oracle(pkg, cuda, A, B, T):
    """Cycle 1 from the zero state, cycle 2 from the state cycle 1 left (reset by its last terminals)."""
    agent, env = _agent(pkg, cuda, B, T, A)
    net = agent.network
    params = lo.init_params(A, seed=41)
    net.set_weights(params)
    agent.before_train()
    agent.step = 100
    for cycle in range(2):
        h0, c0 = (s.cpu().numpy() for s in net.lstm_state())
        reset0 = agent.batch_terminal[T - 1].cpu().numpy().astype(bool)
        params = {k: v.cpu().numpy().copy() for k, v in net.w.items()}
        rms = {k: net.rms[net.offsets[i]:net.offsets[i + 1]].view(net.w[k].shape).cpu().numpy().copy()
               for i, k in enumerate(net.param_names)}
        screens, rews, terms = _rollout(agent, env)
        agent.step -= 1
        masks = gpu_masks(net)
        logits = net.policy_logits.cpu().numpy().copy()
        state_after = tuple(s.cpu().numpy() for s in net.lstm_state())
        acts = agent.batch_action.cpu().numpy().copy()
        agent.batch_update()
        agent.step += 1
        torch.cuda.synchronize()
        new_p, _, aux = lo.lstm_cycle(params, rms, np.stack(screens), acts, rews, terms, agent.step - T, (h0, c0),
                                      reset0, num_envs=B, masks=masks)
        assert rel_err(logits, aux["logits"].reshape(T * B, A)) <= REL_TOL
        assert rel_err(state_after[0], aux["state"][0]) <= REL_TOL and rel_err(state_after[1], aux["state"][1]) <= REL_TOL
        assert rel_err(net.R.cpu().numpy().reshape(T, B), aux["R"]) <= REL_TOL
        # the bootstrap did not advance the state
        assert all(torch.equal(a, torch.as_tensor(b, device=cuda)) for a, b in zip(net.lstm_state(), state_after))
        errs = {k: rel_err(net.g[k].cpu(), aux["grads"][k]) for k in lo.LSTM_NAMES}
        errs["d_h_fc"] = rel_err(net.d_h().cpu().numpy(), aux["d_h_fc"].reshape(T * B, 256))
        print("lstm cycle", cycle, "A=%d B=%d T=%d" % (A, B, T), "terminals", int(terms.sum()), "rel-err", errs)
        assert max(errs.values()) <= REL_TOL, errs
        errs = {k: rel_err(net.w[k].cpu(), new_p[k]) for k in lo.LSTM_NAMES}
        assert max(errs.values()) <= REL_TOL, errs
    assert terms.any()


# ---- 5. graph replay == eager loop, determinism, 18 432 envs -------------------------------------
def _loop(pkg, cuda, graphs, cycles, B=24, T=5, A=6):
    random.seed(123)
    agent, env = _agent(pkg, cuda, B, T, A, over={"cuda_graphs": graphs}, pool=T, p_terminal=0.1, seed=5)
    agent.network.set_weights(lo.init_params(A, seed=9))
    agent.before_train()
    acts, snaps = [], []
    for _ in range(cycles):
        for _ in range(agent.t_max):
            a = agent.predict()
            acts.append(a.clone())
            scr, rew, term = env.act(a, is_training=True, fused=True)
            agent.observe(scr, rew, a, term)
            agent.step += 1
        n = agent.network
        snaps.append((n.params.clone(), n.rms.clone(), n.state_h.clone(), n.state_c.clone()))
    torch.cuda.synchronize()
    return agent, torch.stack(acts), snaps


def test_graph_replay_equals_eager_loop(pkg, cuda):
    eager, acts_e, snaps_e = _loop(pkg, cuda, False, 9)
    graph, acts_g, snaps_g = _loop(pkg, cuda, True, 9)
    assert eager.graph_replays == 0 and graph.graph_replays > 0
    assert torch.equal(acts_e, acts_g)
    for a, b in zip(snaps_e, snaps_g):
        assert all(torch.equal(x, y) for x, y in zip(a, b))
    lw = slice(graph.network.offsets[10], graph.network.offsets[11])
    assert not torch.equal(snaps_g[8][0][lw], snaps_g[0][0][lw])        # lstm_w trained


@pytest.mark.parametrize("B,T", [(4096, 5), (18432, 2)])
def test_full_size_is_finite_and_deterministic(pkg, cuda, B, T):
    """18 432 envs: the trunk runs in env ranges (arl_a2_block_rows), the LSTM over all envs."""
    runs = []
    for _ in range(2):
        agent, acts, snaps = _loop(pkg, cuda, True, 3, B=B, T=T)
        g = agent.network.grads.clone()
        assert bool(torch.isfinite(g).all()) and float(agent.network.g["lstm_w"].abs().max()) > 0
        runs.append((acts, g, snaps[-1]))
        del agent
        torch.cuda.empty_cache()
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    assert all(torch.equal(x, y) for x, y in zip(runs[0][2], runs[1][2]))


def test_chunked_forward_keeps_the_state_continuous(pkg, cuda):
    """At 18 432 envs (two env ranges of 9 216) the step equals the float64 cell on every env."""
    B, A = 18432, 6
    assert pkg._cabi.a2_block_rows(B) < B
    agent, env = _agent(pkg, cuda, B, 2, A, pool=3)
    net = agent.network
    net.set_weights(lo.init_params(A, seed=7))
    agent.before_train()
    for t in range(2):
        h0, c0 = net.lstm_state()
        agent.predict()
        torch.cuda.synchronize()
        d = lambda k: net.w[k].double()
        hr, cr = lo.cell(net.l4[net._rows(t)].double(), h0.double(), c0.double(), d("lstm_w"), d("lstm_b"),
                         torch.ones(B, dtype=torch.bool, device=cuda))
        assert kr.rel_err(net.state_h, hr) <= REL_TOL and kr.rel_err(net.state_c, cr) <= REL_TOL
        agent.t += 1


# ---- 6. checkpoints, play, refusals --------------------------------------------------------------
def test_checkpoint_round_trip_and_cross_kind_refusal(pkg, cuda, tmp_path):
    B, T, A = 8, 2, 6
    lstm, env = _agent(pkg, cuda, B, T, A)
    lstm.network.set_weights(lo.init_params(A, seed=2))
    plain = pkg.Agent(pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T}), env, device=cuda)
    l_dir, p_dir = tmp_path / "lstm", tmp_path / "plain"
    z_l = np.load(lstm.save_checkpoint(str(l_dir)))
    z_p = np.load(plain.save_checkpoint(str(p_dir)))
    assert bool(z_l["lstm"]) and "lstm" not in z_p.files and "lstm_w" in z_l.files
    twin, _ = _agent(pkg, cuda, B, T, A)
    assert twin.load_checkpoint(str(l_dir))
    assert torch.equal(twin.network.params, lstm.network.params)
    before = plain.network.params.clone()
    with pytest.raises(ValueError, match="lstm"):
        plain.load_checkpoint(str(l_dir))
    assert torch.equal(plain.network.params, before)
    with pytest.raises(ValueError, match="non-lstm"):
        twin.load_checkpoint(str(p_dir))


def test_play_resets_its_own_state_per_episode(pkg, cuda):
    B, T, A = 6, 2, 6
    agent, env = _agent(pkg, cuda, B, T, A, p_terminal=0.3)
    agent.network.set_weights(lo.init_params(A, seed=4))
    agent.before_train()
    agent.predict()
    train_state = agent.network.lstm_state()
    calls = []
    orig = agent.network.reset_lstm_state

    def spy(play=False):
        calls.append(play)
        orig(play)
    agent.network.reset_lstm_state = spy
    agent.play(n_step=4, n_episode=3)
    assert calls == [True, True, True]
    assert all(torch.equal(a, b) for a, b in zip(agent.network.lstm_state(), train_state))   # training state kept
    assert bool(agent.network.lstm_state(play=True)[0].abs().max() > 0)


def test_refusals(pkg, cuda):
    def make(mode, kind="nips"):
        cfg = pkg.config.get_config({"model": "m1", "num_envs": 4, "t_max": 2, "loss_mode": mode, "lstm": True,
                                     "DQN_type": kind})
        env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(4, 6, seed=1, pool=4, device=cuda), device=cuda)
        return pkg.Agent(cfg, env, device=cuda)
    for mode in ("async_q", "nstep_q", "sarsa"):
        with pytest.raises(ValueError, match="a3c"):
            make(mode)
    with pytest.raises(NotImplementedError, match="nips"):
        make("a3c", "nature")
    net = pkg.Network(action_size=6, num_envs=4, t_max=2, device=cuda, lstm=True)
    for call in (net.make_target, lambda: net.compute_q_gradients(None, None, None, 1.0)):
        with pytest.raises(ValueError, match="LSTM"):
            call()


# ---- 7. N ranks ----------------------------------------------------------------------------------
@pytest.mark.parametrize("collective", ["p2p", "library"])
def test_multi_gpu_run_equals_single_gpu_union_batch(cuda, collective):
    import json
    import os
    import socket
    import subprocess
    import sys
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (one rank per GPU)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    world = 2 if n < 4 else 4
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(root, "tests", "dist_gpu_check_lstm.py"), "--collective", collective]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["ok"] and line["actions_bit_identical"] and line["replica_max_minus_min"] == 0.0
