"""GPU: the dueling streams (dueling_streams=True: a hidden layer per stream) on the async-Q, n-step Q and
Sarsa learners -- the fc forward of both streams on both sides of the cluster / streaming switch, the
composed forward against float64 and against arl_forward_dueling, the heads and
fc backward against float64, one cycle per learner (and with double Q) against the reference, graph
replay against the eager loop, determinism, checkpoints and refusals."""
import random

import numpy as np
import pytest
import torch

import dueling_streams_oracle as so
import kernel_ref as kr
from oracle import a3c
from test_gpu_network import gpu_masks, ring_stacks
from util import REL_TOL, rel_err

pytestmark = pytest.mark.gpu
MODES = ("async_q", "nstep_q", "sarsa")


def _net_mod(pkg):
    from importlib import import_module
    return import_module(pkg.__name__ + ".src.network")


def _params(pkg, cuda, A, seed, same_la=False):
    p = so.init_streams_params(A, seed=seed, scale=2.0, bias_std=0.3)
    if same_la:
        p["la_w"], p["la_b"] = p["l4_w"].copy(), p["l4_b"].copy()
    return p, torch.as_tensor(so.flatten(p), device=cuda)


def _prepare(pkg, cuda, flat, A):
    prep = torch.empty(pkg._cabi.prepared_floats(True), device=cuda)
    pkg._cabi.call("arl_prepare_weights_streams", pkg._cabi.ptr(flat), pkg._cabi.ptr(prep), A,
                   pkg._cabi.stream_ptr())
    return prep


# ---- 1. the fc forward of both streams -----------------------------------------------------------
def _mc(cuda):
    return 128 * (torch.cuda.get_device_properties(cuda).multi_processor_count // 4)


@pytest.mark.parametrize("where", ["mc", "mc+1", "4096x5"])
def test_fc_forward_both_streams(pkg, cuda, where):
    A = 6
    M = {"mc": _mc(cuda), "mc+1": _mc(cuda) + 1, "4096x5": 4096 * 5}[where]
    net = _net_mod(pkg)
    p, flat = _params(pkg, cuda, A, seed=M)
    prep = _prepare(pkg, cuda, flat, A)
    g = torch.Generator(device=cuda).manual_seed(M)
    a2 = torch.relu(torch.randn(M, 2592, device=cuda, generator=g) * 2.0)
    a2s = net.encode_split(a2)
    a2d = net.decode_split(a2s, M, 2592).double()                    # the values the kernels read
    P, st = pkg._cabi.ptr, pkg._cabi.stream_ptr()
    outs = []
    for _ in range(2):
        buf, h = kr.canary(M * 512 * 4, cuda)
        pkg._cabi.call("arl_fc_forward_streams", P(prep), P(a2s), P(buf), M, st)
        torch.cuda.synchronize()
        kr.check_canary(buf, M * 512 * 4, torch.float32, "fc streams forward")
        outs.append(h.reshape(M, 512).clone())
    assert kr.same_bits(outs[0], outs[1])                            # bit-identical repeat
    d = lambda k: torch.as_tensor(p[k], device=cuda).double()
    ref = torch.cat([torch.relu(a2d @ d("l4_w") + d("l4_b")), torch.relu(a2d @ d("la_w") + d("la_b"))], 1)
    report = {}
    kr.check("h_v", outs[0][:, :256], ref[:, :256], (0,), REL_TOL, report)
    kr.check("h_a", outs[0][:, 256:], ref[:, 256:], (0,), REL_TOL, report)
    kr.show("fc streams forward M=%d" % M, report)


# ---- 2. the composed forward ---------------------------------------------------------------------
class Fwd:
    def __init__(self, pkg, cuda, B, A, steps, seed, same_la=False):
        g = torch.Generator(device=cuda).manual_seed(seed)
        self.pkg, self.cuda, self.B, self.A, self.steps = pkg, cuda, B, A, steps
        self.slots = steps + 3
        self.ring = torch.randint(0, 256, (B, self.slots, 84 * 84), dtype=torch.uint8, device=cuda, generator=g)
        self.p, self.flat = _params(pkg, cuda, A, seed + 31, same_la)
        N = B * steps
        f32 = dict(device=cuda, dtype=torch.float32)
        self.l1, self.l2 = torch.empty(N, 3200, **f32), torch.empty(N, 2592, **f32)

    def run(self, entry, actions=None, ep=0.0, step=0, seed=0):
        P, N, A, c = self.pkg._cabi.ptr, self.B * self.steps, self.A, self.pkg._cabi
        f32 = dict(device=self.cuda, dtype=torch.float32)
        streams = entry == "arl_forward_streams"
        params = self.flat if streams else self.flat[:c.param_layout(A)[-1]]
        prep = torch.empty(c.prepared_floats(streams), **f32)
        h = torch.empty(N, 512 if streams else 256, **f32)
        q, probs, v = torch.empty(N, A, **f32), torch.empty(N, A, **f32), torch.empty(N, **f32)
        c.call(entry, P(params), P(prep), 1, A, P(self.ring), self.B, self.slots, 0, self.steps, P(self.l1),
               P(self.l2), P(h), P(q), P(probs), P(v), P(actions), 0, int(step), None, int(seed), float(ep),
               0.0, 0.0, 1.0, 0.0, c.stream_ptr())
        torch.cuda.synchronize()
        return h, q, probs, v


@pytest.mark.parametrize("B,A,steps", [(4096, 6, 5), (18432, 18, 1)])
def test_forward_against_float64_and_the_fused_draw(pkg, cuda, B, A, steps):
    f = Fwd(pkg, cuda, B, A, steps, seed=B + A)
    h, q, probs, v = f.run("arl_forward_streams")
    h2, q2, _, v2 = f.run("arl_forward_streams")
    assert kr.same_bits(q, q2) and kr.same_bits(h, h2) and kr.same_bits(v, v2)
    assert float((probs - torch.softmax(q, 1)).abs().max()) <= 1e-6
    ring = f.ring.cpu().numpy().reshape(B, f.slots, 84, 84)
    envs = np.r_[0:128, B - 128:B]
    stacks = ring_stacks(ring[envs], 0, steps)
    qr, vr, advr, hvr, har = (x.numpy() for x in so.forward(a3c.to_torch(f.p), stacks))
    rows = np.concatenate([t * B + envs for t in range(steps)])
    hc = h.cpu().numpy()[rows]
    errs = dict(h_v=rel_err(hc[:, :256], hvr), h_a=rel_err(hc[:, 256:], har), v=rel_err(v.cpu().numpy()[rows], vr),
                q=rel_err(q.cpu().numpy()[rows], qr),
                adv=rel_err((q - v[:, None]).cpu().numpy()[rows], advr - advr.mean(1, keepdims=True)))
    print("streams forward", B, A, steps, errs)
    assert max(errs.values()) <= REL_TOL, errs
    # the epsilon-greedy draw inside the heads launch == arl_egreedy_actions on the written Q
    acts, ref = torch.empty(B, dtype=torch.int32, device=cuda), torch.empty(B, dtype=torch.int32, device=cuda)
    one = Fwd(pkg, cuda, B, A, 1, seed=B + A)
    for ep in (0.0, 0.3):
        _, q1, _, _ = one.run("arl_forward_streams", acts, ep, 7, 99)
        pkg._cabi.call("arl_egreedy_actions", pkg._cabi.ptr(q1), pkg._cabi.ptr(ref), B, A, ep, 0, 7, 99,
                       pkg._cabi.stream_ptr())
        torch.cuda.synchronize()
        assert torch.equal(acts, ref), ep


@pytest.mark.parametrize("B,steps", [(_B, 1) for _B in (4096, 4737)] + [(4096, 5)])
def test_with_la_equal_to_l4_q_is_the_shared_fc_dueling_q(pkg, cuda, B, steps):
    f = Fwd(pkg, cuda, B, 6, steps, seed=B, same_la=True)
    h, q, _, v = f.run("arl_forward_streams")
    _, qd, _, vd = f.run("arl_forward_dueling")
    assert kr.same_bits(h[:, :256], h[:, 256:])
    assert kr.same_bits(q, qd) and kr.same_bits(v, vd)


# ---- 3. the backward -----------------------------------------------------------------------------
@pytest.mark.parametrize("A", [6, 18, 32])
def test_heads_and_fc_backward_against_float64(pkg, cuda, A):
    B, T = 4096, 5
    N = B * T
    net = _net_mod(pkg)
    p, flat = _params(pkg, cuda, A, seed=A)
    prep = _prepare(pkg, cuda, flat, A)
    g = torch.Generator(device=cuda).manual_seed(A)
    a2 = torch.relu(torch.randn(N, 2592, device=cuda, generator=g))
    a2s = net.encode_split(a2)
    a2d = net.decode_split(a2s, N, 2592).double()
    h = torch.relu(torch.randn(N, 512, device=cuda, generator=g))    # relu pattern forced: exact zeros
    dl = torch.randn(N, A, device=cuda, generator=g) * 1e-3
    dv = torch.randn(N, device=cuda, generator=g) * 1e-3
    S = 2.0 ** 14
    off = pkg._cabi.streams_param_layout(A)
    grads = torch.full((off[-1],), float("nan"), device=cuda)
    d_h = torch.empty(N + (N + 7) // 8 * 8, 512, device=cuda)
    d_a2 = torch.empty(N, 2592, device=cuda)
    ws = torch.empty(pkg._cabi.workspace_bytes(A, True), dtype=torch.uint8, device=cuda)
    P, st = pkg._cabi.ptr, pkg._cabi.stream_ptr()
    outs = []
    for _ in range(2):
        pkg._cabi.call("arl_heads_backward_streams", P(flat), A, P(h), P(dl), P(dv), P(d_h), P(grads), P(ws), N, S, st)
        pkg._cabi.call("arl_fc_backward_streams", P(prep), P(a2s), N, P(d_h), P(d_a2), P(grads), P(ws), N, 1.0 / S,
                       A, st)
        torch.cuda.synchronize()
        outs.append((grads.clone(), d_a2.clone(), d_h.clone()))
    for x, y in zip(outs[0], outs[1]):
        assert kr.same_bits(x, y)
    assert not bool(grads[off[4]:].isnan().any())
    dh_dev = net.decode_split(d_h[:N], N, 512).double() / S
    hd, dld, dvd = h.double(), dl.double(), dv.double()
    w = lambda k: torch.as_tensor(p[k], device=cuda).double()
    dhv = dvd[:, None] * w("q_w").reshape(1, -1) * (hd[:, :256] > 0)
    dha = (dld @ w("p_w").T) * (hd[:, 256:] > 0)
    dhr = torch.cat([dhv, dha], 1)
    G = lambda i: grads[off[i]:off[i + 1]]
    # the fc backward against the d_h it reads (the split block, as tests/test_gpu_fc.py does): the column
    # sums of the bias gradients would otherwise carry the split's rounding of d_h through cancellation
    dhk = dh_dev
    ref = {"p_w": (hd[:, 256:].T @ dld, G(6).reshape(256, A)), "p_b": (dld.sum(0), G(7)),
           "q_w": (hd[:, :256].T @ dvd, G(8)), "q_b": (dvd.sum().reshape(1), G(9)),
           "l4_w": (a2d.T @ dhk[:, :256], G(4).reshape(2592, 256)), "l4_b": (dhk[:, :256].sum(0), G(5)),
           "la_w": (a2d.T @ dhk[:, 256:], G(10).reshape(2592, 256)), "la_b": (dhk[:, 256:].sum(0), G(11))}
    report = {}
    kr.check("d_h", dh_dev, dhr, (0,), REL_TOL, report)
    for k, (r, x) in ref.items():
        kr.check(k, x, r, (-1,), REL_TOL, report)
    d_a2r = (dhk @ torch.cat([w("l4_w"), w("la_w")], 1).T) * (a2d > 0)
    kr.check("d_a2", d_a2 / S, d_a2r, (0,), REL_TOL, report)
    kr.show("streams backward A=%d" % A, report)
    assert bool((G(10) != 0).any()) and bool((G(8) != 0).any())


# ---- Agent helpers -------------------------------------------------------------------------------
def _agent(pkg, cuda, mode, B, T, A, over=None, pool=None, p_terminal=0.2, seed=3):
    cfg = pkg.config.get_config(dict({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": mode,
                                      "dueling": True, "dueling_streams": True}, **(over or {})))
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=seed, pool=pool or T + 3, device=cuda,
                                                         p_terminal=p_terminal), device=cuda)
    return pkg.Agent(cfg, env, device=cuda), env


# ---- 4. one cycle per learner --------------------------------------------------------------------
@pytest.mark.parametrize("mode,double", [(m, False) for m in MODES] + [("async_q", True), ("nstep_q", True)])
@pytest.mark.parametrize("A,B,T", [(6, 9, 4), (18, 5, 2)])
def test_cycle_vs_oracle(pkg, cuda, mode, double, A, B, T):
    agent, env = _agent(pkg, cuda, mode, B, T, A, over={"double_q": double})
    net = agent.network
    assert net.dueling and net.dueling_streams and net.double_q == double
    params = so.init_streams_params(A, seed=41, scale=2.0, bias_std=0.1)
    tparams = so.init_streams_params(A, seed=42, scale=2.0, bias_std=0.1)
    net.set_weights(params)
    agent.before_train()
    net.target_params.copy_(torch.as_tensor(so.flatten(tparams), device=cuda))
    agent.step = 100
    hist = agent.history
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
    agent.step -= 1
    masks = gpu_masks(net)
    q_roll = net.q.cpu().numpy().copy()
    agent.batch_update()
    torch.cuda.synchronize()
    acts = (net.sarsa_actions.cpu().numpy().reshape(T + 1, B) if mode == "sarsa"
            else agent.batch_action.cpu().numpy().copy())
    stacks = a3c.stacks_from_screens(np.stack(screens), T)
    scale = 1.0 / (T * B) if mode == "async_q" else 1.0 / B
    grads, aux = so.streams_gradients(mode, params, tparams, stacks, acts, np.stack(rews), np.stack(terms), 0.99,
                                      scale=scale, masks=masks, double_q=double)
    assert rel_err(q_roll, aux["q"]) <= REL_TOL
    assert rel_err((net.R if mode == "nstep_q" else net.target_q_t).cpu(), aux["target"]) <= REL_TOL
    errs = {k: rel_err(net.g[k].cpu(), grads[k]) for k in so.STREAMS_PARAM_NAMES}
    print("streams", mode, double, "grad rel-err", errs)
    assert max(errs.values()) <= REL_TOL, errs
    assert float(net.g["la_w"].abs().max()) > 0 and float(net.g["q_w"].abs().max()) > 0


# ---- 5. graph replay == eager loop ---------------------------------------------------------------
def _loop(pkg, cuda, mode, graphs, cycles, B=24, T=5, A=6, start_step=0, over=None, agent_env=None):
    random.seed(123)
    if agent_env is None:
        o = dict({"cuda_graphs": graphs, "ep_end_t": 30, "learn_start": 5,
                  "target_q_update_step": 3 * T * B}, **(over or {}))
        agent, env = _agent(pkg, cuda, mode, B, T, A, over=o, pool=T, p_terminal=0.1, seed=5)
        agent.step_op = start_step
        agent.network.set_weights(so.init_streams_params(A, seed=9, scale=2.0, bias_std=0.1))
        agent.before_train()
    else:
        agent, env = agent_env
    acts, snaps = [], []
    for _ in range(cycles):
        for _ in range(agent.t_max):
            a = agent.predict()
            acts.append(a.clone())
            scr, rew, term = env.act(a, is_training=True, fused=True)
            agent.observe(scr, rew, a, term)
            agent.step += 1
        n = agent.network
        snaps.append((n.params.clone(), n.rms.clone(), n.target_params.clone()))
    torch.cuda.synchronize()
    return agent, torch.stack(acts), snaps


@pytest.mark.parametrize("mode", ["nstep_q", "sarsa"])
def test_graph_replay_equals_eager_loop(pkg, cuda, mode):
    cycles = 9
    eager, acts_e, snaps_e = _loop(pkg, cuda, mode, False, cycles)
    graph, acts_g, snaps_g = _loop(pkg, cuda, mode, True, cycles)
    assert eager.graph_replays == 0 and graph.graph_replays > 0
    assert torch.equal(acts_e, acts_g)
    for (pe, re_, te), (pg, rg, tg) in zip(snaps_e, snaps_g):
        assert torch.equal(pe, pg) and torch.equal(re_, rg) and torch.equal(te, tg)
    la = slice(graph.network.offsets[10], graph.network.offsets[11])
    assert not torch.equal(snaps_g[8][0][la], snaps_g[0][0][la])      # la_w trained


def test_async_q_eager_cycles_train_both_streams(pkg, cuda):
    agent, _, snaps = _loop(pkg, cuda, "async_q", False, 3, over={"double_q": True})
    off = agent.network.offsets
    for i in (4, 8, 10):
        assert not torch.equal(snaps[-1][0][off[i]:off[i + 1]], snaps[0][0][off[i]:off[i + 1]])
    assert bool(torch.isfinite(agent.network.params).all())


# ---- 6. full size --------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
def test_full_size_is_finite_and_deterministic(pkg, cuda, mode):
    B, T, A = 4096, 5, 6
    runs = []
    for _ in range(2):
        agent, acts, snaps = _loop(pkg, cuda, mode, mode != "async_q", 3, B=B, T=T, A=A, start_step=1000,
                                   over={"ep_end_t": 400 * 10000, "learn_start": 32,
                                         "target_q_update_step": 2 * T * B})
        g = agent.network.grads.clone()
        assert bool(torch.isfinite(g).all()) and float(agent.network.g["la_w"].abs().max()) > 0
        runs.append((acts, g, snaps[-1]))
        del agent
        torch.cuda.empty_cache()
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for x, y in zip(runs[0][2], runs[1][2]):
        assert torch.equal(x, y)


# ---- 7. checkpoints and refusals -----------------------------------------------------------------
def test_checkpoint_round_trip_and_cross_kind_refusal(pkg, cuda, tmp_path):
    B, T, A = 8, 2, 6
    streams, _ = _agent(pkg, cuda, "nstep_q", B, T, A)
    streams.network.set_weights(so.init_streams_params(A, seed=2, scale=2.0, bias_std=0.1))
    cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": "nstep_q", "dueling": True})
    shared = pkg.Agent(cfg, streams.env, device=cuda)
    s_dir, d_dir = tmp_path / "streams", tmp_path / "shared"
    z_s = np.load(streams.save_checkpoint(str(s_dir)))
    z_d = np.load(shared.save_checkpoint(str(d_dir)))
    assert bool(z_s["dueling_streams"]) and "dueling_streams" not in z_d.files and "la_w" in z_s.files
    twin, _ = _agent(pkg, cuda, "nstep_q", B, T, A)
    assert twin.load_checkpoint(str(s_dir))
    assert torch.equal(twin.network.params, streams.network.params)
    before = shared.network.params.clone()
    with pytest.raises(ValueError, match="dueling_streams"):
        shared.load_checkpoint(str(s_dir))
    assert torch.equal(shared.network.params, before)
    with pytest.raises(ValueError, match="non-dueling_streams"):
        twin.load_checkpoint(str(d_dir))


def test_refusals(pkg, cuda):
    def make(mode, kind="nips", dueling=True):
        cfg = pkg.config.get_config({"model": "m1", "num_envs": 4, "t_max": 2, "loss_mode": mode,
                                     "dueling": dueling, "dueling_streams": True, "DQN_type": kind})
        env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(4, 6, seed=1, pool=4, device=cuda), device=cuda)
        return pkg.Agent(cfg, env, device=cuda)
    for mode in MODES:
        with pytest.raises(ValueError, match="dueling=True"):
            make(mode, dueling=False)
        with pytest.raises(NotImplementedError, match="nips"):
            make(mode, "nature")
    with pytest.raises(ValueError, match="a3c"):
        make("a3c")
    with pytest.raises(ValueError, match="dueling=True"):
        pkg.Network(action_size=6, num_envs=4, t_max=2, device=cuda, dueling_streams=True)


# ---- 8. N ranks ----------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["nstep_q", "sarsa"])
def test_multi_gpu_run_equals_single_gpu_union_batch(cuda, mode):
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
           os.path.join(root, "tests", "dist_gpu_check_dueling_streams.py"), "--mode", mode]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["ok"] and line["actions_bit_identical"] and line["replica_max_minus_min"] == 0.0
