"""GPU: dueling Q heads (dueling=True, Wang et al. 2016) on the async-Q, n-step Q and Sarsa learners:
the forward and its fused epsilon-greedy draw against arl_forward / arl_egreedy_actions and the
float64 reference, the three loss entries against their plain entries, one cycle per learner against
the reference, graph replay against the eager loop, determinism, checkpoints, play, refusals and
N ranks."""
import json
import os
import random
import socket
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from dueling_oracle import dueling_gradients, q_forward
from oracle import a3c
from test_gpu_network import gpu_masks, make_params, ring_stacks
from util import REL_TOL, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = ("async_q", "nstep_q", "sarsa")


# ---- 1. the forward ------------------------------------------------------------------------------
class Fwd:
    """Device buffers of a forward of B envs x ``steps`` from a random ring, under random parameters."""

    def __init__(self, pkg, cuda, B, A, steps=1, seed=0):
        g = torch.Generator(device=cuda).manual_seed(seed)
        self.pkg, self.B, self.A, self.steps = pkg, B, A, steps
        self.slots = steps + 3
        self.ring = torch.randint(0, 256, (B, self.slots, 84 * 84), dtype=torch.uint8, device=cuda, generator=g)
        self.params_np = make_params(A, seed=seed + 31, scale=2.0, bias_std=0.3)
        self.params = torch.as_tensor(a3c.flatten_params(self.params_np), device=cuda)
        f32 = dict(device=cuda, dtype=torch.float32)
        N = B * steps
        self.prep = torch.empty(pkg._cabi.prepared_floats(), **f32)
        self.l1, self.l2, self.l4 = (torch.empty(N, n, **f32) for n in (3200, 2592, 256))
        self.cuda = cuda

    def run(self, entry, actions=None, env_id_base=0, step=0, step_dev=None, seed=0, ep=0.0,
            sched=(0.0, 0.0, 1.0, 0.0)):
        P, N, A = self.pkg._cabi.ptr, self.B * self.steps, self.A
        f32 = dict(device=self.cuda, dtype=torch.float32)
        logits, probs, value = torch.empty(N, A, **f32), torch.empty(N, A, **f32), torch.empty(N, **f32)
        head = (P(self.params), P(self.prep), 1, A, P(self.ring), self.B, self.slots, 0, self.steps, P(self.l1),
                P(self.l2), P(self.l4), P(logits), P(probs), P(value))
        if entry == "arl_forward":
            self.pkg._cabi.call(entry, *head, self.pkg._cabi.stream_ptr())
        else:
            self.pkg._cabi.call(entry, *head, P(actions), int(env_id_base), int(step), P(step_dev), int(seed),
                                float(ep), *sched, self.pkg._cabi.stream_ptr())
        torch.cuda.synchronize()
        return logits, probs, value


@pytest.mark.parametrize("B,A,steps", [(4096, 6, 1), (18432, 18, 1), (512, 6, 3)])
def test_forward_is_the_dueling_combine(pkg, cuda, B, A, steps):
    """18 432 envs take two env ranges (arl_a2_block_rows); steps 3 is the target forward's form."""
    f = Fwd(pkg, cuda, B, A, steps, seed=B + A)
    logits, probs, value = f.run("arl_forward")
    q, qprobs, v = f.run("arl_forward_dueling")
    assert torch.equal(v, value)                                      # the value head: the same bits
    ref = value[:, None] + (logits - logits.mean(dim=1, keepdim=True))
    ulp = torch.finfo(torch.float32).eps * (value.abs() + logits.abs().max(dim=1).values)[:, None]
    assert bool(((q - ref).abs() <= 4 * ulp).all()), float(((q - ref).abs() / ulp).max())
    assert not torch.equal(q, logits)
    assert float((qprobs - torch.softmax(q, dim=1)).abs().max()) <= 1e-6
    # the float64 reference on the first and last 128 envs of every step (both env ranges)
    ring = f.ring.cpu().numpy().reshape(B, f.slots, 84, 84)
    envs = np.r_[0:128, B - 128:B]
    stacks = ring_stacks(ring[envs], 0, steps)
    ref64 = q_forward(a3c.to_torch(f.params_np), stacks).numpy()
    rows = np.concatenate([t * B + envs for t in range(steps)])
    assert rel_err(q.cpu().numpy()[rows], ref64) <= REL_TOL


@pytest.mark.parametrize("B", [4096, 18432])
def test_fused_draw_equals_egreedy_actions_on_the_written_q(pkg, cuda, B):
    A, seed, base, step = 6, 77, 1000, (1 << 33) + 5
    f = Fwd(pkg, cuda, B, A, 1, seed=B)
    P, st = pkg._cabi.ptr, pkg._cabi.stream_ptr()
    acts = torch.empty(B, dtype=torch.int32, device=cuda)
    ref = torch.empty(B, dtype=torch.int32, device=cuda)
    q0, _, _ = f.run("arl_forward_dueling")
    for ep in (0.0, 0.3, 1.0):
        q, _, _ = f.run("arl_forward_dueling", acts, base, step, None, seed, ep)
        assert torch.equal(q, q0)
        pkg._cabi.call("arl_egreedy_actions", P(q), P(ref), B, A, ep, base, step, seed, st)
        torch.cuda.synchronize()
        assert torch.equal(acts, ref), ep
        if ep == 0.0:
            assert torch.equal(acts.long(), q.argmax(dim=1))
    # the step_dev form: step = 40 + *step_dev, epsilon from the schedule on the device
    sched = (1.0, 0.1, 100.0, 32.0)
    step_dev = torch.tensor([60], dtype=torch.int64, device=cuda)
    q, _, _ = f.run("arl_forward_dueling", acts, base, 40, step_dev, seed, 0.0, sched)
    host = SimpleNamespace(ep_start=1.0, ep_end=0.1, ep_end_t=100.0, learn_start=32.0, step=100)
    ep = pkg.Agent.ep.fget(host)
    pkg._cabi.call("arl_egreedy_actions", P(q), P(ref), B, A, ep, base, 100, seed, st)
    torch.cuda.synchronize()
    assert torch.equal(acts, ref)
    with pytest.raises(pkg._cabi.ArlError, match="steps == 1"):
        Fwd(pkg, cuda, 8, A, 2).run("arl_forward_dueling", torch.empty(16, dtype=torch.int32, device=cuda))


# ---- 2. the loss entries -------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("A,T,B", [(6, 5, 257), (18, 20, 33)])
def test_loss_entry_against_its_plain_entry(pkg, cuda, mode, A, T, B):
    rng = np.random.default_rng(A * T * B)
    N = T * B
    d = lambda x: torch.as_tensor(x, device=cuda)
    q = d(rng.normal(0, 1, (N, A)).astype(np.float32))
    q_next = d(rng.normal(0, 1, (B if mode == "nstep_q" else N, A)).astype(np.float32))
    rew = d(rng.choice([-3.0, -1.0, 0.0, 0.5, 1.0, 2.0], (T, B)).astype(np.float32))
    term = d((rng.random((T, B)) < 0.3).astype(np.uint8))
    act = d(rng.integers(0, A, N + B).astype(np.int32))
    P, st, scale = pkg._cabi.ptr, pkg._cabi.stream_ptr(), 1.0 / B
    size = (N,) if mode == "async_q" else (T, B)
    name = {"async_q": "arl_q_lossgrad", "nstep_q": "arl_nstep_q_lossgrad", "sarsa": "arl_sarsa_lossgrad"}[mode]

    def call(dueling):
        y, dq, sums = torch.empty(N, device=cuda), torch.full((N, A), 7.0, device=cuda), torch.zeros(2, device=cuda)
        dv = torch.full((N,), 7.0, device=cuda)
        head = (P(rew), P(term), P(act), P(q), P(q_next), P(y), P(dq)) + ((P(dv),) if dueling else ())
        pkg._cabi.call(name + ("_dueling" if dueling else ""), *head, P(sums), *size, A, 0.99, -1.0, 1.0, scale, st)
        torch.cuda.synchronize()
        return y, dq, dv, sums

    y0, dq0, _, s0 = call(False)
    y1, dq1, dv1, s1 = call(True)
    a = act[:N].long()
    assert torch.equal(y1, y0)                                        # targets / returns: the same bits
    assert torch.equal(dv1, dq0[torch.arange(N, device=cuda), a])     # d value = the plain dQ[a]
    onehot = torch.nn.functional.one_hot(a, A).float()
    assert torch.equal(dq1, dv1[:, None] * (onehot - torch.tensor(1.0, device=cuda) / A))
    r = s0.double().cpu()
    assert abs(float(s1[0] - s0[0])) <= 1e-5 * float(r[0])
    assert abs(float(s1[1] - s0[1])) <= 1e-5 * float(q.gather(1, a[:, None]).abs().sum())
    with pytest.raises(pkg._cabi.ArlError, match="null pointer"):
        pkg._cabi.call(name + "_dueling", P(rew), P(term), P(act), P(q), P(q_next), P(y0), P(dq1), None, None,
                       *size, A, 0.99, -1.0, 1.0, scale, st)


# ---- Agent helpers -------------------------------------------------------------------------------
def _agent(pkg, cuda, mode, B, T, A, over=None, pool=None, p_terminal=0.2, seed=3):
    cfg = pkg.config.get_config(dict({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": mode,
                                      "dueling": True}, **(over or {})))
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=seed, pool=pool or T + 3, device=cuda,
                                                         p_terminal=p_terminal), device=cuda)
    return pkg.Agent(cfg, env, device=cuda), env


# ---- 3. one cycle per learner --------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("A,B,T", [(6, 9, 4), (18, 5, 2)])
def test_cycle_vs_oracle(pkg, cuda, mode, A, B, T):
    agent, env = _agent(pkg, cuda, mode, B, T, A)
    net = agent.network
    assert net.dueling
    params, tparams = make_params(A, seed=41, scale=2.0, bias_std=0.1), make_params(A, seed=42, scale=2.0, bias_std=0.1)
    net.set_weights(params)
    agent.before_train()                                        # syncs the target (main.py:92) ...
    net.target_params.copy_(torch.as_tensor(a3c.flatten_params(tparams), device=cuda))  # ... then differ
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
    grads, aux = dueling_gradients(mode, params, tparams, stacks, acts, np.stack(rews), np.stack(terms), 0.99,
                                   scale=scale, masks=masks)
    assert rel_err(q_roll, aux["q"]) <= REL_TOL
    assert rel_err((net.q_boot if mode == "nstep_q" else net.target_q).cpu(), aux["q_next"]) <= REL_TOL
    assert rel_err((net.R if mode == "nstep_q" else net.target_q_t).cpu(), aux["target"]) <= REL_TOL
    errs = {k: rel_err(net.g[k].cpu(), grads[k]) for k in a3c.PARAM_NAMES}
    print("dueling", mode, "grad rel-err", errs)
    assert max(errs.values()) <= REL_TOL, errs
    assert float(net.g["q_w"].abs().max()) > 0 and float(net.g["q_b"].abs().max()) > 0


# ---- 4. graph replay == eager loop ---------------------------------------------------------------
def _loop(pkg, cuda, mode, graphs, cycles, B=24, T=5, A=6, start_step=0, over=None, agent_env=None):
    random.seed(123)
    if agent_env is None:
        o = dict({"cuda_graphs": graphs, "ep_end_t": 30, "learn_start": 5,
                  "target_q_update_step": 3 * T * B}, **(over or {}))
        agent, env = _agent(pkg, cuda, mode, B, T, A, over=o, pool=T, p_terminal=0.1, seed=5)
        agent.step_op = start_step
        agent.network.set_weights(make_params(A, seed=9, scale=2.0, bias_std=0.1))
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
    cycles = 9                                                   # 2 eager, then capture / replay
    eager, acts_e, snaps_e = _loop(pkg, cuda, mode, False, cycles)
    graph, acts_g, snaps_g = _loop(pkg, cuda, mode, True, cycles)
    assert eager.graph_replays == 0 and graph.graph_replays > 0
    assert torch.equal(acts_e, acts_g)
    for (pe, re_, te), (pg, rg, tg) in zip(snaps_e, snaps_g):
        assert torch.equal(pe, pg) and torch.equal(re_, rg) and torch.equal(te, tg)
    assert not torch.equal(snaps_g[5][2], snaps_g[8][2])           # a target sync inside the replayed cycles
    assert torch.equal(snaps_g[8][2], snaps_g[8][0])
    assert not torch.equal(snaps_g[8][0][-257:], snaps_g[0][0][-257:])   # q_w / q_b (the last 257) trained


# ---- 5. full size --------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
def test_full_size_is_finite_and_deterministic(pkg, cuda, mode):
    B, T, A = 4096, 5, 6
    runs = []
    for _ in range(2):
        agent, acts, snaps = _loop(pkg, cuda, mode, True, 4, B=B, T=T, A=A, start_step=1000,
                                   over={"ep_end_t": 400 * 10000, "learn_start": 32,
                                         "target_q_update_step": 2 * T * B})
        g = agent.network.grads.clone()
        assert bool(torch.isfinite(g).all()) and float(agent.network.g["q_w"].abs().max()) > 0
        assert bool(torch.isfinite(agent.network.params).all())
        runs.append((acts, g, snaps[-1]))
        del agent
        torch.cuda.empty_cache()
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for x, y in zip(runs[0][2], runs[1][2]):
        assert torch.equal(x, y)


# ---- 6. checkpoints ------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["nstep_q", "sarsa"])
def test_checkpoint_resume_equals_uninterrupted_run(pkg, cuda, tmp_path, mode):
    B, T, A = 12, 5, 6
    over = {"ep_end_t": 200, "learn_start": 5, "target_q_update_step": 3 * T * B}
    full, acts_f, _ = _loop(pkg, cuda, mode, True, 4, B=B, T=T, A=A, over=over)
    full.step_op = full.step
    full.save_checkpoint(str(tmp_path))
    _, acts_f2, snaps_f = _loop(pkg, cuda, mode, True, 4, agent_env=(full, full.env))
    twin, acts_t, _ = _loop(pkg, cuda, mode, True, 4, B=B, T=T, A=A, over=over)
    assert torch.equal(acts_t, acts_f)
    cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": mode, "dueling": True,
                                 **over})
    resumed = pkg.Agent(cfg, twin.env, device=cuda)
    assert resumed.load_checkpoint(str(tmp_path)) and resumed.step_op == full.step_op
    if mode == "sarsa":
        assert resumed.sarsa_pending
    resumed.step, resumed.T = resumed.step_op, resumed.step_op * resumed.global_envs
    resumed.history.ring.copy_(twin.history.ring)
    resumed.history.head = twin.history.head
    _, acts_r, snaps_r = _loop(pkg, cuda, mode, True, 4, agent_env=(resumed, twin.env))
    assert torch.equal(acts_r, acts_f2)
    for (pf, rf, tf), (pr, rr, tr) in zip(snaps_f, snaps_r):
        assert torch.equal(pf, pr) and torch.equal(rf, rr) and torch.equal(tf, tr)


def test_mismatched_checkpoint_load_raises(pkg, cuda, tmp_path):
    B, T, A = 8, 2, 6
    duel, _ = _agent(pkg, cuda, "nstep_q", B, T, A)
    plain_cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": "nstep_q"})
    plain = pkg.Agent(plain_cfg, duel.env, device=cuda)
    d_dir, p_dir = tmp_path / "dueling", tmp_path / "plain"
    z_d = np.load(duel.save_checkpoint(str(d_dir)))
    z_p = np.load(plain.save_checkpoint(str(p_dir)))
    assert bool(z_d["dueling"]) and "dueling" not in z_p.files      # non-dueling files are unchanged
    before = plain.network.params.clone()
    with pytest.raises(ValueError, match="dueling"):
        plain.load_checkpoint(str(d_dir))
    assert torch.equal(plain.network.params, before)                  # nothing was loaded
    with pytest.raises(ValueError, match="non-dueling"):
        duel.load_checkpoint(str(p_dir))
    assert duel.load_checkpoint(str(d_dir)) and plain.load_checkpoint(str(p_dir))


# ---- 7. play, statistics, refusals ---------------------------------------------------------------
def test_play_and_statistics_use_dueling_q(pkg, cuda, tmp_path):
    B, T, A = 12, 5, 6
    random.seed(123)
    agent, env = _agent(pkg, cuda, "sarsa", B, T, A, over={"_test_step": 10}, pool=64, p_terminal=0.1, seed=9)
    agent.network.set_weights(make_params(A, seed=4, scale=2.0, bias_std=0.3))
    recs = agent.train_with_summary(num_steps=20, log_path=str(tmp_path / "stats.jsonl"))
    assert len(recs) == 2 and all(np.isfinite(r["average.q"]) and r["average.loss"] > 0 for r in recs)
    net, hist = agent.network, agent.history
    a = net.evaluate(hist, 3, 5, ep=0.0)
    torch.cuda.synchronize()
    q = net._b["logits"].clone()
    f32 = dict(device=cuda, dtype=torch.float32)
    out = [torch.empty(B, n, **f32) for n in (3200, 2592, 256, A, A)] + [torch.empty(B, **f32)]
    P = pkg._cabi.ptr
    pkg._cabi.call("arl_forward", P(net.params), P(torch.empty_like(net.fc_w)), 1, A, P(hist.ring), B,
                   hist.ring_slots, hist.first_slot(0), 1, *[P(x) for x in out], pkg._cabi.stream_ptr())
    torch.cuda.synchronize()
    logits, value = out[3], out[5]
    assert torch.equal(net._b["value"], value) and not torch.equal(q, logits)
    assert float((q - (value[:, None] + logits - logits.mean(1, keepdim=True))).abs().max()) <= 1e-5 * float(q.abs().max())
    assert torch.equal(a.long(), q.argmax(dim=1))                     # greedy on the dueling Q
    best, _, means = agent.play(n_step=3, n_episode=1)
    assert np.isfinite(best) and len(means) == 1


def test_refusals(pkg, cuda):
    def make(mode, kind):
        cfg = pkg.config.get_config({"model": "m1", "num_envs": 4, "t_max": 2, "loss_mode": mode, "dueling": True,
                                     "DQN_type": kind})
        env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(4, 6, seed=1, pool=4, device=cuda), device=cuda)
        return pkg.Agent(cfg, env, device=cuda)
    with pytest.raises(ValueError, match="a3c"):
        make("a3c", "nips")
    with pytest.raises(ValueError, match="a3c"):
        make("a3c", "nature")
    for mode in MODES:
        with pytest.raises(NotImplementedError, match="nature|nips"):
            make(mode, "nature")
    # a dueling Network driven on the A3C path directly: its policy/value entry points refuse
    net = pkg.Network(action_size=6, num_envs=4, t_max=2, device=cuda, dueling=True)
    agent = make("nstep_q", "nips")
    hist, z = agent.history, torch.zeros(2, 4, device=cuda)
    with pytest.raises(ValueError, match="forward_sample"):
        net.forward_sample(hist, 0, 0, 1)
    with pytest.raises(ValueError, match="bootstrap_value"):
        net.bootstrap_value(hist)
    with pytest.raises(ValueError, match="compute_gradients"):
        net.compute_gradients(hist, z, z.to(torch.uint8), z[0])


# ---- 8. N ranks ----------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["nstep_q", "sarsa"])
def test_multi_gpu_run_equals_single_gpu_union_batch(cuda, mode):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (one rank per GPU)")
    world = 2 if n < 4 else 4
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "dist_gpu_check_dueling.py"), "--mode", mode]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["ok"] and line["actions_bit_identical"] and line["replica_max_minus_min"] == 0.0
