"""GPU: loss_mode 'nstep_q' -- asynchronous n-step Q-learning (Mnih et al. 2016) on the A3C cycle:
the loss kernel and the fused epsilon-greedy draw through the C-ABI, one Agent cycle against the
float64 reference, graph replay against the eager loop, checkpoints, statistics and N ranks."""
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

from nstep_q_oracle import nstep_q_gradients
from oracle import a3c, philox
from test_gpu_network import gpu_masks, make_params
from util import REL_TOL, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def host_ep(pkg, cfg, step):
    """Agent.ep (agent.py:142-144) for ``cfg`` at ``step``, as the host computes it."""
    return pkg.Agent.ep.fget(SimpleNamespace(ep_start=cfg.ep_start, ep_end=cfg.ep_end, ep_end_t=cfg.ep_end_t,
                                             learn_start=cfg.learn_start, step=step))


# ---- 1. the loss kernel --------------------------------------------------------------------------
@pytest.mark.parametrize("T,B", [(5, 257), (20, 33), (1, 1000)])
@pytest.mark.parametrize("A", [4, 6, 18])
def test_nstep_q_lossgrad_vs_oracle(pkg, cuda, A, T, B):
    rng = np.random.default_rng(A * 1000 + T * B)
    N = T * B
    q = rng.normal(0, 1, (N, A)).astype(np.float32)
    q_boot = rng.normal(0, 1, (B, A)).astype(np.float32)
    rew = rng.choice([-3.0, -1.0, 0.0, 0.5, 1.0, 2.0], (T, B)).astype(np.float32)
    term = rng.random((T, B)) < 0.3
    act = rng.integers(0, A, N).astype(np.int32)
    d = lambda x: torch.as_tensor(x, device=cuda)
    ins = [d(rew), d(term.astype(np.uint8)), d(act), d(q), d(q_boot)]
    R, dq, sums = torch.empty(N, device=cuda), torch.empty(N, A, device=cuda), torch.zeros(2, device=cuda)
    scale, P, st = 1.0 / B, pkg._cabi.ptr, pkg._cabi.stream_ptr()
    pkg._cabi.call("arl_nstep_q_lossgrad", *[P(x) for x in ins], P(R), P(dq), P(sums), T, B, A, 0.99, -1.0, 1.0,
                   scale, st)
    # the A3C returns kernel fed v_boot = max_a q_boot: the same recurrence, the same bits
    R3, dl, dv, s3 = (torch.empty(N, device=cuda), torch.empty(N, A, device=cuda), torch.empty(N, device=cuda),
                      torch.zeros(3, device=cuda))
    v_boot = ins[4].max(dim=1).values.contiguous()
    pkg._cabi.call("arl_returns_lossgrad", P(ins[0]), P(ins[1]), P(ins[2]), P(ins[3]), P(torch.zeros(N, device=cuda)),
                   P(v_boot), P(R3), P(dl), P(dv), P(s3), T, B, A, 0.99, 0.01, -1.0, 1.0, 1.0, st)
    torch.cuda.synchronize()
    assert torch.equal(R, R3)
    ref_R = a3c.nstep_returns(a3c.clip_rewards(rew), term, q_boot.astype(np.float64).max(axis=1), 0.99).reshape(-1)
    assert rel_err(R.cpu(), ref_R) <= 1e-6
    delta = ref_R - q[np.arange(N), act].astype(np.float64)
    ref_dq = np.zeros((N, A))
    ref_dq[np.arange(N), act] = -2.0 * delta * scale
    assert rel_err(dq.cpu(), ref_dq) <= 1e-6
    ref_sums = np.array([(delta ** 2).sum(), q[np.arange(N), act].astype(np.float64).sum()])
    assert abs(float(sums[0]) - ref_sums[0]) <= 1e-4 * abs(ref_sums[0])
    assert abs(float(sums[1]) - ref_sums[1]) <= 1e-4 * np.abs(q[np.arange(N), act]).sum()
    # zero-size calls do nothing
    pkg._cabi.call("arl_nstep_q_lossgrad", *[P(x) for x in ins], P(R), P(dq), P(sums), 0, B, A, 0.99, -1.0, 1.0,
                   scale, st)
    pkg._cabi.call("arl_nstep_q_lossgrad", *[P(x) for x in ins], P(R), P(dq), P(sums), T, 0, A, 0.99, -1.0, 1.0,
                   scale, st)
    with pytest.raises(pkg._cabi.ArlError, match="action_size"):
        pkg._cabi.call("arl_nstep_q_lossgrad", *[P(x) for x in ins], P(R), P(dq), P(sums), T, B, 0, 0.99, -1.0,
                       1.0, scale, st)


# ---- 2. the fused draw ---------------------------------------------------------------------------
@pytest.mark.parametrize("B", [4096, 20480])
def test_fused_egreedy_draw_bit_exact(pkg, cuda, B):
    """Actions of arl_forward_egreedy == arl_egreedy_actions on the logits the same call wrote, with
    epsilon from the device counter (below learn_start, mid-anneal, past ep_end_t) and fixed."""
    A = 6
    cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": 1})
    net = pkg.Network(action_size=A, num_envs=B, t_max=1, device=cuda)
    net.set_weights(make_params(A, seed=4, scale=3.0))
    hist = pkg.History(cfg, num_envs=B, device=cuda)
    g = torch.Generator(device=cuda).manual_seed(B)
    hist.ring.copy_(torch.randint(0, 256, tuple(hist.ring.shape), dtype=torch.uint8, device=cuda, generator=g))
    assert (pkg._cabi.a2_block_rows(B) < B) == (B > 16384)              # 20 480: two env ranges
    sched = (cfg.ep_start, cfg.ep_end, cfg.ep_end_t, cfg.learn_start)
    step_dev = torch.zeros(1, dtype=torch.int64, device=cuda)
    ref_act = torch.empty(B, dtype=torch.int32, device=cuda)
    base, seed = 4096, 123
    steps = [10, cfg.learn_start + 1234567, cfg.ep_end_t + cfg.learn_start + 99]
    cases = [(s, None) for s in steps] + [(777, 0.0), (778, 1.0)]
    for step, ep in cases:
        if ep is None:
            step_dev.fill_(step - 5)
            act = net.forward_egreedy(hist, 0, seed, base, step_dev=step_dev, ep_sched=sched, step=5).clone()
            ep = host_ep(pkg, cfg, step)
        else:
            act = net.forward_egreedy(hist, 0, seed, base, step=step, ep=ep).clone()
        pkg._cabi.call("arl_egreedy_actions", pkg._cabi.ptr(net.policy_logits), pkg._cabi.ptr(ref_act), B, A,
                       float(ep), base, step, seed, pkg._cabi.stream_ptr())
        torch.cuda.synchronize()
        assert torch.equal(act, ref_act), (step, ep)
        q = net.policy_logits.cpu().numpy()
        if ep == 0.0:
            assert np.array_equal(act.cpu().numpy(), q.argmax(1))
        elif ep == 1.0:
            ref = philox.egreedy_actions(q, np.arange(base, base + B), step, seed, 1.0)
            assert np.array_equal(act.cpu().numpy(), ref)
            counts = np.bincount(act.cpu().numpy(), minlength=A)
            assert counts.min() > 0.8 * B / A and counts.max() < 1.2 * B / A   # uniform
        else:
            greedy = float((act.cpu().numpy() == q.argmax(1)).mean())
            assert abs((1.0 - greedy) - ep * (A - 1) / A) < 0.05, (step, ep, greedy)


# ---- 3. one Agent cycle --------------------------------------------------------------------------
def _agent(pkg, cuda, B, T, A, over=None, pool=None, p_terminal=0.2, seed=3, env_seed=None):
    cfg = pkg.config.get_config(dict({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": "nstep_q"},
                                     **(over or {})))
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=seed if env_seed is None else env_seed,
                                                         pool=pool or T + 3, device=cuda, p_terminal=p_terminal),
                             device=cuda)
    return pkg.Agent(cfg, env, device=cuda), env


@pytest.mark.parametrize("A,B,T", [(6, 9, 4), (18, 5, 2)])
def test_nstep_q_cycle_vs_oracle(pkg, cuda, A, B, T):
    agent, env = _agent(pkg, cuda, B, T, A)
    net = agent.network
    assert agent.cuda_graphs and not hasattr(net, "target_q")       # no [T*B] target buffers
    params, tparams = make_params(A, seed=31, scale=2.0), make_params(A, seed=32, scale=2.0)
    net.set_weights(params)
    agent.before_train()                                        # syncs the target (main.py:92) ...
    net.target_params.copy_(torch.as_tensor(a3c.flatten_params(tparams), device=cuda))  # ... then differ
    agent.step = 100                                            # inside the anneal
    hist = agent.history
    first = hist.first_slot(0)
    snap = hist.planes().cpu().numpy()
    screens = [snap[:, (first + k) % hist.ring_slots] for k in range(4)]
    rews, terms = [], []
    for t in range(T):
        action = agent.predict()
        ref_a = philox.egreedy_actions(net.q[t * B:(t + 1) * B].cpu().numpy(), np.arange(B), agent.step,
                                       agent.seed, agent.ep)
        assert np.array_equal(action.cpu().numpy(), ref_a)
        scr, rew, term = env.act(action, is_training=True, fused=True)
        hist.add(scr)
        agent.batch_reward[t].copy_(rew)
        agent.batch_terminal[t].copy_(term)
        rews.append(rew.cpu().numpy()); terms.append(term.cpu().numpy())
        screens.append(hist.planes(hist.head).cpu().numpy())
        agent.t += 1
        agent.step += 1
    agent.step -= 1
    acts = agent.batch_action.cpu().numpy().copy()
    masks = gpu_masks(net)
    agent.batch_update()
    torch.cuda.synchronize()
    stacks = a3c.stacks_from_screens(np.stack(screens), T)
    grads, aux = nstep_q_gradients(params, tparams, stacks, acts, np.stack(rews), np.stack(terms), 0.99,
                                   scale=1.0 / B, masks=masks)
    assert rel_err(net.q_boot.cpu(), aux["q_boot"]) <= REL_TOL
    assert rel_err(net.R.cpu(), aux["R"].reshape(-1)) <= REL_TOL
    errs = {k: rel_err(net.g[k].cpu(), grads[k]) for k in a3c.PARAM_NAMES if k not in ("q_w", "q_b")}
    print("n-step Q grad rel-err", errs)
    assert max(errs.values()) <= REL_TOL, errs
    assert float(net.g["q_w"].abs().max()) == 0.0 and float(net.g["q_b"].abs().max()) == 0.0
    rms = {k: np.ones_like(v) for k, v in params.items()}
    new_p, _ = a3c.update(params, rms, grads, a3c.learning_rate(agent.step - (T - 1)))
    perr = {k: rel_err(net.w[k].cpu(), new_p[k]) for k in a3c.PARAM_NAMES}
    assert max(perr.values()) <= REL_TOL, perr
    assert rel_err(net.target_params.cpu(), a3c.flatten_params(tparams)) == 0.0   # untouched until the sync
    agent.update_target_q_network()
    assert bool((net.target_params == net.params).all())


def test_nature_trunk_refuses_nstep_q(pkg, cuda):
    cfg = pkg.config.get_config({"model": "m1", "num_envs": 4, "t_max": 2, "loss_mode": "nstep_q",
                                 "DQN_type": "nature"})
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(4, 6, seed=1, pool=4, device=cuda), device=cuda)
    with pytest.raises(NotImplementedError, match="nstep_q"):
        pkg.Agent(cfg, env, device=cuda)


# ---- 4. graph replay == eager loop ---------------------------------------------------------------
def _loop(pkg, cuda, graphs, cycles, B=24, T=5, A=6, start_step=0, over=None, agent_env=None):
    random.seed(123)
    if agent_env is None:
        o = dict({"cuda_graphs": graphs, "ep_end_t": 30, "learn_start": 5,
                  "target_q_update_step": 3 * T * B}, **(over or {}))
        agent, env = _agent(pkg, cuda, B, T, A, over=o, pool=T, p_terminal=0.1, seed=5)
        agent.step_op = start_step
        agent.network.set_weights(make_params(A, seed=9, scale=2.0))
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


def test_graph_replay_equals_eager_loop(pkg, cuda):
    cycles = 9                                                   # 2 eager, then capture / replay
    eager, acts_e, snaps_e = _loop(pkg, cuda, False, cycles)
    graph, acts_g, snaps_g = _loop(pkg, cuda, True, cycles)
    assert eager.graph_replays == 0 and not eager._graphs
    assert graph.graph_replays > 0
    assert len(graph._graphs) <= 2 * 2 * 2 * 5 * 2, len(graph._graphs)
    assert torch.equal(acts_e, acts_g)
    for (pe, re_, te), (pg, rg, tg) in zip(snaps_e, snaps_g):
        assert torch.equal(pe, pg) and torch.equal(re_, rg) and torch.equal(te, tg)
    # target syncs every 3 cycles: the target moved inside the replayed cycles and equals the
    # parameters right after a sync
    assert not torch.equal(snaps_g[5][2], snaps_g[8][2])
    assert torch.equal(snaps_g[8][2], snaps_g[8][0]) and not torch.equal(snaps_g[7][2], snaps_g[7][0])
    # epsilon annealed from 1 to 0.1 inside the run (steps 5..35 of 45)
    assert graph.ep < 0.2 and eager.update_count == cycles and graph.step_dev.item() == graph.step


# ---- 5. full size --------------------------------------------------------------------------------
@pytest.mark.parametrize("B,T,A", [(4096, 5, 6), (4096, 20, 18)])
def test_full_size_is_finite_and_deterministic(pkg, cuda, B, T, A):
    runs = []
    for _ in range(2):
        agent, acts, snaps = _loop(pkg, cuda, True, 4, B=B, T=T, A=A, start_step=1000,
                                   over={"ep_end_t": 400 * 10000, "learn_start": 32,
                                         "target_q_update_step": 2 * T * B})
        g = agent.network.grads.clone()
        assert bool(torch.isfinite(g).all()) and float(g.abs().max()) > 0
        assert bool(torch.isfinite(agent.network.params).all())
        runs.append((acts, g, snaps[-1]))
        del agent
        torch.cuda.empty_cache()
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for x, y in zip(runs[0][2], runs[1][2]):
        assert torch.equal(x, y)


# ---- 6. checkpoint -------------------------------------------------------------------------------
def test_checkpoint_resume_equals_uninterrupted_run(pkg, cuda, tmp_path):
    """Save after 4 cycles, load into a fresh Agent (target and sync schedule included), continue 4
    cycles: the same actions, parameters, RMSProp slot and target as the run that never stopped.
    The environment side (emulator, frame history) is carried over from a twin run."""
    B, T, A = 12, 5, 6
    over = {"ep_end_t": 200, "learn_start": 5, "target_q_update_step": 3 * T * B}
    full, acts_f, _ = _loop(pkg, cuda, True, 4, B=B, T=T, A=A, over=over)
    full.step_op = full.step
    full.save_checkpoint(str(tmp_path))
    _, acts_f2, snaps_f = _loop(pkg, cuda, True, 4, agent_env=(full, full.env))
    twin, acts_t, _ = _loop(pkg, cuda, True, 4, B=B, T=T, A=A, over=over)   # the environment after 4 cycles
    assert torch.equal(acts_t, acts_f)
    cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": "nstep_q", **over})
    resumed = pkg.Agent(cfg, twin.env, device=cuda)
    assert resumed.load_checkpoint(str(tmp_path)) and resumed.step_op == full.step_op
    resumed.step, resumed.T = resumed.step_op, resumed.step_op * resumed.global_envs   # before_train's counters
    assert resumed._last_target_sync == twin._last_target_sync
    resumed.history.ring.copy_(twin.history.ring)
    resumed.history.head = twin.history.head
    _, acts_r, snaps_r = _loop(pkg, cuda, True, 4, agent_env=(resumed, twin.env))
    assert torch.equal(acts_r, acts_f2)
    for (pf, rf, tf), (pr, rr, tr) in zip(snaps_f, snaps_r):
        assert torch.equal(pf, pr) and torch.equal(rf, rr) and torch.equal(tf, tr)


# ---- 7. statistics -------------------------------------------------------------------------------
def test_train_with_summary_records(pkg, cuda, tmp_path):
    B, T, A = 12, 5, 6
    random.seed(123)
    agent, env = _agent(pkg, cuda, B, T, A, over={"_test_step": 10}, pool=64, p_terminal=0.1, seed=9)
    recs = agent.train_with_summary(num_steps=20, log_path=str(tmp_path / "stats.jsonl"))
    assert len(recs) == 2 and agent.update_count == 4
    for r in recs:
        assert np.isfinite(r["average.loss"]) and np.isfinite(r["average.q"]) and r["average.loss"] > 0
        assert sum(r["episode.actions"]) == 10 * B
    best, _, means = agent.play(n_step=3, n_episode=1)          # evaluation: epsilon-greedy with test_ep
    assert np.isfinite(best) and len(means) == 1


# ---- 8. N ranks ----------------------------------------------------------------------------------
def test_multi_gpu_run_equals_single_gpu_union_batch(cuda):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (one rank per GPU)")
    world = 2 if n < 4 else 4
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "dist_gpu_check_nstep_q.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["ok"] and line["actions_bit_identical"] and line["replica_max_minus_min"] == 0.0
