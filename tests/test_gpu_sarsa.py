"""GPU: loss_mode 'sarsa' -- asynchronous one-step Sarsa (Mnih et al. 2016) on the graph-replayed
cycle: the loss kernel through the C-ABI, the action a_T drawn at the update and taken by the next
step, one Agent cycle against the float64 reference, graph replay against the eager loop,
checkpoints, statistics and N ranks."""
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

from oracle import a3c, philox
from sarsa_oracle import sarsa_gradients, sarsa_targets
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
def test_sarsa_lossgrad_vs_oracle(pkg, cuda, A, T, B):
    rng = np.random.default_rng(A * 1000 + T * B + 7)
    N = T * B
    q = rng.normal(0, 1, (N, A)).astype(np.float32)
    q_next = rng.normal(0, 1, (N, A)).astype(np.float32)
    rew = rng.choice([-3.0, -1.0, 0.0, 0.5, 1.0, 2.0], (T, B)).astype(np.float32)
    term = rng.random((T, B)) < 0.3
    act = rng.integers(0, A, N + B).astype(np.int32)              # a_0 .. a_T
    d = lambda x: torch.as_tensor(x, device=cuda)
    ins = [d(rew), d(term.astype(np.uint8)), d(act), d(q), d(q_next)]
    P, st = pkg._cabi.ptr, pkg._cabi.stream_ptr()
    scale = 1.0 / B

    def sarsa(acts, sums):
        y, dq = torch.empty(N, device=cuda), torch.empty(N, A, device=cuda)
        pkg._cabi.call("arl_sarsa_lossgrad", P(ins[0]), P(ins[1]), P(acts), P(ins[3]), P(ins[4]), P(y), P(dq),
                       P(sums), T, B, A, 0.99, -1.0, 1.0, scale, st)
        return y, dq

    sums = torch.zeros(2, device=cuda)
    y, dq = sarsa(ins[2], sums)
    torch.cuda.synchronize()
    ref_y = sarsa_targets(q_next, act[B:], rew, term, 0.99)
    assert rel_err(y.cpu(), ref_y) <= 1e-6
    qa = q[np.arange(N), act[:N]].astype(np.float64)
    delta = ref_y - qa
    ref_dq = np.zeros((N, A))
    ref_dq[np.arange(N), act[:N]] = -2.0 * delta * scale
    assert rel_err(dq.cpu(), ref_dq) <= 1e-6
    assert abs(float(sums[0]) - (delta ** 2).sum()) <= 1e-4 * (delta ** 2).sum()
    assert abs(float(sums[1]) - qa.sum()) <= 1e-4 * np.abs(qa).sum()

    # greedy next actions: arl_q_lossgrad's targets and gradient, bit for bit
    greedy = ins[2].clone()
    greedy[B:] = ins[4].argmax(dim=1).int()
    g_sums, q_sums = torch.zeros(2, device=cuda), torch.zeros(2, device=cuda)
    gy, gdq = sarsa(greedy, g_sums)
    qy, qdq = torch.empty(N, device=cuda), torch.empty(N, A, device=cuda)
    pkg._cabi.call("arl_q_lossgrad", P(ins[0]), P(ins[1]), P(greedy), P(ins[3]), P(ins[4]), P(qy), P(qdq),
                   P(q_sums), N, A, 0.99, -1.0, 1.0, scale, st)
    torch.cuda.synchronize()
    assert torch.equal(gy, qy) and torch.equal(gdq, qdq)
    # the same per-warp partial sums; the float atomics that add them up run in no fixed order, so
    # the totals agree to rounding (relative to the sum of magnitudes: sum Q cancels)
    g, r = g_sums.double().cpu(), q_sums.double().cpu()
    assert abs(float(g[0] - r[0])) <= 1e-5 * float(r[0]), (g, r)
    q_greedy = q[np.arange(N), greedy[:N].cpu().numpy()].astype(np.float64)
    assert abs(float(g[1] - r[1])) <= 1e-5 * np.abs(q_greedy).sum(), (g, r)

    # zero-size calls do nothing
    before = (y.clone(), dq.clone(), sums.clone())
    for t_, b_ in ((0, B), (T, 0)):
        pkg._cabi.call("arl_sarsa_lossgrad", *[P(x) for x in ins], P(y), P(dq), P(sums), t_, b_, A, 0.99, -1.0,
                       1.0, scale, st)
    torch.cuda.synchronize()
    assert all(torch.equal(x, z) for x, z in zip(before, (y, dq, sums)))
    with pytest.raises(pkg._cabi.ArlError, match="action_size"):
        pkg._cabi.call("arl_sarsa_lossgrad", *[P(x) for x in ins], P(y), P(dq), P(sums), T, B, 0, 0.99, -1.0,
                       1.0, scale, st)


# ---- Agent helpers -------------------------------------------------------------------------------
def _agent(pkg, cuda, B, T, A, over=None, pool=None, p_terminal=0.2, seed=3, env_seed=None):
    cfg = pkg.config.get_config(dict({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": "sarsa"},
                                     **(over or {})))
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=seed if env_seed is None else env_seed,
                                                         pool=pool or T + 3, device=cuda, p_terminal=p_terminal),
                             device=cuda)
    return pkg.Agent(cfg, env, device=cuda), env


def _plain_forward(pkg, net, params, hist, cuda):
    """Q of the current stack under ``params`` through a plain arl_forward into fresh buffers."""
    B, A = net.num_envs, net.action_size
    f32 = dict(device=cuda, dtype=torch.float32)
    prep = torch.empty(pkg._cabi.prepared_floats(), **f32)
    l1, l2, l4 = (torch.empty(B, n, **f32) for n in (3200, 2592, 256))
    logits, probs, value = torch.empty(B, A, **f32), torch.empty(B, A, **f32), torch.empty(B, **f32)
    P = pkg._cabi.ptr
    pkg._cabi.call("arl_forward", P(params), P(prep), 1, A, P(hist.ring), B, hist.ring_slots, hist.first_slot(0),
                   1, P(l1), P(l2), P(l4), P(logits), P(probs), P(value), pkg._cabi.stream_ptr())
    return logits


# ---- 2. the a_T draw -----------------------------------------------------------------------------
def test_next_action_is_drawn_at_the_update_and_taken_by_the_next_step(pkg, cuda):
    """Every update draws a_T (row T) epsilon-greedily on Q(s_T) under the parameters before the
    update, with the step and epsilon of the next rollout's first frame; the next predict() takes
    it, with Q from the updated parameters.  Two eager cycles, then replayed ones."""
    B, T, A = 64, 3, 6
    random.seed(11)
    agent, env = _agent(pkg, cuda, B, T, A, over={"ep_end_t": 30, "learn_start": 2}, pool=T, p_terminal=0.1)
    net, hist, cfg = agent.network, agent.history, agent.config
    net.set_weights(make_params(A, seed=21, scale=2.0))
    agent.before_train()
    assert not agent.sarsa_pending
    P, N = pkg._cabi.ptr, T * B
    kinds, row = set(), None
    for cycle in range(5):
        for t in range(T):
            a = agent.predict()
            if t == 0 and row is not None:
                torch.cuda.synchronize()
                assert torch.equal(a, row), cycle                 # the step after the update takes a_T ...
                assert torch.equal(net.q[:B], _plain_forward(pkg, net, net.params, hist, cuda))   # ... Q from theta
            if t == T - 1:
                theta_old = net.params.clone()
            scr, rew, term = env.act(a, is_training=True, fused=True)
            agent.observe(scr, rew, a, term)
            agent.step += 1
        assert agent.sarsa_pending and agent.t == 0
        row = net.sarsa_actions[N:].clone()
        q_old = _plain_forward(pkg, net, theta_old, hist, cuda)
        ep = host_ep(pkg, cfg, agent.step)
        ref = torch.empty(B, dtype=torch.int32, device=cuda)
        pkg._cabi.call("arl_egreedy_actions", P(q_old), P(ref), B, A, float(ep), agent.env_id_base, agent.step,
                       agent.seed, pkg._cabi.stream_ptr())
        torch.cuda.synchronize()
        assert torch.equal(row, ref), cycle
        assert torch.equal(net._b['logits'], q_old)               # the draw saw the pre-update Q(s_T)
        assert not torch.equal(net.params, theta_old)             # ... and the update did change theta
        greedy = row.cpu().numpy() == q_old.cpu().numpy().argmax(1)
        kinds.add((bool(greedy.all()), bool(greedy.any())))
    assert agent.graph_replays > 0
    assert (False, True) in kinds                                 # some actions random, some greedy


# ---- 3. one Agent cycle --------------------------------------------------------------------------
@pytest.mark.parametrize("A,B,T", [(6, 9, 4), (18, 5, 2)])
def test_sarsa_cycle_vs_oracle(pkg, cuda, A, B, T):
    agent, env = _agent(pkg, cuda, B, T, A)
    net = agent.network
    assert agent.cuda_graphs and net.target_q.shape == (T * B, A) and not hasattr(net, "q_boot")
    assert net.sarsa_actions.shape == ((T + 1) * B,) and agent.batch_action.data_ptr() == net.sarsa_actions.data_ptr()
    params, tparams = make_params(A, seed=41, scale=2.0), make_params(A, seed=42, scale=2.0)
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
    masks = gpu_masks(net)
    agent.batch_update()
    torch.cuda.synchronize()
    acts = net.sarsa_actions.cpu().numpy().reshape(T + 1, B)
    stacks = a3c.stacks_from_screens(np.stack(screens), T)
    grads, aux = sarsa_gradients(params, tparams, stacks, acts, np.stack(rews), np.stack(terms), 0.99,
                                 scale=1.0 / B, masks=masks)
    assert rel_err(net.target_q.cpu(), aux["q_next"]) <= REL_TOL
    assert rel_err(net.target_q_t.cpu(), aux["target"]) <= REL_TOL
    errs = {k: rel_err(net.g[k].cpu(), grads[k]) for k in a3c.PARAM_NAMES if k not in ("q_w", "q_b")}
    print("one-step Sarsa grad rel-err", errs)
    assert max(errs.values()) <= REL_TOL, errs
    assert float(net.g["q_w"].abs().max()) == 0.0 and float(net.g["q_b"].abs().max()) == 0.0
    rms = {k: np.ones_like(v) for k, v in params.items()}
    new_p, _ = a3c.update(params, rms, grads, a3c.learning_rate(agent.step - (T - 1)))
    perr = {k: rel_err(net.w[k].cpu(), new_p[k]) for k in a3c.PARAM_NAMES}
    assert max(perr.values()) <= REL_TOL, perr
    assert rel_err(net.target_params.cpu(), a3c.flatten_params(tparams)) == 0.0   # untouched until the sync
    agent.update_target_q_network()
    assert bool((net.target_params == net.params).all())


def test_nature_trunk_refuses_sarsa(pkg, cuda):
    cfg = pkg.config.get_config({"model": "m1", "num_envs": 4, "t_max": 2, "loss_mode": "sarsa",
                                 "DQN_type": "nature"})
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(4, 6, seed=1, pool=4, device=cuda), device=cuda)
    with pytest.raises(NotImplementedError, match="sarsa"):
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
    assert torch.equal(eager.network.sarsa_actions, graph.network.sarsa_actions)


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
    """Save after 4 cycles, load into a fresh Agent (target, sync schedule and the pending a_T
    included), continue 4 cycles: the same actions, parameters, RMSProp slot and target as the run
    that never stopped.  The environment side (emulator, frame history) is carried over from a twin
    run."""
    B, T, A = 12, 5, 6
    over = {"ep_end_t": 200, "learn_start": 5, "target_q_update_step": 3 * T * B}
    full, acts_f, _ = _loop(pkg, cuda, True, 4, B=B, T=T, A=A, over=over)
    full.step_op = full.step
    full.save_checkpoint(str(tmp_path))
    pending = full.network.sarsa_actions[T * B:].clone()
    _, acts_f2, snaps_f = _loop(pkg, cuda, True, 4, agent_env=(full, full.env))
    twin, acts_t, _ = _loop(pkg, cuda, True, 4, B=B, T=T, A=A, over=over)   # the environment after 4 cycles
    assert torch.equal(acts_t, acts_f)
    cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": "sarsa", **over})
    resumed = pkg.Agent(cfg, twin.env, device=cuda)
    assert not resumed.sarsa_pending
    assert resumed.load_checkpoint(str(tmp_path)) and resumed.step_op == full.step_op
    assert resumed.sarsa_pending and torch.equal(resumed.network.sarsa_actions[T * B:], pending)
    resumed.step, resumed.T = resumed.step_op, resumed.step_op * resumed.global_envs   # before_train's counters
    assert resumed._last_target_sync == twin._last_target_sync
    resumed.history.ring.copy_(twin.history.ring)
    resumed.history.head = twin.history.head
    _, acts_r, snaps_r = _loop(pkg, cuda, True, 4, agent_env=(resumed, twin.env))
    assert torch.equal(acts_r[0], pending)                        # the first step took the saved a_T
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
           os.path.join(ROOT, "tests", "dist_gpu_check_sarsa.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["ok"] and line["actions_bit_identical"] and line["replica_max_minus_min"] == 0.0
