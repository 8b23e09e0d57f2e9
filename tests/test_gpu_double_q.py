"""GPU: double Q-learning targets (double_q=True, van Hasselt et al. 2016) on the async-Q and n-step Q
learners: the loss entries against their plain entries, one cycle per learner against the float64
reference, theta^- = theta against double_q=False, graph replay against the eager loop, full size,
checkpoints, refusals and N ranks."""
import json
import os
import random
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from double_q_oracle import double_q_gradients
from oracle import a3c
from test_gpu_network import gpu_masks, make_params
from util import REL_TOL, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = ("async_q", "nstep_q")


# ---- 1. the loss entries -------------------------------------------------------------------------
@pytest.mark.parametrize("dueling", [False, True])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("A,T,B", [(6, 5, 257), (18, 20, 33)])
def test_loss_entry_against_its_plain_entry(pkg, cuda, mode, dueling, A, T, B):
    rng = np.random.default_rng(A * T * B + dueling)
    N = T * B
    d = lambda x: torch.as_tensor(x, device=cuda)
    nboot = B if mode == "nstep_q" else N                      # rows of q_next (q_boot)
    q_np = rng.normal(0, 1, (N, A)).astype(np.float32)
    q_next_np = rng.normal(0, 1, (nboot, A)).astype(np.float32)
    rew = d(rng.choice([-3.0, -1.0, 0.0, 0.5, 1.0, 2.0], (T, B)).astype(np.float32))
    term = d((rng.random((T, B)) < 0.3).astype(np.uint8))
    act = d(rng.integers(0, A, N).astype(np.int32))
    P, st, scale = pkg._cabi.ptr, pkg._cabi.stream_ptr(), 1.0 / B
    plain_name = "arl_q_lossgrad" if mode == "async_q" else "arl_nstep_q_lossgrad"
    suffix = "_dueling" if dueling else ""

    def call(q, q_next, q_online_T=None):
        """The plain entry (q_online_T None) or the double entry; returns targets, dq, dvalue, loss_sums."""
        y, dq, sums = torch.empty(N, device=cuda), torch.full((N, A), 7.0, device=cuda), torch.zeros(2, device=cuda)
        dv = torch.full((N,), 7.0, device=cuda)
        extra = (P(dv),) if dueling else ()
        if q_online_T is None:
            size = (N,) if mode == "async_q" else (T, B)
            pkg._cabi.call(plain_name + suffix, P(rew), P(term), P(act), P(q), P(q_next), P(y), P(dq), *extra,
                           P(sums), *size, A, 0.99, -1.0, 1.0, scale, st)
        else:
            name = ("arl_double_q_lossgrad" if mode == "async_q" else "arl_double_nstep_q_lossgrad") + suffix
            pkg._cabi.call(name, P(rew), P(term), P(act), P(q), P(q_next), P(q_online_T), P(y), P(dq), *extra,
                           P(sums), T, B, A, 0.99, -1.0, 1.0, scale, st)
        torch.cuda.synchronize()
        return y, dq, dv, sums

    def online_rows(q_np, q_online_T_np):
        """The rows a* is taken from, one per bootstrap row: q rows 1..T-1 then Q(s_T; theta) for the
        1-step learner, Q(s_T; theta) for the n-step learner."""
        return np.concatenate([q_np[B:], q_online_T_np]) if mode == "async_q" else q_online_T_np

    # online Q == target Q: the double entry is the plain entry, bit for bit
    if mode == "async_q":
        q_same = q_np.copy()
        q_same[B:] = q_next_np[:N - B]                          # the online rows of s_1..s_{T-1}
        online_T = q_next_np[N - B:]
    else:
        q_same, online_T = q_np, q_next_np
    y0, dq0, dv0, s0 = call(d(q_same), d(q_next_np))
    y1, dq1, dv1, s1 = call(d(q_same), d(q_next_np), d(online_T.copy()))
    assert torch.equal(y1, y0) and torch.equal(dq1, dq0)
    if dueling:
        assert torch.equal(dv1, dv0)
    assert abs(float(s1[0] - s0[0])) <= 1e-5 * abs(float(s0[0]))

    # online Q != target Q, with tied online maxima on every third row: the double entry on q_next equals
    # the plain entry on q_next' (every entry of row n = q_next[n][a*_n], a* the first index of the max)
    online_T = rng.normal(0, 1, (B, A)).astype(np.float32)
    on = online_rows(q_np, online_T)
    tied = np.arange(0, nboot, 3)
    j, k = rng.integers(0, A - 1, tied.size), np.full(tied.size, A - 1)
    top = on.max(axis=1)[tied] + 1.0
    on[tied, j], on[tied, k] = top, top                         # tied maxima at j < k
    q_next_np[tied, k] = q_next_np[tied, j] + 2.0               # ... with different target values
    if mode == "async_q":
        q_np[B:], online_T = on[:N - B], on[N - B:]
    else:
        online_T = on
    a_star = np.argmax(on, axis=1)                              # ties -> the first index
    assert np.array_equal(a_star[tied], j)
    chosen = q_next_np[np.arange(nboot), a_star]
    assert float((chosen != q_next_np.max(axis=1)).mean()) >= 0.3
    y_ref, dq_ref, dv_ref, _ = call(d(q_np), d(np.repeat(chosen[:, None], A, axis=1)))
    y2, dq2, dv2, _ = call(d(q_np), d(q_next_np), d(online_T.copy()))
    assert torch.equal(y2, y_ref) and torch.equal(dq2, dq_ref)
    if dueling:
        assert torch.equal(dv2, dv_ref)
    y_max, _, _, _ = call(d(q_np), d(q_next_np))
    assert not torch.equal(y2, y_max)

    with pytest.raises(pkg._cabi.ArlError, match="null pointer"):
        name = ("arl_double_q_lossgrad" if mode == "async_q" else "arl_double_nstep_q_lossgrad") + suffix
        pkg._cabi.call(name, P(rew), P(term), P(act), P(d(q_np)), P(d(q_next_np)), None, P(y2), P(dq2),
                       *((P(dv2),) if dueling else ()), None, T, B, A, 0.99, -1.0, 1.0, scale, st)


# ---- Agent helpers -------------------------------------------------------------------------------
def _agent(pkg, cuda, mode, B, T, A, dueling=False, double_q=True, over=None, pool=None, p_terminal=0.2, seed=3):
    cfg = pkg.config.get_config(dict({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": mode,
                                      "dueling": dueling, "double_q": double_q}, **(over or {})))
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=seed, pool=pool or T + 3, device=cuda,
                                                         p_terminal=p_terminal), device=cuda)
    return pkg.Agent(cfg, env, device=cuda), env


def _rollout(agent, env, T, record=False):
    """One rollout driven by hand (Agent.observe without the update trigger); returns the screens,
    rewards and terminals the reference needs when ``record``."""
    hist = agent.history
    first = hist.first_slot(0)
    snap = hist.planes().cpu().numpy() if record else None
    screens = [snap[:, (first + k) % hist.ring_slots] for k in range(4)] if record else []
    rews, terms = [], []
    for t in range(T):
        action = agent.predict()
        scr, rew, term = env.act(action, is_training=True, fused=True)
        hist.add(scr)
        agent.batch_reward[t].copy_(rew)
        agent.batch_terminal[t].copy_(term)
        if record:
            rews.append(rew.cpu().numpy()); terms.append(term.cpu().numpy())
            screens.append(hist.planes(hist.head).cpu().numpy())
        agent.t += 1
        agent.step += 1
    agent.step -= 1
    return screens, rews, terms


# ---- 2. one cycle per learner --------------------------------------------------------------------
@pytest.mark.parametrize("dueling", [False, True])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("A,B,T", [(6, 40, 4), (18, 12, 2)])
def test_cycle_vs_oracle(pkg, cuda, mode, dueling, A, B, T):
    agent, env = _agent(pkg, cuda, mode, B, T, A, dueling=dueling)
    net = agent.network
    assert net.double_q and net.dueling == dueling
    params, tparams = make_params(A, seed=41, scale=2.0, bias_std=0.1), make_params(A, seed=42, scale=2.0, bias_std=0.1)
    net.set_weights(params)
    agent.before_train()                                        # syncs the target (main.py:92) ...
    net.target_params.copy_(torch.as_tensor(a3c.flatten_params(tparams), device=cuda))  # ... then differ
    agent.step = 100
    screens, rews, terms = _rollout(agent, env, T, record=True)
    masks = gpu_masks(net)
    q_roll = net.q.cpu().numpy().copy()
    agent.batch_update()
    torch.cuda.synchronize()
    acts = agent.batch_action.cpu().numpy().copy()
    q_online_T = net.q_online_T.cpu().numpy()
    # the device's a*: the first index of the max of the device's online rows
    online = np.concatenate([q_roll[B:], q_online_T]) if mode == "async_q" else q_online_T
    a_star = np.argmax(online, axis=1)
    stacks = a3c.stacks_from_screens(np.stack(screens), T)
    scale = 1.0 / (T * B) if mode == "async_q" else 1.0 / B
    grads, aux = double_q_gradients(mode, params, tparams, stacks, acts, np.stack(rews), np.stack(terms), 0.99,
                                    scale=scale, masks=masks, dueling=dueling, a_star=a_star)
    # a* is an argmax of Q(s'; theta) up to the forward's tolerance, and it is not the target's argmax
    q64 = aux["q_online"]
    gap = q64.max(axis=1) - q64[np.arange(q64.shape[0]), a_star]
    assert float(gap.max()) <= REL_TOL * float(np.abs(q64).max()), float(gap.max())
    share = float((a_star != aux["q_next"].argmax(axis=1)).mean())
    print("double_q", mode, "dueling" if dueling else "plain", "A=%d B=%d T=%d" % (A, B, T),
          "share of rows with a* != argmax Q(s'; theta^-): %.3f" % share)
    assert share >= 0.3, share
    assert rel_err(q_roll, aux["q"]) <= REL_TOL
    assert rel_err(q_online_T, q64[-B:]) <= REL_TOL
    assert rel_err((net.q_boot if mode == "nstep_q" else net.target_q).cpu(), aux["q_next"]) <= REL_TOL
    assert rel_err((net.R if mode == "nstep_q" else net.target_q_t).cpu(), aux["target"]) <= REL_TOL
    errs = {k: rel_err(net.g[k].cpu(), grads[k]) for k in a3c.PARAM_NAMES}
    g = aux["delta"]                                            # q_b's gradient (dueling): one sum over the samples
    print("double_q", mode, "grad rel-err", errs, "q_b sum conditioning sum|delta| / |sum delta|: %.1f"
          % (np.abs(g).sum() / max(abs(g.sum()), 1e-30)))
    assert max(errs.values()) <= REL_TOL, errs


# ---- 3. theta^- = theta: double_q on == off --------------------------------------------------------
@pytest.mark.parametrize("dueling", [False, True])
@pytest.mark.parametrize("mode", MODES)
def test_double_equals_plain_when_target_is_online(pkg, cuda, mode, dueling):
    """Right after before_train the target is the online network: the online and target forwards of
    s_T are the same launches on equal weights, so a* is the target's argmax and one cycle is bit for
    bit the plain one.  async_q also takes the online rows of s_1..s_{T-1} from the rollout's 1-step
    forwards while the target rows come from one T-step forward."""
    B, T, A = 40, 5, 6
    out = []
    for double_q in (False, True):
        random.seed(321)
        agent, env = _agent(pkg, cuda, mode, B, T, A, dueling=dueling, double_q=double_q, seed=8)
        agent.network.set_weights(make_params(A, seed=17, scale=2.0, bias_std=0.1))
        agent.before_train()
        agent.step = 100
        _rollout(agent, env, T)
        agent.batch_update()
        torch.cuda.synchronize()
        n = agent.network
        out.append((n.params.clone(), n.rms.clone(), (n.R if mode == "nstep_q" else n.target_q_t).clone()))
        if double_q and mode == "async_q":                     # the rows a* came from are the target's rows
            on = torch.cat([n.q[B:], n.q_online_T])
            print("async_q rollout rows == target rows:", bool(torch.equal(on, n.target_q)),
                  "max |diff|:", float((on - n.target_q).abs().max()))
        del agent, env
    (p0, r0, y0), (p1, r1, y1) = out
    assert torch.equal(y0, y1)
    assert torch.equal(p0, p1) and torch.equal(r0, r1)


# ---- 4. graph replay == eager loop ---------------------------------------------------------------
def _loop(pkg, cuda, mode, graphs, cycles, B=24, T=5, A=6, dueling=False, start_step=0, over=None, agent_env=None):
    random.seed(123)
    if agent_env is None:
        o = dict({"cuda_graphs": graphs, "ep_end_t": 30, "learn_start": 5,
                  "target_q_update_step": 3 * T * B}, **(over or {}))
        agent, env = _agent(pkg, cuda, mode, B, T, A, dueling=dueling, over=o, pool=T, p_terminal=0.1, seed=5)
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


@pytest.mark.parametrize("dueling", [False, True])
def test_graph_replay_equals_eager_loop(pkg, cuda, dueling):
    cycles = 9                                                   # 2 eager, then capture / replay
    eager, acts_e, snaps_e = _loop(pkg, cuda, "nstep_q", False, cycles, dueling=dueling)
    graph, acts_g, snaps_g = _loop(pkg, cuda, "nstep_q", True, cycles, dueling=dueling)
    assert eager.graph_replays == 0 and graph.graph_replays > 0
    assert graph.network.double_q
    assert torch.equal(acts_e, acts_g)
    for (pe, re_, te), (pg, rg, tg) in zip(snaps_e, snaps_g):
        assert torch.equal(pe, pg) and torch.equal(re_, rg) and torch.equal(te, tg)
    assert not torch.equal(snaps_g[5][2], snaps_g[8][2])           # a target sync inside the replayed cycles
    assert torch.equal(snaps_g[8][2], snaps_g[8][0])


# ---- 5. full size --------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("T,A", [(5, 6), (20, 18)])
def test_full_size_is_finite_and_deterministic(pkg, cuda, mode, T, A):
    B = 4096
    runs = []
    for _ in range(2):
        agent, acts, snaps = _loop(pkg, cuda, mode, True, 4, B=B, T=T, A=A, start_step=1000,
                                   over={"ep_end_t": 400 * 10000, "learn_start": 32,
                                         "target_q_update_step": 2 * T * B})
        g = agent.network.grads.clone()
        assert bool(torch.isfinite(g).all()) and float(agent.network.g["p_w"].abs().max()) > 0
        assert bool(torch.isfinite(agent.network.params).all())
        assert bool(torch.isfinite(agent.network.q_online_T).all())
        runs.append((acts, g, snaps[-1]))
        del agent
        torch.cuda.empty_cache()
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for x, y in zip(runs[0][2], runs[1][2]):
        assert torch.equal(x, y)


# ---- 6. checkpoints ------------------------------------------------------------------------------
def test_checkpoint_resume_equals_uninterrupted_run(pkg, cuda, tmp_path):
    B, T, A, mode = 12, 5, 6, "nstep_q"
    over = {"ep_end_t": 200, "learn_start": 5, "target_q_update_step": 3 * T * B}
    full, acts_f, _ = _loop(pkg, cuda, mode, True, 4, B=B, T=T, A=A, over=over)
    full.step_op = full.step
    full.save_checkpoint(str(tmp_path))
    _, acts_f2, snaps_f = _loop(pkg, cuda, mode, True, 4, agent_env=(full, full.env))
    twin, acts_t, _ = _loop(pkg, cuda, mode, True, 4, B=B, T=T, A=A, over=over)
    assert torch.equal(acts_t, acts_f)
    cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": mode, "double_q": True,
                                 **over})
    resumed = pkg.Agent(cfg, twin.env, device=cuda)
    assert resumed.load_checkpoint(str(tmp_path)) and resumed.step_op == full.step_op
    resumed.step, resumed.T = resumed.step_op, resumed.step_op * resumed.global_envs
    resumed.history.ring.copy_(twin.history.ring)
    resumed.history.head = twin.history.head
    _, acts_r, snaps_r = _loop(pkg, cuda, mode, True, 4, agent_env=(resumed, twin.env))
    assert torch.equal(acts_r, acts_f2)
    for (pf, rf, tf), (pr, rr, tr) in zip(snaps_f, snaps_r):
        assert torch.equal(pf, pr) and torch.equal(rf, rr) and torch.equal(tf, tr)


@pytest.mark.parametrize("mode", MODES)
def test_checkpoints_are_the_plain_files(pkg, cuda, tmp_path, mode):
    """double_q stores nothing: a double_q=False checkpoint loads into a double_q=True agent and both
    write the same entries."""
    B, T, A = 8, 2, 6
    plain, env = _agent(pkg, cuda, mode, B, T, A, double_q=False)
    plain.network.set_weights(make_params(A, seed=23, scale=2.0, bias_std=0.1))
    double, _ = _agent(pkg, cuda, mode, B, T, A, double_q=True)
    z_p = np.load(plain.save_checkpoint(str(tmp_path / "plain")))
    z_d = np.load(double.save_checkpoint(str(tmp_path / "double")))
    assert sorted(z_p.files) == sorted(z_d.files)
    assert double.load_checkpoint(str(tmp_path / "plain"))
    assert torch.equal(double.network.params, plain.network.params)
    assert torch.equal(double.network.target_params, plain.network.target_params)
    assert plain.load_checkpoint(str(tmp_path / "double"))


# ---- 7. refusals ---------------------------------------------------------------------------------
def test_refusals(pkg, cuda):
    def make(mode, kind="nips"):
        cfg = pkg.config.get_config({"model": "m1", "num_envs": 4, "t_max": 2, "loss_mode": mode, "double_q": True,
                                     "DQN_type": kind})
        env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(4, 6, seed=1, pool=4, device=cuda), device=cuda)
        return pkg.Agent(cfg, env, device=cuda)
    for mode in ("a3c", "sarsa"):
        for kind in ("nips", "nature"):
            with pytest.raises(ValueError, match=mode):
                make(mode, kind)
    for mode in MODES:
        with pytest.raises(NotImplementedError, match="nature|nips"):
            make(mode, "nature")
        assert make(mode).network.double_q


# ---- 8. N ranks ----------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
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
           os.path.join(ROOT, "tests", "dist_gpu_check_double_q.py"), "--mode", mode]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["ok"] and line["actions_bit_identical"] and line["replica_max_minus_min"] == 0.0
