"""Cycle time of the four learners on one GPU: a3c, nstep_q and sarsa replayed from CUDA graphs,
async_q eager (its own path: host epsilon, a separate draw launch, a target forward over all T*B next
states; sarsa runs that target forward too, inside its graph).

    python tools/bench_nstep_q.py [--rounds R] [--cycles K] [--modes a3c,nstep_q,...] [--dueling off|on|both]
                                  [--double off|on|both] [--dueling-streams off|on|both] [--lstm off|on|both]
                                  [--out FILE]

For each shape (envs x t_max x actions: 4096 x 5 x 6 and 16384 x 20 x 18) one agent per mode is built
and warmed up until a whole ring period has replayed without a new graph capture; then the modes take
turns, R rounds of K whole cycles each (t_max x (predict, act, observe) + the update), with a CUDA
event pair around every K-cycle block.  Reported per mode: ms per cycle (median, min, max over the
rounds) and env frames/s (envs x t_max / median cycle time).  The card's name and power limit are
read in the same run and written beside the numbers.  Synthetic frames, resident in HBM; the frame
pool is larger than L2 at both shapes.

--dueling on runs the Q learners with dueling Q heads (dueling=True; reported as "<mode>+dueling"),
--dueling both runs every Q learner both ways, all of them alternating.
--double on|both does the same with double Q-learning targets (double_q=True) for async_q and nstep_q,
reported as "<mode>+double" or "<mode>+dueling+double".
"""
import argparse
import importlib
import json
import os
import random
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODES = ("a3c", "nstep_q", "sarsa", "async_q")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                       # report, never guess
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % str(e)[:80]}


def lstm_entry_times(pkg, agent, reps):
    """GPU time of each new LSTM entry on the network's own buffers after the timed cycles (a CUDA event pair
    around ``reps`` back-to-back calls; the state is not advanced), with the bytes each must move at the
    least, counted from the shapes, and the rate that gives.  Per row of B envs (one step) or N = T*B samples:
      arl_lstm_step      read h_fc, h (2 KB), write xh (2 KB); GEMM read xh (2 KB), write z (4 KB); cell read
                         z, c (5 KB), write gates, c_prev, c, h (7 KB)                                = 22 KB
      arl_heads_backward_lstm  read h (1 KB), write d_h_lstm (1 KB)                                 =  2 KB
      arl_lstm_backward  cell bwd read d_h_lstm, dh_rec, dc, gates, c_prev, c (9 KB), write dz, dc (5 KB);
                         dgrad read dz (4 KB), write dxh (2 KB); wgrad read xh, dz (6 KB); dx hand-over read
                         dx, h_fc (2 KB), write d_h twice (2 KB)                                      = 30 KB
    (+ the 4 MB of weight images and the wgrad's 8 MB of partials, read back once)."""
    P, st, net = pkg._cabi.ptr, pkg._cabi.stream_ptr(), agent.network
    B, T, A = net.num_envs, net.t_max, net.action_size
    N, b = B * T, net._b
    calls = {
        "arl_lstm_step": (lambda: pkg._cabi.call(
            "arl_lstm_step", P(net.params), P(net.fc_w), A, P(net.l4[:B]), P(net.state_h), P(net.state_c), None, 0,
            P(b["xh"]), P(net.lstm_z), P(net.gates[:B]), P(net.c_prev[:B]), P(b["c"]), P(b["h"]), B, st),
            B * 22 * 1024 + 4 * 2 ** 20),
        "arl_heads_backward_lstm": (lambda: pkg._cabi.call(
            "arl_heads_backward_lstm", P(net.params), A, P(net.h_lstm), P(net.d_logits), P(net.d_value),
            P(net.d_h_lstm), P(net.grads), P(net.workspace), N, 64.0, st), N * 2 * 1024),
        "arl_lstm_backward": (lambda: pkg._cabi.call(
            "arl_lstm_backward", P(net.params), P(net.fc_w), A, B, T, P(agent.batch_terminal), P(net.l4), P(net.xh),
            P(net.gates), P(net.c_prev), P(net.c_seq), P(net.d_h_lstm), P(net.dz), P(net.dxh), P(net.dc),
            P(net.d_l4), P(net.grads), P(net.workspace), 64.0, st), N * 30 * 1024 + 12 * 2 ** 20),
    }
    out = {}
    for name, (fn, nbytes) in calls.items():
        fn()                                                     # warm
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out[name] = {"ms": round(ms, 4), "min_bytes": nbytes, "GB_per_s": round(nbytes / ms / 1e6, 1),
                     "launches_per_call": {"arl_lstm_step": 3, "arl_heads_backward_lstm": 2,
                                           "arl_lstm_backward": 2 * T + 4}[name]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cycles", type=int, default=20, help="cycles per timed block")
    ap.add_argument("--shapes", default="4096x5x6,16384x20x18", help="envs x t_max x actions, comma separated")
    ap.add_argument("--modes", default=",".join(MODES))
    ap.add_argument("--dueling", default="off", choices=("off", "on", "both"),
                    help="dueling Q heads for the Q learners: off, on, or both (each Q learner twice)")
    ap.add_argument("--double", default="off", choices=("off", "on", "both"),
                    help="double Q-learning targets for async_q and nstep_q: off, on, or both")
    ap.add_argument("--dueling-streams", default="off", choices=("off", "on", "both"),
                    help="a hidden layer per dueling stream (reported as \"<mode>+streams\"): off, on, or both "
                         "(each Q learner plain, with dueling heads and with dueling streams)")
    ap.add_argument("--lstm", default="off", choices=("off", "on", "both"),
                    help="the A3C LSTM agent for the a3c mode (reported as \"a3c+lstm\"): off, on, or both; with the "
                         "flag on, the GPU time of each new LSTM entry is recorded too")
    ap.add_argument("--out", default=None, help="default: profiles/r05_sarsa_bench.json, "
                                                "profiles/r06_dueling_bench.json with --dueling on|both, "
                                                "profiles/r08_double_q_bench.json with --double on|both, or "
                                                "profiles/r09_dueling_streams_bench.json with --dueling-streams on|both, "
                                                "or profiles/r11_lstm_bench.json with --lstm on|both")
    args = ap.parse_args()
    if args.out is None:
        args.out = os.path.join(ROOT, "profiles", "r11_lstm_bench.json" if args.lstm != "off"
                                else "r09_dueling_streams_bench.json" if args.dueling_streams != "off"
                                else "r08_double_q_bench.json" if args.double != "off"
                                else "r05_sarsa_bench.json" if args.dueling == "off" else "r06_dueling_bench.json")
    if not torch.cuda.is_available():
        sys.exit("bench_nstep_q: needs a CUDA device")
    pkg = importlib.import_module("async-rl-tensorflow_b200")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    modes = []
    for m in args.modes.split(","):
        heads = ({"off": [""], "on": ["+lstm"], "both": ["", "+lstm"]}[args.lstm] if m == "a3c"
                 else {"off": [""], "on": ["+dueling"], "both": ["", "+dueling"]}[args.dueling])
        if m != "a3c" and args.dueling_streams != "off":
            heads = {"on": ["+streams"], "both": ["", "+dueling", "+streams"]}[args.dueling_streams]
        targets = ([""] if m not in ("async_q", "nstep_q")
                   else {"off": [""], "on": ["+double"], "both": ["", "+double"]}[args.double])
        modes += [m + h + d for h in heads for d in targets]
    result = {"card": card(), "rounds": args.rounds, "cycles_per_block": args.cycles, "shapes": []}

    for shape in args.shapes.split(","):
        B, T, A = (int(x) for x in shape.split("x"))
        pool = max(2, min(T, int(24e9 // (B * 100800) // len(modes))))   # frames kept per agent
        agents = {}
        for mode in modes:
            cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": mode.split("+")[0],
                                         "dueling": "+dueling" in mode or "+streams" in mode,
                                         "dueling_streams": "+streams" in mode, "double_q": mode.endswith("+double"),
                                         "lstm": "+lstm" in mode})
            env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=123, pool=pool, device=dev), device=dev)
            agent = pkg.Agent(cfg, env, device=dev)
            random.seed(cfg.seed)
            agent.before_train()
            agents[mode] = (agent, env)

        def cycles(mode, k):
            agent, env = agents[mode]
            for _ in range(k):
                for _ in range(T):
                    a = agent.predict()
                    scr, rew, term = env.act(a, is_training=True, fused=True)
                    agent.observe(scr, rew, a, term)
                    agent.step += 1

        for mode in modes:                                       # warm-up: every graph captured
            agent = agents[mode][0]
            cycles(mode, 3)
            seen, quiet = len(agent._graphs), 0
            for _ in range(64):
                if not agent.cuda_graphs or quiet >= 3:
                    break
                cycles(mode, 1)
                quiet = quiet + 1 if len(agent._graphs) == seen else 0
                seen = len(agent._graphs)
        torch.cuda.synchronize()
        ms = {m: [] for m in modes}
        for _ in range(args.rounds):
            for mode in modes:                                   # the modes alternate
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                cycles(mode, args.cycles)
                e1.record()
                torch.cuda.synchronize()
                ms[mode].append(e0.elapsed_time(e1) / args.cycles)
        entry = {"envs": B, "t_max": T, "actions": A, "frame_pool_steps": pool, "modes": {}}
        for mode in modes:
            med = statistics.median(ms[mode])
            agent = agents[mode][0]
            entry["modes"][mode] = {"ms_per_cycle": round(med, 4), "ms_min": round(min(ms[mode]), 4),
                                    "ms_max": round(max(ms[mode]), 4), "frames_per_sec": round(B * T / med * 1e3),
                                    "graph_replayed": bool(agent.graph_replays), "graphs": len(agent._graphs)}
        for mode in modes:
            if "+lstm" in mode:
                entry["modes"][mode]["entries"] = lstm_entry_times(pkg, agents[mode][0], args.cycles)
        if "a3c" in modes:
            for mode in modes:
                entry["modes"][mode]["vs_a3c"] = round(entry["modes"][mode]["ms_per_cycle"] /
                                                       entry["modes"]["a3c"]["ms_per_cycle"], 4)
        result["shapes"].append(entry)
        print(json.dumps(entry), flush=True)
        del agents
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
        f.write("\n")
    print(json.dumps({"card": result["card"], "out": args.out}))


if __name__ == "__main__":
    main()
