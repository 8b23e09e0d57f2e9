"""GPU time per C-ABI entry in one cycle of each learner, to compare the learners' cycles entry by entry.

    python tools/learner_entry_times.py [--modes sarsa,async_q,...] [--shapes 4096x5x6,...] [--cycles K]
                                        [--out FILE]

Every library call (``_cabi.call``) is bracketed by a CUDA event pair; CUDA graphs are off, so every
call is launched on its own.  For each mode and shape: 3 warm-up cycles, then K cycles recorded.
Reported per entry: summed event time per cycle (ms) and calls per cycle.  ``arl_forward`` is split by
its step count (steps = 1: one env step of B samples; steps = T: T*B samples).  Torch copies and fills
between the calls are not counted.  The card's name and power limit are written beside the numbers.
"""
import argparse
import importlib
import json
import os
import random
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_nstep_q import card                                   # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--modes", default="a3c,nstep_q,sarsa,async_q")
    ap.add_argument("--shapes", default="4096x5x6,16384x20x18", help="envs x t_max x actions, comma separated")
    ap.add_argument("--cycles", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_sarsa_entry_times.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("learner_entry_times: needs a CUDA device")
    pkg = importlib.import_module("async-rl-tensorflow_b200")
    cabi = pkg._cabi
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    events = []
    plain = cabi.call

    def timed_call(name, *a):
        key = "%s[steps=%d]" % (name, a[8]) if name == "arl_forward" else name
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        plain(name, *a)
        e1.record()
        events.append((key, e0, e1))

    result = {"card": card(), "cycles": args.cycles, "shapes": []}
    for shape in args.shapes.split(","):
        B, T, A = (int(x) for x in shape.split("x"))
        entry = {"envs": B, "t_max": T, "actions": A, "modes": {}}
        for mode in args.modes.split(","):
            cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": mode,
                                         "cuda_graphs": False})
            env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=123, pool=T, device=dev), device=dev)
            agent = pkg.Agent(cfg, env, device=dev)
            random.seed(cfg.seed)
            agent.before_train()

            def cycles(k):
                for _ in range(k * T):
                    a = agent.predict()
                    scr, rew, term = env.act(a, is_training=True, fused=True)
                    agent.observe(scr, rew, a, term)
                    agent.step += 1

            cycles(3)
            torch.cuda.synchronize()
            events.clear()
            cabi.call = timed_call
            try:
                cycles(args.cycles)
            finally:
                cabi.call = plain
            torch.cuda.synchronize()
            per = {}
            for key, e0, e1 in events:
                ms, n = per.get(key, (0.0, 0))
                per[key] = (ms + e0.elapsed_time(e1), n + 1)
            rows = {k: {"ms_per_cycle": round(ms / args.cycles, 4), "calls_per_cycle": n / args.cycles}
                    for k, (ms, n) in sorted(per.items(), key=lambda kv: -kv[1][0])}
            entry["modes"][mode] = {"entries": rows,
                                    "sum_ms_per_cycle": round(sum(ms for ms, _ in per.values()) / args.cycles, 4)}
            print(json.dumps({"shape": shape, "mode": mode, **entry["modes"][mode]}), flush=True)
            del agent, env
            torch.cuda.empty_cache()
        result["shapes"].append(entry)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
        f.write("\n")
    print(json.dumps({"card": result["card"], "out": args.out}))


if __name__ == "__main__":
    main()
