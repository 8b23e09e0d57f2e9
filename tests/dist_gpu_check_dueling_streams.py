"""Multi-GPU parity check of the dueling streams (dueling_streams=True), run under torchrun, one rank per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P tests/dist_gpu_check_dueling_streams.py [--mode nstep_q|sarsa|async_q] [--envs B] [--cycles C]

Every rank runs C cycles of the learner on its env shard (the default exchange of the world size),
with a target sync inside the run.  Rank 0 then repeats the run in-process on the UNION batch (N*B envs, no
collective) and checks

  * epsilon-greedy actions on the dueling Q: bit-identical to the union run's columns of every rank
    (Philox keyed by the global env id, epsilon from the per-env step),
  * parameters + RMSProp slot + target parameters after C updates: within 1e-5 of the union run,
  * replicas: bit-identical across ranks.

Prints one JSON line on rank 0 and exits non-zero on failure.  tests/test_gpu_dueling_streams.py launches it
when the box has >= 2 GPUs.
"""
import argparse
import importlib
import json
import os
import random
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def run(pkg, dev, mode, B, T, A, cycles, shard, weights, standalone, world):
    random.seed(123)                                           # main.py:41
    cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "loss_mode": mode, "dueling": True,
                                 "dueling_streams": True, "ep_end_t": 4 * T, "learn_start": 2,
                                 # global frames: a sync after every second cycle
                                 "target_q_update_step": 2 * T * B * (1 if standalone else world)})
    env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(
        B, A, seed=77, pool=cycles * T + 40, device=dev, p_terminal=0.1, shard=shard), device=dev)
    agent = pkg.Agent(cfg, env, device=dev)
    if standalone:                                             # union batch, no collective
        agent.rank, agent.world_size, agent.env_id_base, agent.global_envs = 0, 1, 0, B
    agent.network.set_weights(weights)
    agent.before_train()
    actions = []
    for _ in range(cycles):
        for _ in range(T):
            a = agent.predict()
            actions.append(a.clone())
            scr, rew, term = env.act(a, is_training=True, fused=True)
            agent.observe(scr, rew, a, term)
            agent.step += 1
    torch.cuda.synchronize()
    n = agent.network
    return torch.stack(actions), n.params.clone(), n.rms.clone(), n.target_params.clone()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="nstep_q", choices=("async_q", "nstep_q", "sarsa"))
    ap.add_argument("--envs", type=int, default=24, help="envs per rank")
    ap.add_argument("--t-max", type=int, default=5)
    ap.add_argument("--actions", type=int, default=6)
    ap.add_argument("--cycles", type=int, default=5)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    pkg = importlib.import_module("async-rl-tensorflow_b200")
    B, T, A = args.envs, args.t_max, args.actions
    weights = pkg.src.network.initial_weights(A, seed=5, stddev=0.05, streams=True)

    acts, params, rms, target = run(pkg, dev, args.mode, B, T, A, args.cycles, (rank, world), weights, False,
                                       world)

    hi, lo = params.clone(), params.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    replica_diff = float((hi - lo).abs().max())
    all_acts = [torch.empty_like(acts) for _ in range(world)]
    dist.all_gather(all_acts, acts)
    ok = True
    if rank == 0:
        u_acts, u_params, u_rms, u_target = run(pkg, dev, args.mode, B * world, T, A, args.cycles, None, weights,
                                                 True, world)
        acts_equal = bool(torch.equal(torch.cat(all_acts, dim=1), u_acts))
        scale = float(u_params.abs().max())
        p_err = float((params - u_params).abs().max()) / scale
        r_err = float((rms - u_rms).abs().max()) / float(u_rms.abs().max())
        t_err = float((target - u_target).abs().max()) / float(u_target.abs().max())
        synced = bool(not torch.equal(u_target, torch.cat([torch.as_tensor(w).reshape(-1) for w in
                                                            weights.values()]).to(dev)))
        ok = acts_equal and p_err <= 1e-5 and r_err <= 1e-5 and t_err <= 1e-5 and replica_diff == 0.0 and synced
        print(json.dumps({"world": world, "envs_per_rank": B, "cycles": args.cycles, "loss_mode": args.mode,
                          "dueling_streams": True, "actions_bit_identical": acts_equal, "param_rel_err": p_err, "rms_rel_err": r_err,
                          "target_rel_err": t_err, "target_synced_in_run": synced,
                          "replica_max_minus_min": replica_diff, "ok": ok}), flush=True)
    flag = torch.tensor([0 if ok else 1], device=dev)
    dist.all_reduce(flag)
    dist.destroy_process_group()
    sys.exit(1 if int(flag.item()) else 0)


if __name__ == "__main__":
    main()
