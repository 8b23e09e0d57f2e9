"""Multi-GPU parity check of the A3C LSTM agent (lstm=True), run under torchrun, one rank per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P tests/dist_gpu_check_lstm.py [--envs B] [--cycles C] [--collective auto|p2p|library]

Every rank runs C a3c cycles on its env shard (the exchange of the world size: the NCCL all-reduce of all
12 tensors inside arl_backward_lstm, or the peer-memory exchange over 13 offsets), with terminals inside
and at the end of rollouts.  Rank 0 then repeats the run in-process on the UNION batch (N*B envs, no
collective) and checks

  * policy samples: bit-identical to the union run's columns of every rank (Philox keyed by the global
    env id), which needs every rank's (h, c) to follow the union run's,
  * parameters + RMSProp slot after C updates: within 1e-5 of the union run, and each rank's LSTM state
    within 1e-5 of the union run's rows of its envs,
  * replicas: bit-identical across ranks.

Prints one JSON line on rank 0 and exits non-zero on failure.  tests/test_gpu_lstm.py launches it when the
box has >= 2 GPUs.
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


def run(pkg, dev, collective, B, T, A, cycles, shard, weights, standalone):
    random.seed(123)                                           # main.py:41
    cfg = pkg.config.get_config({"model": "m1", "num_envs": B, "t_max": T, "lstm": True, "collective": collective})
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
    return torch.stack(actions), n.params.clone(), n.rms.clone(), n.state_h.clone(), n.state_c.clone()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--collective", default="auto", choices=("auto", "p2p", "library"))
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
    weights = pkg.src.network.initial_weights(A, seed=5, stddev=0.05, lstm=True)

    acts, params, rms, sh, sc = run(pkg, dev, args.collective, B, T, A, args.cycles, (rank, world), weights, False)

    hi, lo = params.clone(), params.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    replica_diff = float((hi - lo).abs().max())
    all_acts = [torch.empty_like(acts) for _ in range(world)]
    dist.all_gather(all_acts, acts)
    all_h, all_c = [torch.empty_like(sh) for _ in range(world)], [torch.empty_like(sc) for _ in range(world)]
    dist.all_gather(all_h, sh)
    dist.all_gather(all_c, sc)
    ok = True
    if rank == 0:
        u_acts, u_params, u_rms, u_h, u_c = run(pkg, dev, args.collective, B * world, T, A, args.cycles, None, weights,
                                                True)
        acts_equal = bool(torch.equal(torch.cat(all_acts, dim=1), u_acts))
        p_err = float((params - u_params).abs().max()) / float(u_params.abs().max())
        r_err = float((rms - u_rms).abs().max()) / float(u_rms.abs().max())
        s_err = max(float((torch.cat(all_h) - u_h).abs().max()) / float(u_h.abs().max()),
                    float((torch.cat(all_c) - u_c).abs().max()) / float(u_c.abs().max()))
        ok = acts_equal and p_err <= 1e-5 and r_err <= 1e-5 and s_err <= 1e-5 and replica_diff == 0.0
        print(json.dumps({"world": world, "envs_per_rank": B, "cycles": args.cycles, "lstm": True,
                          "collective": args.collective, "actions_bit_identical": acts_equal, "param_rel_err": p_err,
                          "rms_rel_err": r_err, "state_rel_err": s_err, "replica_max_minus_min": replica_diff,
                          "ok": ok}), flush=True)
    flag = torch.tensor([0 if ok else 1], device=dev)
    dist.all_reduce(flag)
    dist.destroy_process_group()
    sys.exit(1 if int(flag.item()) else 0)


if __name__ == "__main__":
    main()
