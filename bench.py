"""bench.py -- env-frames/sec through preprocess + forward + backward + update.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W

One "step" = one A3C cycle of the hot path: t_max env steps for every env of this rank
(K1 preprocess+ring push, forward, action sampling), the bootstrap forward, n-step returns +
loss gradients, the backward over the t_max*envs samples, [NCCL all-reduce of the gradient at
N>1], per-tensor clip + RMSProp.  Workload at N=1: BASELINE.json configs[2]/[3] -- 4096 envs
per GPU, 6-action head, t_max 5, synthetic 210x160x3 uint8 frames (weak scaling: 4096 per GPU).

Prints ONE JSON line (contract in the task statement): value = device-resident throughput,
e2e = the same cycle through the public API with frames in pinned HOST memory (H2D of every
frame and D2H of the actions/loss inside the timed region), roofline = the dominant kernel
timed live with CUDA events, cpu_baseline = the CPU port of the reference path on this box.

    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

also writes what the last timed cycle of the device-resident arm computed as DIR/<name>.npy
(see dump_outputs).  Frames, weights, random starts and action draws are all seeded, so the same
arguments give the same inputs on every run and two builds can be compared output for output.
"""
import argparse
import importlib
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env_frames_per_sec"
UNIT = "frames/s"

# Work per unit (SURVEY.md §8d, DESIGN.md kernel table).  Two byte counts per entry:
#   "bytes"      ALGORITHMIC, layout-independent: every distinct tensor the entry touches counted
#                once at its natural size (u8 frames / stack, float32 activations and gradients as
#                the reference holds them, no padding, no second read) -- what a fused
#                implementation of the entry cannot avoid.  roofline.frac uses this.
#   "impl_bytes" what the kernels behind the entry move as built (a tensor read by two kernels
#                counts twice, padded grids count their padding) -- the ncu DRAM traffic tracks it.
def entry_work(A):
    stack, a1, a2, h = 28224, 25600, 10368, 1024
    a1s, da1s = 12800, 14112          # a1 and d_a1 (21x21 grid) as stored: one fp16 per value (a2, d_a2, h, d_h: 4 bytes)
    heads_out = 4 * (2 * A + 1)
    dhead = 4 * (A + 1)
    return {
        # entry: (kernels, flop per unit (one exact pass), algorithmic bytes, bytes as built)
        "arl_preprocess_push": ("preprocess_kernel", 0.0, 80640 + 7056, 80640 + 7056),
        "arl_conv1_forward": ("tc_kernel<Conv1Fwd> (kind::i8, bulk-copied ring)", 2.0 * 1638400,
                              stack + a1, stack + a1s),
        "arl_conv2_forward": ("tc_kernel<Conv2Fwd> (bulk-copied fp16 a1s, split-bf16 a2 blocks out)",
                              2.0 * 663552, a1 + a2, a1s + a2),
        # fc256, then heads + softmax + Philox draw as one warp-per-sample launch
        "arl_fc_heads_forward": ("tc_kernel<FcFwdCluster> (bulk-copied split-bf16 operands) + heads_fwd_kernel (heads + sampling)",
                                 2.0 * 663552 + 2.0 * 256 * (A + 1), a2 + h + heads_out + 4, a2 + h + heads_out + 4),
        "arl_heads_forward": ("heads_fwd_kernel", 2.0 * 256 * (A + 1), h + heads_out, h + heads_out),
        "arl_sample_actions": ("sample_actions_kernel", 0.0, 4 * A + 4, 4 * A + 4),
        "arl_returns_lossgrad": ("returns_lossgrad_kernel", 0.0, 4 * (A + 1) + 9 + 4 + 4 * (A + 1),
                                 4 * (A + 1) + 9 + 4 + 4 * (A + 1)),
        # d_h is written twice (block + transposed copy for the weight gradient)
        "arl_heads_backward": ("heads_bwd_kernel", 4.0 * 256 * (A + 1), h + dhead + h, h + dhead + 2 * h),
        # algorithmic: d_h + a2 (operand and relu mask) in, d_a2 out.  As built: dgrad reads d_h + the
        # hi half of a2 (mask) and writes d_a2; wgrad reads a2 + d_h again
        "arl_fc_backward": ("tc_kernel<BulkGemm fc dgrad> + <fc wgrad>", 4.0 * 663552,
                            h + a2 + a2, h + a2 // 2 + a2 + a2 + h),
        # algorithmic: a1 + d_a2 in, d_a1 out (VERDICT r1: 61 568).  As built: wgrad reads a1 (fp16) +
        # d_a2, dgrad reads d_a2 again + a1 (relu mask) and writes d_a1 on the padded 21x21 grid
        "arl_conv2_backward": ("tc_kernel<Conv2Wgrad> + <Conv2Dgrad>", 4.0 * 663552,
                               a1 + a2 + a1, a1s + a2 + a2 + a1s + da1s),
        "arl_conv1_backward": ("tc_kernel<Conv1Wgrad> (bulk-copied d_a1 grid)", 2.0 * 1638400,
                               stack + a1, stack + da1s),
        # per PARAMETER (unit = one parameter): grad, rms, param read; rms, param written
        "arl_clip_rmsprop": ("sumsq_kernel + rmsprop_kernel", 6.0, 20, 24),
        # N > 2 GPUs (collective 'library'): the sum of the flat gradient over the ranks, per PARAMETER
        # (one read + one write of the local buffer; the time is launch + NVLink latency + rank skew)
        "arl_allreduce_grads": ("ncclAllReduce (launched by the library)", 1.0, 8, 8),
    }


def load_traffic():
    """DRAM bytes per launch of each entry's kernels from the committed ncu capture
    (profiles/r02_traffic.json, written by tools/ncu_traffic.py) -- null when absent."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(path):
        return json.load(open(path))
    return {}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tensor=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json; bf16 figure = sustained)")
    return dict(hbm=6650.0, tensor=1590.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._halt.is_set():
            self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for n, b in bits.items():
                if r & b:
                    self.reasons.add(n)
            self._halt.wait(0.01)

    def run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.2)

    def finish(self):
        self._halt.set()
        self.join(timeout=6)
        busy = [s for s in self.samples if s > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_reference(workers, t_max, actions, steps, warmup, cycles_per_step):
    """The reference's CPU ps/worker path (oracle/cpu_ref.py port), in a subprocess tree."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "cpu_ref.py"), "--workers", str(workers),
           "--t-max", str(t_max), "--actions", str(actions), "--steps", str(steps),
           "--warmup", str(warmup), "--cycles-per-step", str(cycles_per_step)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="1", MKL_NUM_THREADS="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    if out.returncode != 0:
        raise RuntimeError("cpu_ref failed: " + out.stderr[-2000:])
    return json.loads(out.stdout.strip().splitlines()[-1])


def run_reference(args, rank):
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    cyc = args.ref_cycles_per_step
    res = cpu_reference(cores, args.t_max, args.actions, args.steps, max(args.warmup, 1), cyc)
    total_t = sum(res["step_seconds"])
    value = res["frames_per_step"] * len(res["step_seconds"]) / total_t
    sample = ("%d worker processes (1 env, 1 torch thread each, shared hogwild parameter block) x "
              "%d cycles of t_max=%d frames per step" % (cores, cyc, args.t_max))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_t / len(res["step_seconds"]), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, ref=True),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, net, T, B, A):
    """Write what one A3C cycle hands back, float32, as out_dir/<name>.npy: the actions sampled at
    its t_max env steps, the logits / policy / values of its rollout forward ([T, B, ...]), the
    loss sums, the gradient its backward produced and the parameters and RMSProp state its update
    left.  Above DUMP_BYTES in all, the per-env arrays keep a fixed, seeded sample of the envs,
    whose indices go to env_index.npy.  The loss sums are accumulated with float atomics, so they
    may differ in the last bits from run to run; the other arrays repeat bit for bit."""
    out = {"params": net.params, "rms": net.rms, "grads": net.grads, "loss_sums": net.loss_sums}
    out = {k: v.float().cpu().numpy() for k, v in out.items()}
    rollout = {"actions": net.sampled_action.view(T, B), "logits": net.policy_logits.view(T, B, A),
               "policy": net.policy.view(T, B, A), "value": net.value.view(T, B)}
    rollout = {k: v.float().cpu().numpy() for k, v in rollout.items()}
    fixed = sum(v.nbytes for v in out.values()) + 4096                # + room for the .npy headers
    per_env = sum(v[:, :1].nbytes for v in rollout.values())
    if fixed + B * per_env > DUMP_BYTES:
        keep = (DUMP_BYTES - fixed) // (per_env + 8)
        idx = np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
        rollout = {k: v[:, idx] for k, v in rollout.items()}
        out["env_index"] = idx.astype(np.float64)
    out.update(rollout)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def workload_config(args, ref=False):
    return {"workload": "A3C full update, %d envs/GPU, conv16-conv32-fc256, %d-action head, "
                        "t_max %d, history 4, shared RMSProp (BASELINE.json configs[2]/[3])"
                        % (args.envs, args.actions, args.t_max),
            "envs_per_gpu": args.envs, "t_max": args.t_max, "action_size": args.actions,
            "frame": "210x160x3 uint8", "frames_per_step_per_gpu": args.envs * args.t_max,
            "l2_policy": "inputs larger than L2: each env step reads %d MB of fresh frames (pool of %s steps)"
                         % (args.envs * 100800 // 2 ** 20, getattr(args, "pool_used", "t_max")),
            "parallelism": "dp%d (env-sharded; the 2.7 MB gradient is summed over the ranks once per step: "
                           "%s)" % (args.gpus, {"p2p": "read over NVLink peer memory inside the update kernel",
                                                "library": "ncclAllReduce inside the library",
                                                "torch": "torch.distributed all_reduce"}[
                                                    (getattr(args, "collective", None) or "auto").replace(
                                                        "auto", "p2p" if args.gpus == 2 else "library")])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="environments per GPU")
    ap.add_argument("--t-max", type=int, default=5)
    ap.add_argument("--actions", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--ref-cycles-per-step", type=int, default=40)
    ap.add_argument("--profile-all", action="store_true", help="print per-entry times to stderr")
    ap.add_argument("--collective", default=None, choices=[None, "auto", "p2p", "library", "torch"],
                    help="gradient exchange at N>1 (default: config.collective = auto)")
    ap.add_argument("--pool", type=int, default=0, help="steps of synthetic frames kept (0: t_max, capped to ~24 GB)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    # CPU baseline first (rank 0 at N=1 only), before this process touches CUDA
    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        cores = len(os.sched_getaffinity(0))
        try:
            res = cpu_reference(cores, args.t_max, args.actions, 2, 1, 250)   # ~10 s of CPU work
            cpu_base = {"value": res["frames_per_sec"], "unit": UNIT, "cores": cores,
                        "kind": "port",
                        "sample": "%d workers x 2 timed steps x 250 cycles x t_max %d = %d frames "
                                  "(%.1f s)" % (cores, args.t_max, 2 * res["frames_per_step"],
                                                sum(res["step_seconds"]))}
        except Exception as e:                                  # report, never fake
            cpu_base = {"value": None, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "failed: %s" % str(e)[:200]}

    import torch
    import torch.distributed as dist
    try:
        # pin this rank to the CPUs next to its GPU BEFORE any pinned host buffer is allocated
        # (first touch decides the NUMA node the end-to-end arm uploads from)
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
    except Exception:
        pass
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pkg = importlib.import_module("async-rl-tensorflow_b200")
    cabi = pkg._cabi
    peaks = load_peaks()
    B, T, A, K, W = args.envs, args.t_max, args.actions, args.steps, args.warmup
    over = {"model": "m1", "num_envs": B, "t_max": T}
    if args.collective:
        over["collective"] = args.collective
    cfg = pkg.config.get_config(over)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # the frame pool rotates over `pool` env steps (> L2 in any case: one step of 1024 envs is 103 MB);
    # default t_max, capped so that the pool stays under ~24 GB at the large sweep points
    pool = args.pool if args.pool > 0 else max(2, min(T, int(24e9 // (B * 100800))))
    args.pool_used = pool

    def make_agent(host):
        env = pkg.GymEnvironment(cfg, env=pkg.SyntheticAtari(B, A, seed=123 + rank, pool=pool,
                                                             device=dev, host=host), device=dev)
        agent = pkg.Agent(cfg, env, device=dev)
        random.seed(cfg.seed)                    # the random-start no-ops of new_random_game
        agent.before_train()
        return agent, env

    def cycle(agent, env, d2h=None):
        for _ in range(T):
            action = agent.predict()
            if d2h is not None:                                  # a host-side emulator needs them
                d2h["actions"].copy_(action, non_blocking=True)
            scr, rew, term = env.act(action, is_training=True, fused=True)
            agent.observe(scr, rew, action, term)
            agent.step += 1
        if d2h is not None:
            d2h["loss"].copy_(agent.network.loss_sums, non_blocking=True)
            torch.cuda.current_stream().synchronize()           # the caller reads the loss

    def timed(agent, env, d2h=None, sampler=None):
        for _ in range(W):
            cycle(agent, env, d2h)
        # the loop runs from CUDA graphs captured on first sight of each distinct launch-argument
        # set (ring position x buffer parity: a short period); keep warming up until a whole
        # period has replayed without a new capture so that no capture falls into the timed region
        seen, quiet = len(agent._graphs), 0
        for _ in range(64):
            if not agent.cuda_graphs or quiet >= 3:
                break
            cycle(agent, env, d2h)
            quiet = quiet + 1 if len(agent._graphs) == seen else 0
            seen = len(agent._graphs)
        barrier()
        if sampler:
            sampler.start()
        cabi.launch_count(reset=True)
        replays0, nodes0 = agent.graph_replays, agent.graph_kernels_replayed
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            cycle(agent, env, d2h)
        e1.record()
        barrier()
        # kernels of the library launched in the region: eagerly (counted by the library) + as
        # nodes of replayed graphs (counted when each graph was captured)
        launches = cabi.launch_count() + agent.graph_kernels_replayed - nodes0
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), launches, agent.graph_replays - replays0

    # ---- arm 1: inputs resident in HBM ----------------------------------------------------
    agent, env = make_agent(host=False)
    net = agent.network
    work = entry_work(A)
    n_params = int(net.params.numel())
    # (a) per-entry pass, untimed region: a CUDA-event pair around EVERY C-ABI entry of the cycle
    # (the composed arl_forward / arl_backward are issued as their per-layer entries: the same
    # kernels in the same order) for PROFILE_CYCLES cycles -> roofline.entries
    net.timed, net.events = {"*"}, {}
    k1_events = []

    k1_graph_events = []

    def k1_timer(name, *a):
        # while a CUDA graph is being captured the pair becomes two event-record NODES around K1's
        # kernel node: every replay re-records them, so after the timed region each captured pair
        # holds the timing of K1's last launch from that graph
        cap = torch.cuda.is_current_stream_capturing()
        kw = {"external": True} if cap else {}
        ea, eb = torch.cuda.Event(enable_timing=True, **kw), torch.cuda.Event(enable_timing=True, **kw)
        ea.record(); cabi.call(name, *a); eb.record()
        (k1_graph_events if cap else k1_events).append((ea, eb))

    def graph_events_ok():
        """Can a timing event pair live inside a captured graph on this torch / driver?"""
        try:
            x = torch.zeros(1 << 20, device=dev)
            g = torch.cuda.CUDAGraph()
            ea = torch.cuda.Event(enable_timing=True, external=True)
            eb = torch.cuda.Event(enable_timing=True, external=True)
            with torch.cuda.graph(g):
                ea.record(); x.add_(1.0); eb.record()
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            t = ea.elapsed_time(eb)
            return 0.0 < t < 5.0
        except Exception as e:                                   # noqa: BLE001 - any failure = fall back
            print("bench: event nodes inside a graph unavailable (%s); K1 is launched eagerly "
                  "between its events" % (str(e).splitlines()[0][:120],), file=sys.stderr)
            return False
    agent.history.timer = k1_timer
    for _ in range(2):
        cycle(agent, env)
    torch.cuda.synchronize()
    net.events, k1_events[:] = {}, []
    PROFILE_CYCLES = 5
    for _ in range(PROFILE_CYCLES):
        cycle(agent, env)
    torch.cuda.synchronize()
    launch_ms = {n: [a.elapsed_time(b) for a, b in ev] for n, ev in net.events.items()}
    for alias in ("arl_clip_rmsprop_sched", "arl_exchange_clip_rmsprop"):      # K5 under its other entry names
        if alias in launch_ms:
            launch_ms.setdefault("arl_clip_rmsprop", []).extend(launch_ms.pop(alias))
    launch_ms["arl_preprocess_push"] = [a.elapsed_time(b) for a, b in k1_events]
    per_entry = {n: sum(v) / PROFILE_CYCLES for n, v in launch_ms.items()}
    traffic_all = load_traffic()

    def units_of(entry):
        if entry in ("arl_clip_rmsprop", "arl_allreduce_grads"):
            return n_params
        if entry.endswith("_backward") or entry == "arl_returns_lossgrad":
            return B * T
        # above 16 384 envs the forward entries run once per env range (arl_a2_block_rows)
        return cabi.a2_block_rows(B) if entry.endswith("_forward") else B

    def roof(entry, avg_ms):
        kname, flop_per, bytes_per, impl_per = work[entry]
        units = units_of(entry)
        t_hbm = bytes_per * units / (peaks["hbm"] * 1e9)
        t_tensor = flop_per * units / (peaks["tensor"] * 1e12)
        gbs = bytes_per * units / (avg_ms * 1e-3) / 1e9
        tfs = flop_per * units / (avg_ms * 1e-3) / 1e12
        # the bound is whichever roof gives the LONGER ideal time for the entry's algorithmic work
        hbm = t_hbm >= t_tensor
        return {"kernel": kname, "bound": "hbm" if hbm else "tensor",
                "achieved": gbs if hbm else tfs, "peak": peaks["hbm"] if hbm else peaks["tensor"],
                "unit": "GB/s" if hbm else "TFLOP/s",
                "frac": (gbs / peaks["hbm"]) if hbm else (tfs / peaks["tensor"]),
                "frac_impl_bytes": impl_per * units / (avg_ms * 1e-3) / 1e9 / peaks["hbm"],
                "avg_launch_ms": avg_ms, "units_per_launch": units,
                "algorithmic_bytes_per_unit": bytes_per, "impl_bytes_per_unit": impl_per,
                "algorithmic_flop_per_unit": flop_per, "hbm_gbs": gbs, "tensor_tflops": tfs,
                "traffic": (traffic_all.get(entry) or {}).get("dram_bytes_per_launch")}

    entries = {}
    for n, v in sorted(launch_ms.items(), key=lambda x: -per_entry[x[0]]):
        if n in work and v:
            e = roof(n, sum(v) / len(v))
            e["launches_per_step"] = len(v) // PROFILE_CYCLES
            e["ms_per_step"] = per_entry[n]
            entries[n] = e
    # fused floors of the chains (VERDICT r1 #5): only what enters / must be kept leaves a count
    fwd = ["arl_conv1_forward", "arl_conv2_forward", "arl_fc_heads_forward"]
    bwd = ["arl_heads_backward", "arl_fc_backward", "arl_conv2_backward", "arl_conv1_backward"]
    fwd_bytes = 28224 + 25600 + 10368 + 1024 + 4 * (2 * A + 1)      # stack in; a1, a2, h, heads kept
    bwd_bytes = 1024 + 4 * (A + 1) + 10368 + 25600 + 28224          # h, d heads, a2, a1, stack in
    chains = {}
    if all(k in per_entry for k in fwd + bwd):
        f_ms, b_ms = sum(per_entry[k] for k in fwd), sum(per_entry[k] for k in bwd)
        k1_ms, k5_ms = per_entry["arl_preprocess_push"], per_entry.get("arl_clip_rmsprop", 0.0)
        chains["forward_chain"] = {"ms_per_step": f_ms, "bytes_per_sample": fwd_bytes,
                                   "frac": fwd_bytes * B * (T + 1) / (f_ms * 1e-3) / 1e9 / peaks["hbm"]}
        chains["backward_chain"] = {"ms_per_step": b_ms, "bytes_per_sample": bwd_bytes,
                                    "frac": bwd_bytes * B * T / (b_ms * 1e-3) / 1e9 / peaks["hbm"]}
        cyc_bytes = 87696 * B * T + fwd_bytes * B * (T + 1) + bwd_bytes * B * T + 20 * n_params
        chains["cycle"] = {"bytes_per_step": cyc_bytes, "sum_of_entries_ms": sum(per_entry.values())}
    dominant = max(entries, key=lambda k: entries[k]["ms_per_step"])
    if world > 1:
        # every rank must take the same path below (the eager re-run contains collectives): rank 0 decides
        box = [dominant]
        dist.broadcast_object_list(box, src=0)
        dominant = box[0]
    if args.profile_all and rank == 0:
        print("per-entry ms per step:", json.dumps({k: round(v, 4) for k, v in
                                                    sorted(per_entry.items(), key=lambda x: -x[1])}),
              file=sys.stderr)
    # (b) timed region: the loop as a user runs it (CUDA graphs on).  Kernels inside a captured
    # graph cannot carry event pairs, so the dominant entry is timed live in the region only when
    # it is K1 (launched eagerly between its events, the rest of the step still replayed); for any
    # other dominant entry the K steps are run once more eagerly with events around that entry.
    net.timed, net.events, k1_events[:] = None, {}, []
    agent.history.timer = k1_timer if dominant == "arl_preprocess_push" else None
    in_graph = dominant == "arl_preprocess_push" and agent.cuda_graphs and graph_events_ok()
    agent.history.timer_in_graph = in_graph
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_total, launches, replays = timed(agent, env, sampler=sampler)
    clocks = sampler.finish() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, net, T, B, A)
    value = world * B * T * K / (ms_total * 1e-3)
    timed_in = "timed region (K1 launched between events, everything else replayed from CUDA graphs)"
    if dominant == "arl_preprocess_push" and in_graph and k1_graph_events:
        # one pair per captured observe graph (ring position x buffer parity: a period of two
        # cycles = 2 T launches): the values left by each graph's LAST replay, i.e. by the last
        # two cycles of the timed region
        ev = k1_graph_events
        timed_in = ("timed region, whole step replayed from CUDA graphs: the event pair around K1 is a pair "
                    "of event-record nodes inside each captured graph; the %d launches timed are those of "
                    "the region's last two cycles" % len(ev))
    elif dominant == "arl_preprocess_push":
        ev = k1_events[-T * K:]
    else:
        agent.history.timer = None
        net.timed, net.events = {dominant}, {}
        for _ in range(K):
            cycle(agent, env)
        torch.cuda.synchronize()
        ev = net.events.get(dominant, [])
        timed_in = "eager re-run of the K steps right after the timed region (event pairs cannot sit inside a captured graph)"
    dom_ms = [a.elapsed_time(b) for a, b in ev]
    net.timed, agent.history.timer = None, None
    if "cycle" in chains:
        chains["cycle"]["ms_per_step"] = ms_total / K
        chains["cycle"]["frac"] = chains["cycle"]["bytes_per_step"] / (ms_total / K * 1e-3) / 1e9 / peaks["hbm"]

    roofline = roof(dominant, sum(dom_ms) / len(dom_ms)) if dom_ms else dict(entries[dominant])
    roofline.update({"entry": dominant, "launches_timed": len(dom_ms), "timed_in": timed_in,
                     "share_of_step": per_entry[dominant] / sum(per_entry.values()),
                     "peak_source": peaks["source"], "entries": entries, "chains": chains,
                     "entries_ms_per_step": {k: round(v, 4) for k, v in
                                             sorted(per_entry.items(), key=lambda x: -x[1])},
                     "note": "top level = the dominant entry timed live with CUDA events inside the "
                             "timed region; entries = every C-ABI entry of the cycle timed the same "
                             "way over %d cycles just before it.  frac = ALGORITHMIC bytes (each "
                             "tensor once, natural size) / time / peak; frac_impl_bytes = the bytes "
                             "the kernels move as built; traffic = ncu DRAM bytes per launch "
                             "(profiles/r02_traffic.json); flop = one exact pass" % PROFILE_CYCLES})
    params_checksum = float(net.params.double().sum().item())
    replica_spread = 0.0
    if world > 1:
        # every rank holds a replica: max - min over ranks of every parameter must be exactly 0
        lo, hi = net.params.clone(), net.params.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        replica_spread = float((hi - lo).abs().max().item())
    del agent, env, net
    torch.cuda.empty_cache()

    # ---- arm 2: end to end through the public API with HOST frames --------------------------
    e2e = None
    if not args.no_e2e:
        agent, env = make_agent(host=True)
        d2h = {"actions": torch.empty(B, dtype=torch.int32, pin_memory=True),
               "loss": torch.empty(3, dtype=torch.float32, pin_memory=True)}
        ms_e2e, _, _ = timed(agent, env, d2h=d2h)
        # what the host->device path of THIS box gives when nothing else runs (VERDICT r1 #7): every
        # rank copies its own pinned pool at the same time -- plain whole-frame cudaMemcpyAsync, and
        # the rows-only strided copy the loop uses -- max time over ranks
        syn = env.env
        def upload_rate(fn, nbytes, reps=10):
            for _ in range(2):
                fn(0)
            barrier()
            u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            u0.record()
            for i in range(reps):
                fn(i)
            u1.record()
            barrier()
            t = torch.tensor([u0.elapsed_time(u1)], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return nbytes * reps / (float(t.item()) * 1e-3) / 1e9
        plain = upload_rate(lambda i: syn._stage[i & 1].copy_(syn._frames[i % syn.pool], non_blocking=True),
                            B * 100800)
        rows = upload_rate(lambda i: cabi.call("arl_upload_frames", syn._frames[i % syn.pool].data_ptr(),
                                               cabi.ptr(syn._stage[i & 1]), B, cabi.stream_ptr()), B * 80640)
        e2e_value = world * B * T * K / (ms_e2e * 1e-3)
        e2e = {"value": e2e_value, "unit": UNIT,
               "h2d_bytes_per_step": T * B * 80640, "d2h_bytes_per_step": T * B * 4 + 12,
               "ms_per_step": ms_e2e / K,
               "upload": {"plain_memcpy_gbs_per_gpu": plain, "rows_only_copy_gbs_per_gpu": rows,
                          "aggregate_rows_only_gbs": rows * world,
                          "ceiling_frames_per_s": rows * world * 1e9 / 80640,
                          "e2e_fraction_of_ceiling": e2e_value * 80640 / (rows * world * 1e9),
                          "note": "all ranks copy at once from their own pinned pools, nothing else running; "
                                  "the e2e arm needs 80 640 B per frame over this path"},
               "note": "frames in pinned host memory, double-buffered upload of the 168 of 210 rows "
                       "the resize reads (arl_upload_frames: one 2-D copy per step); PCIe-bound"}
        del agent, env

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "dtype_note": "fp32 parameters, gradients, optimizer state and accumulation; tcgen05 operands as 16-bit "
                          "hi/lo pairs, conv1's output and the gradient w.r.t. it stored as one fp16 per value "
                          "(logits / values <= 6.4e-4, gradients <= 4e-4 vs the float64 oracle; bar 1e-3)",
            "config": workload_config(args), "clocks": clocks, "e2e": e2e,
            "gpu_launches": launches, "cuda_graph_replays": replays, "roofline": roofline,
            "parity": {"replica_max_minus_min": replica_spread, "params_checksum": params_checksum},
        }
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
