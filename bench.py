#!/usr/bin/env python
"""bench.py -- env-steps/s of the TaskEnv step on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA path through the C ABI); --steps / --warmup are its
                                                                  timed / untimed passes and are refused by the other arms below
  python bench.py --dump-outputs DIR [...]                        our arm, then what its last timed pass returned, as DIR/<name>.npy
                                                                  (this arm only: rollout / train / reference have no dump)
  python bench.py --impl reference [...]                          the reference's CPU implementation of the path
  torchrun --nproc-per-node N bench.py --gpus N ...               N > 1 (one rank per GPU, env shards, no collective on the data path);
                                                                  launched plainly with --gpus N > 1 it re-executes itself under torchrun
  python bench.py --total-envs 1048576 --agents A --tasks T --gpus N     BASELINE configs[3]: a fixed job sharded evenly (strong scaling)
  python bench.py --mode rollout|train [--fused|--amp] --gpus N           BASELINE configs[4]: the attention policy in the loop (--fused: the rollouts
                                                                          call policy_fused.FusedPolicy; --no-compact: every decision forwards every env)

A "step" is one pass of the hot path over one batch: ONE leader decision for every env of the batch (dcm_step:
apply the choice, coalition/feasibility update, agent update, slot advance, leader choice, observation + mask for the
next leader), B env-steps per GPU per step.  Workload = BASELINE.json configs[2]: 65,536 synthetic 20A/50T envs per GPU,
uniform-random policy over unmasked actions (in-kernel Philox), auto-reset, fp64 event clock, fp32 observations.  The timed passes
always see the STEADY STATE: an untimed pre-roll (--preroll, 400 passes) desynchronises the envs after the reset, and config.phase
reports how many episodes ended per timed pass.

  value        whole-job env-steps/s, state resident in HBM (CUDA events, max over ranks)
  e2e          same metric through the host-buffer C-ABI call (dcm_step_host): actions from pinned host memory (read in place by the
               step kernel), reward/done/next-leader D2H every step, observations written to the device-resident policy buffers
  e2e_full_obs as e2e but the observations and mask are also copied to pinned host memory every step (PCIe-bound)
  roofline     HBM: algorithmic bytes/step (SURVEY 8(d), w=8) x B / average duration of one pass (k_step, then k_episode_list on a
               side stream beside k_obs_tile; CUDA events on the launching stream, which joins the side stream before the next pass)
               vs MEASURED_PEAKS.json; traffic / dram_frac = the DRAM bytes ncu counted for one steady-state pass (profiles/traffic.json)
  cpu_baseline the C oracle port of the reference TaskEnv on the host cores, bounded sample of the same workload
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "env-steps/sec at 20A/50T"          # the headline shape; other --agents/--tasks name theirs (metric_name)
UNIT = "env-steps/s"
FALLBACK_HBM_GBS = 6650.0           # /opt/skills/guides/B200_PROFILING.md fallback


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, help="timed passes of the env step (default 2000; --mode env, --impl ours only)")
    p.add_argument("--warmup", type=int, help="untimed passes before them (default 200; --mode env, --impl ours only)")
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--envs", type=int, default=65536, help="envs per GPU (weak scaling)")
    p.add_argument("--total-envs", type=int, default=0, help="BASELINE configs[3]: this many envs in total, sharded evenly over the GPUs "
                                                              "(strong scaling; overrides --envs)")
    p.add_argument("--preroll", type=int, default=400, help="untimed passes after reset and before the warm-up, so that the timed passes see "
                                                            "the steady state (envs desynchronised, episodes ending every pass) whatever --warmup is")
    p.add_argument("--no-e2e", action="store_true", help="skip the e2e legs (shape sweeps)")
    p.add_argument("--agents", type=int, default=20)
    p.add_argument("--tasks", type=int, default=50)
    p.add_argument("--policy", default="random", choices=["random", "greedy"])
    p.add_argument("--e2e-steps", type=int, default=200)
    p.add_argument("--cpu-seconds", type=float, default=12.0)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--mode", default="env", choices=["env", "rollout", "train"],
                   help="env: the headline metric (step kernels only).  rollout / train: BASELINE configs[4], the same env-steps/s with the "
                        "PyTorch attention policy in the loop (rollout) and with the REINFORCE update + gradient all-reduce (train)")
    p.add_argument("--iters", type=int, default=3, help="--mode rollout/train: timed iterations (one episode per env each)")
    p.add_argument("--amp", action="store_true", help="--mode rollout/train: the rollouts call a bf16 shadow copy of the policy (the update stays fp32)")
    p.add_argument("--fused", action="store_true", help="--mode rollout/train: the rollouts call policy_fused.FusedPolicy (bf16 GEMMs + the sm_100a "
                   "kernels of include/dcmrta_policy.h between them); the update stays fp32 PyTorch")
    p.add_argument("--no-compact", action="store_true", help="--mode rollout/train: every decision forwards the whole batch (default: only the envs "
                   "that are still playing, at the fractions of the batch TrainerConfig.rollout_fractions names)")
    p.add_argument("--eager", action="store_true", help="--mode rollout/train: eager decision loop instead of the CUDA-graph replay")
    p.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned to its caller as DIR/<name>.npy "
                   "(float32; a fixed sample of the envs of rank 0 when the batch would exceed 64 MB), so that two builds can be compared output for output.  "
                   "--mode env, --impl ours only: the rollout / train modes and the reference arm have no dump")
    args = p.parse_args()
    if args.mode != "env" or args.impl != "ours":
        # the rollout / train modes time --iters iterations and the reference arm runs for --cpu-seconds
        given = [f for f, v in (("--steps", args.steps), ("--warmup", args.warmup), ("--dump-outputs", args.dump_outputs)) if v is not None]
        if given:
            p.error(f"{', '.join(given)}: --mode env --impl ours only (--mode rollout/train time --iters iterations, --impl reference "
                    "runs for --cpu-seconds)")
    args.steps = 2000 if args.steps is None else args.steps
    args.warmup = 200 if args.warmup is None else args.warmup
    return args


def metric_name(args):
    return METRIC if (args.agents, args.tasks) == (20, 50) else f"env-steps/sec at {args.agents}A/{args.tasks}T"


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.load(open(f))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(A, T, M=5, w=8):
    s_static = 2 * w * T + 2 * w + T + w * T
    s_dyn = T * (M * (1 + w) + 2 * w + 5) + A * (3 * w + 4) + 40
    s_obs = 4 * 6 * A + 4 * 5 * (T + 1) + (T + 1)
    return s_static + 2 * s_dyn + s_obs + 16


DUMP_LIMIT = 64_000_000


def dump_outputs(out_dir, env, first_gid):
    """What BatchedTaskEnv.step() hands its caller, as left by the last timed step: the next leader's agent / task observation and
    mask, the next leader, the step reward and done flag, and the action the in-kernel policy took.  All float32 (the integer and
    uint8 outputs are small enough to be exact).  When the whole batch would pass DUMP_LIMIT, the same envs are kept every run: a
    sample drawn from a fixed seed; env_index.npy (float64) holds their global ids."""
    import numpy as np
    import torch
    outs = {"agent_obs": env.agent_obs, "task_obs": env.task_obs, "mask": env.mask_u8, "next_leader": env.leader,
            "reward": env.reward, "done": env.done_u8, "action": env.used_action}
    per_env = 8 + 4 * sum(t[0].numel() for t in outs.values())
    n = min(env.B, (DUMP_LIMIT - 4096) // per_env)                 # 4 KB of room for the .npy headers
    idx = np.arange(env.B) if n == env.B else np.sort(np.random.default_rng(0).choice(env.B, n, replace=False))
    sel = torch.from_numpy(idx).to(env.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), (idx + first_gid).astype(np.float64))
    for name, t in outs.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.index_select(0, sel).float().cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                mx = float(f[1])
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(f[0]))
                    for n, v in zip(names, f[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(n)
            except ValueError:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores
# ----------------------------------------------------------------------------------------------------------------------
def python_reference_note():
    """The Python reference cannot run on the GPU box (its tree does not travel): the factor between it and the C port was measured in the
    build container by tools/time_python_reference.py and is quoted from the committed result."""
    f = ROOT / "profiles" / "r09_python_reference_rate.json"
    try:
        d = json.load(open(f))
        return (f"the Python reference itself: {d['python_reference_decisions_per_s']:.0f} decisions/s on 1 core in the build container, "
                f"{d['port_over_python']:.0f}x slower than this port on the same core (tools/time_python_reference.py, {f.name})")
    except Exception:
        return "the Python reference ran 455-541 decisions/s/core in the build container (SURVEY.md 6)"


def cpu_rollout(A, T, policy, seconds, threads=None, steps_per_thread=None):
    """All host cores, one env pool per thread (ctypes releases the GIL); returns (steps/s, cores, steps, elapsed)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle.oracle import OracleEnv, synthetic_instance
    n = threads or os.cpu_count() or 1
    pol = 1 if policy == "random" else 2
    envs = []
    for t in range(n):
        pool = []
        for q in range(8):
            ia = synthetic_instance(A, T, 5, seed=1234 + 8 * t + q)
            o = OracleEnv.make(**ia)
            o.seed(1234, gid=8 * t + q, episode=0)
            pool.append(o)
        envs.append(pool)
    # calibrate on one thread
    t0 = time.perf_counter()
    c = envs[0][0].rollout_bench(pol, 20000, seed=1)
    rate1 = c / (time.perf_counter() - t0)
    per_env = steps_per_thread // 8 if steps_per_thread else max(2000, int(rate1 * seconds / 8))

    def work(pool):
        return sum(o.rollout_bench(pol, per_env, seed=2) for o in pool)

    t0 = time.perf_counter()
    with ThreadPoolExecutor(n) as ex:
        total = sum(ex.map(work, envs))
    dt = time.perf_counter() - t0
    return total / dt, n, total, dt, rate1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    # warm-up
    cpu_rollout(args.agents, args.tasks, args.policy, 0.5)
    # a bounded sample of the workload: the run is sized to ~args.cpu_seconds of wall time on all host threads (it has no passes to
    # count, so the line reports no steps / ms_per_step)
    rate, cores, total, dt, rate1 = cpu_rollout(args.agents, args.tasks, args.policy, args.cpu_seconds)
    line = {
        "metric": metric_name(args), "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": None, "warmup": None,
        "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "impl": "reference",
        "config": {"workload": f"synthetic {args.agents}A/{args.tasks}T TaskEnv, {args.policy} policy, obs+mask built every decision",
                   "env_steps_timed": total, "threads": cores},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{total} decisions of the C oracle port (oracle/taskenv_oracle.c) over {cores} threads x 8 envs in {dt:.1f}s; "
                                   f"1-thread rate {rate1:.0f}/s; " + python_reference_note()},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from dcmrta_b200 import BatchedTaskEnv
    from dcmrta_b200.sharding import dist_env, reduce_job_totals, shard_range

    rank, local, world = dist_env()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    A, T = args.agents, args.tasks
    strong = args.total_envs > 0
    # weak scaling: args.envs per GPU; strong (--total-envs, BASELINE configs[3]): a fixed job sharded evenly.  Global ids are shard-invariant.
    first_gid, B = shard_range(args.total_envs if strong else args.envs * world, rank, world)
    env = BatchedTaskEnv(B, A, T, M=5, device=local, auto_reset=True, seed=1234, first_gid=first_gid)
    env.generate(max_duration=5.0)
    env.reset()
    # Pre-roll to the steady state (SURVEY 8(d) config 3: ">= 200 steps warm-up").  After a synchronised reset every env is in its
    # first slot and no episode ends for ~130 passes; the workload the metric is quoted on has the envs desynchronised, with ~B/150
    # episodes ending (accounting + restart) in every pass.  Untimed, ~50 ms.
    for _ in range(max(args.preroll, 0)):
        env.step(policy=args.policy)
    launches0 = env.launch_count()
    for _ in range(args.warmup):
        env.step(policy=args.policy)
    barrier()
    steps0 = env.total_steps()
    episodes0 = env.total_episodes()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches1 = env.launch_count()
    w0 = time.time()
    ev0.record()
    prof_at = int(os.environ.get("DCM_PROFILE_AT", "-1"))        # ncu --profile-from-start off: capture a few steady-state steps
    for k in range(args.steps):
        if k == prof_at:
            torch.cuda.synchronize(); torch.cuda.cudart().cudaProfilerStart()
        env.step(policy=args.policy)
        if k == prof_at + 1:
            torch.cuda.synchronize(); torch.cuda.cudart().cudaProfilerStop()
    ev1.record()
    torch.cuda.synchronize()
    w1 = time.time()
    launched = env.launch_count() - launches1
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    if args.dump_outputs and rank == 0:                              # before the e2e legs re-seed and reset the env
        dump_outputs(args.dump_outputs, env, first_gid)
    env_steps = env.total_steps() - steps0
    episodes_timed = env.total_episodes() - episodes0
    total_steps, ms_max = reduce_job_totals(env_steps, ms)          # env-steps summed over the ranks, time = max over the ranks
    ep_timed_all, _ = reduce_job_totals(episodes_timed, 0.0)
    ep_before_all, _ = reduce_job_totals(episodes0, 0.0)
    value = total_steps / (ms_max * 1e-3)

    # ---- end-to-end through the host-buffer C-ABI call ---------------------------------------------------------------
    def e2e(full_obs):
        K = args.e2e_steps
        env.seed(4321, first_gid=first_gid)
        env.reset()
        acts = torch.empty(K + 8, B, dtype=torch.int32).pin_memory()
        for k in range(K + 8):                      # record a valid action trace (deterministic given the Philox contract)
            env.step(policy=args.policy)
            acts[k].copy_(env.used_action, non_blocking=True)
        torch.cuda.synchronize()
        env.seed(4321, first_gid=first_gid)
        env.reset()
        torch.cuda.synchronize()
        out = {"next_leader": torch.empty(B, dtype=torch.int32).pin_memory(), "reward": torch.empty(B, dtype=torch.float32).pin_memory(),
               "done": torch.empty(B, dtype=torch.uint8).pin_memory()}
        if full_obs:
            out.update(agent_obs=torch.empty(B, A, 6, dtype=torch.float32).pin_memory(),
                       task_obs=torch.empty(B, T + 1, 5, dtype=torch.float32).pin_memory(),
                       mask=torch.empty(B, T + 1, dtype=torch.uint8).pin_memory())
        for k in range(8):
            env.step_host(acts[k], out)
        barrier()
        t0 = time.perf_counter()
        for k in range(8, K + 8):
            env.step_host(acts[k], out)             # H2D actions, step, D2H results; returns when the outputs are valid
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        d2h = sum(v.numel() * v.element_size() for v in out.values())
        return world * B * K / float(tt.item()), 4 * B, d2h

    if args.no_e2e:
        e_val = f_val = None; e_h2d = f_h2d = e_d2h = f_d2h = 0
    else:
        e_val, e_h2d, e_d2h = e2e(False)
        f_val, f_h2d, f_d2h = e2e(True)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    bytes_step = algorithmic_bytes(A, T)
    per_launch_s = ms_max * 1e-3 / args.steps
    achieved = bytes_step * B / per_launch_s / 1e9
    traffic, traffic_source = None, None
    tf = ROOT / "profiles" / "traffic.json"
    if tf.exists():
        try:
            tj = json.load(open(tf))
            traffic = tj.get(f"{A}x{T}x{B}")
            if traffic is not None:
                traffic_source = tj.get("_source", "ncu --set full capture of one steady-state pass of this workload (profiles/), not of the timed passes")
        except Exception:
            traffic = None
    dram = {}
    if traffic is not None:                                          # the same pass against the bytes ncu counted: the honest distance to the HBM limit
        dram = {"dram_achieved": traffic / per_launch_s / 1e9, "dram_frac": traffic / per_launch_s / 1e9 / peak}
    line = {
        "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": (f"{args.total_envs} synthetic {A}A/{T}T envs sharded evenly over {world} GPU(s) (BASELINE configs[3])" if strong else
                                f"{B} synthetic {A}A/{T}T envs per GPU (BASELINE configs[2])") +
                               f", {args.policy} policy (in-kernel Philox), auto-reset, fp64 event clock, fp32 obs; one step = one leader decision per env",
                   "envs_per_gpu": B, "total_envs": args.total_envs if strong else B * world, "agents": A, "tasks": T, "max_coalition": 5,
                   "phase": {"preroll_passes": args.preroll, "episodes_completed_before_timing": ep_before_all,
                             "ended_envs_per_pass": ep_timed_all / max(args.steps, 1),
                             "what": "steady state: envs desynchronised by the pre-roll, episode accounting + restart inside every timed pass"},
                   "l2": f"state {B * (env.record_bytes() + env.layout['sta_bytes']) / 1e6:.0f} MB + obs {B * 1551 / 1e6:.0f} MB per GPU > 126 MB L2, streamed every step (no flush needed)",
                   "parallelism": f"env shards x{world}, no data-path collective"},
        "e2e": {"value": e_val, "unit": UNIT, "h2d_bytes_per_step": e_h2d, "d2h_bytes_per_step": e_d2h,
                "what": "dcm_step_host: actions from pinned host memory, reward/done/next_leader to pinned host memory every step; obs stay in the device policy buffers"},
        "e2e_full_obs": {"value": f_val, "unit": UNIT, "h2d_bytes_per_step": f_h2d, "d2h_bytes_per_step": f_d2h,
                         "what": "as e2e plus agent_obs/task_obs/mask copied to pinned host memory every step"},
        "gpu_launches": launched, "env_steps_timed": total_steps,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source,
                     "kernel": "one pass = k_step, then k_episode_list (priority side stream) beside k_obs_tile", "algorithmic_bytes_per_env_step": bytes_step, "units_per_launch": B, "peak_source": peak_src,
                     "launch_us": per_launch_s * 1e6, **dram},
        "clocks": clocks,
    }
    if not args.no_cpu_baseline and world == 1:
        rate, cores, total, dt, rate1 = cpu_rollout(A, T, args.policy, args.cpu_seconds)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{total} decisions of the C oracle port over {cores} threads x 8 synthetic {A}A/{T}T envs in {dt:.1f}s "
                                          f"(1 thread: {rate1:.0f}/s); " + python_reference_note()}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_training(args):
    """BASELINE configs[4]: env-steps/s with the policy in the loop.  rollout: one sampled episode per env (policy forward +
    sampling + dcm_step per decision).  train: a full trainer iteration (sampled rollout, greedy baseline rollout, REINFORCE
    updates with the NCCL gradient all-reduce); env-steps counted = decisions of the sampled rollout only."""
    import torch
    import torch.distributed as dist
    from dcmrta_b200.sharding import dist_env
    from dcmrta_b200.trainer import ReinforceTrainer, TrainerConfig

    rank, local, world = dist_env()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.envs if args.envs != 65536 else 8192
    amp = "fused" if args.fused else args.amp
    cfg = TrainerConfig(agents=args.agents, tasks=args.tasks, envs_per_rank=B, amp=amp, seed=1234, eval_instances=max(world, 64),
                        graph_rollout=not args.eager, **({"rollout_fractions": (1.0,)} if args.no_compact else {}))
    tr = ReinforceTrainer(cfg, device=local)

    forwarded = [0, 0]                                               # policy rows forwarded / of them live, sampled rollouts of the timed iterations

    def one():
        if args.mode == "train":
            return tr.iteration()["decisions"]
        tr.env.generate(max_duration=5.0)
        ep = tr.rollout.run(tr.net, "sample", None if cfg.graph_rollout else tr.gen, amp=cfg.amp)
        n = int(ep.active.sum())
        forwarded[0] += ep.forwarded; forwarded[1] += n
        return n

    one()                                                            # warm-up (allocator, cuBLAS handles, autotune)
    forwarded[:] = [0, 0]
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    decisions = sum(one() for _ in range(args.iters))
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([float(decisions)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    if rank == 0:
        print(json.dumps({
            "metric": f"env-steps/sec at {args.agents}A/{args.tasks}T with the attention policy in the loop ({args.mode})",
            "value": float(cnt.item()) / (float(t.item()) * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.iters, "warmup": 1,
            "ms_per_step": float(t.item()) / args.iters, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 env / " + ("bf16 fused-kernel" if args.fused else "bf16" if args.amp else "fp32") + " policy", "data": "synthetic",
            "config": {"workload": f"BASELINE configs[4]: {B} synthetic {args.agents}A/{args.tasks}T envs per GPU, one episode per env per iteration, "
                                   f"AttentionNet(128) in PyTorch" + (", rollout forward = torch.mm GEMMs + libdcmrta_policy.so kernels" if args.fused else "") + f", mode={args.mode}, decision loop " + ("eager" if args.eager else "replayed from a CUDA graph"), "envs_per_gpu": B, "iterations": args.iters,
                       "parallelism": f"env shards x{world}" + (", one flat NCCL gradient all-reduce per update" if args.mode == "train" else "")},
            "env_steps_timed": float(cnt.item()),
            "policy_rows": ({"forwarded": forwarded[0], "live_fraction": forwarded[1] / forwarded[0], "fractions": list(cfg.rollout_fractions) if cfg.graph_rollout else [1.0]}
                            if forwarded[0] else None)}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # not launched under torchrun: re-exec ourselves with one rank per GPU (the driver launches torchrun itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29533", __file__] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    if args.impl == "reference":
        run_reference(args)
    elif args.mode != "env":
        run_training(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
