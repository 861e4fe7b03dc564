"""tools/ia_rate.py -- rates of the individual-agent (IA) protocol beside leader-follower (LF), in one process on one GPU.

  env    env-steps/s of the step path at --envs envs, 20A/50T synthetic instances, in-kernel random policy, auto-reset, after an
         untimed pre-roll to the steady state as bench.py does.  An env-step is one decision: one leader (LF) or one agent (IA).
         LF and IA alternate --repeats times; every figure is reported, the median is the summary.
  eval   wall time of dcmrta_b200.evaluate.evaluate over the 50 bundled instances (tests/golden/instances_20A_50T.npz) with a
         randomly initialised AttentionNet, for {LF, IA} x {fp32 module, fused forward}; one untimed run first, median of --repeats.
The card's name and power limit are read in the same process.  One JSON object is printed.

    python tools/ia_rate.py [--envs 65536] [--steps 1000] [--repeats 3]
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (x.strip() for x in q.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def env_rate(protocol, B, A, T, preroll, warmup, steps):
    import torch
    from dcmrta_b200 import BatchedTaskEnv
    env = BatchedTaskEnv(B, A, T, M=5, auto_reset=True, seed=1234, first_gid=0, protocol=protocol)
    env.generate(max_duration=5.0)
    env.reset()
    for _ in range(preroll + warmup):
        env.step(policy="random")
    torch.cuda.synchronize()
    s0, e0 = env.total_steps(), env.total_episodes()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        env.step(policy="random")
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    n, ep = env.total_steps() - s0, env.total_episodes() - e0
    env.close()
    return {"env_steps_per_s": n / (ms * 1e-3), "us_per_step": 1e3 * ms / steps, "episodes_ended_per_step": ep / steps}


def eval_time(net, inst, method, amp, repeats):
    import torch
    from dcmrta_b200.evaluate import evaluate
    m = evaluate(net, inst, method=method, amp=amp)               # untimed: builds, allocations, the fused weights
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m = evaluate(net, inst, method=method, amp=amp)
        times.append(time.perf_counter() - t0)
    return {"seconds": statistics.median(times), "all_seconds": times, "decisions": int(m[:, 7].sum()),
            "longest_episode": int(m[:, 7].max()), "makespan_mean": float(m[:, 2].mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--agents", type=int, default=20)
    ap.add_argument("--tasks", type=int, default=50)
    ap.add_argument("--preroll", type=int, default=600, help="untimed passes after the reset (IA episodes are ~185 decisions long)")
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    import torch
    from dcmrta_b200.evaluate import load_test_set
    from dcmrta_b200.policy import AttentionNet
    assert torch.cuda.is_available(), "tools/ia_rate.py measures on a CUDA device"
    out = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "envs": args.envs, "shape": f"{args.agents}A/{args.tasks}T",
           "steps": args.steps, "preroll": args.preroll, "warmup": args.warmup, "env": {"LF": [], "IA": []}}
    for _ in range(args.repeats):
        for p in ("LF", "IA"):
            out["env"][p].append(env_rate(p, args.envs, args.agents, args.tasks, args.preroll, args.warmup, args.steps))
    for p in ("LF", "IA"):
        out["env"][p + "_median_env_steps_per_s"] = statistics.median(r["env_steps_per_s"] for r in out["env"][p])
    torch.manual_seed(0)
    net = AttentionNet(6, 5, 128).cuda().eval()
    inst = load_test_set(ROOT / "tests" / "golden" / "instances_20A_50T.npz")
    out["eval"] = {f"{m}/{name}": eval_time(net, inst, m, amp, args.repeats) for m in ("LF", "IA") for name, amp in (("fp32", False), ("fused", "fused"))}
    out["card_after"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
