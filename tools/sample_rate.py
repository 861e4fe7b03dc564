"""tools/sample_rate.py -- what the Philox action sampler (policy_fused.sample, dcmp_sample) costs on one GPU, in one process:

  1. dcmp_sample against policy.sample_actions (torch.multinomial) on [B, 51] log-probabilities, B = 8,192 and 65,536 (CUDA events over
     500 calls after 50 untimed ones; the inputs stay resident in L2, as the log-probabilities a forward just wrote are);
  2. GraphedRollout with the fused forward and the trainer's compaction fractions at 8,192 synthetic 20A/50T envs, sampled with either
     sampler, alternated three times (env-steps = decisions played, summed over the envs);
  3. evaluate_sampled (LF) on the 50 bundled instances at K = 1, 128 and 1,024 with the fused forward and the fp32 module: wall time of the
     call after one untimed call at the same K, and torch.cuda.max_memory_allocated at the default max_envs.

The card's name and power limit are read in the same process.  One JSON object per line on stdout and in --out.

    python tools/sample_rate.py --out sample_rate.jsonl
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

from dcmrta_b200 import BatchedTaskEnv  # noqa: E402
from dcmrta_b200.evaluate import evaluate_sampled, load_test_set  # noqa: E402
from dcmrta_b200.policy import AttentionNet, sample_actions  # noqa: E402
from dcmrta_b200.policy_fused import draw_tensor, sample  # noqa: E402
from dcmrta_b200.rollout import GraphedRollout  # noqa: E402

FRACTIONS = (1.0, 0.85, 0.7, 0.5, 0.35, 0.2, 0.1, 0.03)                     # TrainerConfig.rollout_fractions


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn, iters=500, warm=50):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3                                   # us per call


def kernel_rates(emit):
    for B in (8192, 65536):
        g = torch.Generator(device="cuda").manual_seed(0)
        logp = torch.log_softmax(torch.randn(B, 51, device="cuda", generator=g) * 2, 1)
        mask = (torch.rand(B, 51, device="cuda", generator=g) < 0.3).to(torch.uint8)
        mask[:, 0] = 0
        logp = logp.masked_fill(mask.bool(), -1e4)
        draw = draw_tensor(1, 0, 0, logp.device)
        out = torch.empty(B, dtype=torch.int32, device="cuda")
        us_philox = timed(lambda: sample(logp, mask, draw, None, 0, out))
        us_multi = timed(lambda: sample_actions(logp))
        emit(dict(what="sampler", B=B, n=51, dcmp_sample_us=round(us_philox, 2), multinomial_us=round(us_multi, 2)))


def rollout_rates(emit, B=8192, repeats=3):
    torch.manual_seed(0)
    net = AttentionNet(6, 5, 128).cuda().eval()
    env = BatchedTaskEnv(B, 20, 50, M=5, auto_reset=False, seed=5, first_gid=0)
    env.generate(max_duration=5.0)
    ro = GraphedRollout(env, 280, record=False, fractions=FRACTIONS)
    arms = {"multinomial": None, "philox": (7, 0)}
    for s in arms.values():                                                  # captures and a first untimed rollout per arm
        ro.run(net, "sample", amp="fused", sampler=s)
    rates = {k: [] for k in arms}
    for _ in range(repeats):
        for name, s in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ep = ro.run(net, "sample", amp="fused", sampler=s)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            rates[name].append(float(ep.metrics[:, 7].sum()) / dt)
    env.close()
    emit(dict(what="graphed_rollout", B=B, shape="20A/50T", forward="fused", fractions=list(FRACTIONS),
              env_steps_per_s={k: [round(v, -3) for v in r] for k, r in rates.items()}))


def evaluation_rates(emit):
    sets = load_test_set(ROOT / "tests" / "golden" / "instances_20A_50T.npz")
    torch.manual_seed(0)
    net = AttentionNet(6, 5, 128).cuda().eval()
    for amp in ("fused", False):
        for K in (1, 128, 1024):
            evaluate_sampled(net, sets, K, amp=amp)                           # untimed: allocator, cuBLAS algorithms, the fused re-layout
            torch.cuda.reset_peak_memory_stats()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m = evaluate_sampled(net, sets, K, amp=amp)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            emit(dict(what="evaluate_sampled", method="LF", forward="fused" if amp else "fp32", K=K, envs=50 * K, seconds=round(dt, 3),
                      decisions=int(m[:, :, 7].sum()), max_memory_allocated_GB=round(torch.cuda.max_memory_allocated() / 1e9, 2),
                      best_reward_mean=round(float(m[:, :, 0].max(1).mean()), 4), reward_mean=round(float(m[:, :, 0].mean()), 4)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/sample_rate.py measures on a GPU; there is none here")
    lines = []

    def emit(d):
        d = dict(card=card(), **d)
        print(json.dumps(d), flush=True)
        lines.append(d)
    kernel_rates(emit)
    rollout_rates(emit)
    evaluation_rates(emit)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
