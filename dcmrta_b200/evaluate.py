"""dcmrta_b200/evaluate.py -- test-set evaluation of a checkpoint on the device: what the reference's RL_test.py does, in one batch.

RL_test.py loads `checkpoint["model"]` into the attention network, plays ONE greedy episode (argmax of the policy, worker.py:222)
on every instance of a test set, one instance after the other, and writes the per-instance perf_metrics (worker.py:103-108) to
<method>.csv.  It does so under either decision protocol:
  LF  leader-follower, Worker.run_test: a leader drawn per location group, followers drawn to fill the chosen task;
  IA  individual agent, Worker.run_test_IS (worker.py:159-198): every decider of a slot acts alone, in ascending id order.
Here all instances are played at once by one BatchedTaskEnv (protocol "LF" or "IA") driven by dcmrta_b200.rollout.  LF leader and
follower draws come from the Philox contract (DESIGN.md 5) keyed by `seed`, instance i being global env i; IA draws nothing.

    python -m dcmrta_b200.evaluate --checkpoint model/REINFORCE/checkpoint.pth --test-set testSet_20A_50T_CONDET \\
        --method IA --out REINFORCE_IA.csv

The default forward is the fp32 module, as in the reference; --amp fused (policy_fused.FusedPolicy) or --amp bf16 are opt-in.

--samples K (which the reference does not have) plays K sampled episodes per instance instead, all N K of them on the device, and reports
the best of the K per instance: the usual second number after greedy decoding for a learned routing / allocation policy.  Actions come from
the Philox sampler (policy_fused.sample, DESIGN.md 5) keyed by --sample-seed and the global env id, so the result does not depend on how
the N K envs are split into batches (--max-envs).
"""
from __future__ import annotations

import argparse
import pickle
import re
import sys
from pathlib import Path

import numpy as np

from .instance_io import METRIC_COLUMNS, write_metrics_csv

MAX_WAITING_TIME = 10           # RL_test.py:39
MAX_TIME = 100.0                # parameters.py:19: the reference loop stops at finished or this clock


# ---- test sets -------------------------------------------------------------------------------------------------------------
def load_test_set(path) -> dict:
    """Instances as dict(A, task_xy [N,T,2] f64, depot_xy [N,2] f64, req [N,T] i32, dur [N,T] f64).

    path: an .npz with those keys (the layout of tests/golden/instances_20A_50T.npz), or a directory of reference env_<i>.pkl files,
    taken in ascending i.  A pickle is imported by the drop-in TaskEnv (its __setstate__ reads the reference's dicts; this needs a
    CUDA device) and normalised as RL_test.py:34-44 does: max_waiting_time = 10, reset with its own dicts, clear_decisions."""
    p = Path(path)
    if p.is_dir():
        return _load_pickles(p)
    z = np.load(p)
    inst = dict(A=int(z["A"]), task_xy=np.asarray(z["task_xy"], np.float64), depot_xy=np.asarray(z["depot_xy"], np.float64),
                req=np.asarray(z["req"], np.int32), dur=np.asarray(z["dur"], np.float64))
    N, T = inst["task_xy"].shape[:2]
    if inst["depot_xy"].shape != (N, 2) or inst["req"].shape != (N, T) or inst["dur"].shape != (N, T):
        raise ValueError(f"{p}: expected task_xy [N,T,2], depot_xy [N,2], req [N,T], dur [N,T]")
    return inst


def _load_pickles(d: Path) -> dict:
    from .task_env import TaskEnv

    class Unpickler(pickle.Unpickler):          # RL_test.py:35 pickles name the reference class: hand out the drop-in instead
        def find_class(self, module, name):
            return TaskEnv if name == "TaskEnv" else super().find_class(module, name)

    files = sorted((f for f in d.iterdir() if re.fullmatch(r"env_\d+\.pkl", f.name)), key=lambda f: int(f.stem[4:]))
    if not files:
        raise FileNotFoundError(f"{d}: no env_<i>.pkl files")
    envs = []
    for f in files:
        with open(f, "rb") as fh:
            env = Unpickler(fh).load()
        env.max_waiting_time = MAX_WAITING_TIME                 # RL_test.py:36-44
        env.reactive_planning = False
        env.reset((env.task_dic, env.agent_dic, env.depot))
        env.clear_decisions()
        envs.append(env)
    A = {e.agents_num for e in envs}
    T = {e.tasks_num for e in envs}
    if len(A) != 1 or len(T) != 1:
        raise ValueError(f"{d}: one batch needs one shape, found agents {sorted(A)} and tasks {sorted(T)}")
    inst = dict(A=A.pop(), task_xy=np.stack([e._xy for e in envs]), depot_xy=np.stack([e._depot_xy for e in envs]),
                req=np.stack([e._req for e in envs]).astype(np.int32), dur=np.stack([e._dur for e in envs]))
    for e in envs:
        e._be.close()
    return inst


# ---- evaluation ------------------------------------------------------------------------------------------------------------
def evaluate(net, instances: dict, method: str = "LF", amp=False, seed: int = 0, device: int = 0, graphed: bool = False,
             horizon: int | None = None) -> np.ndarray:
    """One greedy episode per instance, all in one batch.  Returns the [N,8] f64 metrics (reward, success_rate, makespan, time_cost,
    waiting_time, travel_dist, efficiency, decisions).

    method "LF" | "IA"; amp False (fp32 module) | True (bf16 shadow copy) | "fused" (policy_fused.FusedPolicy); seed keys the LF leader
    and follower draws; graphed: replay the decision loop from a CUDA graph (rollout.GraphedRollout).  Every episode must end the way
    the reference loop ends one, finished or at MAX_TIME: an episode the horizon would cut raises instead of being scored."""
    import torch

    from .batched_env import BatchedTaskEnv
    from .rollout import BatchedRollout, GraphedRollout

    if method not in ("LF", "IA"):
        raise ValueError(f"method must be 'LF' or 'IA', not {method!r}")
    N, T = instances["task_xy"].shape[:2]
    A = int(instances["A"])
    M = max(5, int(np.max(instances["req"])))                 # member slots: the reference's max_coalition_size, or more if the set needs it
    # Decisions per episode are bounded by the clock, not by the shape; this is twice the longest seen (bundled 20A/50T, greedy: LF 190, IA 259)
    horizon = int(horizon or 8 * (A + T))
    env = BatchedTaskEnv(N, A, T, M=M, device=device, auto_reset=False, max_wait=float(MAX_WAITING_TIME), max_time=MAX_TIME,
                         seed=seed, first_gid=0, protocol=method)
    try:
        env.load_instances(instances["task_xy"], instances["depot_xy"], instances["req"], instances["dur"])
        R = GraphedRollout if graphed else BatchedRollout
        ep = R(env, horizon, record=False, check_every=8).run(net, "greedy", amp=amp)
        if not bool(ep.ended.all()):
            cut = torch.logical_not(ep.ended).nonzero().flatten().tolist()
            raise RuntimeError(f"{len(cut)} episode(s) not over after {ep.length} decisions (instances {cut[:8]}): raise `horizon`")
        return ep.metrics.cpu().numpy()
    finally:
        env.close()


def evaluate_sampled(net, instances: dict, samples: int, method: str = "LF", amp=False, seed: int = 0, sample_seed: int = 0,
                     device: int = 0, graphed: bool = False, horizon: int | None = None, max_envs: int = 32768) -> np.ndarray:
    """K = `samples` sampled episodes per instance.  Returns the [N,K,8] f64 metrics (columns as `evaluate`).

    Env e = i K + k plays instance i, with global id e: LF leader and follower draws come from `seed` as in `evaluate` (so K = 1 keys
    everything exactly as the greedy run does), action draws from `sample_seed`, stream 0.  The N K envs run in contiguous chunks of at most
    `max_envs`, each with first_gid = its first env, so the table does not depend on the chunk size.  An episode the horizon would cut
    raises, as in `evaluate`."""
    import torch

    from .batched_env import BatchedTaskEnv
    from .rollout import BatchedRollout, GraphedRollout

    if method not in ("LF", "IA"):
        raise ValueError(f"method must be 'LF' or 'IA', not {method!r}")
    K, max_envs = int(samples), int(max_envs)
    if K < 1 or max_envs < 1:
        raise ValueError("samples and max_envs must be >= 1")
    N, T = instances["task_xy"].shape[:2]
    A = int(instances["A"])
    M = max(5, int(np.max(instances["req"])))
    horizon = int(horizon or 8 * (A + T))
    out = np.empty((N * K, 8), np.float64)
    R = GraphedRollout if graphed else BatchedRollout
    for e0 in range(0, N * K, max_envs):
        n = min(max_envs, N * K - e0)
        inst = np.arange(e0, e0 + n) // K
        env = BatchedTaskEnv(n, A, T, M=M, device=device, auto_reset=False, max_wait=float(MAX_WAITING_TIME), max_time=MAX_TIME,
                             seed=seed, first_gid=e0, protocol=method)
        try:
            env.load_instances(instances["task_xy"][inst], instances["depot_xy"][inst], instances["req"][inst], instances["dur"][inst])
            ep = R(env, horizon, record=False, check_every=8).run(net, "sample", amp=amp, sampler=(sample_seed, 0))
            if not bool(ep.ended.all()):
                cut = (e0 + torch.logical_not(ep.ended).nonzero().flatten()).tolist()
                raise RuntimeError(f"{len(cut)} episode(s) not over after {ep.length} decisions (envs {cut[:8]}): raise `horizon`")
            out[e0:e0 + n] = ep.metrics.cpu().numpy()
        finally:
            env.close()
    return out.reshape(N, K, 8)


def best_of(metrics):
    """[N,K,8] -> (best [N,8], k [N]): the sample of highest reward per instance, ties to the lowest k."""
    m = np.asarray(metrics, np.float64)
    k = np.argmax(m[:, :, 0], axis=1)                           # first maximum
    return m[np.arange(m.shape[0]), k], k


def metric_rows(metrics) -> list:
    """[N,8] metrics -> the per-instance perf_metrics dicts RL_test.py collects (worker.py:103-108)."""
    m = np.asarray(metrics, np.float64)
    return [dict(zip(METRIC_COLUMNS, (float(v) for v in row[1:7]))) for row in m]


def summary(metrics) -> str:
    """mean +- std (population) of each metric over the instances, one line each (how testSet_*/metrics/metrics.csv reports a method)."""
    m = np.asarray(metrics, np.float64)
    return "\n".join(f"{name:>13}: {m[:, c].mean():.3f} +- {m[:, c].std():.3f}" for c, name in enumerate(METRIC_COLUMNS, start=1))


# ---- command line ----------------------------------------------------------------------------------------------------------
def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="python -m dcmrta_b200.evaluate",
                                 description="Play a checkpoint greedily on a test set, one batch (the reference's RL_test.py), "
                                             "or best of K sampled episodes per instance (--samples K).")
    ap.add_argument("--checkpoint", required=True, help="torch checkpoint with a 'model' state dict (reference or ReinforceTrainer.save)")
    ap.add_argument("--test-set", required=True, help="instances .npz, or a directory of reference env_<i>.pkl files")
    ap.add_argument("--method", choices=("LF", "IA"), default="LF", help="leader-follower (run_test) or individual agent (run_test_IS)")
    ap.add_argument("--amp", choices=("none", "bf16", "fused"), default="none", help="policy forward: fp32 module (default), bf16 copy, fused kernels")
    ap.add_argument("--seed", type=int, default=0, help="Philox key of the LF leader / follower draws")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", required=True, help="per-instance metrics CSV (e.g. REINFORCE_IA.csv); with --samples, each instance's best sample")
    ap.add_argument("--samples", type=int, default=0, help="K sampled episodes per instance, best of K reported (default 0: one greedy episode)")
    ap.add_argument("--sample-seed", type=int, default=0, help="Philox key of the action draws of --samples")
    ap.add_argument("--max-envs", type=int, default=32768, help="envs per batch of --samples (the result does not depend on it)")
    ap.add_argument("--samples-out", help="optional .npz for the whole [N, K, 8] table of --samples (key 'metrics', plus 'best_k')")
    return ap.parse_args(argv)


def load_net(checkpoint, device: int = 0):
    """AttentionNet with checkpoint["model"]; the embedding width is read from the state dict."""
    import torch

    from .policy import AttentionNet
    # a checkpoint is a file of the user's own training run: the reference's also holds optimiser and scheduler state
    ck = torch.load(checkpoint, map_location=torch.device("cuda", device), weights_only=False)
    sd = ck["model"]
    net = AttentionNet(6, 5, int(sd["agent_embedding.weight"].shape[0])).to(torch.device("cuda", device))
    net.load_state_dict(sd)
    return net.eval()


def main(argv=None) -> int:
    args = parse_args(argv)
    amp = {"none": False, "bf16": True, "fused": "fused"}[args.amp]
    net = load_net(args.checkpoint, args.device)
    inst = load_test_set(args.test_set)
    if args.samples > 0:
        table = evaluate_sampled(net, inst, args.samples, method=args.method, amp=amp, seed=args.seed, sample_seed=args.sample_seed,
                                 device=args.device, max_envs=args.max_envs)
        best, k = best_of(table)
        write_metrics_csv(args.out, metric_rows(best))
        if args.samples_out:
            np.savez(args.samples_out, metrics=table, best_k=k)
        print(f"{args.method}: {table.shape[0]} instances x {args.samples} samples, {int(table[:, :, 7].sum())} decisions -> {args.out}")
        print(f"best of {args.samples}:\n{summary(best)}")
        print(f"all samples:\n{summary(table.reshape(-1, 8))}")
        return 0
    metrics = evaluate(net, inst, method=args.method, amp=amp, seed=args.seed, device=args.device)
    write_metrics_csv(args.out, metric_rows(metrics))
    print(f"{args.method}: {metrics.shape[0]} instances, {int(metrics[:, 7].sum())} decisions -> {args.out}")
    print(summary(metrics))
    return 0


if __name__ == "__main__":
    sys.exit(main())
