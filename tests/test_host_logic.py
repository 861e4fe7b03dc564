"""CPU tests of host-side logic that needs no GPU."""
from pathlib import Path

import numpy as np
import pytest

from helpers import quirk_instance, quirk_traces, sweep_instance, sweep_traces


def test_instance_generator_matches_reference_rng_protocol():
    """TaskEnv(seed=s) must be the same instance as the reference's (task_env.py:57-71 draw order).

    The four cases of oracle/make_generator_golden.CASES (tests/golden/generator_cases.npz): agent and task counts drawn from ranges,
    fixed counts given as ranges, plain-int counts with M = 3, and the unseeded path that draws from the global NumPy state.  Their
    stored values are what this generator drew while this test compared it live with the reference TaskEnv in exactly these cases
    (generate_instance has not changed since); the script re-records them from the reference.

    Every instance the reference generator made for the other golden files: the shape sweep of traces_sweep.npz (TaskEnv((A, A),
    (T, T), 1, 5, seed=s), oracle/make_golden.py), the searched quirk fixtures of quirks.npz (M = 2 and 3, oracle/make_quirk_golden.py)
    and the three 10A/20T instances of rollout_golden.npz (oracle/make_rollout_golden.py)."""
    from dcmrta_b200.task_env import generate_instance
    from oracle.make_generator_golden import CASES, FIELDS, GLOBAL_SEED, UNSEEDED_FIELDS
    g = np.load(Path(__file__).resolve().parent / "golden" / "generator_cases.npz")
    for i, (ar, tr, M, s) in enumerate(CASES):
        if s is None:
            np.random.seed(GLOBAL_SEED)
        A, xy, dep, req, dur, cost = generate_instance(ar, tr, M, 5, None if s is None else np.random.default_rng(s))
        got = dict(A=A, task_xy=xy, depot_xy=dep, req=req, dur=dur)
        for k in (UNSEEDED_FIELDS if s is None else FIELDS):
            assert np.array_equal(got[k], g[f"case{i}/{k}"]), (i, k)

    cases = []
    tr = sweep_traces()
    for name in dict.fromkeys(n.rsplit("/", 1)[0] for n in tr.names):
        inst = sweep_instance(tr, name + "/random")
        cases.append((inst, len(inst["req"]), 5, int(name.split("/")[1])))
    q = quirk_traces()
    for name in q.names:
        if name.startswith("seed"):
            inst = quirk_instance(q, name)
            cases.append((inst, len(inst["req"]), int(q.z[f"inst/{name}/M"]), int(name[4:].split("_")[0])))
    r = np.load(Path(__file__).resolve().parent / "golden" / "rollout_golden.npz")
    for i, s in enumerate((3, 14, 27)):
        cases.append((dict(A=10, **{k: r[f"inst/{k}"][i] for k in ("task_xy", "depot_xy", "req", "dur")}), 20, 5, s))
    assert len(cases) == 17 and {M for _, _, M, _ in cases} == {2, 3, 5}
    for ia, T, M, s in cases:
        A, xy, dep, req, dur, cost = generate_instance((ia["A"], ia["A"]), (T, T), M, 5, np.random.default_rng(s))
        assert A == ia["A"] and np.array_equal(xy, ia["task_xy"]) and np.array_equal(dep, ia["depot_xy"]), (A, T, M, s)
        assert np.array_equal(req, ia["req"]) and np.array_equal(dur, ia["dur"]), (A, T, M, s)


def test_algorithmic_bytes_formula():
    """SURVEY.md 8(d): 10,633 B per env-step at 20A/50T/M5, 4,493 at 10A/20T, 39,733 at 50A/200T."""
    import bench
    assert bench.algorithmic_bytes(20, 50) == 10633
    assert bench.algorithmic_bytes(10, 20) == 4493
    assert bench.algorithmic_bytes(50, 200) == 39733


@pytest.mark.parametrize("B", [65536, 100])
def test_bench_dump_outputs_sample_and_size(tmp_path, B):
    """bench.py --dump-outputs on host tensors shaped like BatchedTaskEnv's buffers (20A/50T): every output as float, at most 64 MB in
    all, rows equal to the buffers they were taken from.  The headline batch (65,536 envs) is over the limit: the same envs are sampled
    every run.  A batch of 100 is written whole."""
    import types
    import torch
    import bench
    A, T = 20, 50
    g = torch.Generator().manual_seed(0)
    env = types.SimpleNamespace(B=B, device=torch.device("cpu"), agent_obs=torch.rand(B, A, 6, generator=g),
                                task_obs=torch.rand(B, T + 1, 5, generator=g), mask_u8=torch.randint(0, 2, (B, T + 1), generator=g, dtype=torch.uint8),
                                leader=torch.randint(0, A, (B,), generator=g, dtype=torch.int32), reward=torch.rand(B, generator=g),
                                done_u8=torch.randint(0, 2, (B,), generator=g, dtype=torch.uint8),
                                used_action=torch.randint(0, T + 1, (B,), generator=g, dtype=torch.int32))
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, env, first_gid=100)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["action.npy", "agent_obs.npy", "done.npy", "env_index.npy", "mask.npy", "next_leader.npy", "reward.npy", "task_obs.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64_000_000
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert idx.dtype == np.float64 and np.all(np.diff(idx) > 0)
    assert 30000 < len(idx) < B if B == 65536 else np.array_equal(idx, np.arange(B) + 100.0)
    rows = idx.astype(np.int64) - 100
    for name, t in (("agent_obs", env.agent_obs), ("task_obs", env.task_obs), ("mask", env.mask_u8), ("next_leader", env.leader),
                    ("reward", env.reward), ("done", env.done_u8), ("action", env.used_action)):
        a = np.load(tmp_path / "a" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy()[rows].astype(np.float32)), name
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{name}.npy")), name


def test_rollout_sub_batch_sizes_keep_the_forwarded_rows_live():
    """rollout.GraphedRollout forwards only the envs that are still playing, at the captured sizes of TrainerConfig.rollout_fractions, re-chosen
    at a poll every 8 decisions.  Host logic only: episode lengths come from the oracle playing the random policy on synthetic 20A/50T
    instances (120 +- 9 decisions); the schedule of sizes is simulated exactly as GraphedRollout.run walks it.  This is how the default
    fractions were chosen (DESIGN.md 9): forwarding every env at every decision keeps < 85 % of the forwarded rows live (400 envs; the longest of
    8,192 episodes is longer still), the default > 93 %
    (measured on 8,192 envs on a B200: 77.1 % and 95.5 %, profiles/r14*)."""
    import numpy as np
    from dcmrta_b200.rollout import rows_for, sub_batch_sizes
    from dcmrta_b200.trainer import TrainerConfig
    from oracle.oracle import OracleEnv, synthetic_instance
    assert sub_batch_sizes(300, (1.0, 0.75, 0.5, 0.25, 0.05)) == [15, 75, 150, 225, 300]
    assert sub_batch_sizes(8, (1.0, 0.85, 0.7, 0.5, 0.35, 0.2, 0.1, 0.03)) == [1, 2, 3, 4, 6, 7, 8]
    assert sub_batch_sizes(64, (1.0,)) == [64] and sub_batch_sizes(64, ()) == [64]
    assert rows_for([15, 75, 150, 225, 300], 76) == 150 and rows_for([15, 75, 150], 15) == 15 and rows_for([8], 1) == 8
    B = 400
    lengths = []
    for s in range(B):
        inst = synthetic_instance(20, 50, 5, 5000 + s)
        o = OracleEnv.make(20, inst["task_xy"], inst["depot_xy"], inst["req"], inst["dur"])
        o.seed(11, gid=s, episode=0)
        o.fused_reset()
        n = 0
        while not o.done and n < 400:
            o.fused_step(o.policy_action(1))
            n += 1
        lengths.append(n)
    L = np.array(lengths)
    assert 100 < L.mean() < 140 and L.max() < 280                     # inside the trainer's horizon of 4 (A + T)

    def live_fraction(fractions, every=8):
        sizes, rows, forwarded, t = sub_batch_sizes(B, fractions), B, 0, 0
        while True:
            forwarded += rows * every
            t += every
            n = int((L > t).sum())
            if n == 0:
                return L.sum() / forwarded
            rows = rows_for(sizes, n)
    full, default = live_fraction((1.0,)), live_fraction(TrainerConfig().rollout_fractions)
    assert full < 0.85 and default > 0.93 and default > live_fraction((1.0, 0.75, 0.5, 0.25)) > full + 0.05
