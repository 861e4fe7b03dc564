"""CPU tests of the individual-agent (IA) decision protocol (worker.py:159-198 `run_test_IS`, RL_test.py METHOD = 'IA'): the IA loop restated on
the C oracle's per-method calls (tests/ia_oracle.py) pinned to tests/golden/facade_is.npz (recorded from the real reference's IA loop), IA
episodes of the built-in policies, the fp32 stand-in policy the GPU tests use, the ABI flag, and the evaluation entry point's argument
parsing and CSV."""
import re
from pathlib import Path

import numpy as np
import pytest

from oracle import canon
from oracle.oracle import OracleEnv, synthetic_instance

from helpers import GOLD, pickle_instances
from ia_oracle import IAOracle

METRICS7 = ("reward", "success_rate", "makespan", "time_cost", "waiting_time", "travel_dist", "efficiency")


def facade_is():
    return np.load(GOLD / "facade_is.npz")


def nearest_open_task(mask, task_obs):
    """The stand-in policy of the GPU tests, on the fp32 observation alone: the open task nearest to the acting agent (task rows,
    columns 3-4 = task - agent), the depot only when nothing is open.  Ties go to the lowest index, as in the oracle's greedy."""
    d2 = task_obs[..., 3] * task_obs[..., 3] + task_obs[..., 4] * task_obs[..., 4]
    return int(np.argmin(np.where(mask.astype(bool), np.float32(np.inf), d2), axis=-1))


def test_ia_oracle_replays_reference_run_test_is():
    """The reference's own IA loop on three bundled instances: at every decision the acting agent, the clock, the observation digest
    and the full-state digest; then the final reward, the finished flags and the six metrics."""
    z = facade_is()
    inst = pickle_instances()
    for i in (int(x) for x in z["instances"]):
        agent, action = z[f"{i}/agent"], z[f"{i}/action"]
        n = len(agent)
        o = IAOracle(**inst[i])
        assert o.leader == int(agent[0]) == 0
        for k in range(n):
            a = int(agent[k])
            assert o.leader == a, (i, k)
            assert a == (o.pending & -o.pending).bit_length() - 1, (i, k)          # the lowest pending decider acts
            assert o.current_time == z[f"{i}/now"][k], (i, k)
            mask, ag, tk = o.mask(), o.agent_status(a).astype(np.float32), o.task_status(a).astype(np.float32)
            assert canon.obs_digest(mask, ag, tk) == int(z[f"{i}/dig_obs"][k]), (i, k)
            assert canon.state_digest(o.export()) == int(z[f"{i}/dig_state"][k]), (i, k)
            r, done, used, mover = o.step(int(action[k]))
            assert used == int(action[k]) and mover == a, (i, k)
            assert done == (k == n - 1), (i, k)
        assert o.n_steps == n and not o.stuck
        m, fin = o.episode_metrics()
        gold = z[f"{i}/metrics"]
        assert m["reward"] == gold[0]
        assert np.array_equal(fin, z[f"{i}/finished"])
        for c, key in enumerate(METRICS7[1:], start=1):
            assert m[key] == pytest.approx(gold[c], rel=1e-12, abs=0), (i, key)
        assert m["n_steps"] == n


@pytest.mark.parametrize("policy", [-1, -2])
def test_ia_builtin_policies_one_mover_per_decision(policy):
    """Synthetic 20A/50T instances, the random (-1) and greedy-nearest (-2) policies of the RNG contract: every IA episode ends, every
    decision moves the lowest pending decider, and its reward is -travel_time of that one agent."""
    for s in range(12):
        inst = synthetic_instance(20, 50, 5, seed=100 + s, random_duration=bool(s % 2))
        o = IAOracle(**inst)
        o.seed(77, gid=s, episode=0)
        assert o.reset() == 0
        k = 0
        while not o.done:
            a, pending = o.leader, o.pending
            assert a == (pending & -pending).bit_length() - 1
            frm = o.position(a)
            before = o.export()["has_route"].copy()
            r, done, used, mover = o.step(policy)
            assert mover == a and np.flatnonzero(o.export()["has_route"] != before).tolist() in ([], [a]), (s, k)
            to = inst["depot_xy"] if used == 0 else inst["task_xy"][used - 1]
            assert r == pytest.approx(-np.hypot(*(np.asarray(to) - np.asarray(frm))) / 0.2, rel=1e-12, abs=1e-15), (s, k)
            k += 1
            assert k < 2000
        assert o.n_steps == k and o.episode_metrics()[0]["n_steps"] == k and not o.stuck


def test_stand_in_policy_is_the_oracle_greedy_on_fp32_observations():
    """The nearest-open-task stand-in reads only what the network reads (fp32 rows); on every IA and every LF decision of the 50 bundled
    instances it picks the fp64 greedy-nearest action of the in-kernel policy, and on the reference's IA run (facade_is.npz) the recorded
    action -- so a torch module computing it checks the batched evaluation exactly."""
    n = 0
    for gid, inst in enumerate(pickle_instances()):
        o = IAOracle(**inst)
        while not o.done:
            want = o.policy_action(2)
            assert nearest_open_task(o.mask(), o.task_status(o.leader).astype(np.float32)) == want, ("IA", gid)
            o.step(want)
            n += 1
        o = OracleEnv.make(**inst)                                   # LF: the leader / follower draws of tests/test_gpu_individual_agent.py
        o.seed(17, gid=gid, episode=0)
        o.fused_reset()
        while not o.done:
            want = o.policy_action(2)
            assert nearest_open_task(o.mask(), o.task_status(o.leader).astype(np.float32)) == want, ("LF", gid)
            assert o.fused_step(want)[0] == 0
            n += 1
    assert n > 5000 + 4000
    z = facade_is()
    inst = pickle_instances()
    for i in (int(x) for x in z["instances"]):
        o = IAOracle(**inst[i])
        for act in z[f"{i}/action"]:
            assert nearest_open_task(o.mask(), o.task_status(o.leader).astype(np.float32)) == int(act)
            o.step(int(act))


def test_ia_episodes_are_longer_than_lf():
    """Callers size rollout horizons from this: on the bundled 20A/50T instances an IA episode takes more env steps than an LF one."""
    lf, ia = [], []
    for inst in pickle_instances()[:10]:
        o = OracleEnv.make(**inst)
        o.seed(0, gid=0, episode=0)
        o.fused_reset()
        while not o.done:
            o.fused_step(-2)
        lf.append(o.n_steps)
        o = IAOracle(**inst)
        while not o.done:
            o.step(-2)
        ia.append(o.n_steps)
    assert min(ia) > max(lf) * 0.9 and np.mean(ia) > 1.3 * np.mean(lf), (lf, ia)
    assert max(ia) < 8 * 70                                  # dcmrta_b200.evaluate's default horizon, 8 (A + T)


def test_abi_knows_the_individual_flag():
    from dcmrta_b200 import _lib
    hdr = (Path(__file__).resolve().parent.parent / "include" / "dcmrta.h").read_text()
    m = re.search(r"#define\s+DCM_FLAG_INDIVIDUAL\s+(\d+)u", hdr)
    assert m and int(m.group(1)) == _lib.FLAG_INDIVIDUAL == 4
    assert _lib.PROTOCOL == {"LF": 0, "IA": 4}
    assert not _lib.FLAG_INDIVIDUAL & (_lib.FLAG_AUTO_RESET | _lib.FLAG_REGENERATE)


def test_evaluate_cli_arguments_and_csv(tmp_path):
    from dcmrta_b200 import evaluate as ev
    a = ev.parse_args(["--checkpoint", "ck.pth", "--test-set", "set.npz", "--method", "IA", "--amp", "fused", "--seed", "3",
                       "--out", "REINFORCE_IA.csv"])
    assert (a.checkpoint, a.test_set, a.method, a.amp, a.seed, a.out) == ("ck.pth", "set.npz", "IA", "fused", 3, "REINFORCE_IA.csv")
    d = ev.parse_args(["--checkpoint", "c", "--test-set", "s", "--out", "o"])
    assert (d.method, d.amp, d.seed, d.device) == ("LF", "none", 0, 0)
    with pytest.raises(SystemExit):
        ev.parse_args(["--checkpoint", "c", "--test-set", "s", "--out", "o", "--method", "XY"])
    # the test set in the bundled layout
    inst = ev.load_test_set(GOLD / "instances_20A_50T.npz")
    assert inst["A"] == 20 and inst["task_xy"].shape == (50, 50, 2) and inst["req"].dtype == np.int32
    rng = np.random.default_rng(0)
    met = rng.random((50, 8))
    out = tmp_path / "REINFORCE_IA.csv"
    import pandas as pd
    from dcmrta_b200.instance_io import write_metrics_csv
    write_metrics_csv(out, ev.metric_rows(met))
    df = pd.read_csv(out, index_col=0)
    assert list(df.columns) == ["success_rate", "makespan", "time_cost", "waiting_time", "travel_dist", "efficiency"]
    assert df.shape == (50, 6) and list(df.index) == list(range(50))
    np.testing.assert_allclose(df.to_numpy(), met[:, 1:7], rtol=1e-12, atol=0)
    s = ev.summary(met).splitlines()
    assert len(s) == 6 and s[1].split(":")[0].strip() == "makespan" and f"{met[:, 2].mean():.3f} +- {met[:, 2].std():.3f}" in s[1]
