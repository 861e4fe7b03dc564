"""GPU tests of the individual-agent (IA) protocol on the fused step path (DCM_FLAG_INDIVIDUAL, BatchedTaskEnv(protocol="IA")) and of the
batched test-set evaluation (dcmrta_b200.evaluate): against tests/golden/facade_is.npz (the real reference's run_test_IS loop), against the
IA loop restated on the C oracle (tests/ia_oracle.py), and against the step path's own variants (serial pass, host buffers, shards)."""
from contextlib import closing

import numpy as np
import pytest

from dcmrta_b200._lib import ENV_DONE, ENV_ERR_FOLLOW, ENV_ERR_LEADER, ENV_ERR_MASK
from oracle import canon
from oracle.oracle import OracleEnv

from gpu_env import (assert_metrics_match, check_shard_invariance, lockstep, make_env, stack_instances, step_host_equals_step, twin_handles,
                     twin_steps)
from helpers import GOLD, METRIC_KEYS, EnvelopeShape, pickle_instances
from ia_oracle import IAOracle

pytestmark = pytest.mark.gpu


def facade_is():
    return np.load(GOLD / "facade_is.npz")


def nearest_task_module():
    """A torch stand-in for the attention network that reads only its fp32 inputs: the open task nearest to the acting agent (task rows,
    columns 3-4), the depot only when nothing is open.  It returns scores, not log-probabilities (argmax is all a greedy episode
    uses; a log_softmax could merge nearly equal scores).  tests/test_individual_agent.py shows it picks the oracle's greedy action."""
    import torch

    class NearestTask(torch.nn.Module):
        def forward(self, tasks, agents, mask):
            d2 = tasks[..., 3] * tasks[..., 3] + tasks[..., 4] * tasks[..., 4]
            return (-d2).masked_fill(mask, float("-inf"))

    return NearestTask().cuda()


def oracle_metrics(inst, protocol, seed=0, gid=0):
    """greedy-nearest episode of the CPU reference: the IA loop, or the oracle's leader-follower driver with the LF draws of (seed, gid)"""
    if protocol == "IA":
        o = IAOracle(**inst)
        while not o.done:
            o.step(-2)
    else:
        o = OracleEnv.make(**inst)
        o.seed(seed, gid=gid, episode=0)
        o.fused_reset()
        while not o.done:
            assert o.fused_step(-2)[0] == 0
    m, _ = o.episode_metrics()
    return np.array([m[k] for k in METRIC_KEYS])


def test_replay_reference_run_test_is_through_dcm_step():
    """The three recorded IA episodes in one batch of three, external actions, leaders chosen by the kernel: at every decision the acting
    agent, the clock, the observation digest and the state digest; then the metrics and no contract bit."""
    from dcmrta_b200 import BatchedTaskEnv
    z = facade_is()
    ids = [int(x) for x in z["instances"]]
    inst = pickle_instances()
    insts = [inst[i] for i in ids]
    B, A, T = len(ids), 20, 50
    n = np.array([len(z[f"{i}/agent"]) for i in ids])
    env = BatchedTaskEnv(B, A, T, M=5, protocol="IA")
    env.load_instances(*stack_instances(insts))
    env.reset()
    for k in range(int(n.max())):
        ag, tk, mk = env.agent_obs.cpu().numpy(), env.task_obs.cpu().numpy(), env.mask_u8.cpu().numpy()
        leaders = env.leader.cpu().numpy()
        states = env.export_state()
        act = np.zeros(B, np.int32)
        for b, i in enumerate(ids):
            if k >= n[b]:
                assert states[b]["flags"] & ENV_DONE and leaders[b] == -1, (i, k)
                continue
            assert leaders[b] == z[f"{i}/agent"][k], (i, k)
            st = states[b]
            assert st["now"] == z[f"{i}/now"][k], (i, k)
            assert canon.obs_digest(mk[b], ag[b], tk[b]) == int(z[f"{i}/dig_obs"][k]), (i, k)
            assert canon.state_digest(st) == int(z[f"{i}/dig_state"][k]), (i, k)
            act[b] = z[f"{i}/action"][k]
        env.step(act)
        done = env.done_u8.cpu().numpy()
        for b in range(B):
            if k < n[b]:
                assert bool(done[b]) == (k == n[b] - 1), (ids[b], k)
    assert not (env.env_flags().cpu().numpy() & ENV_ERR_MASK).any()
    met = env.episode_metrics().cpu().numpy()
    states = env.export_state()
    for b, i in enumerate(ids):
        gold = z[f"{i}/metrics"]
        assert met[b, 0] == gold[0]
        np.testing.assert_allclose(met[b, 1:7], gold[1:], rtol=1e-12, atol=0, err_msg=str(i))
        assert met[b, 7] == n[b]
        assert np.array_equal(states[b]["finished"], z[f"{i}/finished"])
    assert env.total_steps() == n.sum()
    env.close()


@pytest.mark.parametrize("policy", ["random", "greedy"])
def test_inkernel_ia_policy_matches_oracle(policy):
    """In-kernel random / greedy IA with auto-reset against the CPU IA loop on the same Philox contract: a sample of a batch of 1,003
    checked at every decision (observations, reward, done, the next acting agent) over at least two episodes each."""
    shape = EnvelopeShape(20, 50, 5, 1003, policy, None, 640, "", [])
    sample = [0, 1, 2, 31, 32, 500, 1001, 1002]
    with closing(make_env(shape, "IA", seed=4321, first_gid=7_000)) as env:
        env.reset()
        assert (env.leader[sample] == 0).all()                          # an IA episode starts with agent 0
        lockstep(env, shape, sample, shape.ia_steps, seed=4321, first_gid=7_000)


@pytest.mark.parametrize("shape,policy", [((20, 50), "random"), ((20, 50), "greedy"), ((30, 100), "random"), ((50, 200), "greedy")])
def test_ia_fused_pass_equals_serial_pass(shape, policy):
    """IA: the default pass against DCM_PASS_SERIAL (k_step, episode kernel, k_obs one after the other) on 4,099 envs, raw records of
    every env and every output at checkpoints; one shape per mask width (k_step_ia<1>, <2>, <4>)."""
    A, T = shape
    B = 4099
    steps = 10 * (A + T)                                            # about four IA episodes per env at every shape (50A/200T: ~650 decisions each)
    sh = EnvelopeShape(A, T, 5, B, policy, None, steps, "", [])
    with twin_handles(lambda: make_env(sh, "IA", seed=13, first_gid=5), "DCM_PASS_SERIAL") as (fused, other):
        ended = twin_steps(fused, other, policy, steps, lambda k: k % 50 == 49 or k < 3 or k == steps - 1)
        assert ended > 2 * B                                        # restarts were exercised
        assert not (fused.env_flags().cpu().numpy() & ENV_ERR_MASK).any()


def test_ia_step_host_matches_device_step():
    shape = EnvelopeShape(20, 50, 5, 1003, "random", None, 450, "", [])

    def restarts_with_agent_0(k, out):                              # a restarted IA episode starts with agent 0
        assert (out["next_leader"][out["done"] > 0] == 0).all(), k

    with twin_handles(lambda: make_env(shape, "IA", seed=23, first_gid=3)) as (dev, host):
        assert step_host_equals_step(dev, host, shape.ia_steps, after_step=restarts_with_agent_0) > shape.B


def test_ia_shard_invariance():
    check_shard_invariance("IA", 300)


def test_ia_contract_bits():
    """Followers given for a task move -> ERR_FOLLOW and no step; an injected leader that is not the lowest pending decider (or, at a
    reset, not agent 0) -> ERR_LEADER; a leader-follower record whose group holds every agent, imported into an IA handle, moves one."""
    from dcmrta_b200 import BatchedTaskEnv
    inst = pickle_instances()
    insts = [inst[0], inst[1], inst[2]]
    env = BatchedTaskEnv(3, 20, 50, M=5, protocol="IA")
    env.load_instances(*stack_instances(insts))
    env.reset(leaders=np.array([0, 4, -1], np.int32))
    flags = env.env_flags().cpu().numpy()
    assert not flags[0] & ENV_ERR_LEADER and flags[1] & ENV_ERR_LEADER and not flags[2] & ENV_ERR_LEADER
    assert env.leader.cpu().numpy().tolist() == [0, 0, 0]
    env.reset()
    fol = np.full((3, 4), -1, np.int32)
    fol[0, 0] = 1                                                        # env 0: a follower under IA
    env.step(np.array([1, 1, 1], np.int32), fol, np.array([-1, 2, 1], np.int32))
    flags = env.env_flags().cpu().numpy()
    assert flags[0] & ENV_ERR_FOLLOW and not flags[1] & ENV_ERR_FOLLOW and not flags[2] & ENV_ERR_FOLLOW
    assert int(env.used_action[0]) == -1 and env.export_state([0])[0]["has_route"].sum() == 0     # env 0 did not step
    assert flags[1] & ENV_ERR_LEADER and not flags[2] & ENV_ERR_LEADER                         # agent 1 acts next, not agent 2
    assert env.leader.cpu().numpy()[1:].tolist() == [1, 1]
    env.close()

    lf = BatchedTaskEnv(2, 20, 50, M=5, seed=3)
    lf.load_instances(*stack_instances(insts[:2]))
    lf.reset()
    raw = lf.export_raw()
    assert all(bin(s["group"]).count("1") == 20 for s in lf.export_state())
    ia = BatchedTaskEnv(2, 20, 50, M=5, protocol="IA")
    ia.load_instances(*stack_instances(insts[:2]))
    ia.import_raw(raw)
    leader = lf.leader.cpu().numpy()
    ia.step(np.array([1, 0], np.int32))                                  # env 0: a task of requirement > 1; env 1: the depot (Q11 in LF)
    assert int(insts[0]["req"][0]) > 1
    for b, st in enumerate(ia.export_state()):
        assert st["has_route"].sum() == 1 and st["has_route"][leader[b]] == 1, b
        assert st["n_steps"] == 1
    assert ia.leader.cpu().numpy().tolist() == [0 if leader[0] else 1, 0 if leader[1] else 1]
    d = np.hypot(*(insts[0]["task_xy"][0] - insts[0]["depot_xy"]))
    assert float(ia.reward[0]) == pytest.approx(-d / 0.2, rel=1e-6) and float(ia.reward[1]) == 0.0
    assert not (ia.env_flags().cpu().numpy() & ENV_ERR_MASK).any()
    lf.step(np.array([1, 0], np.int32))                                  # the same records under LF move a coalition / the whole group
    assert [s["has_route"].sum() for s in lf.export_state()] == [int(insts[0]["req"][0]), 20]
    lf.close(); ia.close()


def test_evaluate_matches_inkernel_greedy_oracle_and_reference():
    """evaluate() with the nearest-task stand-in on the 50 bundled instances: IA equals the in-kernel greedy IA run and the oracle, and
    instances 0/5/9 the reference's run_test_IS (facade_is.npz); LF equals the oracle's LF greedy with the same seed and global ids;
    the eager and the graphed loop agree; a recorded IA rollout's `leader` is the acting agent of each decision."""
    import torch
    from dcmrta_b200 import BatchedTaskEnv
    from dcmrta_b200.evaluate import evaluate, load_test_set
    from dcmrta_b200.rollout import BatchedRollout
    sets = load_test_set(GOLD / "instances_20A_50T.npz")
    inst = pickle_instances()
    net = nearest_task_module()
    ia = evaluate(net, sets, method="IA")
    assert ia.shape == (50, 8)
    env = BatchedTaskEnv(50, 20, 50, M=5, protocol="IA")
    env.load_instances(sets["task_xy"], sets["depot_xy"], sets["req"], sets["dur"])
    env.reset()
    while not bool(env.done.all()):
        env.step(policy="greedy")
    assert np.array_equal(ia, env.episode_metrics().cpu().numpy())
    env.close()
    for i in range(50):
        assert_metrics_match(ia[i], oracle_metrics(inst[i], "IA"), ("IA", i))
    z = facade_is()
    for i in (int(x) for x in z["instances"]):
        gold = z[f"{i}/metrics"]
        assert ia[i, 0] == gold[0] and ia[i, 7] == len(z[f"{i}/agent"])
        np.testing.assert_allclose(ia[i, 1:7], gold[1:], rtol=1e-12, atol=0)
    seed = 17
    lf = evaluate(net, sets, method="LF", seed=seed)
    for i in range(50):
        assert_metrics_match(lf[i], oracle_metrics(inst[i], "LF", seed=seed, gid=i), ("LF", i))
    assert (ia[:, 7] > lf[:, 7]).mean() > 0.9
    assert np.array_equal(evaluate(net, sets, method="IA", graphed=True), ia)
    assert np.array_equal(evaluate(net, sets, method="LF", seed=seed, graphed=True), lf)
    # Episodes.leader under IA: the acting agent of each decision
    env = BatchedTaskEnv(50, 20, 50, M=5, protocol="IA")
    env.load_instances(sets["task_xy"], sets["depot_xy"], sets["req"], sets["dur"])
    ep = BatchedRollout(env, 320, record=True).run(net, "greedy")        # IA greedy: up to 259 decisions on these instances
    assert bool(ep.ended.all()) and torch.equal(ep.metrics.cpu(), torch.from_numpy(ia))
    for i in (int(x) for x in z["instances"]):
        act = ep.active[:, i].cpu().numpy()
        assert np.array_equal(ep.leader[:, i].cpu().numpy()[act], z[f"{i}/agent"])
        assert np.array_equal(ep.action[:, i].cpu().numpy()[act], z[f"{i}/action"])
    env.close()
    with pytest.raises(RuntimeError):
        evaluate(net, sets, method="IA", horizon=40)             # an episode the horizon would cut is an error, never a score


@pytest.mark.parametrize("method", ["LF", "IA"])
def test_trainer_checkpoint_through_evaluate_cli(method, tmp_path, capsys):
    """ReinforceTrainer.save -> python -m dcmrta_b200.evaluate -> the per-instance CSV, fp32 module and fused forward."""
    import pandas as pd
    from dcmrta_b200.evaluate import evaluate, load_test_set, main
    from dcmrta_b200.trainer import ReinforceTrainer, TrainerConfig
    tr = ReinforceTrainer(TrainerConfig(envs_per_rank=32, eval_instances=8, graph_rollout=False, seed=5))
    ck = tmp_path / "checkpoint.pth"
    tr.save(ck)
    out = tmp_path / f"REINFORCE_{method}.csv"
    test_set = str(GOLD / "instances_20A_50T.npz")
    assert main(["--checkpoint", str(ck), "--test-set", test_set, "--method", method, "--seed", "2", "--out", str(out)]) == 0
    printed = capsys.readouterr().out
    assert "makespan" in printed and "+-" in printed
    df = pd.read_csv(out, index_col=0)
    assert df.shape == (50, 6) and list(df.columns) == ["success_rate", "makespan", "time_cost", "waiting_time", "travel_dist", "efficiency"]
    want = evaluate(tr.net, load_test_set(test_set), method=method, seed=2)
    np.testing.assert_allclose(df.to_numpy(), want[:, 1:7], rtol=1e-12, atol=0)
    fused = tmp_path / f"REINFORCE_{method}_fused.csv"
    assert main(["--checkpoint", str(ck), "--test-set", test_set, "--method", method, "--amp", "fused", "--out", str(fused)]) == 0
    f = pd.read_csv(fused, index_col=0)
    assert f.shape == (50, 6) and np.isfinite(f.to_numpy()).all() and (f["success_rate"] <= 1).all()
