"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C ABI, against
  * golden vectors recorded from the real reference (tests/golden/, digests of every decision), and
  * the C oracle stepped in lock-step on the same inputs (full state diff, used for readable failures and for
    synthetic instances at the bench's full batch size).
Bar (BASELINE.json north_star): discrete state bit-exact; times/distances/rewards within 1e-5 relative.  The fp64 event
clock makes the float state bit-exact too, so the digests are compared exactly; REL documents the contractual tolerance."""
from contextlib import closing

import numpy as np
import pytest

from dcmrta_b200._lib import ENV_DONE, ENV_ERR_MASK, ENV_FINISHED, ENV_STUCK
from oracle import canon
from oracle.oracle import OracleEnv

from gpu_env import (assert_same_outputs, assert_same_records, check_shard_invariance, instances, lockstep, make_env, stack_instances,
                     step_host_equals_step, twin_handles, twin_steps)
from helpers import (METRIC_KEYS, EnvelopeShape, ctasd, pickle_instances, pickle_traces, quirk_instance, quirk_traces, sweep_instance,
                     sweep_traces)

pytestmark = pytest.mark.gpu
REL = 1e-5


def replay_batch(insts, eps, tr, max_wait=10.0):
    """Replay B recorded episodes in one batch, checking every decision of every env."""
    import torch
    from dcmrta_b200 import BatchedTaskEnv
    B, A, T = len(eps), insts[0]["A"], insts[0]["task_xy"].shape[0]
    env = BatchedTaskEnv(B, A, T, M=5, max_wait=max_wait)
    env.load_instances(*stack_instances(insts))
    n = np.array([len(e["leader"]) for e in eps])
    FS = 8
    first = np.array([int(e["leader"][0]) for e in eps], np.int32)
    env.reset(leaders=first)
    oracles = [None] * B

    def oracle_at(b, k):
        """replay env b on the oracle up to decision k (only used to explain a mismatch)."""
        o = OracleEnv.make(**insts[b], max_wait=max_wait)
        e = eps[b]
        o.fused_reset(int(e["leader"][0]))
        for q in range(k):
            o.fused_step(int(e["action"][q]), tr.followers(e, q), int(e["leader"][q + 1]) if q + 1 < len(e["leader"]) else -1)
        return o

    for k in range(int(n.max())):
        ag, tk, mk = env.agent_obs.cpu().numpy(), env.task_obs.cpu().numpy(), env.mask_u8.cpu().numpy()
        leaders = env.leader.cpu().numpy()
        states = env.export_state()
        for b in range(B):
            if k >= n[b]:
                assert states[b]["flags"] & ENV_DONE, f"env {b} should be done after {n[b]} decisions"
                continue
            e = eps[b]
            assert leaders[b] == e["leader"][k]
            st = states[b]
            assert st["now"] == e["now"][k], (e["name"], k)
            if canon.obs_digest(mk[b], ag[b], tk[b]) != int(e["dig_obs"][k]):
                o = oracle_at(b, k)
                l = int(e["leader"][k])
                np.testing.assert_array_equal(mk[b], o.mask(), err_msg=f"{e['name']} mask @ {k}")
                np.testing.assert_array_equal(ag[b], o.agent_status(l).astype(np.float32), err_msg=f"{e['name']} agent obs @ {k}")
                np.testing.assert_array_equal(tk[b], o.task_status(l).astype(np.float32), err_msg=f"{e['name']} task obs @ {k}")
                raise AssertionError(f"{e['name']}: obs digest differs from the reference at decision {k} but matches the oracle")
            if canon.state_digest(st) != int(e["dig_state"][k]):
                d = canon.diff_states(st, oracle_at(b, k).export(canon.MC_CANON))
                raise AssertionError(f"{e['name']}: state differs at decision {k}: {d}")
        act = np.zeros(B, np.int32)
        fol = np.full((B, FS), -1, np.int32)
        nxt = np.full(B, -1, np.int32)
        for b in range(B):
            if k < n[b]:
                e = eps[b]
                act[b] = e["action"][k]
                f = tr.followers(e, k)
                fol[b, :len(f)] = f
                if k + 1 < n[b]:
                    nxt[b] = e["leader"][k + 1]
        env.step(act, fol, nxt)
        rew, done = env.reward.cpu().numpy(), env.done_u8.cpu().numpy()
        for b in range(B):
            if k < n[b]:
                assert rew[b] == np.float32(eps[b]["reward"][k]), (eps[b]["name"], k)
                assert bool(done[b]) == (k == n[b] - 1), (eps[b]["name"], k)
    flags = env.env_flags().cpu().numpy()
    assert not (flags & ENV_ERR_MASK).any(), "contract-violation bits set during a legal replay"
    met = env.episode_metrics().cpu().numpy()
    states = env.export_state()
    for b in range(B):
        gold = eps[b]["metrics"]
        np.testing.assert_allclose(met[b], gold, rtol=1e-12, atol=0, err_msg=eps[b]["name"])
        for c in (0, 1, 2, 3, 5, 6, 7):                      # everything but waiting_time is bit-exact
            assert met[b, c] == gold[c], (eps[b]["name"], METRIC_KEYS[c])
        assert canon.state_digest(states[b]) == eps[b]["final_digest"], eps[b]["name"]
    env.close()
    return met


def test_replay_50_pickles_random_and_greedy():
    """BASELINE config 2: all 50 testSet_20A_50T_CONDET instances x {random, greedy}, every decision, one batch of 100."""
    inst = pickle_instances()
    tr = pickle_traces()
    eps = [tr.episode(i) for i in range(len(tr))]
    insts = [inst[int(e["name"].split("/")[0])] for e in eps]
    met = replay_batch(insts, eps, tr)
    fin = tr.finished
    assert np.array_equal(met[:, 1], fin.sum(1) / fin.shape[1])


@pytest.mark.parametrize("shape", ["10x20", "20x50", "30x100", "50x200"])
def test_replay_shape_sweep(shape):
    tr = sweep_traces()
    idx = [i for i, nm in enumerate(tr.names) if nm.startswith(shape + "/")]
    eps = [tr.episode(i) for i in idx]
    insts = [sweep_instance(tr, e["name"]) for e in eps]
    replay_batch(insts, eps, tr)


def test_replay_quirk_fixtures():
    """SURVEY 4 item 3 / App. A: the hand-built and searched quirk fixtures recorded from the real reference (oracle/make_quirk_golden.py),
    every decision.  q10_groups has one slot with FOUR location groups: the leaders arrive in np.unique(axis=0) order (x, then y), which
    is not agent-id order, and an injected leader outside the current group raises DCM_ENV_ERR_LEADER -- so a green replay proves the
    lexicographic multi-location branch of get_unique_group (t_current_group), which no other trace reaches.  q11_depot_stuck ends
    in the state where the reference loop would spin forever: DCM_ENV_STUCK."""
    from dcmrta_b200 import BatchedTaskEnv
    tr = quirk_traces()
    for e in range(len(tr)):
        ep = tr.episode(e)
        replay_batch([quirk_instance(tr, ep["name"])], [ep], tr)
    # the stuck fixture once more, for the status bit
    ep = tr.episode(tr.names.index("q11_depot_stuck"))
    inst = quirk_instance(tr, "q11_depot_stuck")
    env = BatchedTaskEnv(1, inst["A"], inst["task_xy"].shape[0], M=5)
    env.load_instances(*stack_instances([inst]))
    env.reset(leaders=np.array([int(ep["leader"][0])], np.int32))
    fol = np.full((1, 8), -1, np.int32); f = tr.followers(ep, 0); fol[0, :len(f)] = f
    env.step(np.array([int(ep["action"][0])], np.int32), fol, np.array([-1], np.int32))
    flags = int(env.env_flags()[0])
    assert flags & ENV_DONE and flags & ENV_STUCK and not flags & ENV_FINISHED
    env.close()


def test_ctasd_routes_known_answer():
    """SURVEY 8(c)(i): CTAS-D routes through execute_by_route reproduce the reference's CTAS-D_300s.csv."""
    import torch
    from dcmrta_b200 import BatchedTaskEnv
    inst = pickle_instances()
    gold = ctasd()
    B, A, T = 50, 20, 50
    Lmax = max(len(r) for g in gold for r in g["routes"].values())
    routes = np.zeros((B, A, Lmax), np.int32)
    rlen = np.zeros((B, A), np.int32)
    for b, g in enumerate(gold):
        for a, r in g["routes"].items():
            routes[b, int(a), :len(r)] = r
            rlen[b, int(a)] = len(r)
    env = BatchedTaskEnv(B, A, T, M=8)      # preset routes ignore the mask: coalitions may exceed max_coalition_size
    env.load_instances(*stack_instances(inst))
    env.reset()
    mk = env.execute_by_route(routes, rlen).cpu().numpy()
    env.set_params(max_wait=100.0)                   # execute_by_route leaves max_waiting_time = 100 (task_env.py:564)
    met = env.compute_metrics().cpu().numpy()
    flags = env.env_flags().cpu().numpy()
    assert not (flags & ENV_ERR_MASK).any()
    states = env.export_state()
    for b, g in enumerate(gold):
        for k, v in g["csv"].items():
            assert met[b, METRIC_KEYS.index(k)] == pytest.approx(v, rel=1e-14, abs=0), (b, k)
        for k in ("success_rate", "makespan", "time_cost", "travel_dist", "efficiency", "reward"):
            assert met[b, METRIC_KEYS.index(k)] == g["ref_here"][k], (b, k)
        assert met[b, 4] == pytest.approx(g["ref_here"]["waiting_time"], rel=1e-13)
        assert states[b]["finished"].tolist() == g["finished"]
        assert str(canon.state_digest(states[b])) == g["final_digest"], b
    env.close()


@pytest.mark.parametrize("policy", ["random", "greedy"])
def test_inkernel_policy_matches_oracle_on_synthetic(policy):
    """In-kernel Philox policies + generator vs the oracle running the same RNG contract, synthetic 20A/50T instances,
    auto-reset across several episodes; sample of envs out of a batch that is not a multiple of the CTA size."""
    shape = EnvelopeShape(20, 50, 5, 1003, policy, 400, None, "", [])
    with closing(make_env(shape, seed=1234, first_gid=10_000)) as env:
        env.reset()
        orcs = lockstep(env, shape, [0, 1, 2, 3, 4, 500, 1001, 1002], shape.steps, seed=1234, first_gid=10_000)
        assert env.total_episodes() >= sum(o.episodes for o in orcs)     # dcm_total_episodes: every accounted episode of the batch (bench.py's phase report)


def test_shard_invariance():
    """SURVEY 8(e): the trajectory of global env k does not depend on the batch it lives in (leader-follower, 200 decisions)."""
    check_shard_invariance("LF", 200)


@pytest.mark.parametrize("variant", ["DCM_PASS_SERIAL"])
@pytest.mark.parametrize("shape,policy", [((20, 50), "random"), ((20, 50), "greedy"), ((10, 20), "random"), ((50, 200), "random"), ((30, 100), "greedy")])
def test_fused_pass_equals_split_kernels(shape, policy, variant):
    """The default pass (k_step, then k_episode on a side stream writing the restarted envs' observations from registers
    beside k_obs) against the three kernels one after the other with k_obs building every observation from memory: raw records (every field, bookkeeping bits included), observations, rewards, leaders and metrics identical on a batch
    that is not a multiple of the tile size."""
    B = 4099
    sh = EnvelopeShape(*shape, 5, B, policy, 600, None, "", [])
    with twin_handles(lambda: make_env(sh, seed=11, first_gid=5), variant) as (fused, other):
        assert fused.launch_count() == other.launch_count()
        twin_steps(fused, other, policy, sh.steps, lambda k: k % 50 == 49 or k < 3)
        assert fused.total_steps() == other.total_steps() == B * sh.steps


@pytest.mark.parametrize("variant", [None, "DCM_OBS_RESET_BY_EPISODE", "DCM_OBS_CHUNKED"])
def test_step_host_matches_device_step(variant):
    """dcm_step_host (host buffers; next_leader / reward / done leave for the host when k_step ends, beside the episode and
    observation kernels) against dcm_step with device buffers replaying the same actions: every output of every decision,
    restarts included (the first leader and the first observation of a restarted episode come from k_step / k_obs_tile in the
    default pass and from the episode kernel in the variants, which the host-buffer handle is created with)."""
    shape = EnvelopeShape(20, 50, 5, 1003, "random", 450, None, "", [])

    def every_env_has_a_leader(k, out):                                          # auto-reset: after every decision
        assert (out["next_leader"] >= 0).all(), k

    with twin_handles(lambda: make_env(shape, seed=21, first_gid=3), variant) as (dev, host):
        restarts = step_host_equals_step(dev, host, shape.steps, pinned=True, after_step=every_env_has_a_leader)
        assert restarts > shape.B                                                # the restart path was exercised


def test_regenerate_restarts_on_fresh_instances():
    """DCM_FLAG_REGENERATE: an env whose episode ended restarts on a NEW instance drawn in the episode kernel's registers (same
    Philox streams as dcm_generate, instance counter + 1), and that kernel writes the first observation of the new episode
    beside k_obs_tile.  Checked against (a) the serial pass, where k_obs builds that observation from memory after the
    restart, and (b) the closed form of a reset observation on the instance read back from the device."""
    from dcmrta_b200 import BatchedTaskEnv
    B, A, T = 1003, 20, 50

    def make():
        e = BatchedTaskEnv(B, A, T, auto_reset=True, regenerate=True, seed=31, first_gid=9)
        e.generate(max_duration=5.0)
        return e

    with twin_handles(make, "DCM_PASS_SERIAL") as (env, ser):
        first_xy = stack_instances(instances(env))[0]
        restarted = np.zeros(B, bool)

        def reset_observations(k):
            done = env.done_u8.cpu().numpy().astype(bool)
            ag, tk, mk = env.agent_obs.cpu().numpy(), env.task_obs.cpu().numpy(), env.mask_u8.cpu().numpy()
            ended = np.flatnonzero(done)[:8]
            for b, inst in zip(ended, instances(env, ended)):
                assert not ag[b].any(), (k, b)                                         # nobody has a route (:165-180)
                want = np.zeros((T + 1, 5), np.float32)
                want[1:, 0] = inst["req"]; want[1:, 1] = inst["req"]; want[1:, 2] = inst["dur"].astype(np.float32)
                want[1:, 3:] = (inst["task_xy"] - inst["depot_xy"]).astype(np.float32)
                assert np.array_equal(tk[b], want), (k, b)                              # :182-190 seen from the depot
                assert mk[b, 0] == 1 and not mk[b, 1:].any(), (k, b)                    # only the depot is masked
            restarted[done] = True

        twin_steps(env, ser, "random", 450, lambda k: True, after_step=reset_observations)
        assert restarted.sum() > B // 2
        xy, depot, req, dur = stack_instances(instances(env))
        moved = (xy != first_xy).any(axis=(1, 2))
        assert np.array_equal(moved, restarted)                                         # new instances exactly where an episode ended
        assert (xy >= 0).all() and (xy < 1).all() and (depot >= 0).all() and (depot < 1).all()
        assert req.min() >= 1 and req.max() <= 5 and (dur == 5.0).all()


def test_bench_configuration_at_its_own_size():
    """The configuration the headline number is measured on (BASELINE configs[2]: 65,536 synthetic 20A/50T envs, in-kernel random
    policy, auto-reset) checked AT THAT SIZE through its steady state (k_step appends ~450 ended envs per pass to the episode list,
    2,048 observation blocks share the SMs with the episode blocks):
      * 64 random envs against the oracle at every one of 340 decisions -- observations, mask, reward, done, next leader;
      * the default pass against the serial pass (DCM_PASS_SERIAL: k_step, k_episode_list, k_obs one after the other on one
        stream, observations always built from memory) on every output at checkpoints and on the raw records of all envs."""
    import torch
    shape = EnvelopeShape(20, 50, 5, 65536, "random", 340, None, "", [])
    B, STEPS = shape.B, shape.steps
    rng = np.random.default_rng(5)
    sample = sorted(int(x) for x in rng.choice(B, 64, replace=False))
    sample[0], sample[-1] = 0, B - 1
    with twin_handles(lambda: make_env(shape, seed=1234, first_gid=0), "DCM_PASS_SERIAL") as (env, ser):
        ended = []

        def serial_pass(k):
            ser.step(policy="random")
            if k % 20 == 19 or k >= STEPS - 3:
                ended.append(int(env.done_u8.sum()))
                assert_same_outputs(env, ser, k)

        lockstep(env, shape, sample, STEPS, seed=1234, first_gid=0, min_episodes=1, metrics=False, after_step=serial_pass)
        assert sum(ended) > 20 * 100                                # the steady state was reached: hundreds of episode ends per pass
        assert_same_records(env, ser, "default against serial pass")
        assert torch.equal(env.episode_metrics(), ser.episode_metrics())
