"""CPU tests: pin the C oracle (oracle/taskenv_oracle.c) against the reference's own golden vectors and against
vectors recorded from the real reference (tests/golden/, made by oracle/make_golden.py)."""
import numpy as np
import pytest

from oracle import canon
from oracle.oracle import OracleEnv, philox

from helpers import METRIC_KEYS, ctasd, full_dump, pickle_instances, pickle_traces, quirk_census, quirk_instance, quirk_traces, sweep_instance, sweep_traces


def replay_on_oracle(inst, ep, tr, check_full=None):
    o = OracleEnv.make(**inst)
    n = len(ep["leader"])
    assert o.fused_reset(int(ep["leader"][0])) == int(ep["leader"][0])
    for k in range(n):
        leader = int(ep["leader"][k])
        assert o.leader == leader
        assert o.current_time == ep["now"][k]
        mask, ag, tk = o.mask(), o.agent_status(leader).astype(np.float32), o.task_status(leader).astype(np.float32)
        assert canon.obs_digest(mask, ag, tk) == int(ep["dig_obs"][k]), f"obs digest, decision {k}"
        st = o.export(canon.MC_CANON)
        assert canon.state_digest(st) == int(ep["dig_state"][k]), f"state digest, decision {k}"
        if check_full is not None:
            check_full(k, mask, ag, tk, st)
        nl = int(ep["leader"][k + 1]) if k + 1 < n else -1
        rc, r, done, _, mem = o.fused_step(int(ep["action"][k]), tr.followers(ep, k), nl)
        assert rc == 0
        assert r == ep["reward"][k]
        assert done == (k == n - 1)
    m, fin = o.episode_metrics()
    got = np.array([m[k] for k in METRIC_KEYS[:7]] + [float(o.n_steps)])
    assert np.array_equal(got, ep["metrics"]), (got, ep["metrics"])
    assert canon.state_digest(o.export(canon.MC_CANON)) == ep["final_digest"]
    return o, fin


def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32-10
    assert philox([0, 0, 0, 0], [0, 0]).tolist() == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert philox([0xffffffff] * 4, [0xffffffff] * 2).tolist() == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]).tolist() == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_ctasd_known_answer_csv():
    """SURVEY 8(c)(i): CTAS-D routes -> execute_by_route -> the reference's own CTAS-D_300s.csv (time_cost is stale)."""
    inst = pickle_instances()
    for i, g in enumerate(ctasd()):
        o = OracleEnv.make(**inst[i])
        for a, r in g["routes"].items():
            o.pre_set_route(r, int(a))
        o.execute_by_route()
        m, fin = o.episode_metrics()
        assert fin.tolist() == g["finished"]
        for k, v in g["csv"].items():
            assert m[k] == pytest.approx(v, rel=1e-15, abs=0), (i, k)
        for k in ("success_rate", "makespan", "time_cost", "waiting_time", "travel_dist", "efficiency", "reward"):
            assert m[k] == g["ref_here"][k], (i, k)          # bit-exact against the reference run in the build container
        assert str(canon.state_digest(o.export(canon.MC_CANON))) == g["final_digest"]


def test_pickle_traces_digest_exact():
    """SURVEY 8(c)(iv): 50 instances x {random, greedy}: every decision's obs/mask/state digests, rewards, metrics."""
    inst = pickle_instances()
    tr = pickle_traces()
    for e in range(len(tr)):
        ep = tr.episode(e)
        i = int(ep["name"].split("/")[0])
        _, fin = replay_on_oracle(inst[i], ep, tr)
        assert np.array_equal(fin, tr.finished[e])


def test_full_dump_undigested():
    inst = pickle_instances()[0]
    tr = pickle_traces()
    fd = full_dump()
    for e in range(len(tr)):
        ep = tr.episode(e)
        i, policy = ep["name"].split("/")
        if int(i) != 0:
            continue

        def chk(k, mask, ag, tk, st):
            assert np.array_equal(mask, fd[f"{policy}/mask"][k])
            assert np.array_equal(ag, fd[f"{policy}/agent_obs"][k])
            assert np.array_equal(tk, fd[f"{policy}/task_obs"][k])
            ref = {key: fd[f"{policy}/state/{key}"][k] for key in canon.normalise(st) if key != "now"}
            ref["now"] = float(fd[f"{policy}/state/now"][k])
            assert not canon.diff_states(st, ref)

        replay_on_oracle(inst, ep, tr, check_full=chk)


def test_sweep_traces_digest_exact():
    tr = sweep_traces()
    for e in range(len(tr)):
        ep = tr.episode(e)
        _, fin = replay_on_oracle(sweep_instance(tr, ep["name"]), ep, tr)
        assert np.array_equal(fin, tr.z[f"finished/{ep['name']}"])


def test_builtin_policies_terminate_and_are_deterministic():
    inst = pickle_instances()[5]
    runs = []
    for _ in range(2):
        o = OracleEnv.make(**inst)
        o.seed(1234, gid=42, episode=0)
        assert o.fused_reset() >= 0
        acts = []
        while not o.done:
            rc, r, done, ua, mem = o.fused_step(-1)
            assert rc == 0
            acts.append((ua, tuple(mem)))
        runs.append((acts, o.episode_metrics()[0]))
    assert runs[0] == runs[1]
    assert 60 < len(runs[0][0]) < 400


def test_quirk_fixtures_digest_exact():
    """SURVEY 4 item 3: small fixtures recorded from the real reference, one per quirk of App. A -- four location groups in one slot
    ordered by np.unique(axis=0) (Q10), the group that follows its leader to the depot (Q11), the clock jump when nobody can decide
    (Q13), members skipped while the list they are removed from is iterated (Q2), stale status (Q3), spread removals (Q4), sticky
    `assigned` (Q5), ghost members (Q1), re-visits (Q8), and the state in which the reference loop would spin forever (STUCK)."""
    tr = quirk_traces()
    seen = dict.fromkeys(tr.census_keys, 0)
    for e in range(len(tr)):
        ep = tr.episode(e)
        inst = quirk_instance(tr, ep["name"])
        o, fin = replay_on_oracle(inst, ep, tr)
        assert np.array_equal(fin, tr.z[f"finished/{ep['name']}"])
        assert o.stuck == (ep["name"] == "q11_depot_stuck")
        for k, v in quirk_census(tr, ep["name"]).items():
            seen[k] = max(seen[k], v) if k == "q10_max_groups" else seen[k] + v
    assert seen["q10_max_groups"] == 4 and seen["q10_multi_group_slot"] >= 3
    for k in ("q1_ghost_member_decides", "q2_skipped_after_removal", "q3_stale_status", "q4_spread_removal", "q5_sticky_assigned",
              "q8_revisit", "q11_group_follows_to_depot", "q13_clock_jump"):
        assert seen[k] >= 1, k
