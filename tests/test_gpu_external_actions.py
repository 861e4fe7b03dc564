"""GPU tests of dcm_step on caller-supplied inputs (DCM_POLICY_EXTERNAL) over the supported shape range (include/dcmrta.h:
1 <= A <= 64, 1 <= T <= 254, 1 <= M <= 8), every env of each batch against its own oracle.

The built-in policies only ever pick unmasked actions.  A caller may pick any action in [0, T], as TaskEnv.step allows
(task_env.py:326-342), and the step's shortcuts (the decider rule and the xfin / xamin bounds of t_task_update, the movers'
observation cache AOBS2, the lazy `assigned` of t_agent_update) were argued for legal play.  So the actions here are
helpers.ExternalOracle's: masked joins of running, finished and satisfied-waiting tasks (within M members), masked depot moves,
re-visits of feasible tasks, with followers drawn by the test on part of the decisions.  The file also checks the contract bits
DCM_ENV_ERR_ACTION / _FOLLOW / _LEADER (a refused step leaves the env as it was; a bad injected leader falls back to the lowest id of
the group), DCM_ENV_ERR_OVERFLOW on envs that pile M + 1 agents on one task, and dcm_step_host against dcm_step.
tests/test_external_actions_oracle.py replays the same trajectories on the oracle alone and checks their census."""
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import canon

from helpers import ENVELOPE_SHAPES, ExternalOracle, envelope_shape, external_census_needs, external_steps, inject_followers_at
from test_gpu_shape_envelope import ERR_BITS, assert_metrics_match, assert_same_records, make_env, outputs, with_finish

pytestmark = pytest.mark.gpu
ERR_OVERFLOW, ERR_ACTION, ERR_FOLLOW, ERR_LEADER = 16, 32, 64, 128


def batch_instances(env):
    inst = {k: v.cpu().numpy() for k, v in env.get_instances().items()}
    return [{k: inst[k][b] for k in inst} for b in range(env.B)]


def flags_offset(env):
    from dcmrta_b200.batched_env import _HDR_DTYPE
    return env.layout["o_hdr"] + _HDR_DTYPE.fields["flags"][1]


def check_obs(env, orcs, skip, what):
    """mask, agent rows and task rows of every env not in `skip` against its oracle's leader"""
    ag, tk, mk = env.agent_obs.cpu().numpy(), env.task_obs.cpu().numpy(), env.mask_u8.cpu().numpy()
    for b, o in enumerate(orcs):
        if b in skip:
            continue
        assert np.array_equal(mk[b], o.env.mask()), (what, b, "mask")
        assert np.array_equal(ag[b], o.env.agent_status(o.leader).astype(np.float32)), (what, b, "agent rows")
        assert np.array_equal(tk[b], o.env.task_status(o.leader).astype(np.float32)), (what, b, "task rows")


def step_outputs(env):
    return (env.reward.cpu().numpy(), env.done_u8.cpu().numpy(), env.leader.cpu().numpy(), env.used_action.cpu().numpy())


def check_result(out, b, o, res, action, what):
    """reward (f32 of the oracle's f64), done, next leader and used_action of env b, bit for bit"""
    rew, done, lead, ua = out
    r, d, _ = res
    assert rew[b] == np.float32(r), (what, b, "reward", rew[b], r)
    assert bool(done[b]) == d, (what, b, "done")
    assert lead[b] == o.leader, (what, b, "next leader", lead[b], o.leader)
    assert ua[b] == action, (what, b, "used_action", ua[b], action)


def assert_episode_metrics(got, want, M, what):
    """assert_metrics_match, but at M = 8 `efficiency` to 1e-12 only: the episode kernel sums the waits of an 8-member coalition one after
    the other, NumPy pairwise (DESIGN.md, known deviations), and masked joins fill 8 slots far more often than legal play"""
    if M < 8:
        return assert_metrics_match(got, want, what)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0, err_msg=str(what))
    for c in (0, 1, 2, 3, 5, 7):
        assert got[c] == want[c], (what, c, got[c], want[c])


def final_checks(env, orcs, insts, skip, what):
    """metrics of every env's last episode, decoded state against oracle.export"""
    met = env.episode_metrics().cpu().numpy()
    states = env.export_state()
    for b, o in enumerate(orcs):
        if b in skip:
            continue
        if o.last_metrics is not None:
            assert_episode_metrics(met[b], o.last_metrics, o.shape.M, (what, b))
        d = canon.diff_states(with_finish(states[b], insts[b]["dur"]), o.o.export(canon.MC_CANON))
        assert not d, (what, b, d)


def run_external(shape, protocol, steps):
    """auto-reset, DCM_POLICY_EXTERNAL, ExternalOracle's actions and followers, every env of the batch against its oracle at every
    decision; then the last episode's metrics, the state, the error bits and the step counter.  Returns (env, oracles)."""
    env = make_env(shape, protocol)
    insts = batch_instances(env)
    env.reset()
    orcs = [ExternalOracle(shape, b, insts[b], protocol) for b in range(shape.B)]
    for b, o in enumerate(orcs):
        assert o.leader == int(env.leader[b]), (shape.name, b)
    for k in range(steps):
        what = (shape.name, protocol, k)
        check_obs(env, orcs, (), what)
        dec = [o.decide(k, shape.M) for o in orcs]
        acts = np.array([d[0] for d in dec], np.int32)
        rows = np.stack([d[1] for d in dec]) if dec[0][1] is not None else None
        env.step(acts, followers=rows)
        out = step_outputs(env)
        for b, (o, (a, _, fol, kind)) in enumerate(zip(orcs, dec)):
            check_result(out, b, o, o.apply(a, fol, kind=kind), a, what)
    final_checks(env, orcs, insts, (), (shape.name, protocol))
    assert not (env.env_flags().cpu().numpy() & ERR_BITS).any()
    assert env.total_steps() == shape.B * steps
    return env, orcs


@pytest.mark.parametrize("shape", ENVELOPE_SHAPES, ids=lambda s: s.name)
def test_external_actions_match_oracle(shape):
    """leader-follower, followers injected on every third decision"""
    env, orcs = run_external(shape, "LF", external_steps(shape))
    missing = external_census_needs(shape) - set.union(*(o.ext_census for o in orcs))
    assert not missing, (shape.name, missing)
    assert max(o.max_joined for o in orcs) <= shape.M
    env.close()


@pytest.mark.parametrize("shape", [s for s in ENVELOPE_SHAPES if s.ia_steps], ids=lambda s: s.name)
def test_external_actions_ia_match_oracle(shape):
    """the individual-agent protocol (tests/ia_oracle.py) on the same kinds of actions"""
    env, orcs = run_external(shape, "IA", external_steps(shape, "IA"))
    missing = external_census_needs(shape, "IA") - set.union(*(o.ext_census for o in orcs))
    assert not missing, (shape.name, missing)
    env.close()


# ---- contract bits -------------------------------------------------------------------------------------------------------------------
# case -> (bit, least M at which it can be built).  Each case has its own env of one mixed batch.
CONTRACT_CASES = {
    "action_minus_one": (ERR_ACTION, 1), "action_T_plus_1": (ERR_ACTION, 1), "action_int_max": (ERR_ACTION, 1),
    "follow_too_few": (ERR_FOLLOW, 2), "follow_too_many": (ERR_FOLLOW, 2), "follow_duplicate": (ERR_FOLLOW, 3),
    "follow_id_ge_A": (ERR_FOLLOW, 2), "follow_other_group": (ERR_FOLLOW, 2), "follow_not_pending": (ERR_FOLLOW, 2),
    "follow_fstride": (ERR_FOLLOW, 3),
    "leader_outside_group": (ERR_LEADER, 1), "leader_ge_A": (ERR_LEADER, 1), "leader_restart_ge_A": (ERR_LEADER, 1),
    "depot_with_followers": (0, 2),
}
CASE_FROM = 4                           # first decision at which a case may fire (follow_other_group: when its slot comes)
DRIVE_HOME_AFTER = 3                    # decisions after a case fired at which its env starts to play the depot, to see its episode end


def case_env(i):
    return 3 * i + 2


def bits(m):
    return [i for i in range(64) if m >> i & 1]


def other_group_instance(inst):
    """tasks 0 and 1 at the same distance from the depot, two agents each, equal durations: both coalitions finish at the same clock at
    two locations, so that slot has two location groups (task 0's sorts first, task_env.py:293)"""
    inst = {k: np.array(v, copy=True) for k, v in inst.items()}
    inst["depot_xy"][:] = (0.5, 0.5)
    inst["task_xy"][0], inst["task_xy"][1] = (0.25, 0.5), (0.75, 0.5)
    inst["req"][:2], inst["dur"][:2] = 2, 1.0
    return inst


def task_with_want(o, need):
    """an open task whose vacancy gives the leader `need` or more followers from its group -> (action, want), or (None, 0)"""
    st, mask = o.env.export(o.shape.M), o.env.mask()
    g = bin(o.o.current_group()).count("1") - 1
    for j in np.flatnonzero(mask[1:] == 0):
        want = min(int(st["status"][j]) - 1, g)
        if want >= need:
            return int(j) + 1, want
    return None, 0


def alone_action(o):
    """a task the leader moves to alone (vacancy <= 1): an open task of status 1, else a masked one with fewer than M members"""
    st, mask, L = o.env.export(o.shape.M), o.env.mask(), o.o.leader
    free = (st["n_mem"] < o.shape.M) & ~(st["members"] == L).any(1)
    for j in list(np.flatnonzero((mask[1:] == 0) & (st["status"] == 1))) + list(np.flatnonzero((mask[1:] > 0) & free)):
        return int(j) + 1
    return None


def plan_case(case, o, k):
    """the bad input of `case` for env o at decision k, or None while its precondition does not hold.  -> dict with the GPU's
    action / followers row / next leader, what the oracle is given and whether it refuses"""
    s, L = o.shape, o.o.leader
    A, M = s.A, s.M
    if case == "follow_other_group":
        if k < 2:
            return None
        other = o.o.pending & ~o.o.current_group()
        action, want = task_with_want(o, 1)
        if not other or action is None:
            return None
        row, fol = o.draw_followers(k, action, M)
        row[0] = bits(other)[0]
        return dict(action=action, row=row, oracle=(action, [int(x) for x in row[:want]], -1), refused=True)
    if case == "leader_restart_ge_A":
        st = o.env.export(M)
        home = sum(1 << i for i in range(A) if st["node"][i] < 0 and st["has_route"][i])
        if (o.o.current_group() | home) != (1 << A) - 1:
            return None                                           # the depot would not end the episode: go home meanwhile
        return dict(action=0, leader=A + 5, oracle=(0, None, -1), refused=False, restart_leader=0)
    if k < CASE_FROM:
        return None
    if case.startswith("action_"):
        action = {"action_minus_one": -1, "action_T_plus_1": s.T + 1, "action_int_max": 2 ** 31 - 1}[case]
        return dict(action=action, oracle=None if action < 0 else (action, None, -1), refused=True)
    if case in ("leader_outside_group", "leader_ge_A"):
        g = o.o.current_group()
        action = alone_action(o)
        if bin(g).count("1") < 3 or action is None:
            return None
        rest = g & ~(1 << L)                                      # the group that decides next: nobody else moved, nobody new is pending
        bad = L if case == "leader_outside_group" else A + 7
        return dict(action=action, leader=bad, oracle=(action, None, bits(rest)[0]), refused=False)
    if case == "depot_with_followers":
        if bin(o.o.current_group()).count("1") < 2:
            return None
        return dict(action=0, row=np.arange(M, dtype=np.int32) % A, oracle=(0, None, -1), refused=False)
    need = 2 if case in ("follow_duplicate", "follow_fstride") else 1
    action, want = task_with_want(o, need)
    if action is None:
        return None
    row, fol = o.draw_followers(k, action, M)
    if case == "follow_not_pending":
        out = [i for i in range(A) if not o.o.pending >> i & 1]
        if not out:
            return None
        row[0] = out[0]
    elif case == "follow_too_few":
        row[want - 1] = -1
        return dict(action=action, row=row, oracle=(action, fol[:-1], -1), refused=True)
    elif case == "follow_too_many":
        row[want] = next(i for i in range(A) if i != L and i not in fol)
        return dict(action=action, row=row, oracle=(action, fol + [int(row[want])], -1), refused=True)
    elif case == "follow_duplicate":
        row[1] = row[0]
    elif case == "follow_id_ge_A":
        row[0] = A
    elif case == "follow_fstride":
        return dict(action=action, row=row, fstride=1, oracle=(action, fol[:1], -1), refused=True)
    return dict(action=action, row=row, oracle=(action, [int(x) for x in row[:want]], -1), refused=True)


@pytest.mark.parametrize("name", ["7A_63T_2M_B100_greedy", "64A_254T_8M_B100_random"])
def test_contract_bits_in_a_mixed_batch(name):
    """each case of CONTRACT_CASES on its own env of one auto-reset batch; every other env plays ExternalOracle's actions.
      - a refused step (ERR_ACTION, ERR_FOLLOW) leaves the raw record as it was except the flags word, the observation, the next
        leader and dcm_total_steps too, and outputs reward 0, used_action -1, done 0; the oracle refuses the same input (rc < 0; an
        action of -1 means the built-in policy to the oracle, so that one is refused on the GPU side only);
      - a bad injected next leader (ERR_LEADER) applies the decision and falls back to the lowest id of the group, which the oracle is
        given; at an auto-reset restart only an id >= A is outside the group (everybody starts in it) and agent 0 starts;
      - the depot with followers given sets no bit: the whole group goes, the followers are ignored;
      - the bit stays set for the rest of the episode and the restart clears it (a restart with a bad injected leader sets
        ERR_LEADER for the new episode): each env's bits are checked after every decision, and each case env goes home a few
        decisions after its case to end its episode;
      - every env, the case envs included, stays bit-exact with its oracle at every decision."""
    shape = envelope_shape(name)
    B, A, M = shape.B, shape.A, shape.M
    cases = [c for c, (_, m) in CONTRACT_CASES.items() if M >= m]
    owner = {case_env(i): c for i, c in enumerate(cases)}
    env = make_env(shape)
    insts = batch_instances(env)
    b_og = next((b for b, c in owner.items() if c == "follow_other_group"), None)
    if b_og is not None:
        insts[b_og] = other_group_instance(insts[b_og])
        env.load_instances(*(np.stack([i[k] for i in insts]) for k in ("task_xy", "depot_xy", "req", "dur")))
    env.reset()
    orcs = [ExternalOracle(shape, b, insts[b]) for b in range(B)]
    fired, home, cleared, expect = {}, set(), set(), np.zeros(B, np.int64)
    off = flags_offset(env)
    steps = 160
    for k in range(steps):
        what = (name, k)
        check_obs(env, orcs, (), what)
        plans = {}
        for b, c in owner.items():
            if b not in fired:
                p = plan_case(c, orcs[b], k)
                if p is not None:
                    plans[b] = p
        fstride = min(p.get("fstride", M) for p in plans.values()) if plans else M
        if fstride < M:                                               # the short stride is the only row case of its decision
            plans = {b: p for b, p in plans.items() if "fstride" in p or "row" not in p}
        inject = inject_followers_at(k) or any("row" in p for p in plans.values())
        dec = [o.decide(k, M, inject) for o in orcs]
        if b_og is not None and b_og not in fired and k < 2:          # tasks 0 and 1 first, two agents each, from the depot at t = 0
            o = orcs[b_og]
            dec[b_og] = (k + 1, *(o.draw_followers(k, k + 1, M) if inject else (None, None)), "legal")
        for b in home:                                                # a case env on its way home: the depot until the episode ends
            dec[b] = (0, np.full(M, -1, np.int32) if inject else None, None, "depot")
        for b, (a, row, fol, kind) in enumerate(dec):
            if fstride < M and b not in plans and fol and len(fol) > fstride:
                dec[b] = (0, np.full(M, -1, np.int32), None, "depot")    # the one decision with a short stride: nobody else injects past it
        acts = np.array([d[0] for d in dec], np.int32)
        rows = np.stack([d[1][:fstride] for d in dec]) if inject else None
        lead_in = np.full(B, -1, np.int32)
        for b, p in plans.items():
            acts[b] = p["action"]
            if inject:
                rows[b] = p["row"][:fstride] if "row" in p else -1
            if "leader" in p:
                lead_in[b] = p["leader"]
        raw0, total0 = env.export_raw(), env.total_steps()
        obs0 = outputs(env)
        env.step(acts, followers=rows, next_leaders=lead_in if (lead_in >= 0).any() else None)
        out = step_outputs(env)
        raw1, flags = env.export_raw(), env.env_flags().cpu().numpy()
        obs1 = outputs(env)
        refused = set()
        for b, o in enumerate(orcs):
            p = plans.get(b)
            if p is not None:
                fired[b] = k
                bit = CONTRACT_CASES[owner[b]][0]
                expect[b] |= bit
                if p["refused"]:
                    refused.add(b)
                    n0 = o.o.n_steps
                    if p["oracle"] is not None:
                        rc = o.o.fused_step(*p["oracle"])[0]
                        assert rc < 0, (what, owner[b], rc)
                    assert o.o.n_steps == n0 and not o.o.done
                    rew, done, lead, ua = out
                    assert rew[b] == 0 and ua[b] == -1 and done[b] == 0, (what, owner[b])
                    assert lead[b] == o.leader == obs0["leader"][b], (what, owner[b])
                    x, y = raw0[b].copy(), raw1[b].copy()
                    x[off:off + 4] = y[off:off + 4] = 0
                    assert np.array_equal(x, y), (what, owner[b], "raw record", np.flatnonzero(x != y)[:8])
                    for n in ("agent_obs", "task_obs", "mask_u8"):
                        assert np.array_equal(obs0[n][b], obs1[n][b]), (what, owner[b], n)
                    continue
                a, fol, nl = p["oracle"]
                res = o.apply(a, fol, nl, restart_leader=p.get("restart_leader", -1))
                if owner[b] == "leader_restart_ge_A":
                    assert res[1] and o.leader == 0, (what, "the depot of the whole remaining group ends the episode")
                    expect[b] = ERR_LEADER
                elif owner[b].startswith("leader_"):
                    assert not res[1] and o.leader == nl, (what, owner[b])
                check_result(out, b, o, res, a, what)
                continue
            a, _, fol, kind = dec[b]
            res = o.apply(a, fol, kind=kind if kind != "depot" else "legal")
            check_result(out, b, o, res, a, what)
            if res[1]:
                if b in fired and expect[b]:
                    cleared.add(b)
                expect[b] = 0                                         # the restart clears the bits
                home.discard(b)
        for b, k0 in fired.items():
            if k == k0 + DRIVE_HOME_AFTER and expect[b]:
                home.add(b)
        assert env.total_steps() == total0 + B - len(refused), what
        for b in range(B):
            assert flags[b] & ERR_BITS == expect[b], (what, b, owner.get(b), flags[b], expect[b])
    assert set(fired) == set(owner), ("cases that never fired", sorted(owner[b] for b in set(owner) - set(fired)))
    kept = [owner[b] for b in owner if CONTRACT_CASES[owner[b]][0] and b not in cleared]
    assert not kept, ("case envs whose episode did not end after their case, so no restart was seen to clear the bit", kept)
    final_checks(env, orcs, insts, (), name)
    env.close()


@pytest.mark.parametrize("name", ["7A_63T_2M_B100_greedy", "64A_254T_8M_B100_random"])
def test_done_env_ignores_any_input(name):
    """without auto-reset a finished env is left untouched whatever it is given: actions -5 and T + 9, followers and leaders out
    of range set no bit; the outputs are done = 1, next_leader = -1, reward = 0, used_action = -1"""
    shape = envelope_shape(name)
    B, A, T = shape.B, shape.A, shape.T
    env = make_env(shape, auto_reset=False)
    env.reset()
    env.step(np.zeros(B, np.int32))          # the depot for the first group, which is everybody: every episode ends (stuck)
    assert env.done_u8.cpu().numpy().all()
    raw0, flags0, total0 = env.export_raw(), env.env_flags().cpu().numpy(), env.total_steps()
    for k, junk in enumerate((-5, T + 9)):
        env.step(np.full(B, junk, np.int32), followers=np.full((B, 3), A + k, np.int32), next_leaders=np.full(B, A + 3, np.int32))
        rew, done, lead, ua = step_outputs(env)
        assert (done == 1).all() and (lead == -1).all() and (rew == 0).all() and (ua == -1).all(), junk
        assert np.array_equal(env.env_flags().cpu().numpy(), flags0) and not (flags0 & ERR_BITS).any(), junk
        assert np.array_equal(env.export_raw(), raw0), junk
    assert env.total_steps() == total0
    env.close()


def norm_distance(ax, ay, bx, by):
    """np.linalg.norm of the 2-vector: sqrt(fma(dy, dy, dx * dx)), one rounding in the fma"""
    dx, dy = ax - bx, ay - by
    return math.sqrt(float(Fraction(dy) * Fraction(dy) + Fraction(dx * dx)))


@pytest.mark.parametrize("name", ["7A_63T_2M_B100_greedy", "64A_254T_8M_B100_random"])
def test_overflow_bit_on_its_envs_only(name):
    """every 25th env sends each of its leaders (with the followers step() draws) to one task until M agents are members, then one
    more with a masked join: DCM_ENV_ERR_OVERFLOW is set on that env at that decision and on no other env; the extra agent moved
    (node, travel distance as the oracle, which has no member cap, moved it) and is not a member.  The other envs stay bit-exact
    with their oracles; the overflowed envs are not compared after their overflow."""
    shape = envelope_shape(name)
    B, A, M = shape.B, shape.A, shape.M
    piles = {b: 0 for b in range(5, B, 25)}                         # env -> the task it piles agents on
    env = make_env(shape)
    insts = batch_instances(env)
    env.reset()
    orcs = [ExternalOracle(shape, b, insts[b]) for b in range(B)]
    over = {}
    for k in range(400):
        what = (name, k)
        check_obs(env, orcs, over, what)
        inject = inject_followers_at(k)
        dec = [o.decide(k, M) if b not in piles else None for b, o in enumerate(orcs)]
        now = set()
        for b, j in piles.items():
            if b in over:
                dec[b] = (0, np.full(M, -1, np.int32) if inject else None, None, "legal")
                continue
            o = orcs[b]
            st = o.env.export(M)
            if st["n_mem"][j] >= M and o.leader not in st["members"][j]:
                now.add(b)
            dec[b] = (j + 1, *(o.draw_followers(k, j + 1, M) if inject else (None, None)), "legal")
        acts = np.array([d[0] for d in dec], np.int32)
        env.step(acts, followers=np.stack([d[1] for d in dec]) if inject else None)
        out, flags = step_outputs(env), env.env_flags().cpu().numpy()
        states = env.export_state(sorted(now)) if now else []
        for b, o in enumerate(orcs):
            if b in over:
                continue
            a, _, fol, kind = dec[b]
            L = o.leader
            if b in now:
                before = o.env.export(M)
                o.apply(a, fol)
                st, want = states[sorted(now).index(b)], o.env.export(M)
                j = a - 1
                assert flags[b] & ERR_OVERFLOW, (what, b)
                assert st["node"][L] == j and st["travel_dist"][L] == want["travel_dist"][L], (what, b)
                xy = insts[b]["task_xy"]
                src = insts[b]["depot_xy"] if before["node"][L] < 0 else xy[before["node"][L]]
                assert st["travel_dist"][L] == before["travel_dist"][L] + norm_distance(*src, *xy[j]), (what, b)
                assert st["n_mem"][j] == M and L not in st["members"][j][:M], (what, b)
                over[b] = k
                continue
            check_result(out, b, o, o.apply(a, fol, kind=kind), a, what)
            assert not flags[b] & ERR_BITS, (what, b, flags[b])
        if len(over) == len(piles):
            break
    assert set(over) == set(piles), ("envs that never overflowed", set(piles) - set(over))
    final_checks(env, orcs, insts, over, name)
    env.close()


def test_step_host_equals_step_on_masked_actions():
    """dcm_step_host (action buffers pageable and pinned on alternate calls) against dcm_step on a twin handle, with ExternalOracle's
    masked action stream at the largest shape: every output at every decision, then the raw records"""
    import torch
    shape = envelope_shape("64A_254T_8M_B100_random")
    B, A, T = shape.B, shape.A, shape.T
    a, h = make_env(shape), make_env(shape)
    insts = batch_instances(a)
    a.reset(); h.reset()
    orcs = [ExternalOracle(shape, b, insts[b]) for b in range(B)]
    pinned = torch.empty(B, dtype=torch.int32).pin_memory()
    out = dict(agent_obs=np.empty((B, A, 6), np.float32), task_obs=np.empty((B, T + 1, 5), np.float32),
               mask=np.empty((B, T + 1), np.uint8), next_leader=np.empty(B, np.int32), reward=np.empty(B, np.float32),
               done=np.empty(B, np.uint8))
    for k in range(200):
        dec = [o.decide(k, inject=False) for o in orcs]
        acts = np.array([d[0] for d in dec], np.int32)
        a.step(acts)
        if k % 2:
            pinned.copy_(torch.from_numpy(acts))
            h.step_host(pinned, out)
        else:
            h.step_host(acts.copy(), out)
        want = outputs(a)
        for n, m in (("agent_obs", "agent_obs"), ("task_obs", "task_obs"), ("mask_u8", "mask"), ("leader", "next_leader"),
                     ("reward", "reward"), ("done_u8", "done")):
            assert np.array_equal(want[n], out[m]), (k, n)
        for b, (o, (x, _, _, kind)) in enumerate(zip(orcs, dec)):
            r, d, _ = o.apply(x, kind=kind)
            assert out["reward"][b] == np.float32(r) and bool(out["done"][b]) == d and out["next_leader"][b] == o.leader, (k, b)
    assert_same_records(a, h, "after 200 decisions")
    a.close(); h.close()
