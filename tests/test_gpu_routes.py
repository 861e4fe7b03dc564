"""GPU tests of dcm_execute_by_route (k_routes: pre_set_route + execute_by_route, task_env.py:562-599, a whole episode per env in one
launch) against the C oracle, every env of every batch: makespan, final state, status bits, the metrics and the per-element waiting sums
of dcm_compute_metrics.  The routes (helpers.make_routes) finish, wait and give up, run into the 200-unit clock, end stuck, re-visit
tasks, go home in the middle, are empty, or fill their row; tests/test_routes_oracle.py checks on the CPU that the batches reach each
of those events.  The edges: coalitions above M, entries outside [0, T], lengths above the row stride (C ABI, guard memory), a
non-default velocity and the individual-agent handle."""
import ctypes as C

import numpy as np
import pytest

from dcmrta_b200._lib import ENV_DONE, ENV_ERR_ACTION, ENV_ERR_MASK, ENV_ERR_OVERFLOW, ENV_FINISHED, ENV_STUCK
from oracle import canon

from gpu_env import instances
from helpers import (ENVELOPE_SHAPES, METRIC_KEYS, ROUTE_MAX_DURATION, envelope_shape, make_routes, pack_routes, route_batch_sizes,
                     route_family, route_oracle, route_seed)

pytestmark = pytest.mark.gpu


def route_env(shape, B, protocol="LF", velocity=0.2):
    """a handle on the instances dcm_generate draws for the shape's envs 0..B-1, reset; -> (env, per-env instances)"""
    from dcmrta_b200 import BatchedTaskEnv
    env = BatchedTaskEnv(B, shape.A, shape.T, M=shape.M, seed=shape.seed, first_gid=shape.first_gid(), protocol=protocol,
                         velocity=velocity)
    env.generate(max_duration=ROUTE_MAX_DURATION, random_duration=shape.random_duration)
    env.reset()
    return env, instances(env)


def batch_routes(shape, insts):
    return [make_routes(route_seed(shape, b), inst, shape.A, shape.M, route_family(b)) for b, inst in enumerate(insts)]


def check_against_oracle(env, insts, makespan, played, envs, velocity=0.2):
    """env b of `envs` against the oracle running routes played[b]: makespan, state and status bits, then dcm_compute_metrics with
    max_wait = 100 (what execute_by_route leaves, task_env.py:564) against the oracle's metrics and waiting sums"""
    A = env.A
    mk = makespan.cpu().numpy()
    flags = env.env_flags().cpu().numpy()
    states = env.export_state(envs)
    env.set_params(velocity=velocity, max_wait=100.0)
    met, tw, aw = (x.cpu().numpy() for x in env.compute_metrics(per_element=True))
    ends = set()
    for q, b in enumerate(envs):
        what = (env.A, env.T, env.M, env.B, b)
        o, want_mk = route_oracle(A, insts[b], played[b], velocity)
        assert mk[b] == want_mk, (what, mk[b], want_mk)
        ref = o.export(canon.MC_CANON)
        d = canon.diff_states(states[q], ref)
        assert not d, (what, d)
        f = int(flags[b])
        assert f & ENV_DONE, (what, f)                                        # always
        assert bool(f & ENV_FINISHED) == ref["env_finished"], (what, f)
        assert bool(f & ENV_STUCK) == o.stuck, (what, f)
        ends.add("finished" if ref["env_finished"] else ("stuck" if o.stuck else "clock_cap"))
        want = o.episode_metrics()[0]
        for c in (0, 1, 2, 3, 5, 6):
            assert met[b, c] == want[METRIC_KEYS[c]], (what, METRIC_KEYS[c], met[b, c], want[METRIC_KEYS[c]])
        # the per-agent sums add W per give-up after the per-task terms instead of interleaved (DESIGN.md §2): 1e-12 relative
        assert met[b, 4] == pytest.approx(want["waiting_time"], rel=1e-12, abs=0), what
        # the oracle counts fused decisions only; the device counts every agent step of the routes, which is every entry of the
        # route lists the oracle's agents recorded (task_env.py:314), the final trips home included
        assert met[b, 7] == sum(len(r) for r, _ in o.routes()), what
        want_aw, want_tw = o.agent_scalars()
        assert np.array_equal(tw[b], want_tw), (what, np.flatnonzero(tw[b] != want_tw)[:8])
        np.testing.assert_allclose(aw[b], want_aw, rtol=1e-12, atol=0, err_msg=str(what))
    return flags, ends


@pytest.mark.parametrize("shape,B", [(s, B) for s in ENVELOPE_SHAPES for B in route_batch_sizes(s)],
                         ids=lambda x: getattr(x, "name", f"B{x}"))
def test_routes_match_oracle(shape, B):
    """every env of the batch, the four route families side by side; no error bits"""
    env, insts = route_env(shape, B)
    R = batch_routes(shape, insts)
    routes, rlen = pack_routes(R, shape.A)
    mk = env.execute_by_route(routes, rlen)
    flags, ends = check_against_oracle(env, insts, mk, R, list(range(B)))
    assert not (flags & ENV_ERR_MASK).any()
    if B == max(route_batch_sizes(shape)) and shape.M > 1:                 # the batch tests/test_routes_oracle.py takes the census of
        assert {"finished", "stuck", "clock_cap"} <= ends, ends
    env.close()


@pytest.mark.parametrize("name", ["24A_64T_8M_B100_random", "33A_129T_5M_B100_greedy"])
def test_route_errors_stay_in_their_env(name):
    """in one batch of 48: envs where M + 1 agents start with the same task get DCM_ENV_ERR_OVERFLOW, envs with entries below 0 or
    above T (one of them first on its route, so that it is played) get DCM_ENV_ERR_ACTION and equal the oracle run with those entries
    replaced by 0 (the depot, as the kernel plays them), and every other env equals the oracle with no error bit"""
    shape = envelope_shape(name)
    B, A, T, M = 48, shape.A, shape.T, shape.M
    env, insts = route_env(shape, B)
    R = batch_routes(shape, insts)
    played = [[list(r) for r in Rb] for Rb in R]
    rng = np.random.default_rng(7)
    overflow, bad = set(range(0, B, 6)), set(range(3, B, 6))
    for b in overflow:
        for a in rng.choice(A, M + 1, replace=False):
            R[b][a] = [1 + b % T] + R[b][a]
    for b in bad:
        for i, a in enumerate(rng.choice([a for a in range(A) if len(R[b][a]) > 1], 2, replace=False)):
            k = 0 if i == 0 else int(rng.integers(len(R[b][a])))               # the first bad entry is played at time 0 for sure
            R[b][a] = list(R[b][a])
            R[b][a][k] = -1 - int(rng.integers(3)) if a % 2 else T + 1 + int(rng.integers(3))
            played[b][a] = [x if 0 <= x <= T else 0 for x in R[b][a]]
    routes, rlen = pack_routes(R, A)
    mk = env.execute_by_route(routes, rlen)
    ok = [b for b in range(B) if b not in overflow]
    flags, _ = check_against_oracle(env, insts, mk, played, ok)
    for b in range(B):
        want = ENV_ERR_OVERFLOW if b in overflow else (ENV_ERR_ACTION if b in bad else 0)
        assert flags[b] & ENV_ERR_MASK == want, (name, b, flags[b])
        assert flags[b] & ENV_DONE
    env.close()


def own_tasks(Rb, a, M):
    """the tasks on agent a's route, or else the first task fewer than M agents are routed to (so that no member list overflows)"""
    own = [x for x in Rb[a] if x > 0]
    if own:
        return own
    count = {}
    for r in Rb:
        for x in set(r):
            count[x] = count.get(x, 0) + 1
    return [next(j for j in range(1, 1000) if count.get(j, 0) < M)]


def test_route_lengths_beyond_the_row_stride():
    """dcm_execute_by_route through the C ABI.  `routes` is the front of a larger tensor whose tail holds live task ids; some route_len
    entries exceed rstride, among them the last agent of the last env, and those rows are filled to rstride with re-visits of the
    agent's own tasks.  Each env plays at most rstride entries of its rows: it equals the oracle on the rows truncated to rstride,
    with DCM_ENV_ERR_ACTION on the envs with a long entry and nothing else.  The makespan lies inside a sentinel frame that survives
    bit for bit."""
    import torch
    from dcmrta_b200._lib import check, lib
    shape = envelope_shape("25A_65T_8M_B100_greedy")
    B, A, T = 37, shape.A, shape.T
    env, insts = route_env(shape, B)
    R = batch_routes(shape, insts)
    L = max(len(r) for Rb in R for r in Rb)
    assert L < 200
    rng = np.random.default_rng(11)
    long = {(b, a) for b in range(2, B, 5) for a in rng.choice(A, 3, replace=False)} | {(B - 1, A - 1)}
    rlen = np.zeros((B, A), np.int32)
    played = [[list(r) for r in Rb] for Rb in R]
    for b in range(B):
        for a in range(A):
            r = R[b][a]
            if (b, a) in long:
                own = own_tasks(played[b], a, shape.M)                       # counts the padding already given
                played[b][a] = r + [own[int(rng.integers(len(own)))] for _ in range(L - len(r))]
                rlen[b, a] = min(L + 1 + int(rng.integers(40)), 255)
            else:
                rlen[b, a] = len(r)
    routes, _ = pack_routes(played, A, L)
    TAIL = 255
    big = torch.empty(B * A * L + TAIL, dtype=torch.int32, device="cuda")
    big[:B * A * L] = torch.from_numpy(routes.reshape(-1)).cuda()
    big[B * A * L:] = torch.from_numpy(rng.integers(1, T + 1, TAIL).astype(np.int32)).cuda()
    before = big.cpu().numpy()
    n_d = torch.from_numpy(rlen).cuda()
    G = 64
    SENT = np.int64(0x7FF4_DEAD_BEEF_0001)                                    # a NaN payload no double the kernel computes carries
    frame = torch.full((B + 2 * G,), int(SENT), dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    check(lib().dcm_execute_by_route(env._h, C.c_void_p(big.data_ptr()), L, C.c_void_p(n_d.data_ptr()),
                                     C.c_void_p(frame.data_ptr() + 8 * G), C.c_void_p(stream)))
    torch.cuda.synchronize()
    fr = frame.cpu().numpy()
    assert (fr[:G] == SENT).all() and (fr[G + B:] == SENT).all(), "makespan written outside its B entries"
    assert np.array_equal(big.cpu().numpy(), before)
    mk = frame[G:G + B].view(torch.float64)
    flags, _ = check_against_oracle(env, insts, mk, played, list(range(B)))
    long_envs = {b for b, _ in long}
    for b in range(B):
        assert flags[b] & ENV_ERR_MASK == (ENV_ERR_ACTION if b in long_envs else 0), (b, flags[b])
    env.close()


def test_routes_at_a_non_default_velocity():
    """set_params(velocity=0.35) against the oracle built with the same velocity, every env"""
    shape = envelope_shape("20A_55T_5M_B100_random")
    env, insts = route_env(shape, 64, velocity=0.35)
    R = batch_routes(shape, insts)
    mk = env.execute_by_route(*pack_routes(R, shape.A))
    flags, _ = check_against_oracle(env, insts, mk, R, list(range(64)), velocity=0.35)
    assert not (flags & ENV_ERR_MASK).any()
    env.close()


def test_individual_agent_handle_plays_routes_alike():
    """the header says dcm_execute_by_route ignores DCM_FLAG_INDIVIDUAL: a handle created with it leaves the same raw records,
    makespans and status bits as the leader-follower handle"""
    shape = envelope_shape("33A_129T_5M_B100_greedy")
    out = []
    for protocol in ("LF", "IA"):
        env, insts = route_env(shape, 64, protocol=protocol)
        mk = env.execute_by_route(*pack_routes(batch_routes(shape, insts), shape.A))
        out.append((env.export_raw(), mk.cpu().numpy(), env.env_flags().cpu().numpy()))
        env.close()
    (ra, ma, fa), (rb, mb, fb) = out
    assert np.array_equal(ra, rb), np.flatnonzero((ra != rb).any(1))[:8]
    assert np.array_equal(ma, mb) and np.array_equal(fa, fb)
