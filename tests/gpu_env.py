"""The machinery the env's GPU tests share (tests only): handles and their instances, the step outputs, the in-kernel policy in lock-step
with the oracle, a default handle against one built with an environment switch, and dcm_step_host against dcm_step.  Nothing here
imports torch at module level, so the suite still collects without a GPU."""
from __future__ import annotations

import contextlib

import numpy as np
import pytest

from dcmrta_b200._lib import ENV_ERR_MASK
from oracle import canon

from helpers import METRIC_KEYS, EnvelopeOracle

OUTPUTS = ("reward", "leader", "done_u8", "used_action", "agent_obs", "task_obs", "mask_u8")
HOST_OUTPUTS = {"agent_obs": "agent_obs", "task_obs": "task_obs", "mask_u8": "mask", "leader": "next_leader", "reward": "reward",
                "done_u8": "done"}                      # BatchedTaskEnv buffer -> its key in the output dict of step_host


def make_env(shape, protocol="LF", auto_reset=True, seed=None, first_gid=None):
    """a handle of the shape's B, A, T and M on the instances dcm_generate draws for the shape's seed and global ids (or `seed` and
    `first_gid`), not reset"""
    from dcmrta_b200 import BatchedTaskEnv
    env = BatchedTaskEnv(shape.B, shape.A, shape.T, M=shape.M, auto_reset=auto_reset, seed=shape.seed if seed is None else seed,
                         first_gid=shape.first_gid() if first_gid is None else first_gid, protocol=protocol)
    env.generate(max_duration=5.0, random_duration=shape.random_duration)
    return env


def instances(env, envs=None):
    """the instances of envs `envs` (every env when None), one dict of NumPy arrays per env"""
    envs = [int(b) for b in (range(env.B) if envs is None else envs)]
    got = {k: v[envs].cpu().numpy() for k, v in env.get_instances().items()}
    return [{k: got[k][q] for k in got} for q in range(len(envs))]


def stack_instances(insts):
    """per-env instance dicts -> the arguments of BatchedTaskEnv.load_instances"""
    return (np.stack([i["task_xy"] for i in insts]), np.stack([i["depot_xy"] for i in insts]),
            np.stack([i["req"] for i in insts]).astype(np.int32), np.stack([i["dur"] for i in insts]))


def outputs(env):
    """host copies of the step's output buffers, by name"""
    return {n: getattr(env, n).cpu().numpy() for n in OUTPUTS}


def assert_same_outputs(a, b, what):
    import torch
    for n in OUTPUTS:
        assert torch.equal(getattr(a, n), getattr(b, n)), (what, n)


def assert_same_records(a, b, what):
    """the raw records of every env are equal; otherwise name the first env that differs and its decoded fields that do"""
    ra, rb = a.export_raw(), b.export_raw()
    if np.array_equal(ra, rb):
        return
    bad = np.flatnonzero((ra != rb).any(1))
    sa, sb = a.export_state(bad[:1])[0], b.export_state(bad[:1])[0]
    diff = [key for key in sa if not np.array_equal(np.asarray(sa[key]), np.asarray(sb[key]), equal_nan=True)]
    raise AssertionError(f"{what}: {len(bad)} envs differ, first env {bad[0]} in {diff}")


def check_obs(env, oracles, envs, what, leader=None):
    """mask, agent rows and task rows of env envs[q] against oracles[q], seen by the oracle's leader or by leader[envs[q]]"""
    envs = list(envs)
    ag, tk, mk = (getattr(env, n)[envs].cpu().numpy() for n in ("agent_obs", "task_obs", "mask_u8"))
    for q, (b, o) in enumerate(zip(envs, oracles)):
        l = o.leader if leader is None else int(leader[b])
        assert np.array_equal(mk[q], o.env.mask()), (what, b, "mask")
        assert np.array_equal(ag[q], o.env.agent_status(l).astype(np.float32)), (what, b, "agent rows")
        assert np.array_equal(tk[q], o.env.task_status(l).astype(np.float32)), (what, b, "task rows")


def assert_metrics_match(got, want, what):
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0, err_msg=str(what))      # waiting_time: the documented order difference
    for c in (0, 1, 2, 3, 5, 6, 7):
        assert got[c] == want[c], (what, METRIC_KEYS[c], got[c], want[c])


def lockstep(env, shape, sample, steps, seed=None, first_gid=None, min_episodes=2, metrics=True, after_step=None):
    """`steps` decisions of the in-kernel shape.policy on `env` (reset, auto-reset, protocol env.protocol) against an EnvelopeOracle
    per env of `sample` (with `seed` and `first_gid` as the handle's): the mask, agent rows and task rows before every decision,
    reward, done and next leader after it; then at least `min_episodes` episodes per sampled env, the metrics of its last one
    (`metrics`), its state, no error bit in the batch and the step counter.  after_step(k) runs after decision k of `env`.
    -> the oracles"""
    orcs = [EnvelopeOracle(shape, b, inst, env.protocol, seed, first_gid) for b, inst in zip(sample, instances(env, sample))]
    first = env.leader[sample].cpu().numpy()
    for q, o in enumerate(orcs):
        assert o.leader == first[q], (shape.name, env.protocol, sample[q])
    for k in range(steps):
        what = (shape.name, env.protocol, k)
        check_obs(env, orcs, sample, what)
        env.step(policy=shape.policy)
        if after_step:
            after_step(k)
        rew, done, lead = (getattr(env, n)[sample].cpu().numpy() for n in ("reward", "done_u8", "leader"))
        for q, o in enumerate(orcs):
            r, d, _ = o.step()
            assert rew[q] == np.float32(r), (what, sample[q], "reward")
            assert bool(done[q]) == d, (what, sample[q], "done")
            assert lead[q] == o.leader, (what, sample[q], "next leader")
    assert min(o.episodes for o in orcs) >= min_episodes, (shape.name, env.protocol)
    if metrics:
        met = env.episode_metrics()[sample].cpu().numpy()
        for q, o in enumerate(orcs):
            assert_metrics_match(met[q], o.last_metrics, (shape.name, env.protocol, sample[q]))
    for q, (o, st) in enumerate(zip(orcs, env.export_state(sample))):
        d = canon.diff_states(st, o.o.export(canon.MC_CANON))
        assert not d, (shape.name, env.protocol, sample[q], d)
    assert not (env.env_flags().cpu().numpy() & ENV_ERR_MASK).any()
    assert env.total_steps() == env.B * steps
    return orcs


def check_shard_invariance(protocol, steps):
    """SURVEY 8(e): the trajectory of global env k does not depend on the batch it lives in.  Envs 32..47 of a batch of 64 and a batch
    of 16 whose env 0 has global id 32, `steps` decisions of the in-kernel random policy: the same raw records and task rows."""
    from dcmrta_b200 import BatchedTaskEnv
    A, T = 20, 50
    with contextlib.closing(BatchedTaskEnv(64, A, T, auto_reset=True, seed=7, first_gid=0, protocol=protocol)) as big, \
            contextlib.closing(BatchedTaskEnv(16, A, T, auto_reset=True, seed=7, first_gid=32, protocol=protocol)) as small:
        for e in (big, small):
            e.generate()
            e.reset()
        for _ in range(steps):
            big.step(policy="random")
            small.step(policy="random")
        assert np.array_equal(big.export_raw()[32:48], small.export_raw())
        assert np.array_equal(big.task_obs[32:48].cpu().numpy(), small.task_obs.cpu().numpy())


@contextlib.contextmanager
def twin_handles(make, variant=None):
    """two handles from make() (a new handle on generated instances), the second created with the environment switch `variant` set
    to 1 (None: two default handles).  dcm_create reads the switches once, so the switch is set around that construction only.  Both
    are reset, and closed when the block ends, passed or failed."""
    with contextlib.ExitStack() as stack:
        a = stack.enter_context(contextlib.closing(make()))
        with pytest.MonkeyPatch.context() as mp:
            if variant:
                mp.setenv(variant, "1")
            b = stack.enter_context(contextlib.closing(make()))
        a.reset()
        b.reset()
        yield a, b


def twin_steps(a, b, policy, steps, checkpoint, after_step=None):
    """`steps` decisions of the in-kernel `policy` on both handles: every output and the raw records equal at the decisions k for
    which checkpoint(k) holds, the raw records and the last episodes' metrics at the end.  after_step(k) runs after decision k of
    both.  -> the number of episode ends of `a`"""
    ended = 0
    for k in range(steps):
        a.step(policy=policy)
        b.step(policy=policy)
        ended = ended + a.done_u8.sum()                 # on the device: no synchronisation per decision
        if after_step:
            after_step(k)
        if checkpoint(k):
            assert_same_outputs(a, b, k)
            assert_same_records(a, b, k)
    assert_same_records(a, b, "at the end")
    assert np.array_equal(a.episode_metrics().cpu().numpy(), b.episode_metrics().cpu().numpy())
    return int(ended)


def step_host_equals_step(dev, host, steps, actions=None, pinned=False, after_step=None):
    """dcm_step_host on `host` against dcm_step on `dev`, twin handles: every output at every decision, then the raw records.
    actions(k) -> the int32 actions [B] of decision k, which both are given; None plays the in-kernel random policy on `dev` and gives
    `host` the actions it used.  pinned: the action buffer is pinned on odd decisions (the step kernel reads it in place) and pageable on
    even ones (a staged copy).  after_step(k, out) runs after each comparison, `out` holding host's outputs.  -> the number of
    episode ends"""
    import torch
    B, A, T = dev.B, dev.A, dev.T
    out = {"next_leader": np.empty(B, np.int32), "reward": np.empty(B, np.float32), "done": np.empty(B, np.uint8),
           "agent_obs": np.empty((B, A, 6), np.float32), "task_obs": np.empty((B, T + 1, 5), np.float32), "mask": np.empty((B, T + 1), np.uint8)}
    buf = torch.empty(B, dtype=torch.int32).pin_memory() if pinned else None
    ended = 0
    for k in range(steps):
        if actions is None:
            dev.step(policy="random")
            acts = np.array(dev.used_action.cpu().numpy(), np.int32)
        else:
            acts = np.array(actions(k), np.int32)
            dev.step(acts)
        if pinned and k % 2:
            buf.copy_(torch.from_numpy(acts))
            host.step_host(buf, out)
        else:
            host.step_host(acts, out)
        for n, m in HOST_OUTPUTS.items():
            assert np.array_equal(out[m], getattr(dev, n).cpu().numpy()), (k, n)
        ended += int(out["done"].sum())
        if after_step:
            after_step(k, out)
    assert_same_records(dev, host, f"after {steps} decisions")
    return ended
