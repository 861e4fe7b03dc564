"""GPU tests of the CUDA path at the edges of the supported shape range (include/dcmrta.h: 1 <= A <= 64, 1 <= T <= 254, 1 <= M <= 8),
where the kernels change code path: one, two or four 64-bit task-mask words and the last bit of each, agent bit 63, node ids in 32 or
64 bytes, the step's next_decision scratch (A <= 24) or not, ragged agent chunks of the observation kernels, k_obs_tile or the chunked
k_obs, the second 16-entry staging chunk of the step's scans, 8-member coalitions, partial tiles of envs, and metric sums over more than
248 tasks (NumPy splits those twice).  The shapes, their trajectories' census and the CPU side of the same runs are in tests/helpers.py
and tests/test_shape_envelope_oracle.py.  The whole file takes about 16 s on one B200."""
from contextlib import closing

import numpy as np
import pytest

from dcmrta_b200._lib import ENV_DONE, ENV_ERR_MASK, ENV_FINISHED, ENV_STUCK

from gpu_env import (assert_metrics_match, assert_same_outputs, assert_same_records, check_obs, instances, lockstep, make_env,
                     stack_instances, twin_handles, twin_steps)
from helpers import ENVELOPE_SHAPES, EnvelopeOracle, EnvelopeShape, device_instance, envelope_shape

pytestmark = pytest.mark.gpu
OBS_TILE_AGENTS = 20


def obs_tile_switch(A=OBS_TILE_AGENTS):
    """The largest T whose observations k_obs_tile writes at A agents (dcm_kernels.cu: obs_tile_smem and the rule of prepare_obs, with
    this device's shared memory), so that T + 1 is the first served by the chunked k_obs."""
    import torch
    p = torch.cuda.get_device_properties(0)
    optin, per_sm = p.shared_memory_per_block_optin, p.shared_memory_per_multiprocessor

    def smem(T):
        r16 = lambda n: (n + 15) & ~15
        parts = [32 * 6 * A * 4, 32 * 5 * (T + 1) * 4, 32 * (T + 1), 256 * T, 256 * T, 1024 * A, 512 * A, 32 * T, 32 * T, 8]
        return sum(r16(n) for n in parts)

    fits = [T for T in range(1, 255) if smem(T) <= optin and 2 * (smem(T) + 1024) <= per_sm]
    assert fits and fits[-1] < 254, "every T or no T uses k_obs_tile at this A: nothing to straddle"
    return fits[-1]


def test_table_straddles_the_obs_tile_switch():
    """the two 20-agent shapes of the table are the last shape k_obs_tile serves and the first k_obs serves on this device"""
    t = obs_tile_switch()
    tabled = sorted(s.T for s in ENVELOPE_SHAPES if s.A == OBS_TILE_AGENTS)
    assert tabled == [t, t + 1], f"k_obs_tile serves T <= {t} at A = {OBS_TILE_AGENTS} here; update the table's 20-agent shapes"


def test_device_generator_is_the_restated_one():
    """dcm_generate draws what helpers.device_instance restates on the CPU, so the oracle-only runs of the CPU test replay the
    trajectories this file checks"""
    for shape in (ENVELOPE_SHAPES[0], envelope_shape("64A_254T_8M_B100_random"), envelope_shape("33A_129T_5M_B100_greedy")):
        env = make_env(shape)
        for b, got in zip(shape.sample(), instances(env, shape.sample())):
            want = device_instance(shape.A, shape.T, shape.M, shape.seed, shape.first_gid() + b, random_duration=shape.random_duration)
            for k in ("task_xy", "depot_xy", "req", "dur"):
                assert np.array_equal(got[k], want[k]), (shape.name, b, k)
        env.close()


def run_lockstep(shape, protocol, steps):
    """in-kernel policy with auto-reset against the oracle on the shape's sample (gpu_env.lockstep).  -> the oracles"""
    with closing(make_env(shape, protocol)) as env:
        env.reset()
        return lockstep(env, shape, shape.sample(), steps, min_episodes=1 if shape.T > 200 else 2)


@pytest.mark.parametrize("shape", ENVELOPE_SHAPES, ids=lambda s: s.name)
def test_envelope_matches_oracle(shape):
    """leader-follower, and the census events the shape is listed for"""
    orcs = run_lockstep(shape, "LF", shape.steps)
    missing = set(shape.census) - set.union(*(o.census for o in orcs))
    assert not missing, (shape.name, missing)


@pytest.mark.parametrize("shape", [s for s in ENVELOPE_SHAPES if s.ia_steps], ids=lambda s: s.name)
def test_envelope_ia_matches_oracle(shape):
    """the individual-agent protocol (tests/ia_oracle.py's loop) at the shapes of the table that run it"""
    run_lockstep(shape, "IA", shape.ia_steps)


@pytest.mark.parametrize("which", ["tile_last", "chunked_first", "64A_254T_8M"])
def test_envelope_default_pass_equals_serial_pass(which):
    """the default pass against DCM_PASS_SERIAL (k_step, episode kernel and the chunked k_obs one after the other): every output at
    checkpoints and the raw records of every env, on the last shape k_obs_tile serves at 20 agents, the first it does not, and the
    largest shape"""
    if which == "64A_254T_8M":
        shape = EnvelopeShape(64, 254, 8, 1003, "random", 700, None, "", [])      # the table's largest shape at ten times its batch
    else:
        shape = EnvelopeShape(OBS_TILE_AGENTS, obs_tile_switch() + (which == "chunked_first"), 5, 4099, "random", 500, None, "", [])
    with twin_handles(lambda: make_env(shape), "DCM_PASS_SERIAL") as (a, b):
        ended = twin_steps(a, b, shape.policy, shape.steps, lambda k: k % 50 == 49 or k < 3 or k == shape.steps - 1)
        assert ended > shape.B                                              # restarts were exercised
        assert not (a.env_flags().cpu().numpy() & ENV_ERR_MASK).any()


def test_step_without_next_decision_scratch_equals_default():
    """24 agents, the largest count whose next_decision rows the step keeps in shared memory: DCM_STEP_NO_NDS=1 (rows from global
    memory) leaves every raw record as the default does"""
    shape = EnvelopeShape(24, 64, 8, 1003, "random", 400, None, "", [])        # the table's 24-agent shape at ten times its batch
    with twin_handles(lambda: make_env(shape), "DCM_STEP_NO_NDS") as (a, b):
        twin_steps(a, b, shape.policy, shape.steps, lambda k: k % 100 == 99)


@pytest.mark.parametrize("name", ["2A_3T_3M_B100_random", "7A_63T_2M_B100_greedy", "64A_249T_3M_B100_greedy", "64A_254T_8M_B100_random"])
def test_envelope_granular_path(name):
    """without auto-reset: dcm_build_obs (always the chunked k_obs) for several leaders of each checked state against the oracle's
    observations, then, once every sampled episode has ended, dcm_compute_metrics (the thread-per-env np_sum) against the oracle's
    metrics and the DONE / FINISHED / STUCK bits against the oracle's end of the episode.  An episode that finishes but is flagged
    stuck ends at the same decision with the same metrics, so the bits are the only output that tells the two apart; 64A/249T
    finishes its episodes (agent bit 63 of the returned mask), the others end by the clock cap or stuck."""
    import torch
    shape = envelope_shape(name)
    env = make_env(shape, auto_reset=False)
    sample = shape.sample()
    orcs = [EnvelopeOracle(shape, b, inst) for b, inst in zip(sample, instances(env, sample))]
    env.reset()
    B, A = shape.B, shape.A
    ended = [False] * len(sample)
    k = 0
    while not all(ended):
        if k % 20 == 0:
            live = env.leader.cpu().numpy()
            for trial in range(3):
                leaders = (np.arange(B, dtype=np.int32) * 7 + k + trial * (A // 3 + 1)) % A
                if trial == 0:
                    leaders[:] = A - 1
                env.build_obs(leaders)
                playing = [q for q in range(len(sample)) if not ended[q]]
                check_obs(env, [orcs[q] for q in playing], [sample[q] for q in playing], (name, k, trial), leader=leaders)
            env.build_obs(np.where(live >= 0, live, 0).astype(np.int32))       # what the step wrote, for the policy of the next step
        env.step(policy=shape.policy)
        done = env.done_u8[sample].cpu().numpy()
        for q, o in enumerate(orcs):
            if ended[q]:
                assert done[q], (name, sample[q], k)                             # a finished env stays finished
                continue
            r, d, _ = o.step()
            assert bool(done[q]) == d, (name, sample[q], k)
            ended[q] = d
        k += 1
        assert k <= shape.steps, (name, "an episode did not end")
    torch.cuda.synchronize()
    flags = env.env_flags()[sample].cpu().numpy()
    met = env.compute_metrics()[sample].cpu().numpy()
    for q, o in enumerate(orcs):
        finished, stuck = o.first_end
        want = ENV_DONE | (ENV_FINISHED if finished else 0) | (ENV_STUCK if stuck else 0)
        assert flags[q] & (ENV_DONE | ENV_FINISHED | ENV_STUCK) == want, (name, sample[q], flags[q])
        assert_metrics_match(met[q], o.last_metrics, (name, sample[q]))
    assert not (env.env_flags().cpu().numpy() & ENV_ERR_MASK).any()
    env.close()


def test_export_import_at_the_largest_shape():
    """the raw records of a batch in mid-episode copied into a fresh handle with the same instances and seed: 100 more decisions of
    both give the same records and outputs"""
    from dcmrta_b200 import BatchedTaskEnv
    shape = envelope_shape("64A_254T_8M_B100_random")
    a = make_env(shape)
    a.reset()
    for _ in range(150):
        a.step(policy=shape.policy)
    b = BatchedTaskEnv(shape.B, shape.A, shape.T, M=shape.M, auto_reset=True, seed=shape.seed, first_gid=shape.first_gid())
    b.load_instances(*stack_instances(instances(a)))
    b.import_raw(a.export_raw())
    assert_same_records(a, b, "after import")
    for k in range(100):
        a.step(policy=shape.policy)
        b.step(policy=shape.policy)
        assert_same_outputs(a, b, k)
    assert_same_records(a, b, "after 100 decisions")
    assert np.array_equal(a.episode_metrics().cpu().numpy(), b.episode_metrics().cpu().numpy())
    a.close(); b.close()


@pytest.mark.parametrize("name", ["64A_254T_8M_B100_random", "1A_1T_1M_B33_random"])
def test_policy_forward_on_envelope_observations(name):
    """FusedPolicy on the observations the env wrote, with the bounds of test_fused_forward_matches_the_module.  At 64 agents and
    255 task rows the attention's key counts are 64, the largest single-block case of k_attention_mma, and 255, its multi-block path."""
    import torch
    from dcmrta_b200.policy_fused import FusedPolicy, forward_torch
    from test_policy_fused import _net
    shape = envelope_shape(name)
    env = make_env(shape)
    env.reset()
    for _ in range(30):
        env.step(policy=shape.policy)
    net = _net().cuda()
    tasks, agents, mask = env.task_obs, env.agent_obs, env.mask_u8.view(torch.bool)
    with torch.no_grad():
        ref = net(tasks, agents, mask)
    out = FusedPolicy(net)(tasks, agents, mask).clone()
    assert out.shape == ref.shape == (shape.B, shape.T + 1) and bool(torch.isfinite(out).all())
    spec = forward_torch(net, tasks, agents, mask, torch.bfloat16)
    ok = ~mask
    assert float((out - spec).abs()[ok].max()) < 0.08, "CUDA kernels vs the same dataflow in torch bf16"
    assert float((out - ref).abs()[ok].max()) < 0.1, "bf16 fused path vs the fp32 module"
    chosen = ref.gather(1, out.argmax(1, keepdim=True)).squeeze(1)
    assert float((ref.max(1).values - chosen).max()) < 0.1
    assert torch.allclose(out.exp().sum(1), torch.ones(shape.B, device=out.device), atol=1e-3)
    env.close()
