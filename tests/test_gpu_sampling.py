"""GPU tests of the policy's action sampler (dcmp_sample, include/dcmrta_sample.h; DESIGN.md 5): exact cases bit for bit, random and
real log-probabilities against the float64 rule of tests/test_sampling_rule.py inside a derived window, the distribution, the counter, guard
memory, the rollouts' invariance to batching / compaction / graphs / shards, an oracle replay of sampled episodes, and best-of-K evaluation."""
import math

import numpy as np
import pytest

from helpers import GOLD, METRIC_KEYS
from test_sampling_rule import kth_allowed, rule64, sampler_word

pytestmark = pytest.mark.gpu
NS = (1, 2, 31, 32, 33, 51, 64, 65, 255, 256)
ERR_BITS = 0xF0
SENTINEL = 0x5A5A5A5A


def run(x, mask, seed, stream, decision, rows=None, first_gid=0):
    import torch
    from dcmrta_b200.policy_fused import draw_tensor, sample
    x = torch.as_tensor(x).cuda()
    m = None if mask is None else torch.as_tensor(np.ascontiguousarray(mask, np.uint8)).cuda()
    r = None if rows is None else torch.as_tensor(rows, dtype=torch.int64).cuda()
    return sample(x, m, draw_tensor(seed, stream, decision, x.device), r, first_gid).cpu().numpy()


# ---- exact cases ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", NS)
def test_exact_cases(n):
    rng = np.random.default_rng(n)
    B, seed, stream, dec, g0 = 4099, 2 ** 40 + 3, 5, 77, 12345
    x0 = sampler_word(seed, g0 + np.arange(B), stream, dec)
    # all-ones allowed weights (a constant per row), random masks, NaN behind the mask (never read): allowed index number floor(u S)
    mask = rng.random((B, n)) < rng.random((B, 1))
    mask[0] = True
    x = np.repeat(rng.normal(0, 50, (B, 1)).astype(np.float32), n, 1)
    x[mask] = np.nan
    a = run(x, mask, seed, stream, dec, first_gid=g0)
    assert np.array_equal(a, kth_allowed(~mask, x0)), n
    assert a[0] == 0                                                          # no allowed entry
    # a single allowed entry, whatever its value
    one = rng.integers(0, n, B)
    mask = np.ones((B, n), bool)
    mask[np.arange(B), one] = False
    x = rng.normal(0, 1e3, (B, n)).astype(np.float32)
    assert np.array_equal(run(x, mask, seed, stream, dec, first_gid=g0), one)
    # -inf and -1e4-gap entries have weight exactly 0: with equal live entries the choice is again exact, with and without a mask
    c = rng.normal(0, 10, (B, 1)).astype(np.float32)
    x = np.repeat(c, n, 1)
    kind = rng.integers(0, 3, (B, n))                                         # 0 live, 1 -inf, 2 a gap of 1e4 below the live value
    kind[:, rng.integers(0, n)] = 0
    x[kind == 1] = -np.inf
    x[kind == 2] = np.repeat(c - np.float32(1e4), n, 1)[kind == 2]
    for mk in (None, ((rng.random((B, n)) < 0.3) & (kind != 0)) | (rng.random((B, n)) < 0.1)):
        allowed = np.ones((B, n), bool) if mk is None else ~mk
        top = np.where(allowed, x, -np.inf).max(1, keepdims=True)
        live = allowed & (x == top) & (top > -np.inf)                         # (a row whose live entries are all masked: its gap entries)
        a = run(x, mk, seed, stream, dec, first_gid=g0)
        assert np.array_equal(a, kth_allowed(live, x0)), n
        has = (allowed & (kind == 0)).any(1)
        assert (kind[np.arange(B), a][has] == 0).all() and allowed[np.arange(B), a][live.any(1)].all()
    # every allowed entry at -inf: nothing of positive weight, action 0
    x = np.full((B, n), -np.inf, np.float32)
    assert (run(x, None, seed, stream, dec) == 0).all()


# ---- bounded cases ----------------------------------------------------------------------------------------------------------------------
def window(S, n):
    """|C_j(kernel) - C_j(float64)| and |S(kernel) - S(float64)| are both at most E, so the kernel's comparison C_j > theta agrees with the
    float64 one wherever |theta - C_j| > 2 E (theta moves by u |dS| <= E, C_j by E).  E over the row:
      * the subtraction x_j - m rounds once: w_j (1 + |x_j - m| 2^-24) up to second order, and w |x - m| = |x - m| e^-|x - m| <= 1/e;
      * expf has at most 2 ulp of error (CUDA C Programming Guide, single-precision functions): w_j 2^-22;
      * the prefix sum takes each w_j through at most 5 shuffle levels, one carry add per chunk and at most 8 chunks, 13 roundings:
        gamma_13 S with gamma_k = k 2^-24 / (1 - k 2^-24);
      * weights below the fp32 normal range carry absolute errors of at most 2^-126 each.
    E = S (2^-22 + gamma_13) + n (2^-24 / e + 2^-126); the window is 2 E, doubled again for slack."""
    g13 = 13 * 2.0 ** -24 / (1 - 13 * 2.0 ** -24)
    return 4 * (S * (2.0 ** -22 + g13) + n * (2.0 ** -24 / math.e + 2.0 ** -126))


def check_bounded(x, mask, a, x0):
    """The kernel's actions `a` against the float64 rule: equal outside the window, one of the two positive-weight entries either side of
    the boundary inside it.  Returns how many draws fell in the window."""
    ref, C, S, theta, w = rule64(x, mask, x0)
    n = x.shape[1]
    near = 0
    for b in range(x.shape[0]):
        pos = np.flatnonzero(w[b] > 0)
        if pos.size == 0:
            assert a[b] == 0, b
            continue
        tol = window(S[b], n)
        close = pos[np.abs(C[b, pos] - theta[b]) <= tol]
        if close.size == 0:
            assert a[b] == ref[b], (b, a[b], ref[b])
            continue
        near += 1
        ok = {int(ref[b])}
        for j in close:                                                       # boundary after j: j itself or the next positive entry
            ok.add(int(j))
            nxt = pos[pos > j]
            if nxt.size:
                ok.add(int(nxt[0]))
        assert int(a[b]) in ok, (b, a[b], sorted(ok))
    return near


@pytest.mark.parametrize("n", NS)
def test_random_logits_against_float64_rule(n):
    rng = np.random.default_rng(100 + n)
    B = 8192
    x = (rng.normal(0, 2, (B, n)) + rng.normal(0, 30, (B, 1))).astype(np.float32)
    x[rng.random((B, n)) < 0.05] = -np.inf
    mask = rng.random((B, n)) < rng.random((B, 1)) * 0.8
    for dec in (0, 1, 2 ** 30 - 2):
        x0 = sampler_word(9, 500 + np.arange(B), 3, dec)
        near = check_bounded(x, mask, run(x, mask, 9, 3, dec, first_gid=500), x0)
        print(f"n={n} decision={dec}: {near} of {B} draws in the window")


def test_fused_forward_log_probabilities_against_float64_rule():
    """The fused forward's own log-probabilities (with its -1e4 fill) on real observations, sampled with and without the mask."""
    import torch
    from dcmrta_b200 import BatchedTaskEnv
    from dcmrta_b200.policy import AttentionNet
    from dcmrta_b200.policy_fused import FusedPolicy
    torch.manual_seed(3)
    net = AttentionNet(6, 5, 128).cuda().eval()
    env = BatchedTaskEnv(4096, 20, 50, auto_reset=True, seed=8, first_gid=0)
    env.generate()
    env.reset()
    fused = FusedPolicy(net)
    total = 0
    for k in range(40):
        if k % 10 == 0:
            mask = env.mask_u8.clone()
            logp = fused(env.task_obs, env.agent_obs, mask.view(torch.bool)).clone()
            x, m = logp.cpu().numpy(), mask.cpu().numpy().astype(bool)
            for use_mask in (True, False):
                a = run(x, m if use_mask else None, 21, 0, k, first_gid=0)
                total += check_bounded(x, m if use_mask else None, a, sampler_word(21, np.arange(4096), 0, k))
                if use_mask:
                    assert not m[np.arange(4096), a].any()
        env.step(policy="random")
    print(f"fused log-probabilities: {total} of {8 * 4096} draws in the window")
    env.close()


def test_distribution_chi_square():
    """2^20 draws of fixed rows: 4,096 rows (global ids) x 256 decision words; deterministic, so one fixed threshold."""
    import torch
    from scipy.stats import chi2
    from dcmrta_b200.policy_fused import draw_tensor, sample
    rng = np.random.default_rng(7)
    n, B = 51, 4096
    row = rng.normal(0, 1.5, n).astype(np.float32)
    mask = rng.random(n) < 0.25
    mask[3] = False
    x = torch.from_numpy(np.repeat(row[None], B, 0)).cuda()
    m = torch.from_numpy(np.repeat(mask[None], B, 0).astype(np.uint8)).cuda()
    draw = draw_tensor(99, 0, 0, x.device)
    counts = torch.zeros(n, dtype=torch.int64, device=x.device)
    for d in range(256):
        draw[3].fill_(d)
        counts += torch.bincount(sample(x, m, draw).long(), minlength=n)
    counts = counts.cpu().numpy()
    _, _, _, _, w = rule64(row[None], mask[None], np.zeros(1, np.uint32))
    p = w[0] / w[0].sum()
    N = B * 256
    live = p > 0
    assert counts.sum() == N and counts[~live].sum() == 0
    stat = float((((counts - N * p) ** 2)[live] / (N * p[live])).sum())
    limit = chi2.ppf(1 - 1e-6, int(live.sum()) - 1)
    print(f"chi-square {stat:.1f}, {int(live.sum()) - 1} degrees of freedom, limit {limit:.1f}")
    assert stat < limit


# ---- the counter -------------------------------------------------------------------------------------------------------------------------
def test_counter_keys_rows_and_graph_replay():
    import torch
    from dcmrta_b200.policy_fused import draw_tensor, sample
    B, n = 4096, 256                                                          # all-ones weights: the action is x0 >> 24
    x = np.zeros((B, n), np.float32)
    base = dict(seed=5, stream=1, decision=3, first_gid=1000)

    def draws(seed, stream, decision, first_gid, rows=None):
        return run(x if rows is None else x[:len(rows)], None, seed, stream, decision, rows, first_gid)
    a = draws(**base)
    assert np.array_equal(a, (sampler_word(5, 1000 + np.arange(B), 1, 3) >> 24).astype(np.int32))
    assert np.array_equal(draws(**base), a)                                   # the same inputs, the same draws
    for key, val in (("seed", 6), ("seed", 5 + 2 ** 32), ("stream", 2), ("decision", 4), ("first_gid", 1001)):
        b = draws(**{**base, key: val})
        assert (b != a).mean() > 0.9, key
    rows = np.random.default_rng(0).permutation(B)[:1000]
    assert np.array_equal(draws(**base, rows=rows), a[rows])                  # a row reached through rows_d draws its env's draw
    # one captured graph, new draw words between replays
    xt = torch.from_numpy(x).cuda()
    draw = draw_tensor(5, 1, 3, xt.device)
    out = torch.empty(B, dtype=torch.int32, device=xt.device)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        sample(xt, None, draw, None, 1000, out)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        sample(xt, None, draw, None, 1000, out)
        draw[3:].add_(1)
    for seed, stream, dec in ((5, 1, 3), (8, 0, 0), (2 ** 63 + 1, 7, 2 ** 30 - 3)):
        draw.copy_(draw_tensor(seed, stream, dec, xt.device))
        g.replay()
        assert np.array_equal(out.cpu().numpy(), draws(seed, stream, dec, 1000)), (seed, stream, dec)
        assert int(draw[3]) == dec + 1


def test_guard_memory_and_argument_errors():
    import ctypes as C
    import torch
    from dcmrta_b200 import policy_fused as pf
    rng = np.random.default_rng(1)
    B, n, ld, pad = 1001, 51, 64, 32
    x = np.full((B, ld), np.nan, np.float32)                                  # NaN in the unread columns n..ld-1
    x[:, :n] = rng.normal(0, 2, (B, n))
    mask = rng.random((B, n)) < 0.3
    xt = torch.from_numpy(x).cuda()[:, :n]
    assert xt.stride(0) == ld
    m = torch.from_numpy(mask.astype(np.uint8)).cuda()
    frame = torch.full((B + 2 * pad,), SENTINEL, dtype=torch.int32, device="cuda")
    draw = pf.draw_tensor(4, 0, 1, xt.device)
    a = pf.sample(xt, m, draw, None, 0, frame[pad:pad + B]).cpu().numpy()
    f = frame.cpu().numpy()
    assert (f[:pad] == SENTINEL).all() and (f[pad + B:] == SENTINEL).all()
    check_bounded(x[:, :n], mask, a, sampler_word(4, np.arange(B), 0, 1))
    L = pf.lib()
    xp, dp, op = xt.data_ptr(), draw.data_ptr(), frame.data_ptr() + 4 * pad
    s = torch.cuda.current_stream().cuda_stream
    for args, rc in (((None, ld, None, None, 0, dp, op, B, n, s), -1), ((xp, ld, None, None, 0, None, op, B, n, s), -1),
                     ((xp, ld, None, None, 0, dp, None, B, n, s), -1), ((xp, ld, None, None, -1, dp, op, B, n, s), -1),
                     ((xp, ld, None, None, 0, dp, op, -1, n, s), -2), ((xp, ld, None, None, 0, dp, op, B, 0, s), -2),
                     ((xp, ld, None, None, 0, dp, op, B, 257, s), -2), ((xp, n - 1, None, None, 0, dp, op, B, n, s), -2)):
        assert L.dcmp_sample(*args) == rc, args
        assert b"dcmp_sample" in L.dcmp_last_error()
    frame.fill_(SENTINEL)
    assert L.dcmp_sample(xp, ld, None, None, 0, dp, op, 0, n, s) == 0          # B = 0 writes nothing
    torch.cuda.synchronize()
    assert (frame.cpu().numpy() == SENTINEL).all()


# ---- rollouts ------------------------------------------------------------------------------------------------------------------------------
def nearness_module():
    """A stochastic stand-in for the attention network that reads only its fp32 inputs through elementwise ops: log-weights -8 (dx^2 + dy^2)
    from the task rows' columns 3-4 (the offset of each task from the acting agent).  Its rows do not depend on the batch they are in."""
    import torch

    class Nearness(torch.nn.Module):
        def forward(self, tasks, agents, mask):
            return -8.0 * (tasks[..., 3] * tasks[..., 3] + tasks[..., 4] * tasks[..., 4])

    return Nearness().cuda()


def nearness_np(tasks):
    t = np.asarray(tasks, np.float32)
    return np.float32(-8.0) * (t[..., 3] * t[..., 3] + t[..., 4] * t[..., 4])


FRACTIONS = (1.0, 0.85, 0.7, 0.5, 0.35, 0.2, 0.1, 0.03)                     # TrainerConfig.rollout_fractions


def play(protocol, B, first_gid, runner, sampler=(31, 0), horizon=600):
    from dcmrta_b200 import BatchedTaskEnv
    env = BatchedTaskEnv(B, 20, 50, M=5, auto_reset=False, seed=77, first_gid=first_gid, protocol=protocol)
    env.generate(max_duration=5.0, random_duration=True)
    ep = runner(env, horizon).run(nearness_module(), "sample", sampler=sampler)
    assert bool(ep.ended.all())
    L = int(ep.active.any(1).sum())
    out = dict(action=np.where(ep.active[:L].cpu().numpy(), ep.action[:L].cpu().numpy(), -1),
               leader=np.where(ep.active[:L].cpu().numpy(), ep.leader[:L].cpu().numpy(), -1),
               metrics=ep.metrics.cpu().numpy(), inst={k: v.cpu().numpy() for k, v in env.get_instances().items()},
               flags=env.env_flags().cpu().numpy())
    assert not (out["flags"] & ERR_BITS).any()
    env.close()
    return out


def same(a, b):
    return all(np.array_equal(a[k], b[k]) for k in ("action", "leader", "metrics"))


@pytest.mark.parametrize("protocol", ["LF", "IA"])
def test_rollout_invariance_and_oracle_replay(protocol):
    """Eager, graphed, graphed with compaction and two shards give the same sampled episodes bit for bit; stream 1 differs from 0; and the
    C oracle replays a sample of them decision by decision with the stand-in and the float64 rule on its own observations."""
    from dcmrta_b200.rollout import BatchedRollout, GraphedRollout
    B = 512
    eager = play(protocol, B, 0, lambda e, h: BatchedRollout(e, h))
    assert same(play(protocol, B, 0, lambda e, h: BatchedRollout(e, h)), eager)
    graphed = play(protocol, B, 0, lambda e, h: GraphedRollout(e, h, fractions=(1.0,)))
    assert same(graphed, eager)
    compact = play(protocol, B, 0, lambda e, h: GraphedRollout(e, h, fractions=FRACTIONS))
    assert same(compact, eager)
    lo = play(protocol, B // 2, 0, lambda e, h: BatchedRollout(e, h))
    hi = play(protocol, B // 2, B // 2, lambda e, h: GraphedRollout(e, h, fractions=FRACTIONS))
    L = max(lo["action"].shape[0], hi["action"].shape[0], eager["action"].shape[0])
    padded = lambda a: np.pad(a, ((0, L - a.shape[0]), (0, 0)), constant_values=-1)
    for k in ("action", "leader"):
        assert np.array_equal(np.concatenate([padded(lo[k]), padded(hi[k])], 1), padded(eager[k])), k
    assert np.array_equal(np.concatenate([lo["metrics"], hi["metrics"]]), eager["metrics"])
    other = play(protocol, B, 0, lambda e, h: BatchedRollout(e, h), sampler=(31, 1))
    assert not np.array_equal(other["action"][:20], eager["action"][:20])
    # the oracle replays sampled episodes
    from oracle.oracle import OracleEnv
    from ia_oracle import IAOracle
    inst, near = eager["inst"], 0
    for b in (0, 1, 100, 257, 511):
        args = (20, inst["task_xy"][b], inst["depot_xy"][b], inst["req"][b], inst["dur"][b])
        if protocol == "IA":
            o = IAOracle(*args)
        else:
            o = OracleEnv.make(*args)
            o.seed(77, gid=b, episode=0)
            o.fused_reset()
        t = 0
        while not o.done:
            ga = int(eager["action"][t, b])
            assert ga >= 0 and eager["leader"][t, b] == o.leader, (b, t)
            mask = o.mask().astype(bool)
            x = nearness_np(o.task_status(o.leader).astype(np.float32))[None]
            near += check_bounded(x, mask[None], np.array([ga]), sampler_word(31, np.array([b]), 0, t))
            if protocol == "IA":
                o.step(ga)
            else:
                assert o.fused_step(ga)[0] == 0
            t += 1
        assert t == eager["action"].shape[0] or eager["action"][t, b] == -1, (b, t)
        m, _ = o.episode_metrics()
        want = np.array([m[k] for k in METRIC_KEYS])
        got = eager["metrics"][b]
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
        for c in (0, 1, 2, 3, 5, 6, 7):
            assert got[c] == want[c], (b, METRIC_KEYS[c])
    print(f"{protocol}: oracle replay, {near} decisions in the window")


# ---- evaluation -----------------------------------------------------------------------------------------------------------------------------
def test_evaluate_sampled_does_not_depend_on_chunking():
    from dcmrta_b200.evaluate import evaluate_sampled, load_test_set
    sets = load_test_set(GOLD / "instances_20A_50T.npz")
    net = nearness_module()
    for method, chunk in (("LF", 7), ("IA", 37)):
        one = evaluate_sampled(net, sets, 6, method=method, seed=3, sample_seed=4, max_envs=300)
        assert one.shape == (50, 6, 8)
        assert np.array_equal(evaluate_sampled(net, sets, 6, method=method, seed=3, sample_seed=4, max_envs=chunk), one), method
        assert np.array_equal(evaluate_sampled(net, sets, 6, method=method, seed=3, sample_seed=4, max_envs=128, graphed=True), one)
        assert (one[:, :, 0] != one[:, :1, 0]).any()                          # the K samples differ


def test_k1_with_a_greedy_only_stand_in_equals_greedy_evaluate():
    """Non-greedy entries 1e4 below the greedy one have weight exactly 0: K = 1 is the greedy run, bit for bit, under LF (same seed,
    env i = global id i) and IA."""
    import torch
    from dcmrta_b200.evaluate import evaluate, evaluate_sampled, load_test_set

    class GreedyOnly(torch.nn.Module):
        def forward(self, tasks, agents, mask):
            d2 = tasks[..., 3] * tasks[..., 3] + tasks[..., 4] * tasks[..., 4]
            score = (-d2).masked_fill(mask, float("-inf"))
            best = torch.nn.functional.one_hot(score.argmax(1), score.shape[1]).bool()
            return torch.where(best, 0.0, -1e4)

    sets = load_test_set(GOLD / "instances_20A_50T.npz")
    net = GreedyOnly().cuda()
    for method in ("LF", "IA"):
        greedy = evaluate(net, sets, method=method, seed=17)
        sampled = evaluate_sampled(net, sets, 1, method=method, seed=17, sample_seed=123)
        assert np.array_equal(sampled[:, 0], greedy), method


def test_evaluate_cli_samples(tmp_path, capsys):
    import pandas as pd
    import torch
    from dcmrta_b200.evaluate import best_of, evaluate_sampled, load_net, load_test_set, main
    from dcmrta_b200.policy import AttentionNet
    torch.manual_seed(0)
    ck = tmp_path / "ck.pth"
    torch.save({"model": AttentionNet(6, 5, 128).state_dict()}, ck)
    test_set = str(GOLD / "instances_20A_50T.npz")
    out, npz = tmp_path / "best.csv", tmp_path / "all.npz"
    assert main(["--checkpoint", str(ck), "--test-set", test_set, "--method", "LF", "--amp", "fused", "--samples", "3", "--sample-seed", "8",
                 "--max-envs", "64", "--out", str(out), "--samples-out", str(npz)]) == 0
    printed = capsys.readouterr().out
    assert "best of 3" in printed and "all samples" in printed
    z = np.load(npz)
    assert z["metrics"].shape == (50, 3, 8)
    want = evaluate_sampled(load_net(ck), load_test_set(test_set), 3, method="LF", amp="fused", sample_seed=8, max_envs=64)
    assert np.array_equal(z["metrics"], want)
    best, k = best_of(want)
    assert np.array_equal(z["best_k"], k)
    df = pd.read_csv(out, index_col=0)
    np.testing.assert_allclose(df.to_numpy(), best[:, 1:7], rtol=1e-12, atol=0)


@pytest.mark.parametrize("amp", ["fused", False, True])
def test_attention_net_samples_legal_actions(amp):
    """A real AttentionNet (fused forward, fp32 module, bf16 copy), K = 8 on the bundled set: every sampled action is legal."""
    import torch
    from dcmrta_b200 import BatchedTaskEnv
    from dcmrta_b200.evaluate import evaluate_sampled, load_test_set
    from dcmrta_b200.policy import AttentionNet
    from dcmrta_b200.rollout import BatchedRollout
    torch.manual_seed(1)
    net = AttentionNet(6, 5, 128).cuda().eval()
    sets = load_test_set(GOLD / "instances_20A_50T.npz")
    K = 8
    inst = np.arange(50 * K) // K
    env = BatchedTaskEnv(50 * K, 20, 50, M=5, auto_reset=False, max_wait=10.0, max_time=100.0, seed=0, first_gid=0, protocol="LF")
    env.load_instances(sets["task_xy"][inst], sets["depot_xy"][inst], sets["req"][inst], sets["dur"][inst])
    ep = BatchedRollout(env, 560).run(net, "sample", amp=amp, sampler=(2, 0))
    assert bool(ep.ended.all())
    assert not (env.env_flags().cpu().numpy() & ERR_BITS).any()
    act, mask, active = ep.action.long(), ep.mask, ep.active
    chosen = mask.gather(2, act.unsqueeze(2)).squeeze(2)
    assert int(chosen[active].sum()) == 0 and int(active.sum()) > 50 * K * 50
    table = evaluate_sampled(net, sets, K, amp=amp, sample_seed=2, max_envs=50 * K)
    assert np.array_equal(table.reshape(-1, 8), ep.metrics.cpu().numpy())
    env.close()
