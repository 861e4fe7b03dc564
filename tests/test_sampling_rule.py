"""CPU tests of the policy's action-sampling contract (DESIGN.md 5, include/dcmrta_sample.h dcmp_sample): a vectorised NumPy Philox4x32-10
pinned to the oracle's, the sampling rule restated in float64, and the counter region of the sampler against the env's.  The reference code
here is what tests/test_gpu_sampling.py holds the kernel to."""
import math
import re
from pathlib import Path

import numpy as np
import pytest

M32 = np.uint64(0xFFFFFFFF)
SAMPLER_C3 = 0xC0000000              # + decision
MAX_DECISION = 2 ** 30 - 2           # decision < 2^30 - 1: c3 stays below the generator's depot counter 0xFFFFFFFF


def philox_np(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on broadcast uint32 arrays (uint64 arithmetic: a 32 x 32-bit product fits) -> four uint32 arrays."""
    c0, c1, c2, c3, k0, k1 = (np.asarray(v, np.uint64) & M32 for v in np.broadcast_arrays(c0, c1, c2, c3, k0, k1))
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return tuple(c.astype(np.uint32) for c in (c0, c1, c2, c3))


def sampler_word(seed, gid, stream, decision):
    """x0 of the sampler's draw: counter (gid_lo, gid_hi, stream, 0xC0000000 + decision), key (seed_lo, seed_hi)."""
    gid = np.asarray(gid, np.uint64)
    decision = np.asarray(decision, np.uint64)
    return philox_np(gid & M32, gid >> np.uint64(32), stream, np.uint64(SAMPLER_C3) + decision, seed & 0xFFFFFFFF, seed >> 32)[0]


def rule64(x, mask, x0):
    """The sampling rule in float64 on rows x [B, n] (fp32 values), mask [B, n] bool (True = forbidden) or None, x0 [B] uint32.
    -> (action [B], C [B, n] prefix sums, S [B], theta [B], w [B, n]).  Exact where the weights are exactly representable (all ones)."""
    x = np.asarray(x, np.float32).astype(np.float64)
    allowed = np.ones(x.shape, bool) if mask is None else ~np.asarray(mask, bool)
    xa = np.where(allowed, x, -np.inf)
    m = xa.max(1, keepdims=True)
    with np.errstate(invalid="ignore", over="ignore"):
        w = np.where(allowed & (xa > -np.inf), np.exp(xa - np.where(np.isfinite(m), m, 0.0)), 0.0)
    C = np.cumsum(w, 1)
    S = C[:, -1]
    theta = (np.asarray(x0, np.uint64) >> np.uint64(8)).astype(np.float64) * S * 2.0 ** -24
    hit = (w > 0) & (C > theta[:, None])
    action = np.where(hit.any(1), hit.argmax(1), 0).astype(np.int32)
    return action, C, S, theta, w


def kth_allowed(live, x0):
    """All-ones weights on the entries `live` [B, n] bool: allowed index number floor(u S), u = (x0 >> 8) 2^-24, in integer arithmetic."""
    S = live.sum(1).astype(np.uint64)
    k = ((np.asarray(x0, np.uint64) >> np.uint64(8)) * S) >> np.uint64(24)
    out = np.zeros(live.shape[0], np.int32)
    for b in np.flatnonzero(S):
        out[b] = np.flatnonzero(live[b])[int(k[b])]
    return out


def test_philox_np_matches_oracle_on_kat_and_sampler_counters():
    from oracle.oracle import philox
    kat = [([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
           ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
           ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0], [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]
    for c, k, want in kat:
        assert [int(v) for v in philox_np(*c, *k)] == want
        assert philox(c, k).tolist() == want
    rng = np.random.default_rng(1)
    n = 3000
    seed = rng.integers(0, 2 ** 63, n, dtype=np.uint64)
    gid = rng.integers(0, 2 ** 40, n, dtype=np.uint64)
    stream = rng.integers(0, 2 ** 32, n, dtype=np.uint64)
    dec = rng.integers(0, MAX_DECISION + 1, n, dtype=np.uint64)
    dec[:2] = 0, MAX_DECISION
    got = philox_np(gid & M32, gid >> np.uint64(32), stream, np.uint64(SAMPLER_C3) + dec, seed & M32, seed >> np.uint64(32))
    for i in range(n):
        ctr = [int(gid[i]) & 0xFFFFFFFF, int(gid[i]) >> 32, int(stream[i]), SAMPLER_C3 + int(dec[i])]
        key = [int(seed[i]) & 0xFFFFFFFF, int(seed[i]) >> 32]
        assert philox(ctr, key).tolist() == [int(g[i]) for g in got], i
    assert np.array_equal(sampler_word(int(seed[5]), gid[:10], int(stream[5]), dec[5]),
                          philox_np(gid[:10] & M32, gid[:10] >> np.uint64(32), stream[5], SAMPLER_C3 + int(dec[5]),
                                    int(seed[5]) & 0xFFFFFFFF, int(seed[5]) >> 32)[0])


def test_all_ones_weights_pick_allowed_index_floor_u_s():
    rng = np.random.default_rng(2)
    for n in (1, 2, 31, 32, 33, 51, 64, 65, 255, 256):
        B = 2000
        mask = rng.random((B, n)) < rng.random((B, 1))
        mask[:3] = False
        mask[3] = True                                                       # no allowed entry: action 0
        x = np.repeat(rng.normal(size=(B, 1)).astype(np.float32), n, 1)      # a constant per row: every weight is exactly 1
        x0 = sampler_word(7, np.arange(B), 0, n)
        a, *_ = rule64(x, mask, x0)
        assert np.array_equal(a, kth_allowed(~mask, x0)), n
        assert a[3] == 0


def test_rule_never_picks_zero_weight_entries():
    rng = np.random.default_rng(3)
    B, n = 3000, 51
    x = rng.normal(0, 3, (B, n)).astype(np.float32)
    gap = rng.random((B, n)) < 0.3
    x[gap] = np.float32(-1e4)                                                # the fused forward's fill: exp underflows to exactly 0
    x[rng.random((B, n)) < 0.1] = -np.inf
    x[:, 0] = 1.0                                                            # at least one live entry per row
    mask = rng.random((B, n)) < 0.3
    mask[:, 0] = False
    a, _, _, _, w = rule64(x, mask, sampler_word(11, np.arange(B), 2, 9))
    assert (w[np.arange(B), a] > 0).all() and not mask[np.arange(B), a].any() and np.isfinite(x[np.arange(B), a]).all()
    assert (x[np.arange(B), a] > -1e3).all()


def test_rule_distribution_chi_square():
    """2^18 draws of one masked row over gids and decisions; the statistic is deterministic, so one fixed threshold."""
    from scipy.stats import chi2
    rng = np.random.default_rng(4)
    n = 51
    row = rng.normal(0, 1.5, n).astype(np.float32)
    mask = rng.random(n) < 0.25
    mask[0] = False
    gid, dec = np.meshgrid(np.arange(4096, dtype=np.uint64), np.arange(64, dtype=np.uint64))
    x0 = sampler_word(1234, gid.ravel(), 0, dec.ravel())
    N = x0.size
    a, _, _, _, w = rule64(np.broadcast_to(row, (N, n)), np.broadcast_to(mask, (N, n)), x0)
    p = w[0] / w[0].sum()
    live = p > 0
    counts = np.bincount(a, minlength=n)
    assert counts[~live].sum() == 0
    stat = float((((counts - N * p) ** 2)[live] / (N * p[live])).sum())
    assert stat < chi2.ppf(1 - 1e-6, int(live.sum()) - 1), stat


def test_sampler_counter_region_is_disjoint_from_the_env():
    """env decisions: c3 = decision * 8 + block < 2^31; instance generator: 0x80000000 + 2 j + b (j < 254) and 0xFFFFFFFF; the sampler
    0xC0000000 + decision for decision < 2^30 - 1.  Disjoint intervals, so the two may share a seed without sharing a draw."""
    env_decisions = (0, 2 ** 31 - 1)
    generator = (0x80000000, 0x80000000 + 2 * 253 + 1)
    sampler = (SAMPLER_C3, SAMPLER_C3 + MAX_DECISION)
    regions = sorted([env_decisions, generator, sampler, (0xFFFFFFFF, 0xFFFFFFFF)])
    for (a0, a1), (b0, b1) in zip(regions, regions[1:]):
        assert a1 < b0, (hex(a1), hex(b0))
    assert sampler[1] == 0xFFFFFFFE
    from dcmrta_b200.policy_fused import draw_tensor
    with pytest.raises(ValueError):
        draw_tensor(0, 0, MAX_DECISION + 1)
    d = draw_tensor(2 ** 64 - 1, 2 ** 32 - 1, MAX_DECISION)                  # u32 words in int32 storage
    assert (d.numpy().view(np.uint32) == [0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, MAX_DECISION]).all()


def test_best_of_takes_highest_reward_lowest_k_on_ties():
    from dcmrta_b200.evaluate import best_of
    rng = np.random.default_rng(5)
    N, K = 40, 9
    m = rng.normal(size=(N, K, 8))
    m[:, :, 0] = np.round(m[:, :, 0], 1)                                      # many ties
    m[0, :, 0] = -3.0                                                         # all tied: k = 0
    best, k = best_of(m)
    for i in range(N):
        r = m[i, :, 0]
        want = min(j for j in range(K) if r[j] == r.max())
        assert k[i] == want and np.array_equal(best[i], m[i, want])
    assert k[0] == 0 and math.isclose(best[0, 0], -3.0)


def test_sample_header_symbols_are_exported_and_bound():
    """include/dcmrta_sample.h: libdcmrta_policy.so exports what it declares and policy_fused binds exactly that."""
    from dcmrta_b200 import policy_fused as pf
    text = re.sub(r"/\*.*?\*/", "", (Path(__file__).resolve().parent.parent / "include" / "dcmrta_sample.h").read_text(), flags=re.S)
    names = sorted(set(re.findall(r"\b(dcmp_[a-z0-9_]+)\s*\(", text)))
    assert names == ["dcmp_sample"]
    L = pf.lib()
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/dcmrta_sample.h but not exported"
    assert sorted(pf.SAMPLE_SIGNATURES) == names
    assert L.dcmp_sample.argtypes is not None
