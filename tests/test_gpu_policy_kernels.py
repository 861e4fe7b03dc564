"""The six kernels of libdcmrta_policy.so (csrc/policy_kernels.cu) against a float64 reference of the same operation on the kernel's
own bf16 inputs (`TorchOps(acc=torch.float64)`).

(a) Constructed cases, compared bit for bit: inputs for which every approximate instruction returns an exact value, so that the
    kernel's output is known exactly.  One launch reaches every key, head and query row, or every column, of its kernel.
(b) Bounded cases over the shapes where the kernels change code path and the value regimes where they can lose accuracy:
    |out - ref64| <= a per-element bound derived from the kernel's arithmetic (the docstrings of the `*_check` functions below, term by term).  For embed, gate and
    add_layernorm, which round one fp32 value to bf16, also the rounding direction.
(c) Guard memory: every input and output sits inside a larger buffer.  Inputs are surrounded by NaN (a read of it reaches an output),
    outputs by a sentinel bit pattern that must survive unchanged.
(d) Every kernel call of a real forward, on observations the env wrote, through `CheckedOps` (a CudaOps that checks each call
    against the float64 reference with the bounds of (b)).

The largest error/bound ratio of each kernel is printed at the end of the module (pytest -s)."""
import math
from collections import defaultdict

import pytest
import torch

from helpers import EnvelopeShape, envelope_shape

pytestmark = pytest.mark.gpu

E, H, D, HID = 128, 8, 16, 512
SCALE = 1.0 / math.sqrt(D)
U32 = 2.0 ** -24                       # fp32 unit roundoff (round to nearest)
U16 = 2.0 ** -8                        # bf16 unit roundoff: the relative error of rounding to the nearest bf16
TINY = 2.0 ** -126                     # smallest normal fp32: ex2.approx.ftz flushes below it, __fdividef returns 0 above its inverse
SENT16, SENT32 = 0x7FA5, 0x7FA5A5A5    # NaN payloads no kernel writes
RATIOS = defaultdict(float)            # kernel -> largest observed |out - ref64| / bound


@pytest.fixture(scope="module", autouse=True)
def report_margins():
    yield
    if RATIOS:
        print("\nlargest |out - ref64| / bound per kernel: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(RATIOS.items())))


def _ops():
    from dcmrta_b200.policy_fused import CudaOps, TorchOps
    return CudaOps(), TorchOps(acc=torch.float64)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _bf(*shape, seed, scale=1.0):
    return (torch.randn(*shape, generator=_gen(seed), device="cuda") * scale).to(torch.bfloat16)


# ---- (c) framed buffers -----------------------------------------------------------------------------------------------------------
class Frame:
    """A [rows, cols] view inside a larger buffer: `lead` / `trail` rows and `left` / `right` columns around it (multiples of 16 bytes,
    so the view keeps the kernels' alignment).  Inputs are framed by NaN, outputs by a sentinel bit pattern; `outside_unchanged`
    checks that nothing outside the view was written."""

    def __init__(self, rows, cols, dtype, fill, lead=3, trail=5, left=0, right=0):
        n = lead + rows + trail
        ld = left + cols + right
        if fill == "nan":
            self.buf = torch.full((n, ld), float("nan"), dtype=dtype, device="cuda")
        else:                                                                 # sentinel bits
            it = torch.int16 if dtype.itemsize == 2 else torch.int32
            self.buf = torch.full((n, ld), SENT16 if it == torch.int16 else SENT32, dtype=it, device="cuda").view(dtype)
        self.view = self.buf[lead:lead + rows, left:left + cols]
        self.inside = torch.zeros(n, ld, dtype=torch.bool, device="cuda")
        self.inside[lead:lead + rows, left:left + cols] = True
        self.before = None

    def arm(self):
        self.before = self.buf.clone()
        return self.view

    def outside_unchanged(self, what):
        it = torch.int16 if self.buf.dtype.itemsize == 2 else torch.int32
        a, b = self.buf.view(it)[~self.inside], self.before.view(it)[~self.inside]
        assert torch.equal(a, b), f"{what}: {int((a != b).sum())} elements outside the output were written"


def framed_input(t, left=0, right=0):
    """a copy of t inside a NaN frame"""
    f = Frame(t.shape[0], t.shape[1], t.dtype, "nan", left=left, right=right)
    f.view.copy_(t)
    return f.view


def framed_output(rows, cols, dtype, left=0, right=0):
    return Frame(rows, cols, dtype, "sentinel", left=left, right=right)


def bits(t):
    return t.contiguous().view(torch.int16 if t.dtype.itemsize == 2 else torch.int32)


# ---- (b) bounds, each term derived from the kernel's arithmetic ---------------------------------------------------------------------
def record(kernel, err, bound, what):
    if what.startswith("forward"):
        kernel += " (forward)"
    ratio = err / bound
    worst = float(ratio.max()) if ratio.numel() else 0.0
    RATIOS[kernel] = max(RATIOS[kernel], worst)
    if not bool((err <= bound).all()):                                        # (NaN fails too)
        i = int(torch.nan_to_num(ratio, nan=float("inf")).flatten().argmax())
        raise AssertionError(f"{kernel} {what}: error {float(err.flatten()[i]):.4g} > bound {float(bound.flatten()[i]):.4g} "
                             f"(error/bound {worst:.4g}; {int((~(err <= bound)).sum())} of {err.numel()} elements)")


def check_rounded(kernel, out, ref, e, what, min_exact=0.95):
    """out = bf16_rn(v) for an fp32 value v with |v - ref| <= e.  Rounding to nearest is monotone, so
    bf16_rn(ref - e) <= out <= bf16_rn(ref + e): where no rounding midpoint lies within e of ref this pins out to bf16_rn(ref), and a
    kernel that truncates (or rounds the wrong way) fails it on about half the elements.  Of the elements whose fp32 error is below
    2^-10 of their magnitude, at least `min_exact` must be bf16_rn(ref64) itself (a truncating kernel gives about half).  The error
    bound follows: one bf16 rounding of |v| <= |ref| + e, plus e.  (A double's conversion to bf16 goes through fp32 in torch; that keeps the sandwich valid, because v
    is itself an fp32 value inside [ref - e, ref + e].)"""
    o = out.double()
    record(kernel, (o - ref).abs(), U16 * ref.abs() + (1 + U16) * e + TINY, what)
    lo, hi = (ref - e).to(torch.bfloat16).double(), (ref + e).to(torch.bfloat16).double()
    bad = ~((lo <= o) & (o <= hi))
    assert not bool(bad.any()), f"{kernel} {what}: {int(bad.sum())} elements are not the nearest bf16 of a value within the fp32 error"
    pinned = e < 2.0 ** -10 * ref.abs()
    exact = float((out == ref.to(torch.bfloat16))[pinned].double().mean()) if bool(pinned.any()) else 1.0
    assert exact >= min_exact, f"{kernel} {what}: only {exact:.4f} of the elements are bf16_rn(ref64)"


def embed_check(x, w, b, out, what, th=None):
    """y = b + sum_k x_k w_k as a chain of k_in fmas in fp32, then one rounding to bf16.  Each fma rounds once, at most 2^-24 of a
    partial sum, and every partial sum is at most |b| + sum_k |x_k w_k|: e = (k_in + 1) 2^-24 (|b| + sum |x w|), one spare term."""
    th = th or _ops()[1]
    ref = th.embed(x, w, b, torch.empty(out.shape, dtype=torch.float64, device="cuda"))
    S = x.double().abs() @ w.double().abs().t() + b.double().abs()
    check_rounded("embed", out, ref, (x.shape[1] + 1) * U32 * S, what)


def gate_check(wv, out, what, th=None):
    """y = __fdividef(b, 1 + __expf(-a)), a = wv[:, :512], b = wv[:, 512:], in fp32, then one rounding to bf16.  Relative error of the
    fp32 value, term by term:
      __expf(-a): 2 + floor(1.173 |a|) ulp (CUDA C Programming Guide, intrinsic functions; includes the product -a log2(e) that feeds
                  ex2.approx), one ulp <= 2^-23 relative; it enters 1 + t scaled by t / (1 + t) <= 1;
      1 + t:      2^-24;        __fdividef: 2 ulp = 2^-22 for denominators up to 2^126;
      so e_rel = (2 + 1.2 |a|) 2^-23 + 2^-24 + 2^-22 <= (5 + 1.2 |a|) 2^-23.
    Floor: for a < -87.3 the denominator exceeds 2^126 and __fdividef returns 0 (or __expf overflows and the quotient is 0); the true
    value is below |b| 2^-126 there, hence + |b| 2^-125."""
    th = th or _ops()[1]
    ref = th.gate(wv, torch.empty(out.shape, dtype=torch.float64, device="cuda"))
    a, b = wv[:, :HID].double(), wv[:, HID:].double()
    e = (5 + 1.2 * a.abs()) * 2.0 ** -23 * ref.abs() + b.abs() * 2.0 ** -125
    check_rounded("gate", out, ref, e, what)


def layernorm_check(x, res, g, beta, out, eps, what, th=None):
    """k_add_layernorm, warp per row, lane <-> 4 columns, all in fp32:
      s_i = x_i + res_i                 rounds at most 2^-24 |s_i| (bf16 + bf16);
      mean = tree sum of 128 / 128      7 levels (2 in the lane, 5 shuffles) + the rounding of s: |dm| <= e_m = 8 2^-24 mean|s|;
      d_i = s_i - mean                  |d_i - d64_i| <= e_d_i = e_m + 2^-24 (|s_i| + |d_i|);
      var = tree sum of d^2 / 128       a two-pass variance around a mean that is off by dm is var + dm^2, and perturbing every d_i by
                                        e_d moves it by <= 2 sqrt(var) max e_d + max e_d^2 (sum_i d_i = 0 removes the linear term
                                        of dm); the squares and the 7-level sum add 9 2^-24 var:
                                        e_v = 2 sqrt(var) max e_d + max e_d^2 + 10 2^-24 var;
      rstd = rsqrtf(var + eps)          relative e_r = e_v / (2 (var + eps)) + 2^-24 (the + eps) + 2^-22 (rsqrtf, 2 ulp);
      y = fma(d rstd, g, beta)          |g| (rstd e_d_i + |n_i| e_r) for the normalised value n = d rstd, and two roundings
                                        (d rstd, the fma): 2 2^-24 (|g n| + |beta|).
    The value regimes that break a one-pass variance (E[s^2] - mean^2) or a dropped eps land far outside this bound."""
    th = th or _ops()[1]
    ref = th.add_layernorm(x, res, g, beta, torch.empty(out.shape, dtype=torch.float64, device="cuda"), eps)
    s = x.double() + res.double()
    mean = s.mean(1, keepdim=True)
    d = s - mean
    var = (d * d).mean(1, keepdim=True)
    rstd = (var + eps).rsqrt()
    n = d * rstd
    e_m = 8 * U32 * s.abs().mean(1, keepdim=True)
    e_d = e_m + U32 * (s.abs() + d.abs())
    e_dmax = e_d.amax(1, keepdim=True)
    e_v = 2 * var.sqrt() * e_dmax + e_dmax * e_dmax + 10 * U32 * var
    e_r = e_v / (2 * (var + eps)) + U32 + 2.0 ** -22
    gd, bd = g.double(), beta.double()
    e = gd.abs() * (rstd * e_d + n.abs() * e_r) + 2 * U32 * ((gd * n).abs() + bd.abs())
    check_rounded("add_layernorm", out, ref, e, what)


def _attention_ref(q, k, v, mask, B, nq, nk):
    """float64 softmax(scale q k^T) v per (env, head, query row) with the quantities the bounds need: the reference output, A = sum_j
    w_j |v_j| (w the softmax weights), max_j sum_d |q_d k_jd| and max_j |s_j| (raw scores).  Masked keys carry weight 0."""
    hq = q.double().reshape(B, nq, H, D).transpose(1, 2)                     # [B,H,nq,D]
    hk = k.double().reshape(B, nk, H, D).transpose(1, 2)
    hv = v.double().reshape(B, nk, H, D).transpose(1, 2)
    if mask is not None:                                                      # masked rows may hold NaN (they must not be read)
        keep = ~mask.bool().view(B, 1, nk, 1)
        hk, hv = torch.where(keep, hk, 0.0), torch.where(keep, hv, 0.0)
    s = hq @ hk.transpose(2, 3)                                               # raw scores [B,H,nq,nk]
    a = hq.abs() @ hk.abs().transpose(2, 3)
    z = s * SCALE
    if mask is not None:
        z = z.masked_fill(mask.bool().view(B, 1, 1, nk), float("-inf"))
        s = s.masked_fill(mask.bool().view(B, 1, 1, nk), 0.0)
        a = a.masked_fill(mask.bool().view(B, 1, 1, nk), 0.0)
    w = torch.softmax(z, -1).nan_to_num(0.0)                                  # a query whose every key is masked: zeros
    ref, A = w @ hv, w @ hv.abs()
    flat = lambda t: t.transpose(1, 2).reshape(B * nq, E)
    return flat(ref), flat(A), flat(a.amax(-1, keepdim=True).expand(B, H, nq, D)), flat(s.abs().amax(-1, keepdim=True).expand(B, H, nq, D))


def attention_check(q, k, v, out, B, nq, nk, what):
    """k_attention_mma: raw scores S = Q K^T on the tensor cores (fp32 accumulation), online softmax over blocks of 64 keys with
    p = ex2(s c - m), c = scale log2(e) in fp32, P rounded to bf16 for O += P V, l summed from the unrounded p, out = bf16(O / l).
    With w_j the float64 softmax weights, A = sum_j w_j |v_j| and nb = ceil(nk / 64) blocks:
      the relative error eps of each weight, in natural-log units of the exponent:
        score:      the MMA sums 16 exact bf16 products in fp32: |ds| <= 16 ulp = 2^-20 sum_d |q_d k_d|, times scale;
        exponent:   the fma s c - m rounds once (2^-24 |t|, |t| <= 2 c max|s|) and c is fp32 (2^-24 c |s_j - s_max|); ln 2 log2(e) = 1,
                    so each is 2^-23 scale max|s| at most; the rescale ex2(m_old - m_new) of every later block adds one more:
                    (nb + 2) 2^-22 scale max|s| in all;
        ex2.approx: 2 ulp = 2^-22 relative, once per weight and once per rescale: (nb + 1) 2^-21 with margin;
      a relative error eps in every weight moves the normalised weights by <= 2 eps w_j (numerator and denominator): 3 eps A;
      P to bf16:    the numerator uses bf16(p_j) = p_j (1 + d_j), |d_j| <= 2^-8, the denominator the fp32 p: 2^-8 A;
      accumulation: O over ceil(nk / 16) MMA steps and nb rescales, 2^-22 each; l over nk / 4 additions in a lane and 2 shuffles,
                    2^-24 each; 1 / l and the product: 3 2^-24: ((nk / 16 + nb + 4) 2^-22 + (nk / 4 + 6) 2^-24) A;
      output:       one rounding to bf16, 2^-8 |ref| (of the fp32 value, so times 1 + 2^-8 for the terms above);
      floor:        weights below 2^-126 of the maximum flush to zero: nk 2^-126 max|v|, plus 2^-126."""
    ref, A, amax, smax = _attention_ref(q, k, v, None, B, nq, nk)
    nb = -(-nk // 64)
    eps = SCALE * (2.0 ** -20 * amax + (nb + 2) * 2.0 ** -22 * smax) + (nb + 1) * 2.0 ** -21
    acc = ((nk / 16 + nb + 4) * 2.0 ** -22 + (nk / 4 + 6) * U32) * A
    floor = nk * TINY * float(v.double().abs().max()) + TINY
    bound = U16 * ref.abs() + (1 + U16) * (3 * eps * A + U16 * A + acc) + floor
    record("attention", (out.double() - ref).abs(), bound, what)


def attention_q1_check(q, k, v, mask, out, B, nk, what):
    """k_attention_q1: lane per key, q pre-scaled by c = scale log2(e) in fp32, scores by 16 fmas, p = ex2(s - m) in fp32 (no bf16 P),
    per-lane sums over 8 keys and 5 shuffles, out = bf16(acc / l).  As for k_attention_mma, without the bf16 rounding of P and the
    block rescale:
      score:        16 q_d c roundings and 16 fmas: 17 2^-24 <= 2^-19 of c sum_d |q_d k_d|, so 2^-19 scale sum|q k| in natural-log units;
      exponent:     s - m rounds once (2^-24 |s - m| <= 2^-23 c max|s|) and c is fp32: 2 2^-22 scale max|s|;
      ex2.approx:   2^-21 with margin;
      weights:      3 eps A;   accumulation: (8 + 5 + 3) 2^-24 A for acc, l, 1 / l and the product;
      output:       2^-8 |ref|;   floor: nk 2^-126 max|v| + 2^-126.
    Masked keys carry weight 0 (their K and V rows may hold anything: the kernel must not read them); a query whose every key is
    masked gives exactly 0."""
    ref, A, amax, smax = _attention_ref(q, k, v, mask, B, 1, nk)
    eps = SCALE * (2.0 ** -19 * amax + 2 * 2.0 ** -22 * smax) + 2.0 ** -21
    vmax = float(torch.nan_to_num(v.double(), nan=0.0).abs().max())
    bound = U16 * ref.abs() + (1 + U16) * (3 * eps * A + 16 * U32 * A) + nk * TINY * vmax + TINY
    record("attention_q1", (out.double() - ref).abs(), bound, what)
    if mask is not None:
        none = mask.bool().all(1)
        assert bool((bits(out[none]) == 0).all()), f"attention_q1 {what}: a query with every key masked must give +0"


def pointer_check(qk, feat, mask, out, B, n, norm, clip, what):
    """k_pointer, warp per env, fp32: dot = sum_e qk_e f_e (4 fmas per lane, 5 shuffle levels), u = clip tanhf(norm dot), masked
    u = -1e4, m = max u, l = sum expf(u - m) (8 per lane, 5 shuffles), logp = (u - m) - logf(l).  Term by term:
      e_u (unmasked)  dot: 9 roundings of partial sums <= 10 2^-24 sum|qk f|; norm in fp32 and norm dot: 2 2^-24 |norm dot|; tanh has
                      slope <= 1; tanhf 2 ulp (2^-22) and clip * (2^-24), both relative to a value <= 1: 2^-21 with margin;
                      e_u = clip (norm (10 2^-24 sum|qk f| + 2^-23 |dot|) + 2^-21); 0 for masked entries (-1e4 is exact);
      logsumexp       logp is invariant to the shift m, so u errors enter as e_u_j directly and through log l as at most
                      E_u = max e_u (the weights of log-sum-exp sum to 1); the subtraction u - m rounds 2^-24 |u - m|, weighted by
                      the softmax weights inside log l; expf 2 ulp (2^-22), 13 additions (13 2^-24), logf 1 ulp (2^-23 log l);
      output          the last subtraction rounds 2^-24 |logp|.
    Entries at -1e4 carry fp32 rounding at that magnitude (2^-24 1e4 = 6e-4 per rounding): the 2^-24 |u - m| and 2^-24 |logp| terms,
    a relative bound.  Floor: expf terms below 2^-126 of l may be lost: n 2^-126."""
    th = _ops()[1]
    ref = th.pointer(qk, feat, mask, torch.empty(B, n, dtype=torch.float64, device="cuda"), B, n, norm, clip)
    dot = torch.einsum("be,bne->bn", qk.double(), feat.double().view(B, n, E))
    adot = torch.einsum("be,bne->bn", qk.double().abs(), feat.double().abs().view(B, n, E))
    u = clip * torch.tanh(norm * dot)
    e_u = clip * (norm * (10 * U32 * adot + 2.0 ** -23 * dot.abs()) + 2.0 ** -21)
    if mask is not None:
        u = u.masked_fill(mask.bool(), -1e4)
        e_u = e_u.masked_fill(mask.bool(), 0.0)
    m = u.amax(1, keepdim=True)
    w = torch.softmax(u, 1)
    logl = torch.logsumexp(u - m, 1, keepdim=True)
    bound = (e_u + 2 * e_u.amax(1, keepdim=True) + U32 * ((u - m).abs() + ref.abs() + (w * (u - m).abs()).sum(1, keepdim=True))
             + 2.0 ** -23 * logl + 2.0 ** -22 + 13 * U32 + n * TINY)
    record("pointer", (out.double() - ref).abs(), bound, what)


# ---- (d) every call of a real forward ----------------------------------------------------------------------------------------------
def _checked_ops():
    from dcmrta_b200.policy_fused import CudaOps

    class CheckedOps(CudaOps):
        """CudaOps that checks each kernel call against the float64 reference on the same bf16 inputs, with the bounds of (b).  Inputs
        are copied first: an output may alias one of them."""
        calls = defaultdict(int)

        def embed(self, x, w, b, out):
            x, w, b = x.clone(), w.clone(), b.clone()
            super().embed(x, w, b, out)
            embed_check(x, w, b, out, f"forward call {self.calls['embed']}")
            self.calls["embed"] += 1
            return out

        def attention(self, q, k, v, out, B, nq, nk):
            super().attention(q, k, v, out, B, nq, nk)
            attention_check(q, k, v, out, B, nq, nk, f"forward call {self.calls['attention']} ({B}x{nq}x{nk})")
            self.calls["attention"] += 1
            return out

        def attention_q1(self, q, k, v, mask, out, B, nk):
            super().attention_q1(q, k, v, mask, out, B, nk)
            attention_q1_check(q, k, v, mask, out, B, nk, f"forward call {self.calls['attention_q1']} ({B}x{nk})")
            self.calls["attention_q1"] += 1
            return out

        def add_layernorm(self, x, res, gamma, beta, out, eps):
            x, res = x.clone(), res.clone()
            super().add_layernorm(x, res, gamma, beta, out, eps)
            layernorm_check(x, res, gamma, beta, out, eps, f"forward call {self.calls['add_layernorm']}")
            self.calls["add_layernorm"] += 1
            return out

        def gate(self, wv, out):
            super().gate(wv, out)
            gate_check(wv, out, f"forward call {self.calls['gate']}")
            self.calls["gate"] += 1
            return out

        def pointer(self, qk, feat, mask, out, B, n, norm, clip):
            super().pointer(qk, feat, mask, out, B, n, norm, clip)
            pointer_check(qk, feat, mask, out, B, n, norm, clip, f"forward call {self.calls['pointer']}")
            self.calls["pointer"] += 1
            return out

    return CheckedOps()


def _peaked(net, gain=3.0):
    """the network with every attention's query and key projections scaled by `gain` (scores by gain^2) and the pointer's too: peaked
    attention, as a trained network's is"""
    with torch.no_grad():
        for name, p in net.named_parameters():
            if name.endswith("w_query") or name.endswith("w_key"):
                p.mul_(gain)
    return net


@pytest.mark.parametrize("peaked", [False, True], ids=["init", "peaked"])
@pytest.mark.parametrize("name", ["1A_1T_1M_B33_random", "20A_50T", "64A_254T_8M_B100_random"])
def test_every_kernel_call_of_a_forward(name, peaked):
    from dcmrta_b200.policy_fused import FusedPolicy
    from gpu_env import make_env
    from test_policy_fused import _net
    shape = EnvelopeShape(20, 50, 5, 64, "random", 0, None, "", []) if name == "20A_50T" else envelope_shape(name)
    env = make_env(shape)
    env.reset()
    for _ in range(30):
        env.step(policy=shape.policy)
    net = _net().cuda()
    if peaked:
        _peaked(net)
    fused = FusedPolicy(net)
    fused.ops = _checked_ops()
    out = fused(env.task_obs, env.agent_obs, env.mask_u8.view(torch.bool))
    assert out.shape == (shape.B, shape.T + 1) and bool(torch.isfinite(out).all())
    layers = [n for n, _ in fused.names]
    one_query = sum(n.startswith("globalDecoder") for n in layers)          # the global decoders attend with one query
    assert dict(fused.ops.calls) == {"embed": 3, "attention": len(layers) - one_query, "attention_q1": one_query,
                                     "add_layernorm": 2 * len(layers), "gate": len(layers), "pointer": 1}
    env.close()


# ---- (a) attention: one-hot routing, bit for bit ---------------------------------------------------------------------------------------
def one_hot_attention(B, nq, nk, seed, two_hot=False):
    """q, k, v [B * n, 128] (bf16) whose softmax is exactly one-hot.  Query row r of (env b, head h) is 32 sigma e_d with
    d = (r + r // 16 + 3 h) mod 16 (every row of a 16-row tile a different d, rows r and r + 16 different d too) and sigma = +-1
    drawn per (b, h, d); its hot key t = (b + 37 h + 5 d) mod nk has component d equal to 32 sigma; every other key component has
    magnitude <= 16.  So the hot raw score is 1024 and every other is <= 512: 512 c = 184.7 below it in log2 units (c = scale log2(e))
    and ex2 flushes it to 0, while the hot key's exponent 1024 c - fl(1024 c) is exactly 0 (1024 c is exact) and ex2(0) = 1.  Then
    l = 1, P = (1, 0, ...) in bf16, and 1 * V[t] accumulated with zeros is V[t]: the output row is V[t] of that head, bit for bit.
    Keys of an earlier block give it a nonzero running maximum and O; the hot block's rescale ex2(m_old - 1024 c) <= ex2(-184.7) is
    exactly 0.  two_hot: key (t + 64) mod nk, in another block of 64 when nk >= 128, is hot too; both weights are exactly 1, l = 2, and
    the output is bf16_rn((V[t] + V[t'] ) / 2) (the fp32 sum of two bf16 values of like magnitude is exact)."""
    g = _gen(seed)
    k = ((torch.rand(B, nk, H, D, generator=g, device="cuda") * 2 - 1) * 16).to(torch.bfloat16)
    v = torch.randn(B, nk, H, D, generator=g, device="cuda")
    v = torch.where(v.abs() < 2 ** -6, torch.where(v < 0, -(2 ** -6), 2 ** -6), v).to(torch.bfloat16)   # 2^-6 <= |v| < 2^4: the
    # fp32 sum of two is exact (their exponents differ by less than 16), and no zero (a signed zero would not survive a sum)
    sign = torch.where(torch.rand(B, H, D, generator=g, device="cuda") < 0.5, -1.0, 1.0)
    b_ = torch.arange(B, device="cuda").view(B, 1, 1)
    h_ = torch.arange(H, device="cuda").view(1, H, 1)
    d_ = torch.arange(D, device="cuda").view(1, 1, D)
    hot = (b_ + 37 * h_ + 5 * d_) % nk                                        # [B,H,D]
    bi, hi, di = (t.expand(B, H, D).reshape(-1) for t in (b_, h_, d_))
    k[bi, hot.reshape(-1), hi, di] = (32 * sign).reshape(-1).to(torch.bfloat16)
    hot2 = None
    if two_hot:
        hot2 = (hot + 64) % nk
        k[bi, hot2.reshape(-1), hi, di] = (32 * sign).reshape(-1).to(torch.bfloat16)
    r_ = torch.arange(nq, device="cuda").view(1, nq, 1)
    dq = (r_ + r_ // 16 + 3 * h_.view(1, 1, H)).expand(B, nq, H) % 16      # [B,nq,H]
    q = torch.zeros(B, nq, H, D, device="cuda")
    q.scatter_(3, dq.unsqueeze(3), 32 * sign.gather(2, dq.transpose(1, 2)).transpose(1, 2).unsqueeze(3))
    # expected rows
    t = hot.gather(2, dq.transpose(1, 2)).transpose(1, 2)                    # [B,nq,H]
    bb = torch.arange(B, device="cuda").view(B, 1, 1).expand(B, nq, H)
    hh = torch.arange(H, device="cuda").view(1, 1, H).expand(B, nq, H)
    want = v[bb, t, hh]                                                       # [B,nq,H,D]
    if two_hot:
        t2 = hot2.gather(2, dq.transpose(1, 2)).transpose(1, 2)
        want = ((want.float() + v[bb, t2, hh].float()) * 0.5).to(torch.bfloat16)
    return (q.to(torch.bfloat16).reshape(B * nq, E), k.reshape(B * nk, E), v.reshape(B * nk, E), want.reshape(B * nq, E), t)


def run_attention(q, k, v, B, nq, nk):
    """the kernel on q as columns 128..255 of a 384-wide matrix, k and v as columns 8..135 and 256..383 of one 512-wide matrix (NaN in
    every other column and in the rows around them), out as columns 64..191 of a 256-wide sentinel frame; checks the frame"""
    cu = _ops()[0]
    qb = Frame(B * nq, 384, torch.bfloat16, "nan")
    qb.view[:, 128:256] = q
    kvb = Frame(B * nk, 512, torch.bfloat16, "nan")
    kvb.view[:, 8:136] = k
    kvb.view[:, 256:384] = v
    of = framed_output(B * nq, E, torch.bfloat16, left=64, right=64)
    cu.attention(qb.view[:, 128:256], kvb.view[:, 8:136], kvb.view[:, 256:384], of.arm(), B, nq, nk)
    of.outside_unchanged(f"attention {B}x{nq}x{nk}")
    return of.view


SINGLE_BLOCK_NK = [1, 8, 9, 16, 20, 31, 33, 40, 48, 51, 57, 63, 64]           # every NT = ceil(nk / 8) from 1 to 8
MULTI_BLOCK_NK = [65, 128, 129, 192, 193, 255, 256, 399, 400]


@pytest.mark.parametrize("nq", [1, 17])
@pytest.mark.parametrize("nk", SINGLE_BLOCK_NK + MULTI_BLOCK_NK)
def test_attention_one_hot_routing_is_exact(nk, nq):
    """B = max(nk, 16) envs: every key position, head and query row is some row's hot key"""
    B = max(nk, 16)
    q, k, v, want, t = one_hot_attention(B, nq, nk, seed=nk + 1000 * nq)
    assert set(t[..., 0].flatten().tolist()) == set(range(nk))               # every key position is reached (head 0 alone)
    out = run_attention(q, k, v, B, nq, nk)
    assert torch.equal(bits(out), bits(want)), f"{int((bits(out) != bits(want)).sum())} elements differ"


@pytest.mark.parametrize("nq", [15, 16, 255])
@pytest.mark.parametrize("nk", [16, 64, 65, 400])
def test_attention_one_hot_routing_at_query_tile_edges(nk, nq):
    B = 16
    q, k, v, want, _ = one_hot_attention(B, nq, nk, seed=7 * nk + nq)
    out = run_attention(q, k, v, B, nq, nk)
    assert torch.equal(bits(out), bits(want)), f"{int((bits(out) != bits(want)).sum())} elements differ"


@pytest.mark.parametrize("nk", [128, 129, 193, 256, 400])
def test_attention_two_hot_keys_in_different_blocks_average_exactly(nk):
    B, nq = 24, 17
    q, k, v, want, _ = one_hot_attention(B, nq, nk, seed=nk, two_hot=True)
    out = run_attention(q, k, v, B, nq, nk)
    assert torch.equal(bits(out), bits(want)), f"{int((bits(out) != bits(want)).sum())} elements differ"


# ---- (a) attention_q1, pointer, embed, gate, add_layernorm: exact cases --------------------------------------------------------------
def run_attention_q1(q, k, v, mask, B, nk):
    cu = _ops()[0]
    qb = Frame(B, 256, torch.bfloat16, "nan")
    qb.view[:, 128:] = q
    kvb = Frame(B * nk, 384, torch.bfloat16, "nan")
    kvb.view[:, 8:136] = k
    kvb.view[:, 256:384] = v
    of = framed_output(B, E, torch.bfloat16, left=8, right=120)
    cu.attention_q1(qb.view[:, 128:], kvb.view[:, 8:136], kvb.view[:, 256:384], mask, of.arm(), B, nk)
    of.outside_unchanged(f"attention_q1 {B}x{nk}")
    return of.view


@pytest.mark.parametrize("nk", [1, 2, 31, 32, 33, 63, 64, 65, 128, 129, 200, 255, 256])
def test_attention_q1_single_key_and_one_hot_are_exact(nk):
    """env b keeps key t = b mod nk only: p = ex2(s - s) = 1, l = 1, acc = fma(1, V[t], 0) plus zeros from the other lanes, so the
    output is V[t] bit for bit; every other key's K and V rows are NaN (they must not be read).  The same inputs without a mask go
    through the one-hot construction of test_attention_one_hot_routing_is_exact (q pre-scaled by c: 32 c is exact)."""
    B = max(nk, 16)
    q, k, v, want, t = one_hot_attention(B, 1, nk, seed=3 * nk)
    out = run_attention_q1(q, k, v, None, B, nk)
    assert torch.equal(bits(out), bits(want)), f"one-hot: {int((bits(out) != bits(want)).sum())} elements differ"
    keep = torch.arange(B, device="cuda") % nk
    mask = torch.ones(B, nk, dtype=torch.uint8, device="cuda")
    mask[torch.arange(B, device="cuda"), keep] = 0
    rows = torch.arange(B * nk, device="cuda")
    masked_rows = mask.view(-1).bool()
    k2, v2 = k.clone(), v.clone()
    k2[rows[masked_rows]] = float("nan")
    v2[rows[masked_rows]] = float("nan")
    out = run_attention_q1(q, k2, v2, mask, B, nk)
    want = v.view(B, nk, E)[torch.arange(B, device="cuda"), keep]
    assert torch.equal(bits(out), bits(want)), f"single key: {int((bits(out) != bits(want)).sum())} elements differ"


def run_pointer(qk, feat, mask, B, n, norm, clip):
    cu = _ops()[0]
    of = framed_output(B * n, 1, torch.float32)                              # logp must be a contiguous [B, n]: frame its rows
    cu.pointer(framed_input(qk), framed_input(feat), mask, of.arm().view(B, n), B, n, norm, clip)
    of.outside_unchanged(f"pointer {B}x{n}")
    return of.view.view(B, n)


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 51, 64, 65, 200, 255, 256])
def test_pointer_single_allowed_action_at_every_position(n):
    """env b allows action t = b mod n only: m = u_t, l = expf(0) + expf(-1e4 - u_t) ... = 1 + 0, logf(1) = 0, so logp[t] is exactly 0,
    and every other entry is fl(-1e4 - u_t), within the bound of (b)"""
    B = max(n, 8)
    qk, feat = _bf(B, E, seed=n), _bf(B * n, E, seed=n + 1)
    keep = torch.arange(B, device="cuda") % n
    mask = torch.ones(B, n, dtype=torch.uint8, device="cuda")
    mask[torch.arange(B, device="cuda"), keep] = 0
    norm = 1 / math.sqrt(E)
    out = run_pointer(qk, feat, mask, B, n, norm, 10.0)
    assert bool((out[torch.arange(B, device="cuda"), keep] == 0).all())
    pointer_check(qk, feat, mask, out, B, n, norm, 10.0, f"single action, n = {n}")


@pytest.mark.parametrize("k_in", [5, 6])
@pytest.mark.parametrize("rows", [1, 7, 4099, 20011])
def test_embed_one_hot_rows_are_exact(k_in, rows):
    """x = e_(r mod k_in): every fma but one adds 0 w = 0, the other gives fl32(w[:, k] + b); the output is that, rounded to bf16"""
    cu = _ops()[0]
    x = torch.zeros(rows, k_in, device="cuda")
    x[torch.arange(rows, device="cuda"), torch.arange(rows, device="cuda") % k_in] = 1.0
    w, b = torch.randn(E, k_in, generator=_gen(rows), device="cuda"), torch.randn(E, generator=_gen(rows + 1), device="cuda")
    of = framed_output(rows, E, torch.bfloat16)
    cu.embed(framed_input(x), framed_input(w), framed_input(b.view(1, E)).view(E), of.arm())
    of.outside_unchanged("embed")
    want = (w.t()[torch.arange(rows, device="cuda") % k_in] + b).to(torch.bfloat16)
    assert torch.equal(bits(of.view), bits(want))


@pytest.mark.parametrize("rows", [1, 7, 4099, 20011])
def test_gate_with_zero_gate_input_halves_exactly(rows):
    """a = 0: __expf(-0) = ex2(0) = 1, 1 + 1 = 2, and __fdividef(b, 2) = b * rcp.approx(2) = b / 2, exact for bf16 b; so every column
    of both halves lands where it belongs, bit for bit"""
    cu = _ops()[0]
    wv = _bf(rows, 2 * HID, seed=rows, scale=3.0)
    wv[:, :HID] = 0
    of = framed_output(rows, HID, torch.bfloat16)
    cu.gate(framed_input(wv), of.arm())
    of.outside_unchanged("gate")
    assert torch.equal(bits(of.view), bits((wv[:, HID:].float() * 0.5).to(torch.bfloat16)))


@pytest.mark.parametrize("rows", [1, 7, 4099, 20011])
def test_layernorm_of_constant_rows_is_beta(rows):
    """x + res = c per row, exactly (multiples of 1/8 below 32, and c in {0, 1, -3, 0.5, 1024, 2^20}): the mean is c exactly, every
    deviation 0, the variance 0, rstd = rsqrt(eps) finite, and fma(0 rstd, g, beta) = beta: the output is bf16(beta), also with out
    aliasing x or res"""
    cu = _ops()[0]
    g = _gen(rows)
    c = torch.tensor([0.0, 1.0, -3.0, 0.5, 1024.0, 2.0 ** 20], device="cuda")[torch.arange(rows, device="cuda") % 6].view(rows, 1)
    res = (torch.randint(-64, 65, (rows, E), generator=g, device="cuda") / 8.0)
    res = torch.where(c.abs() > 100, torch.zeros_like(res), res)             # bf16 x = c - res must stay exact
    x = (c - res).to(torch.bfloat16)
    res = res.to(torch.bfloat16)
    assert torch.equal(x.double() + res.double(), c.double().expand(rows, E))
    gamma, beta = torch.randn(E, generator=g, device="cuda"), torch.randn(E, generator=g, device="cuda")
    want = beta.to(torch.bfloat16).expand(rows, E)
    for alias in ("none", "x", "res"):
        xx, rr = framed_input(x), framed_input(res)
        of = framed_output(rows, E, torch.bfloat16)
        out = {"none": of.arm(), "x": xx, "res": rr}[alias]
        cu.add_layernorm(xx, rr, framed_input(gamma.view(1, E)).view(E), framed_input(beta.view(1, E)).view(E), out, 1e-5)
        if alias == "none":
            of.outside_unchanged("add_layernorm")
        assert torch.equal(bits(out), bits(want)), alias


# ---- (b) bounded cases ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("regime", ["randn", "large_scores"])
def test_attention_within_derived_bound(regime):
    """every single- and multi-block key count at the tile and block edges, with query counts at the tile edges; randn scores, and raw
    scores in the hundreds (q, k ~ N(0, 36): |s| up to ~700), where the online maximum and the rescale decide the result"""
    sc = 1.0 if regime == "randn" else 6.0
    for nk in SINGLE_BLOCK_NK + MULTI_BLOCK_NK:
        for nq in (1, 15, 16, 17, 255):
            B = 2
            q, k, v = _bf(B * nq, E, seed=nk * 7 + nq, scale=sc), _bf(B * nk, E, seed=nk * 11 + nq, scale=sc), _bf(B * nk, E, seed=nk + nq)
            out = run_attention(q, k, v, B, nq, nk)
            attention_check(q, k, v, out, B, nq, nk, f"{regime} {B}x{nq}x{nk}")


@pytest.mark.parametrize("regime", ["randn", "large_scores"])
def test_attention_q1_within_derived_bound(regime):
    """no mask, a partial mask (masked K / V rows NaN), all masked but one, all masked, at key counts across the 8 lane rounds"""
    sc = 1.0 if regime == "randn" else 6.0
    B = 6
    for nk in (1, 2, 31, 32, 33, 63, 64, 65, 128, 129, 200, 255, 256):
        q, k, v = _bf(B, E, seed=nk, scale=sc), _bf(B * nk, E, seed=nk + 1, scale=sc), _bf(B * nk, E, seed=nk + 2)
        g = _gen(nk)
        mask = (torch.rand(B, nk, generator=g, device="cuda") < 0.5).to(torch.uint8)
        mask[1] = 1                                                           # nothing to attend to
        mask[2] = 1
        mask[2, nk - 1] = 0                                                   # the last key alone
        mask[3] = 0
        for m in (None, mask):
            kk, vv = k.clone(), v.clone()
            if m is not None:
                kk[m.view(-1).bool()] = float("nan")
                vv[m.view(-1).bool()] = float("nan")
            out = run_attention_q1(q, kk, vv, m, B, nk)
            attention_q1_check(q, kk, vv, m, out, B, nk, f"{regime} nk = {nk} mask = {m is not None}")


@pytest.mark.parametrize("regime", ["randn", "saturated"])
def test_pointer_within_derived_bound(regime):
    """no mask, partial masks, all masked but one, all masked; tanh in its linear range (norm = 1/sqrt(128)) and saturated
    (|norm dot| up to ~50)"""
    B = 9
    norm = 1 / math.sqrt(E) * (1.0 if regime == "randn" else 8.0)
    for n in (1, 2, 8, 31, 32, 33, 51, 63, 64, 65, 128, 129, 200, 255, 256):
        qk, feat = _bf(B, E, seed=n, scale=1.0 if regime == "randn" else 4.0), _bf(B * n, E, seed=n + 1)
        mask = (torch.rand(B, n, generator=_gen(n), device="cuda") < 0.4).to(torch.uint8)
        mask[0] = 1
        mask[1] = 1
        mask[1, n // 2] = 0
        mask[2] = 0
        for m in (None, mask):
            out = run_pointer(qk, feat, m, B, n, norm, 10.0)
            pointer_check(qk, feat, m, out, B, n, norm, 10.0, f"{regime} n = {n} mask = {m is not None}")


@pytest.mark.parametrize("rows", [1, 7, 4099, 20011])
def test_embed_within_derived_bound(rows):
    cu = _ops()[0]
    for k_in in (5, 6):
        for sc in (1.0, 300.0):                                               # observations in [-1, 3], and up to 1e3
            x = (torch.rand(rows, k_in, generator=_gen(rows + k_in), device="cuda") * 4 - 1) * sc
            w, b = torch.randn(E, k_in, generator=_gen(k_in), device="cuda"), torch.randn(E, generator=_gen(k_in + 9), device="cuda")
            of = framed_output(rows, E, torch.bfloat16)
            cu.embed(framed_input(x), framed_input(w), framed_input(b.view(1, E)).view(E), of.arm())
            of.outside_unchanged("embed")
            embed_check(x, w, b, of.view, f"rows = {rows} k_in = {k_in} scale = {sc}")


@pytest.mark.parametrize("rows", [1, 7, 4099, 20011])
def test_gate_within_derived_bound(rows):
    """randn gate inputs, and inputs in +-[87, 100] where __expf and __fdividef saturate (sigmoid below the smallest normal)"""
    cu = _ops()[0]
    g = _gen(rows)
    for regime in ("randn", "saturated"):
        wv = _bf(rows, 2 * HID, seed=rows + len(regime), scale=3.0)
        if regime == "saturated":
            mag = 87 + 13 * torch.rand(rows, HID, generator=g, device="cuda")
            sgn = torch.where(torch.rand(rows, HID, generator=g, device="cuda") < 0.5, -1.0, 1.0)
            wv[:, :HID] = (mag * sgn).to(torch.bfloat16)
        of = framed_output(rows, HID, torch.bfloat16)
        cu.gate(framed_input(wv), of.arm())
        of.outside_unchanged("gate")
        gate_check(wv, of.view, f"{regime} rows = {rows}")


def _layernorm_rows(regime, rows, g):
    """(x, res) in bf16 for a value regime"""
    if regime == "randn":
        return (torch.randn(rows, E, generator=g, device="cuda") * 2).to(torch.bfloat16), torch.randn(rows, E, generator=g, device="cuda").to(torch.bfloat16)
    if regime == "tiny_variance":                                             # spread 3e-3 around 0: variance ~ eps
        return (torch.randn(rows, E, generator=g, device="cuda") * 3e-3).to(torch.bfloat16), torch.zeros(rows, E, device="cuda").to(torch.bfloat16)
    if regime == "one_ulp_rows":                                              # 1.0 everywhere but 1..4 columns at 1 + 2^-7: var 5e-7 .. 2e-6
        x = torch.ones(rows, E, device="cuda")
        for j in range(4):
            col = torch.randint(0, E, (rows,), generator=g, device="cuda")
            on = torch.arange(rows, device="cuda") % 4 >= j
            x[torch.arange(rows, device="cuda")[on], col[on]] = 1 + 2 ** -7
        return x.to(torch.bfloat16), torch.zeros(rows, E, device="cuda").to(torch.bfloat16)
    if regime in ("offset_1024", "offset_4096"):                              # unit spread on a large common offset
        off = 1024.0 if regime == "offset_1024" else 4096.0
        return torch.full((rows, E), off, device="cuda").to(torch.bfloat16), torch.randn(rows, E, generator=g, device="cuda").to(torch.bfloat16)
    raise ValueError(regime)


@pytest.mark.parametrize("regime", ["randn", "tiny_variance", "one_ulp_rows", "offset_1024", "offset_4096"])
@pytest.mark.parametrize("rows", [1, 7, 4099, 20011])
def test_add_layernorm_within_derived_bound(regime, rows):
    """and with out aliasing x or res: the same bits"""
    cu = _ops()[0]
    g = _gen(rows)
    x, res = _layernorm_rows(regime, rows, g)
    gamma, beta = torch.randn(E, generator=g, device="cuda"), torch.randn(E, generator=g, device="cuda") * 0.1
    gf, bf = framed_input(gamma.view(1, E)).view(E), framed_input(beta.view(1, E)).view(E)
    of = framed_output(rows, E, torch.bfloat16)
    cu.add_layernorm(framed_input(x), framed_input(res), gf, bf, of.arm(), 1e-5)
    of.outside_unchanged("add_layernorm")
    layernorm_check(x, res, gamma, beta, of.view, 1e-5, f"{regime} rows = {rows}")
    for alias in ("x", "res"):
        xx, rr = framed_input(x), framed_input(res)
        out = xx if alias == "x" else rr
        cu.add_layernorm(xx, rr, gf, bf, out, 1e-5)
        assert torch.equal(bits(out), bits(of.view)), alias


# ---- (c) guard memory with nothing to do ------------------------------------------------------------------------------------------------
def test_empty_batches_write_nothing():
    """B = 0 / rows = 0 with valid pointers (a torch view of no rows has none, so the C entry points are called directly): every kernel
    returns 0 without reading its inputs (NaN) or writing its output buffer"""
    from dcmrta_b200.policy_fused import _stream, lib
    L = lib()
    x = framed_input(_bf(4, 2 * HID, seed=0)).data_ptr()
    of = framed_output(4, 2 * HID, torch.bfloat16)
    p = of.arm().data_ptr()
    s = _stream(of.view)
    g = framed_input(torch.ones(1, E, device="cuda")).data_ptr()
    rc = {"embed": L.dcmp_embed(x, g, g, p, 0, 5, s),
          "attention": L.dcmp_attention(x, 1024, x, x, 1024, p, 1024, 0, 4, 9, SCALE, s),
          "attention_q1": L.dcmp_attention_q1(x, 1024, x, x, 1024, None, p, 1024, 0, 9, SCALE, s),
          "add_layernorm": L.dcmp_add_layernorm(x, x, g, g, p, 0, 1e-5, s),
          "gate": L.dcmp_gate(x, p, 0, s),
          "pointer": L.dcmp_pointer(x, x, None, p, 0, 5, 0.1, 10.0, s)}
    assert all(v == 0 for v in rc.values()), rc
    torch.cuda.synchronize()
    assert torch.equal(bits(of.buf), bits(of.before))
