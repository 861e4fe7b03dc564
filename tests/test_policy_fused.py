"""The rollout forward of dcmrta_b200/policy_fused.py (SURVEY 8(f) row 1: the policy inside the decision loop).

CPU: the re-laid-out dataflow (`forward_torch`) against `AttentionNet` and against the log-probabilities recorded from the UNMODIFIED
reference attention.py (tests/golden/policy_golden.npz); libdcmrta_policy.so builds for sm_100a only and exports exactly what
include/dcmrta_policy.h declares; no CPU fallback.
GPU (-m gpu): every kernel against its torch specification (`TorchOps`) on the same bf16 inputs, the whole fused forward against the
fp32 module, and the rollout loops calling it.  Each kernel against a float64 reference with derived bounds, exact cases and guard
memory: tests/test_gpu_policy_kernels.py."""
import ctypes as C
import math
import re
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"


def _net(seed=0, jitter=0.1):
    from dcmrta_b200.policy import AttentionNet
    torch.manual_seed(seed)
    net = AttentionNet(6, 5, 128).eval()
    with torch.no_grad():                                # LayerNorm parameters off their (1, 0) initial values, so that a swapped pair shows
        for n, p in net.named_parameters():
            if "normalizer" in n:
                p.add_(torch.randn_like(p) * jitter)
    return net


def _obs(B, A, T, seed=1, p_mask=0.4):
    g = torch.Generator().manual_seed(seed)
    tasks, agents = torch.rand(B, T + 1, 5, generator=g), torch.rand(B, A, 6, generator=g)
    mask = torch.rand(B, T + 1, generator=g) < p_mask
    mask[:, 0] &= torch.rand(B, generator=g) < 0.5
    return tasks, agents, mask


# ---- CPU ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("A,T", [(20, 50), (10, 20), (3, 4)])
def test_relayout_matches_the_module(A, T):
    from dcmrta_b200.policy_fused import forward_torch
    net = _net()
    tasks, agents, mask = _obs(9, A, T)
    mask[4] = True                                       # an env whose every action is forbidden: the decoder query attends to nothing
    with torch.no_grad():
        ref = net(tasks, agents, mask)
    out = forward_torch(net, tasks, agents, mask)
    assert out.shape == ref.shape and torch.allclose(out, ref, atol=2e-5, rtol=0), float((out - ref).abs().max())


@pytest.mark.parametrize("A,T", [(20, 50), (3, 4)])
def test_float64_relayout_matches_the_float64_module(A, T):
    """forward_torch in float64 is a float64 reference (every op computes in float64, the log-probabilities too): the reference the
    GPU kernel tests (test_gpu_policy_kernels.py) compare with.  The re-layout reorders sums (heads, the folded pointer matrix, the
    embedding of the mean task), so it agrees with the module to float64 rounding, far below anything fp32 could reach."""
    from dcmrta_b200.policy_fused import forward_torch
    net = _net().double()
    tasks, agents, mask = _obs(9, A, T)
    mask[4] = True
    tasks, agents = tasks.double(), agents.double()
    with torch.no_grad():
        ref = net(tasks, agents, mask)
    out = forward_torch(net, tasks, agents, mask, torch.float64)
    assert out.dtype == torch.float64 and out.shape == ref.shape
    assert float((out - ref).abs().max()) < 1e-12


def test_relayout_matches_the_reference_recording():
    """weights, inputs and log-probabilities recorded from the unmodified attention.py at embedding 16 (oracle/make_policy_golden.py);
    the re-layout is size-generic, the kernels are not"""
    from dcmrta_b200.policy import AttentionNet
    from dcmrta_b200.policy_fused import forward_torch
    g = np.load(GOLD / "policy_golden.npz")
    net = AttentionNet(6, 5, 16).eval()
    net.load_state_dict({k[len("w/"):]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w/")})
    out = forward_torch(net, torch.from_numpy(g["plain/tasks"]), torch.from_numpy(g["plain/agents"]), torch.from_numpy(g["plain/mask"]))
    assert np.allclose(out.numpy(), g["plain/logp"], atol=2e-5, rtol=2e-5)
    assert np.array_equal(out.argmax(1).numpy(), g["plain/logp"].argmax(1))


def test_bf16_dataflow_stays_close():
    """what the CUDA path computes in (bf16 operands and activations, fp32 inside an op): greedy choices survive almost always"""
    from dcmrta_b200.policy_fused import forward_torch
    net = _net()
    tasks, agents, mask = _obs(64, 20, 50)
    with torch.no_grad():
        ref = net(tasks, agents, mask)
    out = forward_torch(net, tasks, agents, mask, torch.bfloat16)
    assert float((out - ref).abs()[~mask].max()) < 0.1
    assert float((out.argmax(1) == ref.argmax(1)).float().mean()) > 0.9


def declared_symbols():
    text = (ROOT / "include" / "dcmrta_policy.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dcmp_[a-z0-9_]+)\s*\(", text)))


def test_policy_header_symbols_are_exported_and_bound():
    from dcmrta_b200 import policy_fused as pf
    L = pf.lib()
    names = declared_symbols()
    assert len(names) == 8
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/dcmrta_policy.h but not exported"
    assert sorted(pf.SIGNATURES) == names
    assert b"sm_100a" in L.dcmp_version()


def test_policy_binary_targets_sm100a_only():
    import subprocess
    from dcmrta_b200 import build
    build.build_policy()
    out = subprocess.run(["cuobjdump", "-lelf", str(build.POLICY_SO)], capture_output=True, text=True).stdout
    assert set(re.findall(r"sm_\d+a?", out)) == {"sm_100a"}


def test_policy_kernels_validate_arguments_and_have_no_cpu_fallback():
    from dcmrta_b200 import policy_fused as pf
    L = pf.lib()
    buf = (C.c_uint16 * 4096)()
    p = C.addressof(buf) + (-C.addressof(buf)) % 16
    assert L.dcmp_attention(p, 128, p, p, 128, p, 128, 1, 1, 401, 0.25, None) == -2          # nk over the shared-memory budget
    assert L.dcmp_attention(p, 100, p, p, 128, p, 128, 1, 1, 4, 0.25, None) == -1            # row stride not a multiple of 8
    assert L.dcmp_attention(p + 2, 128, p, p, 128, p, 128, 1, 1, 4, 0.25, None) == -1        # misaligned
    assert L.dcmp_embed(p, p, p, p, 4, 7, None) == -2
    assert L.dcmp_pointer(p, p, None, p, 1, 257, 0.1, 10.0, None) == -2
    assert L.dcmp_gate(None, p, 1, None) == -1 and b"null" in L.dcmp_last_error()
    if not torch.cuda.is_available():
        assert L.dcmp_gate(p, p, 1, None) == -3 and b"no CPU fallback" in L.dcmp_last_error()
        net = _net()
        with pytest.raises(pf.PolicyKernelError):
            pf.FusedPolicy(net)(*_obs(2, 20, 50))


def test_fused_policy_rejects_other_network_sizes():
    from dcmrta_b200.policy import AttentionNet
    from dcmrta_b200 import policy_fused as pf
    with pytest.raises(pf.PolicyKernelError):
        pf.FusedPolicy(AttentionNet(6, 5, 32))


# ---- GPU ------------------------------------------------------------------------------------------------------------------------------
def _bf(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, generator=g, device="cuda") * scale).to(torch.bfloat16)


def _close(out, ref, atol, what):
    """bf16 outputs: within one rounding step of the fp32 specification (2^-8 relative) plus atol"""
    err = (out.float() - ref.float()).abs()
    tol = atol + ref.float().abs() * 2.0 ** -7
    assert bool((err <= tol).all()), f"{what}: max error {float(err.max()):.4g} at magnitude {float(ref.float().abs().max()):.4g}"


@pytest.mark.gpu
@pytest.mark.parametrize("B,nq,nk", [(5, 51, 51), (3, 20, 20), (4, 51, 20), (2, 101, 30), (2, 64, 201), (1, 1, 1), (3, 33, 7),
                                     (2, 17, 9), (2, 5, 33), (2, 48, 41), (2, 40, 64), (2, 16, 65), (1, 70, 400)])
def test_kernel_attention(B, nq, nk):
    from dcmrta_b200.policy_fused import CudaOps, TorchOps
    qkv = _bf(B * nq, 384, seed=1)                       # q as a column slice of a wider matrix, k / v of another
    kv = _bf(B * nk, 256, seed=2)
    out = torch.full((B * nq, 128), 7.0, dtype=torch.bfloat16, device="cuda")
    CudaOps().attention(qkv[:, 128:256], kv[:, :128], kv[:, 128:], out, B, nq, nk)
    ref = TorchOps().attention(qkv[:, 128:256], kv[:, :128], kv[:, 128:], torch.empty(B * nq, 128, device="cuda"), B, nq, nk)
    _close(out, ref, 4e-3, "attention")                 # P is rounded to bf16 before P V (the A operand of the second MMA)


@pytest.mark.gpu
@pytest.mark.parametrize("B,nk,masked", [(6, 51, True), (6, 20, False), (3, 201, True), (2, 256, True), (2, 1, False)])
def test_kernel_attention_one_query(B, nk, masked):
    from dcmrta_b200.policy_fused import CudaOps, TorchOps
    q, kv = _bf(B, 128, seed=3), _bf(B * nk, 256, seed=4)
    mask = None
    if masked:
        mask = (torch.rand(B, nk, device="cuda") < 0.5).to(torch.uint8)
        mask[1] = 1                                      # nothing to attend to: zeros (attention.py:137-140)
    out = torch.full((B, 128), 7.0, dtype=torch.bfloat16, device="cuda")
    CudaOps().attention_q1(q, kv[:, :128], kv[:, 128:], mask, out, B, nk)
    ref = TorchOps().attention_q1(q, kv[:, :128], kv[:, 128:], mask, torch.empty(B, 128, device="cuda"), B, nk)
    _close(out, ref, 2e-3, "attention_q1")
    if masked:
        assert bool((out[1] == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [1, 7, 4099, 8192 * 51])
def test_kernel_add_layernorm_gate_embed(rows):
    from dcmrta_b200.policy_fused import CudaOps, TorchOps
    cu, th = CudaOps(), TorchOps()
    x, r = _bf(rows, 128, seed=5, scale=2.0), _bf(rows, 128, seed=6)
    g, b = torch.randn(128, device="cuda"), torch.randn(128, device="cuda")
    out = cu.add_layernorm(x, r, g, b, torch.empty_like(x), 1e-5)
    _close(out, th.add_layernorm(x, r, g, b, torch.empty(rows, 128, device="cuda"), 1e-5), 2e-3, "add_layernorm")
    y = x.clone()
    cu.add_layernorm(y, r, g, b, y, 1e-5)                # out aliases x
    assert torch.equal(y, out)
    wv = _bf(rows, 1024, seed=7, scale=3.0)
    _close(cu.gate(wv, torch.empty(rows, 512, dtype=torch.bfloat16, device="cuda")), th.gate(wv, torch.empty(rows, 512, device="cuda")), 1e-6, "gate")
    for k in (5, 6):
        obs = torch.rand(rows, k, device="cuda") * 4 - 1
        w, bias = torch.randn(128, k, device="cuda"), torch.randn(128, device="cuda")
        _close(cu.embed(obs, w, bias, torch.empty(rows, 128, dtype=torch.bfloat16, device="cuda")),
               th.embed(obs, w, bias, torch.empty(rows, 128, device="cuda")), 1e-5, f"embed k={k}")


@pytest.mark.gpu
@pytest.mark.parametrize("B,n", [(11, 51), (8, 21), (3, 201), (2, 256), (9, 1), (5, 33)])
def test_kernel_pointer(B, n):
    from dcmrta_b200.policy_fused import CudaOps, TorchOps
    qk, feat = _bf(B, 128, seed=8), _bf(B * n, 128, seed=9)
    mask = (torch.rand(B, n, device="cuda") < 0.4).to(torch.uint8)
    mask[0] = 1                                          # everything forbidden: uniform over the -1e4 entries, as the reference
    norm = 1 / math.sqrt(128)
    for m in (mask, None):
        out = CudaOps().pointer(qk, feat, m, torch.empty(B, n, device="cuda"), B, n, norm, 10.0)
        ref = TorchOps().pointer(qk, feat, m, torch.empty(B, n, device="cuda"), B, n, norm, 10.0)
        assert torch.allclose(out, ref, atol=2e-4, rtol=1e-5), float((out - ref).abs().max())
    assert torch.allclose(out.exp().sum(1), torch.ones(B, device="cuda"), atol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("A,T,B", [(20, 50, 257), (10, 20, 64), (50, 200, 9)])
def test_fused_forward_matches_the_module(A, T, B):
    """the CUDA path against (i) its own dataflow in torch at bf16 and (ii) the fp32 module"""
    from dcmrta_b200.policy_fused import FusedPolicy, forward_torch
    net = _net().cuda()
    tasks, agents, mask = (t.cuda() for t in _obs(B, A, T))
    mask[2] = True
    with torch.no_grad():
        ref = net(tasks, agents, mask)
    fused = FusedPolicy(net)
    out = fused(tasks, agents, mask).clone()
    assert out.dtype == torch.float32 and out.shape == ref.shape and bool(torch.isfinite(out).all())
    spec = forward_torch(net, tasks, agents, mask, torch.bfloat16)
    ok = ~mask
    assert float((out - spec).abs()[ok].max()) < 0.08, "CUDA kernels vs the same dataflow in torch bf16"
    assert float((out - ref).abs()[ok].max()) < 0.1, "bf16 fused path vs the fp32 module"
    chosen = ref.gather(1, out.argmax(1, keepdim=True)).squeeze(1)       # the fused greedy choice, scored by the fp32 module
    assert float((ref.max(1).values - chosen).max()) < 0.1
    assert torch.allclose(out.exp().sum(1), torch.ones(B, device="cuda"), atol=1e-3)
    # refresh after an update of the parameters: same buffers, new values
    ptrs = {k: v.data_ptr() for k, v in fused.P.items() if torch.is_tensor(v)}
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(1.05)
        ref2 = net(tasks, agents, mask)
    out2 = fused.refresh()(tasks, agents, mask)
    assert ptrs == {k: v.data_ptr() for k, v in fused.P.items() if torch.is_tensor(v)}
    assert float((out2 - ref2).abs()[ok].max()) < 0.12 and not torch.equal(out2, out)


@pytest.mark.gpu
def test_rollouts_with_the_fused_policy():
    """eager and CUDA-graph decision loops calling FusedPolicy: episodes end, chosen actions are legal, and the recorded experience
    re-scored by the fp32 module gives the log-probabilities the fused path sampled from (bf16 tolerance)"""
    from dcmrta_b200 import BatchedTaskEnv
    from dcmrta_b200.rollout import BatchedRollout, GraphedRollout
    B, A, T = 512, 10, 20
    net = _net().cuda()
    for Rollout in (BatchedRollout, GraphedRollout):
        env = BatchedTaskEnv(B, A, T, auto_reset=False, seed=11)
        env.generate()
        more = {"fractions": (1.0, 0.5, 0.25)} if Rollout is GraphedRollout else {}      # the graphed loop also gathers the live envs
        ro = Rollout(env, horizon=4 * (A + T), record=True, **more)
        torch.cuda.manual_seed(5)
        kw = {"keep_logp": True} if Rollout is BatchedRollout else {}
        ep = ro.run(net, "sample", amp="fused", **kw)
        assert bool(ep.ended.all()) and bool((ep.reward < 0).all())
        chosen_masked = ep.mask.gather(2, ep.action.long().unsqueeze(2)).squeeze(2).bool() & ep.active
        assert not bool(chosen_masked.any())
        assert torch.equal(ep.active.sum(0).double(), ep.metrics[:, 7])
        if "keep_logp" in kw:
            t = ep.length // 2
            with torch.no_grad():
                ref = net(ep.task_obs[t], ep.agent_obs[t], ep.mask[t].view(torch.bool))
            ok = ~ep.mask[t].view(torch.bool) & ep.active[t].unsqueeze(1)
            assert float((ep.logp[t] - ref).abs()[ok].max()) < 0.1
        greedy = Rollout(env, horizon=4 * (A + T), record=False, **more).run(net, "greedy", amp="fused")
        assert bool(greedy.ended.all())
        if more:
            assert ep.forwarded < B * ep.length and greedy.forwarded < B * greedy.length
        env.close()
