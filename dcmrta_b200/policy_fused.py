"""dcmrta_b200/policy_fused.py -- the rollout (no-grad) forward of the attention policy, reference attention.py:288-298
`AttentionNet.forward`, for batches of thousands of envs on one B200.

The policy stays a PyTorch module (`policy.AttentionNet`: parameters, training forward / backward, checkpoints).  What the rollout
loop of SURVEY.md 8(f) row 1 calls once per decision is this INFERENCE path over the same parameters: every dense GEMM is one
`torch.mm` on bf16 rows (cuBLASLt), and what sits between the GEMMs -- the head split, softmax(QK^T)V at head dimension 16, residual +
LayerNorm, the sigmoid gate, the pointer's clipped masked log-softmax -- is one hand-written sm_100a kernel each
(include/dcmrta_policy.h, csrc/policy_kernels.cu) instead of the 5-10 eager kernels per op of the module path
(profiles/r09_policy_forward_profile.txt: LayerNorm 32 %, a flash kernel at head dimension 16 30 %, elementwise 22 %, GEMMs 10 %).

Re-layout of the parameters (done in `refresh`, into buffers whose addresses never change, so a captured CUDA graph stays valid):
  * per-head projections w_query / w_key / w_value [H, E, E/H] (attention.py:91-93) -> one [E, 128] matrix each with head h in columns
    16h..16h+15; self-attention layers use the concatenation [E, 384], decoder layers [E, 128] for the target and [E, 256] for the memory;
  * w_out [H, E/H, E] (attention.py:94) -> [128, E];  GateFFNDense W, V (attention.py:159-160) -> one [E, 1024] matrix, W2 -> [512, E];
  * the pointer's U = (q Wq)(h Wk)^T (attention.py:69-72) = q (Wq Wk^T) h^T: the [E, E] product is folded once, so the pointer never
    projects the T+1 keys;
  * compressed_task = mean_t(task_embedding) (attention.py:268-270) = task_embedding(mean_t(tasks)), the layer being affine.

`forward_torch` is the same dataflow in plain torch ops on the same re-laid-out weights: the CPU tests pin it to `AttentionNet`
(fp32, 1e-5; float64, 1e-12), the GPU tests pin the CUDA path to it and each kernel to its float64 form.  The CUDA path has no
fallback: without libdcmrta_policy.so it raises.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.nn.functional as F

from . import build as _build

E, H, D, HID = 128, 8, 16, 512
_LIB = None

vp, i32, f32, i64 = C.c_void_p, C.c_int, C.c_float, C.c_long
# name -> (restype, argtypes); every symbol include/dcmrta_policy.h declares
SIGNATURES = {
    "dcmp_embed": (i32, [vp, vp, vp, vp, i64, i32, vp]),
    "dcmp_attention": (i32, [vp, i32, vp, vp, i32, vp, i32, i32, i32, i32, f32, vp]),
    "dcmp_attention_q1": (i32, [vp, i32, vp, vp, i32, vp, vp, i32, i32, i32, f32, vp]),
    "dcmp_add_layernorm": (i32, [vp, vp, vp, vp, vp, i64, f32, vp]),
    "dcmp_gate": (i32, [vp, vp, i64, vp]),
    "dcmp_pointer": (i32, [vp, vp, vp, vp, i32, i32, f32, f32, vp]),
    "dcmp_last_error": (C.c_char_p, []),
    "dcmp_version": (C.c_char_p, []),
}
# every symbol include/dcmrta_sample.h declares (the action sampler, in the same library)
SAMPLE_SIGNATURES = {
    "dcmp_sample": (i32, [vp, i32, vp, vp, C.c_longlong, vp, vp, i32, i32, vp]),
}


class PolicyKernelError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load libdcmrta_policy.so (built in-tree first when it is missing or stale and nvcc is present)."""
    global _LIB
    if _LIB is None:
        try:
            so = _build.build_policy()
        except Exception as e:
            so = _build.POLICY_SO
            if not so.exists():
                raise PolicyKernelError(f"libdcmrta_policy.so is missing and cannot be built ({e}); there is no CPU fallback")
        L = C.CDLL(str(so))
        for name, (res, args) in {**SIGNATURES, **SAMPLE_SIGNATURES}.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        raise PolicyKernelError(f"{rc}: {lib().dcmp_last_error().decode()}")


def _stream(t: torch.Tensor):
    return torch.cuda.current_stream(t.device).cuda_stream


# ---- the six ops, tensor-level: CUDA (product) and torch (the specification the tests compare against) -----------------------------
class CudaOps:
    """Each method launches one kernel of libdcmrta_policy.so on the current stream.  Column slices of a wider row-major matrix are
    passed as views (data_ptr() carries the offset, stride(0) the row stride)."""

    acc = torch.float32                                                      # the dtype of the log-probabilities dcmp_pointer writes

    @staticmethod
    def _rows(t):
        assert t.dim() == 2 and t.stride(1) == 1 and t.is_cuda
        return t

    def embed(self, x, w, b, out):
        assert x.dtype == torch.float32 and x.is_contiguous() and out.is_contiguous() and out.dtype == torch.bfloat16
        _check(lib().dcmp_embed(x.data_ptr(), w.data_ptr(), b.data_ptr(), out.data_ptr(), out.shape[0], x.shape[-1], _stream(out)))
        return out

    def attention(self, q, k, v, out, B, nq, nk):
        for t in (q, k, v, out):
            self._rows(t)
        assert k.stride(0) == v.stride(0) and q.shape[0] == B * nq and k.shape[0] == B * nk
        _check(lib().dcmp_attention(q.data_ptr(), q.stride(0), k.data_ptr(), v.data_ptr(), k.stride(0), out.data_ptr(), out.stride(0),
                                    B, nq, nk, 1.0 / math.sqrt(D), _stream(out)))
        return out

    def attention_q1(self, q, k, v, mask, out, B, nk):
        for t in (q, k, v, out):
            self._rows(t)
        assert k.stride(0) == v.stride(0) and q.shape[0] == B and k.shape[0] == B * nk
        assert mask is None or (mask.dtype == torch.uint8 and mask.is_contiguous() and mask.shape == (B, nk))
        _check(lib().dcmp_attention_q1(q.data_ptr(), q.stride(0), k.data_ptr(), v.data_ptr(), k.stride(0),
                                       None if mask is None else mask.data_ptr(), out.data_ptr(), out.stride(0), B, nk,
                                       1.0 / math.sqrt(D), _stream(out)))
        return out

    def add_layernorm(self, x, res, gamma, beta, out, eps):
        assert x.is_contiguous() and res.is_contiguous() and out.is_contiguous() and x.shape == res.shape == out.shape and x.shape[1] == E
        _check(lib().dcmp_add_layernorm(x.data_ptr(), res.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), x.shape[0],
                                        float(eps), _stream(out)))
        return out

    def gate(self, wv, out):
        assert wv.is_contiguous() and out.is_contiguous() and wv.shape[1] == 2 * HID and out.shape == (wv.shape[0], HID)
        _check(lib().dcmp_gate(wv.data_ptr(), out.data_ptr(), wv.shape[0], _stream(out)))
        return out

    def pointer(self, qk, feat, mask, out, B, n, norm, clip):
        assert qk.is_contiguous() and feat.is_contiguous() and out.is_contiguous() and out.dtype == torch.float32
        assert mask is None or (mask.dtype == torch.uint8 and mask.is_contiguous() and mask.shape == (B, n))
        _check(lib().dcmp_pointer(qk.data_ptr(), feat.data_ptr(), None if mask is None else mask.data_ptr(), out.data_ptr(), B, n,
                                  float(norm), float(clip), _stream(out)))
        return out

    @staticmethod
    def mm(a, b, out):
        return torch.mm(a, b, out=out)


class TorchOps:
    """The same six ops in torch (any device / dtype, any embedding size): what each kernel must compute.  Test infrastructure and
    documentation, never called by the product path.  Every op computes in `acc` (fp32 as the kernels do, or float64 for a reference
    that rounds nothing the tests can see)."""

    def __init__(self, e=E, h=H, hid=HID, acc=torch.float32):
        self.E, self.H, self.D, self.HID, self.acc = e, h, e // h, hid, acc

    def embed(self, x, w, b, out):
        return out.copy_(F.linear(x.to(self.acc), w.to(self.acc), b.to(self.acc)))

    def _heads(self, t, B, n):
        return t.reshape(B, n, self.H, self.D).transpose(1, 2).to(self.acc)  # [B,H,n,D]

    def attention(self, q, k, v, out, B, nq, nk):
        s = self._heads(q, B, nq) @ self._heads(k, B, nk).transpose(2, 3) / math.sqrt(self.D)
        o = torch.softmax(s, -1) @ self._heads(v, B, nk)
        return out.copy_(o.transpose(1, 2).reshape(B * nq, self.E))

    def attention_q1(self, q, k, v, mask, out, B, nk):
        s = self._heads(q, B, 1) @ self._heads(k, B, nk).transpose(2, 3) / math.sqrt(self.D)     # [B,H,1,nk]
        if mask is not None:
            s = s.masked_fill(mask.bool().view(B, 1, 1, nk), float("-inf"))
        p = torch.softmax(s, -1)
        if mask is not None:
            p = torch.where(mask.bool().view(B, 1, 1, nk), torch.zeros_like(p), p).nan_to_num(0.0)   # attention.py:137-140
        return out.copy_((p @ self._heads(v, B, nk)).transpose(1, 2).reshape(B, self.E))

    def add_layernorm(self, x, res, gamma, beta, out, eps):
        a = self.acc
        return out.copy_(F.layer_norm(x.to(a) + res.to(a), (self.E,), gamma.to(a), beta.to(a), eps))

    def gate(self, wv, out):
        return out.copy_(torch.sigmoid(wv[:, :self.HID].to(self.acc)) * wv[:, self.HID:].to(self.acc))

    def pointer(self, qk, feat, mask, out, B, n, norm, clip):
        u = clip * torch.tanh(norm * torch.einsum("be,bne->bn", qk.to(self.acc), feat.to(self.acc).view(B, n, self.E)))
        if mask is not None:
            u = u.masked_fill(mask.bool(), -1e4)
        return out.copy_(torch.log_softmax(u, -1))

    @staticmethod
    def mm(a, b, out):
        return out.copy_(a @ b)


# ---- parameter re-layout ---------------------------------------------------------------------------------------------------------------
def _flat_heads(w):
    """[H, E, k] (attention.py:91-93) -> [E, H*k], head h in columns h*k .. h*k + k - 1"""
    return w.detach().permute(1, 0, 2).reshape(w.shape[1], -1)


def _layer_names(net):
    """(name, module, self_attention) in the order forward() uses them"""
    out = [("taskEncoder.0", net.taskEncoder.layers[0], True), ("agentEncoder.0", net.agentEncoder.layers[0], True)]
    for dec in ("crossDecoder", "globalDecoder1", "globalDecoder2"):
        for i, layer in enumerate(getattr(net, dec).layers):
            out.append((f"{dec}.{i}", layer, False))
    return out


def pack_parameters(net, dtype=torch.bfloat16, into: dict | None = None) -> dict:
    """The re-laid-out copy of `net`'s parameters (see the module docstring).  GEMM operands in `dtype`; embedding, LayerNorm and
    nothing else in fp32 (float64 when `dtype` is).  into: refresh these tensors in place instead of allocating."""
    P = {}
    f32 = torch.promote_types(dtype, torch.float32)

    def put(name, t, dt=dtype):
        t = t.detach().to(dt).contiguous()
        if into is not None:
            into[name].copy_(t)
            P[name] = into[name]
        else:
            P[name] = t.clone()

    with torch.no_grad():
        put("task_embedding.w", net.task_embedding.weight, f32); put("task_embedding.b", net.task_embedding.bias, f32)
        put("agent_embedding.w", net.agent_embedding.weight, f32); put("agent_embedding.b", net.agent_embedding.bias, f32)
        for name, layer, self_attn in _layer_names(net):
            mha = layer.multiHeadAttention
            wq, wk, wv = _flat_heads(mha.w_query), _flat_heads(mha.w_key), _flat_heads(mha.w_value)
            if self_attn:
                put(name + ".qkv", torch.cat([wq, wk, wv], 1))
                ln1 = layer.normalization1.normalizer
            else:
                put(name + ".q", wq); put(name + ".kv", torch.cat([wk, wv], 1))
                ln1 = layer.normalization.normalizer
            put(name + ".out", mha.w_out.detach().reshape(-1, mha.embedding_dim))
            ffn, ln2 = layer.feedForward.DenseReluDense, layer.feedForward.layer_norm.normalizer
            put(name + ".wv", torch.cat([ffn.W.weight.t(), ffn.V.weight.t()], 1)); put(name + ".w2", ffn.W2.weight.t())
            for tag, ln in (("ln1", ln1), ("ln2", ln2)):
                put(f"{name}.{tag}.g", ln.weight, f32); put(f"{name}.{tag}.b", ln.bias, f32)
                P[f"{name}.{tag}.eps"] = ln.eps
        put("pointer.m", net.pointer.w_query.detach().to(f32) @ net.pointer.w_key.detach().to(f32).t())
        P["pointer.norm"], P["pointer.clip"] = net.pointer.norm_factor, float(net.pointer.tanh_clipping)
        P["E"], P["HID"] = mha.embedding_dim, ffn.W.out_features
    return P


# ---- the forward ----------------------------------------------------------------------------------------------------------------------
def _forward(ops, P, W, tasks, agents, mask_u8, names):
    """W(name, rows, cols, dtype=None) hands out a workspace tensor; `names` = [(layer name, self_attention)]."""
    B, nt, na = tasks.shape[0], tasks.shape[1], agents.shape[1]
    E, HID = P["E"], P["HID"]                                                # 128, 512 on the CUDA path (FusedPolicy checks)
    te = ops.embed(tasks.reshape(B * nt, -1), P["task_embedding.w"], P["task_embedding.b"], W("te", B * nt, E))
    ae = ops.embed(agents.reshape(B * na, -1), P["agent_embedding.w"], P["agent_embedding.b"], W("ae", B * na, E))
    ct = ops.embed(tasks.mean(1), P["task_embedding.w"], P["task_embedding.b"], W("ct", B, E))    # = mean_t(task_embedding), the layer is affine

    def ffn(name, x1, R):
        wv = ops.mm(x1, P[name + ".wv"], W("wv", R, 2 * HID))
        g = ops.gate(wv, W("g", R, HID))
        f = ops.mm(g, P[name + ".w2"], W("f", R, E))
        return ops.add_layernorm(f, x1, P[name + ".ln2.g"], P[name + ".ln2.b"], W(name + ".y", R, E), P[name + ".ln2.eps"])

    def encoder(name, x, n):                                                  # attention.py:200-206
        R = B * n
        qkv = ops.mm(x, P[name + ".qkv"], W("qkv", R, 3 * E))
        heads = ops.attention(qkv[:, :E], qkv[:, E:2 * E], qkv[:, 2 * E:], W("heads", R, E), B, n, n)
        o = ops.mm(heads, P[name + ".out"], W("o", R, E))
        x1 = ops.add_layernorm(o, x, P[name + ".ln1.g"], P[name + ".ln1.b"], W("x1", R, E), P[name + ".ln1.eps"])
        return ffn(name, x1, R)

    def decoder(name, tgt, nq, mem, nk, mask=None):                           # attention.py:217-223
        R = B * nq
        q = ops.mm(tgt, P[name + ".q"], W("q", R, E))
        kv = ops.mm(mem, P[name + ".kv"], W("kv", B * nk, 2 * E))
        if nq == 1:
            heads = ops.attention_q1(q, kv[:, :E], kv[:, E:], mask, W("heads", R, E), B, nk)
        else:
            assert mask is None
            heads = ops.attention(q, kv[:, :E], kv[:, E:], W("heads", R, E), B, nq, nk)
        o = ops.mm(heads, P[name + ".out"], W("o", R, E))
        x1 = ops.add_layernorm(o, tgt, P[name + ".ln1.g"], P[name + ".ln1.b"], W("x1", R, E), P[name + ".ln1.eps"])
        return ffn(name, x1, R)

    tenc = encoder("taskEncoder.0", te, nt)
    aenc = encoder("agentEncoder.0", ae, na)
    taf = tenc
    for name, _ in names:
        if name.startswith("crossDecoder"):
            taf = decoder(name, taf, nt, aenc, na)
    cs = ct
    for name, _ in names:
        if name.startswith("globalDecoder1"):
            cs = decoder(name, cs, 1, aenc, na)
    for name, _ in names:
        if name.startswith("globalDecoder2"):
            cs = decoder(name, cs, 1, taf, nt, mask_u8)
    qk = ops.mm(cs, P["pointer.m"], W("qk", B, E))
    return ops.pointer(qk, taf, mask_u8, W("logp", B, nt, ops.acc), B, nt, P["pointer.norm"], P["pointer.clip"])


class FusedPolicy:
    """Inference-only forward of an `AttentionNet` (see the module docstring).

        fused = FusedPolicy(net)                  # bf16 re-layout of net's parameters on net's device
        logp = fused(tasks, agents, mask)          # fp32 [B,T+1,5], [B,A,6], bool/u8 [B,T+1] -> fp32 log-probabilities [B,T+1]
        fused.refresh()                            # after an optimiser step: same buffers, new values (CUDA-graph safe)

    The result tensor is a workspace that the next call overwrites."""

    def __init__(self, net):
        mha = net.taskEncoder.layers[0].multiHeadAttention
        ffn = net.taskEncoder.layers[0].feedForward.DenseReluDense
        if (mha.embedding_dim, mha.n_heads, ffn.W.out_features) != (E, H, HID):
            raise PolicyKernelError(f"the kernels are built for the reference network (embedding {E}, {H} heads, hidden {HID}: parameters.py:9, "
                                    f"attention.py:157, :251-258), not for embedding {mha.embedding_dim} / {mha.n_heads} heads / hidden {ffn.W.out_features}")
        self.net = net
        self.names = [(n, s) for n, _, s in _layer_names(net)]
        self.P = pack_parameters(net, torch.bfloat16)
        self._ws = {}
        self.ops = CudaOps()

    def refresh(self, net=None):
        pack_parameters(net if net is not None else self.net, torch.bfloat16, into=self.P)
        return self

    def eval(self):
        return self

    def _workspace(self, device):
        ws = self._ws

        def W(name, rows, cols, dtype=torch.bfloat16):
            t = ws.get(name)
            if t is None or t.shape[0] < rows or t.shape[1] != cols or t.device != device:
                t = ws[name] = torch.empty(rows, cols, dtype=dtype, device=device)
            return t[:rows]
        return W

    @torch.no_grad()
    def __call__(self, tasks, agents, mask):
        if not tasks.is_cuda:
            raise PolicyKernelError("FusedPolicy runs on a CUDA device only (there is no CPU fallback); use AttentionNet on the CPU")
        lib()
        mask_u8 = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        return _forward(self.ops, self.P, self._workspace(tasks.device), tasks.float().contiguous(), agents.float().contiguous(),
                        mask_u8.contiguous(), self.names)


# ---- the action sampler --------------------------------------------------------------------------------------------------------------
def draw_tensor(seed: int, stream: int = 0, decision: int = 0, device=None) -> torch.Tensor:
    """The device-side draw words {seed_lo, seed_hi, stream, decision} that `sample` reads when its kernel runs (int32 storage of the u32
    words).  A captured graph that samples from it serves any seed, stream and decision written into it between replays."""
    if not (0 <= seed < 2 ** 64 and 0 <= stream < 2 ** 32 and 0 <= decision < 2 ** 30 - 1):
        raise ValueError("need 0 <= seed < 2^64, 0 <= stream < 2^32, 0 <= decision < 2^30 - 1")
    words = [seed & 0xFFFFFFFF, seed >> 32, stream, decision]
    return torch.tensor([w - (1 << 32) if w >= 1 << 31 else w for w in words], dtype=torch.int32, device=device)


def sample(logw: torch.Tensor, mask: torch.Tensor | None, draw: torch.Tensor, rows: torch.Tensor | None = None, first_gid: int = 0,
           out: torch.Tensor | None = None) -> torch.Tensor:
    """Categorical(softmax(logw)).sample() per row by dcmp_sample (include/dcmrta_sample.h, the contract of DESIGN.md 5): one int32 action
    per row, on the current stream.  logw [B, n] fp32 log-weights (row stride free, columns contiguous; what any of the three forwards
    returns, the bf16 module's after .float()), mask [B, n] bool / u8 (True = forbidden) or None, draw: `draw_tensor`, rows [B] int64 env
    index of each row (None: row r is env r), the env's global id being first_gid + env index."""
    assert logw.dim() == 2 and logw.dtype == torch.float32 and logw.stride(1) == 1 and logw.is_cuda
    B, n = logw.shape
    if mask is not None:
        mask = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        assert mask.dtype == torch.uint8 and mask.is_contiguous() and mask.shape == (B, n)
    assert draw.dtype == torch.int32 and draw.numel() == 4 and draw.is_contiguous() and draw.device == logw.device
    if rows is not None:
        assert rows.dtype == torch.int64 and rows.is_contiguous() and rows.shape == (B,) and rows.device == logw.device
    if out is None:
        out = torch.empty(B, dtype=torch.int32, device=logw.device)
    _check(lib().dcmp_sample(logw.data_ptr(), logw.stride(0) if B > 1 else n, None if mask is None else mask.data_ptr(),
                             None if rows is None else rows.data_ptr(), int(first_gid), draw.data_ptr(), out.data_ptr(), B, n,
                             _stream(logw)))
    return out


@torch.no_grad()
def forward_torch(net, tasks, agents, mask, dtype=torch.float32):
    """The fused dataflow in torch ops on the re-laid-out parameters (activations and GEMM operands in `dtype`; every op computes in
    fp32, or in float64 when `dtype` is float64: then, on `net.double()`, this is a float64 reference of the whole forward)."""
    P = pack_parameters(net, dtype)
    acc = torch.promote_types(dtype, torch.float32)
    names = [(n, s) for n, _, s in _layer_names(net)]

    def W(name, rows, cols, dt=None):
        return torch.empty(rows, cols, dtype=dt or dtype, device=tasks.device)
    mask_u8 = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    mha = net.taskEncoder.layers[0].multiHeadAttention
    return _forward(TorchOps(P["E"], mha.n_heads, P["HID"], acc), P, W, tasks.to(acc), agents.to(acc), mask_u8, names).clone()
