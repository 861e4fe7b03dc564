// dcmrta_b200/csrc/policy_kernels.cu -- libdcmrta_policy.so (include/dcmrta_policy.h): the memory-bound pieces of the attention policy's
// no-grad rollout forward as single sm_100a kernels.  The dense GEMMs stay in cuBLASLt (torch.mm); what PyTorch runs around them as
// several eager kernels each (head split / permute copies, a flash kernel at head dimension 16, add + LayerNorm, sigmoid + mul, the
// pointer's tanh / masked_fill / log_softmax) is one pass over the activations here.  Everything is HBM-bound SIMT work on bf16 rows:
// 16-byte loads and stores, fp32 arithmetic, warp shuffles; no tensor cores (head dimension 16, at most ~200 keys).
//
// Activations: bf16, row-major, row = env * n + token, embedding 128 (parameters.py:9), 8 heads of 16 (attention.py:251-258).
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/dcmrta_policy.h"
#include "../../include/dcmrta_sample.h"
#include "dcm_philox.cuh"

namespace {

constexpr int E = 128, H = 8, D = 16, HID = 512;
constexpr int ATT_MAX_NK = 400, Q1_MAX_NK = 256, PTR_MAX_N = 256;
constexpr float LOG2E = 1.4426950408889634f;

thread_local char g_err[256] = "";

int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
    if (e != cudaSuccess) snprintf(g_err, sizeof g_err, "%s: %s", what, cudaGetErrorString(e));
    else snprintf(g_err, sizeof g_err, "%s", what);
    return code;
}

int launched(const char* what) {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail(-4, what, e);
}

int sm_count() {                                                              // of the current device, asked once per device
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
    if (!cached[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
        cached[dev] = n;
    }
    return cached[dev];
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- bf16 <-> fp32 on packed words ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ void unpack8(const uint4 u, float* f) {
    f[0] = lo(u.x); f[1] = hi(u.x); f[2] = lo(u.y); f[3] = hi(u.y); f[4] = lo(u.z); f[5] = hi(u.z); f[6] = lo(u.w); f[7] = hi(u.w);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {                 // a -> low half (the lower address), round to nearest even
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
    return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}
__device__ __forceinline__ float ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float wsum(float v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float wmaxf(float v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- embedding: nn.Linear(KIN, 128) on fp32 observation rows -> bf16 ----------------------------------------------------------------
// warp per row, lane <-> 4 output columns whose weights stay in registers; one 8-byte store per lane = one 256-byte row per warp
template <int KIN>
__global__ void __launch_bounds__(256) k_embed(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                               uint2* __restrict__ out, long rows) {
    const int lane = threadIdx.x & 31;
    const long warp = (long)blockIdx.x * 8 + (threadIdx.x >> 5), nwarps = (long)gridDim.x * 8;
    float wr[4][KIN], bs[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        bs[c] = bias[lane * 4 + c];
#pragma unroll
        for (int k = 0; k < KIN; ++k) wr[c][k] = w[(lane * 4 + c) * KIN + k];
    }
    for (long r = warp; r < rows; r += nwarps) {
        float xv[KIN];
#pragma unroll
        for (int k = 0; k < KIN; ++k) xv[k] = __ldg(x + r * KIN + k);
        float y[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            y[c] = bs[c];
#pragma unroll
            for (int k = 0; k < KIN; ++k) y[c] = fmaf(xv[k], wr[c][k], y[c]);
        }
        out[r * 32 + lane] = make_uint2(pack2(y[0], y[1]), pack2(y[2], y[3]));
    }
}

// ---- multi-head attention, no mask, on the tensor cores: block per env, warp per head -------------------------------------------------
// Head dimension 16 is exactly one k-step of mma.m16n8k16: S = Q K^T for 16 queries x 64 keys is 8 MMAs, O += P V another 8, with P
// handed from the accumulator layout to the A-operand layout in registers (two adjacent 16x8 accumulator tiles are one 16x16 A tile).
// K and V rows of the env (all heads, 256 bytes per row) are staged in shared memory with coalesced 16-byte loads, rows padded to 272
// bytes so that the fragment reads (8 rows x 4 words per instruction) hit 32 different banks; Q fragments come straight from global
// memory (a 32-byte head slice per row), the next query tile's while this one is computed.  Online softmax over key blocks of 64, so
// any nk that fits in shared memory.
// History (profiles/r13_policy_experiments.txt): a CUDA-core version (lane per query, K / V broadcast from shared memory) and a first
// tensor-core version that loaded every fragment from global memory per query tile both took 298 us for 8,192 envs of 51 x 51.
// (tcgen05 has nothing to offer a 51 x 51 x 16 problem: its smallest tile is M = 64 with operands staged through shared memory by TMA.)
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t ld32(const uint16_t* p) { return __ldg(reinterpret_cast<const uint32_t*>(p)); }

constexpr int KV_LD = 136;                                                   // shared-memory row stride in elements: 256 + 16 bytes

// NT = S tiles (of 8 keys) per key block.  nk <= 64: one block of exactly ceil(nk / 8) tiles whose K and V fragments are read once,
// before the query tiles (ONE) -- a 20-key memory costs 3 tiles of softmax arithmetic and 14 fragment registers, not 8 and 32.
// nk > 64: blocks of 8 tiles, fragments re-read per block and query tile.
template <int NT, bool ONE>
__global__ void __launch_bounds__(256, 2) k_attention_mma(const uint16_t* __restrict__ q, int ldq, const uint16_t* __restrict__ k,
                                                          const uint16_t* __restrict__ v, int ldkv, uint16_t* __restrict__ out, int ldo,
                                                          int nq, int nk, float scale_log2e) {
    extern __shared__ uint4 smem4[];
    uint16_t* Ks = reinterpret_cast<uint16_t*>(smem4);
    uint16_t* Vs = Ks + (size_t)nk * KV_LD;
    const int b = blockIdx.x, h = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
    const uint16_t* qb = q + (size_t)b * nq * ldq + h * D;
    uint16_t* ob = out + (size_t)b * nq * ldo + h * D;
    for (int idx = threadIdx.x; idx < nk * 16; idx += 256) {                  // 16 chunks of 16 bytes per 128-wide row
        const int t = idx >> 4, c = idx & 15;
        const size_t row = ((size_t)b * nk + t) * ldkv;
        *reinterpret_cast<uint4*>(Ks + t * KV_LD + c * 8) = __ldg(reinterpret_cast<const uint4*>(k + row) + c);
        *reinterpret_cast<uint4*>(Vs + t * KV_LD + c * 8) = __ldg(reinterpret_cast<const uint4*>(v + row) + c);
    }
    const uint16_t* kb = Ks + h * D;
    const uint16_t* vb = Vs + h * D;
    constexpr int KK = (NT + 1) / 2;                                         // P V steps of 16 keys
    uint32_t kf[NT][2], vf[KK][2][2];
    auto load_kv = [&](int k0) {
#pragma unroll
        for (int j = 0; j < NT; ++j) {                                        // S tile j: keys k0 + 8j .. + 7; B fragment = K[key 8j + g][dims 2tg.., 8 + 2tg..]
            const int key = k0 + 8 * j + g;
            kf[j][0] = kf[j][1] = 0u;
            if (key < nk) {
                kf[j][0] = *reinterpret_cast<const uint32_t*>(kb + key * KV_LD + tg * 2);
                kf[j][1] = *reinterpret_cast<const uint32_t*>(kb + key * KV_LD + tg * 2 + 8);
            }
        }
#pragma unroll
        for (int kk = 0; kk < KK; ++kk) {                                     // P V step kk: B fragment = V[keys key0, key0 + 1 | key0 + 8, key0 + 9][dim 8nt + g]
            const int key0 = k0 + 16 * kk + tg * 2;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const uint16_t* vp = vb + key0 * KV_LD + nt * 8 + g;
                const uint32_t v00 = key0 < nk ? vp[0] : 0, v01 = key0 + 1 < nk ? vp[KV_LD] : 0;
                const uint32_t v10 = key0 + 8 < nk ? vp[8 * KV_LD] : 0, v11 = key0 + 9 < nk ? vp[9 * KV_LD] : 0;
                vf[kk][nt][0] = v00 | (v01 << 16); vf[kk][nt][1] = v10 | (v11 << 16);
            }
        }
    };
    auto load_q = [&](int m0, uint32_t (&a)[4]) {                             // A fragment: {row r0, dims 2tg..}, {r1, same}, {r0, dims 8 + 2tg..}, {r1, same}
        const int r0 = m0 + g, r1 = r0 + 8;
        a[0] = r0 < nq ? ld32(qb + (size_t)r0 * ldq + tg * 2) : 0u; a[1] = r1 < nq ? ld32(qb + (size_t)r1 * ldq + tg * 2) : 0u;
        a[2] = r0 < nq ? ld32(qb + (size_t)r0 * ldq + tg * 2 + 8) : 0u; a[3] = r1 < nq ? ld32(qb + (size_t)r1 * ldq + tg * 2 + 8) : 0u;
    };
    uint32_t a[4], an[4] = {0u, 0u, 0u, 0u};
    load_q(0, a);
    __syncthreads();
    if (ONE) load_kv(0);
    for (int m0 = 0; m0 < nq; m0 += 16) {
        const int r0 = m0 + g, r1 = r0 + 8;                                   // the two query rows this lane holds pieces of
        if (m0 + 16 < nq) load_q(m0 + 16, an);
        float mrun0 = -1e30f, mrun1 = -1e30f, l0 = 0.f, l1 = 0.f;              // running maxima (quad-uniform), per-lane partial denominators
        float o[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};          // O accumulators: dims 8nt + 2tg + {0,1}, rows r0 (0,1) and r1 (2,3)
        for (int k0 = 0; k0 < nk; k0 += 8 * NT) {
            if (!ONE) load_kv(k0);
            float s[2 * KK][4];                                               // (an odd NT leaves one all-zero tile for the last P V step)
#pragma unroll
            for (int j = 0; j < 2 * KK; ++j) {
                s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
                if (j < NT && k0 + 8 * j < nk) mma16816(s[j], a, kf[j][0], kf[j][1]);   // warp-uniform
            }
            float mx0 = -1e30f, mx1 = -1e30f;                                  // maxima of the RAW scores (the scale is positive); scaled once, below
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                if (!ONE || j == NT - 1) {                                    // only the last tile of a single block can hold keys past nk
                    const int kc = k0 + 8 * j + tg * 2;                       // this lane's two key columns of tile j
                    if (kc >= nk) s[j][0] = s[j][2] = -1e30f;
                    if (kc + 1 >= nk) s[j][1] = s[j][3] = -1e30f;
                }
                mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1])); mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
            }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
            const float mn0 = fmaxf(mrun0, mx0 * scale_log2e), mn1 = fmaxf(mrun1, mx1 * scale_log2e);
            const float c0 = ex2(mrun0 - mn0), c1 = ex2(mrun1 - mn1);          // 0 on the first block, where everything it scales is 0
            mrun0 = mn0; mrun1 = mn1; l0 *= c0; l1 *= c1;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) { o[nt][0] *= c0; o[nt][1] *= c0; o[nt][2] *= c1; o[nt][3] *= c1; }
#pragma unroll
            for (int j = 0; j < NT; ++j) {                                    // p = 2^(s scale log2(e) - m); keys past nk: 2^(-1e30 ...) = 0
                s[j][0] = ex2(fmaf(s[j][0], scale_log2e, -mn0)); s[j][1] = ex2(fmaf(s[j][1], scale_log2e, -mn0));
                s[j][2] = ex2(fmaf(s[j][2], scale_log2e, -mn1)); s[j][3] = ex2(fmaf(s[j][3], scale_log2e, -mn1));
                l0 += s[j][0] + s[j][1]; l1 += s[j][2] + s[j][3];
            }
#pragma unroll
            for (int kk = 0; kk < KK; ++kk) {                                 // O += P V, 16 keys per step: accumulator tiles 2kk, 2kk + 1 -> one A fragment
                if (k0 + 16 * kk < nk) {                                      // warp-uniform
                    uint32_t pa[4];
                    pa[0] = pack2(s[2 * kk][0], s[2 * kk][1]); pa[1] = pack2(s[2 * kk][2], s[2 * kk][3]);
                    pa[2] = pack2(s[2 * kk + 1][0], s[2 * kk + 1][1]); pa[3] = pack2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
                    mma16816(o[0], pa, vf[kk][0][0], vf[kk][0][1]);
                    mma16816(o[1], pa, vf[kk][1][0], vf[kk][1][1]);
                }
            }
        }
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        const float i0 = 1.f / l0, i1 = 1.f / l1;
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
            if (r0 < nq) *reinterpret_cast<uint32_t*>(ob + (size_t)r0 * ldo + nt * 8 + tg * 2) = pack2(o[nt][0] * i0, o[nt][1] * i0);
            if (r1 < nq) *reinterpret_cast<uint32_t*>(ob + (size_t)r1 * ldo + nt * 8 + tg * 2) = pack2(o[nt][2] * i1, o[nt][3] * i1);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = an[i];
    }
}

// ---- one query per env (global decoders), optional key mask: block per env, warp per head, lane per key -------------------------------
__global__ void __launch_bounds__(256) k_attention_q1(const uint16_t* __restrict__ q, int ldq, const uint16_t* __restrict__ k,
                                                      const uint16_t* __restrict__ v, int ldkv, const uint8_t* __restrict__ mask,
                                                      uint16_t* __restrict__ out, int ldo, int nk, float scale_log2e) {
    const int b = blockIdx.x, h = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float qf[16];
    {
        const uint4* qp = reinterpret_cast<const uint4*>(q + (size_t)b * ldq + h * D);
        unpack8(__ldg(qp), qf); unpack8(__ldg(qp + 1), qf + 8);
#pragma unroll
        for (int d = 0; d < 16; ++d) qf[d] *= scale_log2e;
    }
    constexpr int R = Q1_MAX_NK / 32;
    float s[R];
    float m = -1e30f;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int t = r * 32 + lane;
        s[r] = -1e30f;                                                        // no such key, or forbidden (attention.py:130-133)
        if (t < nk && !(mask && mask[(size_t)b * nk + t])) {
            float kf[16];
            const uint4* kp = reinterpret_cast<const uint4*>(k + ((size_t)b * nk + t) * ldkv + h * D);
            unpack8(__ldg(kp), kf); unpack8(__ldg(kp + 1), kf + 8);
            float a = 0.f;
#pragma unroll
            for (int d = 0; d < 16; ++d) a = fmaf(qf[d], kf[d], a);
            s[r] = a;
        }
        m = fmaxf(m, s[r]);
    }
    m = wmaxf(m);
    uint4* op = reinterpret_cast<uint4*>(out + (size_t)b * ldo + h * D);
    if (m < -1e29f) {                                                         // every key forbidden: the query attends to nothing (attention.py:137-140)
        if (lane == 0) { op[0] = make_uint4(0, 0, 0, 0); op[1] = make_uint4(0, 0, 0, 0); }
        return;
    }
    float l = 0.f, acc[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) acc[d] = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int t = r * 32 + lane;
        if (s[r] > -1e29f) {
            const float p = ex2(s[r] - m);
            l += p;
            float vf[16];
            const uint4* vp = reinterpret_cast<const uint4*>(v + ((size_t)b * nk + t) * ldkv + h * D);
            unpack8(__ldg(vp), vf); unpack8(__ldg(vp + 1), vf + 8);
#pragma unroll
            for (int d = 0; d < 16; ++d) acc[d] = fmaf(p, vf[d], acc[d]);
        }
    }
    l = wsum(l);
#pragma unroll
    for (int d = 0; d < 16; ++d) acc[d] = wsum(acc[d]);
    if (lane == 0) {
        const float inv = 1.f / l;
#pragma unroll
        for (int d = 0; d < 16; ++d) acc[d] *= inv;
        op[0] = pack8(acc); op[1] = pack8(acc + 8);
    }
}

// ---- out = LayerNorm(x + res) * gamma + beta: warp per row, lane <-> 4 columns ---------------------------------------------------------
__global__ void __launch_bounds__(256) k_add_layernorm(const uint2* x, const uint2* res, const float4* __restrict__ gamma,
                                                       const float4* __restrict__ beta, uint2* out, long rows, float eps) {
    const int lane = threadIdx.x & 31;
    const long warp = (long)blockIdx.x * 8 + (threadIdx.x >> 5), nwarps = (long)gridDim.x * 8;
    const float4 g = gamma[lane], bt = beta[lane];
    for (long r = warp; r < rows; r += nwarps) {
        const uint2 a = x[r * 32 + lane], c = res[r * 32 + lane];
        float v0 = lo(a.x) + lo(c.x), v1 = hi(a.x) + hi(c.x), v2 = lo(a.y) + lo(c.y), v3 = hi(a.y) + hi(c.y);
        const float mean = wsum((v0 + v1) + (v2 + v3)) * (1.f / E);
        v0 -= mean; v1 -= mean; v2 -= mean; v3 -= mean;
        const float var = wsum((v0 * v0 + v1 * v1) + (v2 * v2 + v3 * v3)) * (1.f / E);   // biased, as nn.LayerNorm
        const float rstd = rsqrtf(var + eps);
        out[r * 32 + lane] = make_uint2(pack2(fmaf(v0 * rstd, g.x, bt.x), fmaf(v1 * rstd, g.y, bt.y)),
                                        pack2(fmaf(v2 * rstd, g.z, bt.z), fmaf(v3 * rstd, g.w, bt.w)));
    }
}

// A version of this fused with its GEMM (mma.m16n8k16, A fragments in registers, weights streamed through shared memory with cp.async,
// B fragments by ldmatrix.x4; commit "ffn_gate: B fragments by ldmatrix.x4") kept the [rows, 1024] pre-activations out of HBM but ran at a
// third of the legacy tensor rate: 1.47 ms per forward against 0.52 (cuBLASLt GEMM) + 0.74 (this kernel); profiles/r13_policy_experiments.txt.
// ---- out = sigmoid(wv[:, :512]) * wv[:, 512:]: thread per 8 columns -----------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_gate(const uint4* __restrict__ wv, uint4* __restrict__ out, long chunks) {
    const long stride = (long)gridDim.x * 256;
    for (long i = (long)blockIdx.x * 256 + threadIdx.x; i < chunks; i += stride) {
        const long r = i >> 6; const int c = (int)(i & 63);                   // 64 chunks of 8 per 512-wide half row
        float a[8], b[8], y[8];
        unpack8(__ldg(wv + r * 128 + c), a); unpack8(__ldg(wv + r * 128 + 64 + c), b);
#pragma unroll
        for (int d = 0; d < 8; ++d) y[d] = __fdividef(b[d], 1.f + __expf(-a[d]));
        out[i] = pack8(y);
    }
}

// ---- pointer head: warp per env; the 128-wide dot products are warp-cooperative (one coalesced 256-byte row per load) ---------------------
__global__ void __launch_bounds__(256) k_pointer(const uint2* __restrict__ qk, const uint2* __restrict__ feat, const uint8_t* __restrict__ mask,
                                                 float* __restrict__ logp, int B, int n, float norm, float clip) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    const uint2 qw = __ldg(qk + (size_t)b * 32 + lane);
    const float q0 = lo(qw.x), q1 = hi(qw.x), q2 = lo(qw.y), q3 = hi(qw.y);
    constexpr int R = PTR_MAX_N / 32;
    float u[R];
    const uint2* fb = feat + (size_t)b * n * 32;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        u[r] = -1e30f;                                                        // no such key: out of the softmax
        if (r * 32 < n) {                                                     // warp-uniform
            const int cnt = min(32, n - r * 32);
            for (int tt = 0; tt < cnt; tt += 4) {                             // four rows in flight
                float d[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int t = r * 32 + min(tt + j, cnt - 1);
                    const uint2 f = __ldg(fb + (size_t)t * 32 + lane);
                    d[j] = fmaf(q3, hi(f.y), fmaf(q2, lo(f.y), fmaf(q1, hi(f.x), q0 * lo(f.x))));
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float dot = wsum(d[j]);
                    if (tt + j < cnt && lane == tt + j) u[r] = dot;
                }
            }
            const int t = r * 32 + lane;
            if (t < n) {
                u[r] = clip * tanhf(norm * u[r]);                             // attention.py:73-74
                if (mask && mask[(size_t)b * n + t]) u[r] = -1e4f;            // :78-80 (stays inside the softmax, as in the reference)
            }
        }
    }
    float m = -1e30f;
#pragma unroll
    for (int r = 0; r < R; ++r) m = fmaxf(m, u[r]);
    m = wmaxf(m);
    float l = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r) if (r * 32 + lane < n) l += expf(u[r] - m);
    l = wsum(l);
    const float logl = logf(l);
#pragma unroll
    for (int r = 0; r < R; ++r) if (r * 32 + lane < n) logp[(size_t)b * n + r * 32 + lane] = (u[r] - m) - logl;   // in this order: -1e4 entries keep their low bits
}

// ---- action sampler: warp per row, the draw a function of (seed, gid, stream, decision) alone (DESIGN.md 5, include/dcmrta_sample.h) -------
// Pass 1 keeps the row in registers (lane <-> columns 32 r + lane), pass 2 turns it into weights and an inclusive prefix sum (a shuffle
// scan per 32-column chunk, carried from chunk to chunk), pass 3 finds the first crossing of the threshold by ballot.
constexpr int SMP_MAX_N = 256;

__global__ void __launch_bounds__(256) k_sample(const float* __restrict__ x, int ldx, const uint8_t* __restrict__ mask,
                                                const int64_t* __restrict__ rows, long long first_gid, const uint32_t* __restrict__ draw,
                                                int32_t* __restrict__ action, int B, int n) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    const unsigned long long gid = (unsigned long long)(first_gid + (rows ? rows[b] : (long long)b));
    const uint4 r4 = dcm::philox((unsigned)gid, (unsigned)(gid >> 32), draw[2], 0xC0000000u + draw[3], draw[0], draw[1]);
    constexpr int R = SMP_MAX_N / 32;
    float v[R];
    float m = -INFINITY;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int j = r * 32 + lane;
        v[r] = -INFINITY;                                                    // no such column, or forbidden: weight 0
        if (j < n && !(mask && mask[(size_t)b * n + j])) v[r] = x[(size_t)b * ldx + j];
        m = fmaxf(m, v[r]);
    }
    m = wmaxf(m);
    float c[R];
    float carry = 0.f, S = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        c[r] = 0.f;
        if (r * 32 < n) {                                                    // warp-uniform
            const float w = v[r] > -INFINITY ? expf(v[r] - m) : 0.f;         // (m is finite whenever some v is)
            v[r] = w;
            float s = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const float t = __shfl_up_sync(0xffffffffu, s, o);
                if (lane >= o) s += t;
            }
            c[r] = carry + s;
            carry = __shfl_sync(0xffffffffu, c[r], 31);
            const unsigned pos = __ballot_sync(0xffffffffu, w > 0.f);
            if (pos) S = __shfl_sync(0xffffffffu, c[r], 31 - __clz(pos));    // C at the last entry of positive weight so far
        }
    }
    int a = 0;                                                               // nothing of positive weight: 0 (the step ignores it)
    if (S > 0.f) {
        const double theta = (double)(r4.x >> 8) * (double)S * 0x1p-24;      // exact: 24 x 24 significant bits
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const unsigned hit = __ballot_sync(0xffffffffu, r * 32 + lane < n && v[r] > 0.f && (double)c[r] > theta);
            if (hit) { a = r * 32 + __ffs(hit) - 1; break; }
        }
    }
    if (lane == 0) action[b] = a;
}

int row_grid(long rows) {                                                     // 8 rows (warps) per block, at most 8 resident blocks per SM
    const long want = (rows + 7) / 8, cap = (long)sm_count() * 8;
    return (int)(want < cap ? want : cap);
}

}  // namespace

extern "C" {

int dcmp_embed(const float* x, const float* w, const float* bias, uint16_t* out, long rows, int k_in, void* stream) {
    if (!x || !w || !bias || !out || rows < 0) return fail(-1, "dcmp_embed: null pointer or negative row count");
    if (!aligned16(out)) return fail(-1, "dcmp_embed: out must be 16-byte aligned");
    if (k_in != 5 && k_in != 6) return fail(-2, "dcmp_embed: k_in must be 5 (task rows) or 6 (agent rows)");
    if (rows == 0) return 0;
    if (!sm_count()) return fail(-3, "dcmp_embed: no CUDA device (there is no CPU fallback)");
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (k_in == 5) k_embed<5><<<row_grid(rows), 256, 0, s>>>(x, w, bias, reinterpret_cast<uint2*>(out), rows);
    else k_embed<6><<<row_grid(rows), 256, 0, s>>>(x, w, bias, reinterpret_cast<uint2*>(out), rows);
    return launched("k_embed");
}

int dcmp_attention(const uint16_t* q, int ldq, const uint16_t* k, const uint16_t* v, int ldkv, uint16_t* out, int ldo, int B, int nq, int nk,
                   float scale, void* stream) {
    if (!q || !k || !v || !out) return fail(-1, "dcmp_attention: null pointer");
    if (B < 0 || nq < 1 || nk < 1 || nk > ATT_MAX_NK) return fail(-2, "dcmp_attention: need B >= 0, nq >= 1, 1 <= nk <= 400");
    if ((ldq | ldkv | ldo) & 7 || ldq < E || ldkv < E || ldo < E || !aligned16(q) || !aligned16(k) || !aligned16(v) || !aligned16(out))
        return fail(-1, "dcmp_attention: row strides must be multiples of 8 elements (>= 128) and pointers 16-byte aligned");
    if (B == 0) return 0;
    if (!sm_count()) return fail(-3, "dcmp_attention: no CUDA device (there is no CPU fallback)");
    const size_t smem = (size_t)2 * nk * KV_LD * sizeof(uint16_t);
    static bool opted[64] = {false};
    int dev = 0; cudaGetDevice(&dev);
    if (!opted[dev]) {
        const int most = 2 * ATT_MAX_NK * KV_LD * (int)sizeof(uint16_t);
        cudaError_t e = cudaFuncSetAttribute(k_attention_mma<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, most);
        if (e != cudaSuccess) return fail(-4, "cudaFuncSetAttribute(k_attention_mma)", e);
        opted[dev] = true;                                                   // (nk <= 64 needs 34 kB at most: no opt-in)
    }
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
#define DCMP_ATT(NT) k_attention_mma<NT, true><<<B, 256, smem, st>>>(q, ldq, k, v, ldkv, out, ldo, nq, nk, scale * LOG2E)
    switch ((nk + 7) / 8) {
        case 1: DCMP_ATT(1); break; case 2: DCMP_ATT(2); break; case 3: DCMP_ATT(3); break; case 4: DCMP_ATT(4); break;
        case 5: DCMP_ATT(5); break; case 6: DCMP_ATT(6); break; case 7: DCMP_ATT(7); break; case 8: DCMP_ATT(8); break;
        default: k_attention_mma<8, false><<<B, 256, smem, st>>>(q, ldq, k, v, ldkv, out, ldo, nq, nk, scale * LOG2E);
    }
#undef DCMP_ATT
    return launched("k_attention_mma");
}

int dcmp_attention_q1(const uint16_t* q, int ldq, const uint16_t* k, const uint16_t* v, int ldkv, const uint8_t* mask, uint16_t* out, int ldo,
                      int B, int nk, float scale, void* stream) {
    if (!q || !k || !v || !out) return fail(-1, "dcmp_attention_q1: null pointer");
    if (B < 0 || nk < 1 || nk > Q1_MAX_NK) return fail(-2, "dcmp_attention_q1: need B >= 0, 1 <= nk <= 256");
    if ((ldq | ldkv | ldo) & 7 || ldq < E || ldkv < E || ldo < E || !aligned16(q) || !aligned16(k) || !aligned16(v) || !aligned16(out))
        return fail(-1, "dcmp_attention_q1: row strides must be multiples of 8 elements (>= 128) and pointers 16-byte aligned");
    if (B == 0) return 0;
    if (!sm_count()) return fail(-3, "dcmp_attention_q1: no CUDA device (there is no CPU fallback)");
    k_attention_q1<<<B, 256, 0, static_cast<cudaStream_t>(stream)>>>(q, ldq, k, v, ldkv, mask, out, ldo, nk, scale * LOG2E);
    return launched("k_attention_q1");
}

int dcmp_add_layernorm(const uint16_t* x, const uint16_t* res, const float* gamma, const float* beta, uint16_t* out, long rows, float eps,
                       void* stream) {
    if (!x || !res || !gamma || !beta || !out || rows < 0) return fail(-1, "dcmp_add_layernorm: null pointer or negative row count");
    if (!aligned16(x) || !aligned16(res) || !aligned16(out) || !aligned16(gamma) || !aligned16(beta))
        return fail(-1, "dcmp_add_layernorm: pointers must be 16-byte aligned");
    if (rows == 0) return 0;
    if (!sm_count()) return fail(-3, "dcmp_add_layernorm: no CUDA device (there is no CPU fallback)");
    k_add_layernorm<<<row_grid(rows), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const uint2*>(x), reinterpret_cast<const uint2*>(res), reinterpret_cast<const float4*>(gamma),
        reinterpret_cast<const float4*>(beta), reinterpret_cast<uint2*>(out), rows, eps);
    return launched("k_add_layernorm");
}

int dcmp_gate(const uint16_t* wv, uint16_t* out, long rows, void* stream) {
    if (!wv || !out || rows < 0) return fail(-1, "dcmp_gate: null pointer or negative row count");
    if (!aligned16(wv) || !aligned16(out)) return fail(-1, "dcmp_gate: pointers must be 16-byte aligned");
    if (rows == 0) return 0;
    if (!sm_count()) return fail(-3, "dcmp_gate: no CUDA device (there is no CPU fallback)");
    const long chunks = rows * (HID / 8);
    const long want = (chunks + 255) / 256, cap = (long)sm_count() * 8;
    k_gate<<<(int)(want < cap ? want : cap), 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint4*>(wv),
                                                                                          reinterpret_cast<uint4*>(out), chunks);
    return launched("k_gate");
}

int dcmp_pointer(const uint16_t* qk, const uint16_t* feat, const uint8_t* mask, float* logp, int B, int n, float norm, float clip, void* stream) {
    if (!qk || !feat || !logp) return fail(-1, "dcmp_pointer: null pointer");
    if (B < 0 || n < 1 || n > PTR_MAX_N) return fail(-2, "dcmp_pointer: need B >= 0, 1 <= n <= 256");
    if (!aligned16(qk) || !aligned16(feat)) return fail(-1, "dcmp_pointer: pointers must be 16-byte aligned");
    if (B == 0) return 0;
    if (!sm_count()) return fail(-3, "dcmp_pointer: no CUDA device (there is no CPU fallback)");
    k_pointer<<<(B + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint2*>(qk), reinterpret_cast<const uint2*>(feat),
                                                                         mask, logp, B, n, norm, clip);
    return launched("k_pointer");
}

int dcmp_sample(const float* x, int ldx, const uint8_t* mask, const int64_t* rows, long long first_gid, const uint32_t* draw, int32_t* action,
                int B, int n, void* stream) {
    if (!x || !draw || !action) return fail(-1, "dcmp_sample: null pointer");
    if (first_gid < 0) return fail(-1, "dcmp_sample: first_gid must be >= 0");
    if (B < 0 || n < 1 || n > SMP_MAX_N || ldx < n) return fail(-2, "dcmp_sample: need B >= 0, 1 <= n <= 256, ldx >= n");
    if (B == 0) return 0;
    if (!sm_count()) return fail(-3, "dcmp_sample: no CUDA device (there is no CPU fallback)");
    k_sample<<<(B + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, ldx, mask, rows, first_gid, draw, action, B, n);
    return launched("k_sample");
}

const char* dcmp_last_error(void) { return g_err; }
const char* dcmp_version(void) { return "dcmrta_policy 1 (sm_100a)"; }

}  // extern "C"
