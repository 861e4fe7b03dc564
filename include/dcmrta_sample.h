/*
 * include/dcmrta_sample.h -- C ABI of the policy's action sampler, exported by libdcmrta_policy.so beside the rollout-forward kernels of
 * include/dcmrta_policy.h, whose conventions it shares: return 0 or a negative code (-1 argument, -2 shape, -3 no device, -4 CUDA;
 * dcmp_last_error() of include/dcmrta_policy.h has the text), plain device pointers, `stream` a cudaStream_t passed as void*, every call
 * asynchronous on it and capturable in a CUDA graph.  A header of its own: the forward maps the policy's observations to log-probabilities,
 * the sampler maps any row of log-weights to an action under the RNG contract of DESIGN.md 5 (the env's Philox, keyed by global env id).
 */
#ifndef DCMRTA_SAMPLE_H
#define DCMRTA_SAMPLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* worker.py:70 Categorical(logp.exp()).sample(), with a draw that is a function of (seed, gid, stream, decision) alone, so a sampled
 * trajectory does not depend on the batch, the shard layout, compaction or graph capture (DESIGN.md 5):
 *   x_d     [B, ldx] fp32 log-weights (log-probabilities or any scores: a constant per row does not matter), finite or -inf; the first n
 *           columns are read, n <= 256
 *   mask_d  [B, n] u8, 1 = forbidden, or NULL
 *   rows_d  [B] i64 env index of row r, or NULL for row r = env r; gid = first_gid + env index
 *   draw_d  [4] u32 on the device, {seed_lo, seed_hi, stream, decision}, read when the kernel runs (one captured graph serves every draw);
 *           decision < 2^30 - 1
 *   action_d [B] i32
 * Philox4x32-10 counter (gid_lo, gid_hi, stream, 0xC0000000 + decision), key (seed_lo, seed_hi); x0 = word 0.  Weights: w_j = 0 for a
 * forbidden entry, else expf(x_j - m) in fp32 with m the maximum over allowed entries (-inf and entries far enough below m underflow to
 * exactly 0).  C_j = inclusive fp32 prefix sum of w in index order (the kernel's association), S = C_l at the last entry l of positive
 * weight, theta = (x0 >> 8) * S * 2^-24 in fp64 (exact).  action = the smallest j with w_j > 0 and C_j > theta; 0 when no entry has
 * positive weight.  All-ones weights: exactly allowed index number floor(u S), u = (x0 >> 8) 2^-24. */
int dcmp_sample(const float* x_d, int ldx, const uint8_t* mask_d, const int64_t* rows_d, long long first_gid, const uint32_t* draw_d,
                int32_t* action_d, int B, int n, void* stream);

#ifdef __cplusplus
}
#endif
#endif
