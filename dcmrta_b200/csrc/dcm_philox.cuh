// dcm_philox.cuh -- the one Philox4x32-10 of the project (Salmon et al. 2011), shared by the env kernels (dcm_thread.cuh: leaders,
// followers, the in-kernel policies, the instance generator) and the policy's action sampler (policy_kernels.cu k_sample).  Both key their
// streams by global env id; DESIGN.md 5 lists the counter regions, which are disjoint, so the two may share a seed.
#pragma once
#include <cuda_runtime.h>

namespace dcm {

__device__ __forceinline__ uint4 philox(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        unsigned h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        unsigned h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        unsigned n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

}  // namespace dcm
