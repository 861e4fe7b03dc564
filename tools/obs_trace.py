#!/usr/bin/env python
"""tools/obs_trace.py [B] [passes] -- globaltimer stamps of steady-state passes (DCM_PASS_TRACE=1): per k_obs_tile block
entry, scalars landed, input copies landed, rows staged, output copies read, and the SM it ran on; per k_episode_list block
entry, exit and SM.  Prints the phase percentiles of the last pass and, per pass, how long both kernels took and how many obs
blocks each SM had resident while episode blocks were alive."""
import os, sys
os.environ["DCM_PASS_TRACE"] = "1"
import ctypes as C
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dcmrta_b200 import BatchedTaskEnv
from dcmrta_b200._lib import lib, check
B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
PASSES = int(sys.argv[2]) if len(sys.argv) > 2 else 4
env = BatchedTaskEnv(B, 20, 50, auto_reset=True, seed=1234)
env.generate(); env.reset()
for _ in range(700): env.step(policy="random")
torch.cuda.synchronize()
NT = (B + 31) // 32
EB = 148 * 8 + 8   # warps of k_episode_list (one env each): EPI_LIST_WARPS_PER_SM = 8 per SM (csrc/dcm_kernels.cu)
pc = lambda x: np.percentile(x, [0, 10, 50, 90, 99, 100]).round(2)
for p in range(PASSES):
    env.step(policy="random"); torch.cuda.synchronize()
    full = np.zeros(NT * 64 * 4, np.uint64)
    check(lib().dcm_debug_pass_trace(env._h, full.ctypes.data_as(C.c_void_p), full.size))
    buf = full[:NT * 8 + 4 * EB]
    ks0, ks1 = int(full[-2]), int(full[-1])                     # k_step: earliest block entry, latest warp exit
    tr = buf[:NT * 8].reshape(NT, 8)
    ep = buf[NT * 8:].reshape(EB, 4).astype(np.int64)
    ep = ep[ep[:, 0] > 0]
    slow = (tr[:, 3] >> np.uint64(63)).astype(bool)
    sm = tr[:, 5].astype(np.int64)
    tr = (tr & np.uint64((1 << 63) - 1)).astype(np.int64)
    t0 = tr[:, 0].min()
    t = (tr - t0) / 1e3
    line = "pass %d: k_step %.1f us, gap to first obs block %.1f us; k_obs_tile span %.1f us (%d of %d tiles copied env by env)" % (
        p, (ks1 - ks0) / 1e3, (int(t0) - ks1) / 1e3, t[:, 3].max(), int(slow.sum()), NT)
    if p > 0:
        line += "; previous pass end -> this k_step start %.1f us" % ((ks0 - prev_end) / 1e3)
    prev_end = int(t0) + int(t[:, 3].max() * 1e3)
    if len(ep):
        e0, e1 = (ep[:, 0] - t0) / 1e3, (ep[:, 1] - t0) / 1e3
        per_sm = np.bincount(ep[:, 2], minlength=148)
        line += "; k_episode_list %d blocks with work, enter %.1f, last exit %.1f us, per SM min/median/max %d/%d/%d" % (
            len(ep), e0.min(), e1.max(), per_sm.min(), int(np.median(per_sm)), per_sm.max())
        # obs blocks resident per SM at the middle of the episode kernel's life
        mid = 0.5 * (e0.min() + e1.max())
        res = np.bincount(sm[(t[:, 0] <= mid) & (t[:, 3] > mid)], minlength=148)
        line += "; obs blocks resident per SM at t=%.0f us: %s" % (mid, dict(zip(*np.unique(res, return_counts=True))))
    print(line)
print("B", B, "tiles", NT, "last pass:")
print("entry                 p0/10/50/90/99/100", pc(t[:, 0]))
print("scalars landed - entry                  ", pc(t[:, 1] - t[:, 0]))
print("copies landed - entry                   ", pc(t[:, 4] - t[:, 0]))
print("rows staged - entry                     ", pc(t[:, 2] - t[:, 0]))
print("outputs read - rows staged  (bulk)      ", pc((t[:, 3] - t[:, 2])[~slow]))
if slow.any(): print("outputs written - rows staged (by env)  ", pc((t[:, 3] - t[:, 2])[slow]))
print("block lifetime                          ", pc(t[:, 3] - t[:, 0]))
if len(ep):
    print("episode block lifetime                  ", pc(e1 - e0))
