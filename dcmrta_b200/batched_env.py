"""dcmrta_b200/batched_env.py -- device-resident batch of TaskEnv instances (host side of the hot path).

`BatchedTaskEnv` owns one dcm_env handle (include/dcmrta.h) and the policy-input tensors the step kernel writes
into: agent rows [B,A,6] fp32, task rows [B,T+1,5] fp32, mask [B,T+1] bool -- exactly what
AttentionNet.forward(tasks, agents, mask) consumes (reference attention.py:288, worker.py:62-69).  One `step()`
is one leader decision for every env (reference worker.py:45-85) -- or, with protocol="IA", one individual decision
(worker.py:159-198 run_test_IS: every decider acts alone, in ascending id order).  PyTorch is used only for device memory and
streams; all simulation work happens in the CUDA library.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import POLICY, check, lib

METRIC_NAMES = ("reward", "success_rate", "makespan", "time_cost", "waiting_time", "travel_dist", "efficiency", "n_steps")

_LAYOUT_KEYS = ("A", "T", "M", "MC", "Tp", "Ap", "o_arr", "o_tstart", "o_alast", "o_and", "o_adist", "o_hdr", "o_tnab", "o_anab",
                "o_mem", "o_nmem", "o_status", "o_tflags", "o_anode", "o_aflags", "dyn_bytes",
                "s_tx", "s_ty", "s_dur", "s_depot", "s_req", "sta_bytes", "stage_bytes", "warps_per_cta")

_HDR_DTYPE = np.dtype([("now", "<f8"), ("pending", "<u8"), ("group", "<u8"), ("n_steps", "<u4"), ("episode", "<u4"),
                       ("leader", "<i4"), ("flags", "<u4"), ("instance", "<u4"), ("total_steps", "<u4")])


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


class BatchedTaskEnv:
    """B environments of A agents / T tasks stepped in lock-step on one GPU.

    protocol: "LF" leader-follower (worker.py:45-85, what training plays) or "IA" individual agent (worker.py:159-198,
    DCM_FLAG_INDIVIDUAL): `leader` is then the agent that acts next, followers must not be given, and an episode takes one
    step per individual decision: with the greedy policy on the bundled 20A/50T instances 185 on average (at most 259) against
    99 (at most 190) under LF, so size rollout horizons accordingly."""

    def __init__(self, B, A, T, M=5, device=0, auto_reset=False, regenerate=False, velocity=0.2, max_wait=10.0,
                 max_time=100.0, seed=0, first_gid=0, protocol="LF"):
        if protocol not in _lib.PROTOCOL:
            raise ValueError(f"protocol must be 'LF' or 'IA', not {protocol!r}")
        if not torch.cuda.is_available():
            raise _lib.DcmError(-3, "BatchedTaskEnv needs a CUDA device; there is no CPU fallback")
        self.B, self.A, self.T, self.M = int(B), int(A), int(T), int(M)
        self.device = torch.device("cuda", int(device) if not isinstance(device, torch.device) else device.index or 0)
        self.auto_reset = bool(auto_reset)
        self.protocol = protocol
        flags = (_lib.FLAG_AUTO_RESET if auto_reset else 0) | (_lib.FLAG_REGENERATE if regenerate else 0) | _lib.PROTOCOL[protocol]
        h = C.c_void_p()
        check(lib().dcm_create(C.byref(h), self.device.index, self.B, self.A, self.T, self.M, flags))
        self._h = h
        self.set_params(velocity, max_wait, max_time)
        self.seed(seed, first_gid)
        lay = (C.c_int32 * len(_LAYOUT_KEYS))()
        lib().dcm_layout(self._h, lay, len(_LAYOUT_KEYS))
        self.layout = dict(zip(_LAYOUT_KEYS, list(lay)))
        dev = self.device
        # policy input buffers (written in place by every reset/step)
        self.agent_obs = torch.zeros(self.B, self.A, 6, dtype=torch.float32, device=dev)
        self.task_obs = torch.zeros(self.B, self.T + 1, 5, dtype=torch.float32, device=dev)
        self.mask_u8 = torch.ones(self.B, self.T + 1, dtype=torch.uint8, device=dev)
        self.leader = torch.full((self.B,), -1, dtype=torch.int32, device=dev)
        self.reward = torch.zeros(self.B, dtype=torch.float32, device=dev)
        self.done_u8 = torch.zeros(self.B, dtype=torch.uint8, device=dev)
        self.used_action = torch.full((self.B,), -1, dtype=torch.int32, device=dev)
        self._keep = []

    # ---- lifetime ---------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            lib().dcm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_output_buffers(self, agent_obs=None, task_obs=None, mask_u8=None):
        """Make reset()/step() write the next observation straight into caller-owned tensors (e.g. the slot of an episode
        buffer, dcmrta_b200/rollout.py): fp32 [B,A,6], fp32 [B,T+1,5], uint8 [B,T+1], contiguous, on this device."""
        for name, t, shape, dt in (("agent_obs", agent_obs, (self.B, self.A, 6), torch.float32),
                                   ("task_obs", task_obs, (self.B, self.T + 1, 5), torch.float32),
                                   ("mask_u8", mask_u8, (self.B, self.T + 1), torch.uint8)):
            if t is None:
                continue
            if tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous() or t.device != self.device:
                raise _lib.DcmError(-1, f"set_output_buffers: {name} must be a contiguous {dt} tensor of shape {shape} on {self.device}")
            setattr(self, name, t)

    @property
    def mask(self):
        """bool view of the mask buffer, True = forbidden (reference worker.py:57-61)."""
        return self.mask_u8.view(torch.bool)

    @property
    def done(self):
        return self.done_u8.view(torch.bool)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, x, dtype):
        """numpy / tensor -> contiguous device tensor of dtype (None passes through)."""
        if x is None:
            return None
        t = torch.as_tensor(x)
        t = t.to(device=self.device, dtype=dtype).contiguous()
        return t

    # ---- configuration ---------------------------------------------------------------------------------------
    def set_params(self, velocity=0.2, max_wait=10.0, max_time=100.0):
        check(lib().dcm_set_params(self._h, float(velocity), float(max_wait), float(max_time)))
        self.velocity, self.max_wait, self.max_time = float(velocity), float(max_wait), float(max_time)

    def seed(self, seed, first_gid=0):
        check(lib().dcm_seed(self._h, int(seed), int(first_gid)))
        self.first_gid = int(first_gid)                  # global id of env 0, which the policy's action sampler keys its draws by too

    def load_instances(self, task_xy, depot_xy, req, dur):
        """reset(test_env=...) of the reference (task_env.py:116-127) for the whole batch.  Arrays [B,T,2], [B,2], [B,T], [B,T]."""
        xy = self._dev(task_xy, torch.float64).reshape(self.B, self.T, 2)
        dp = self._dev(depot_xy, torch.float64).reshape(self.B, 2)
        rq = self._dev(req, torch.int32).reshape(self.B, self.T)
        du = self._dev(dur, torch.float64).reshape(self.B, self.T)
        if int(rq.min()) < 1 or int(rq.max()) > self.M:
            raise _lib.DcmError(-1, "requirements must lie in [1, M]")
        check(lib().dcm_load_instances(self._h, _ptr(xy), _ptr(dp), _ptr(rq), _ptr(du), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()     # inputs may be freed after return

    def generate(self, max_duration=5.0, random_duration=False):
        """generate_env (task_env.py:57-114) distributions, on device."""
        check(lib().dcm_generate(self._h, float(max_duration), int(bool(random_duration)), self._stream()))

    def get_instances(self):
        dev = self.device
        xy = torch.empty(self.B, self.T, 2, dtype=torch.float64, device=dev)
        dp = torch.empty(self.B, 2, dtype=torch.float64, device=dev)
        rq = torch.empty(self.B, self.T, dtype=torch.int32, device=dev)
        du = torch.empty(self.B, self.T, dtype=torch.float64, device=dev)
        check(lib().dcm_get_instances(self._h, _ptr(xy), _ptr(dp), _ptr(rq), _ptr(du), self._stream()))
        return dict(task_xy=xy, depot_xy=dp, req=rq, dur=du)

    # ---- fused path ------------------------------------------------------------------------------------------
    def reset(self, which=None, leaders=None):
        """clear_decisions + first slot + first leader + its observation.  Returns (agent_obs, task_obs, mask, leader)."""
        w = self._dev(which, torch.uint8)
        l = self._dev(leaders, torch.int32)
        check(lib().dcm_reset(self._h, _ptr(w), _ptr(l), _ptr(self.agent_obs), _ptr(self.task_obs), _ptr(self.mask_u8),
                              _ptr(self.leader), self._stream()))
        self._keep = [w, l]
        # dcm_reset does not write the per-step outputs: a restarted env is not done and has earned nothing yet
        if w is None:
            self.done_u8.zero_(); self.reward.zero_()
        else:
            sel = w.view(torch.bool)
            self.done_u8.masked_fill_(sel, 0); self.reward.masked_fill_(sel, 0.0)
        return self.agent_obs, self.task_obs, self.mask, self.leader

    def step(self, actions=None, followers=None, next_leaders=None, policy="external"):
        """One leader decision per env.  actions [B] int32 (0 = depot, j+1 = task j).
        Returns (agent_obs, task_obs, mask, next_leader, reward, done) -- views of the persistent buffers."""
        a = self._dev(actions, torch.int32)
        f = self._dev(followers, torch.int32)
        nl = self._dev(next_leaders, torch.int32)
        fstride = 0
        if f is not None:
            f = f.reshape(self.B, -1)
            fstride = f.shape[1]
        check(lib().dcm_step(self._h, _ptr(a), _ptr(f), fstride, _ptr(nl), POLICY[policy] if isinstance(policy, str) else int(policy),
                             _ptr(self.agent_obs), _ptr(self.task_obs), _ptr(self.mask_u8), _ptr(self.leader), _ptr(self.reward),
                             _ptr(self.done_u8), _ptr(self.used_action), self._stream()))
        self._keep = [a, f, nl]          # keep inputs alive until the stream has consumed them
        return self.agent_obs, self.task_obs, self.mask, self.leader, self.reward, self.done

    def step_host(self, actions, out, policy="external"):
        """dcm_step_host: host buffers in, host buffers out (numpy arrays or pinned tensors), synchronous.
        out: dict with optional keys agent_obs, task_obs, mask, next_leader, reward, done (preallocated, C-contiguous)."""
        def hp(x):
            if x is None:
                return None
            if isinstance(x, torch.Tensor):
                return C.c_void_p(x.data_ptr())
            return x.ctypes.data_as(C.c_void_p)
        check(lib().dcm_step_host(self._h, hp(actions), POLICY[policy] if isinstance(policy, str) else int(policy),
                                  hp(out.get("agent_obs")), hp(out.get("task_obs")), hp(out.get("mask")),
                                  hp(out.get("next_leader")), hp(out.get("reward")), hp(out.get("done"))))
        return out

    def episode_metrics(self):
        """[B,8] fp64: reward, success_rate, makespan, time_cost, waiting_time, travel_dist, efficiency, decisions of the last finished episode."""
        out = torch.empty(self.B, 8, dtype=torch.float64, device=self.device)
        check(lib().dcm_episode_metrics(self._h, _ptr(out), self._stream()))
        return out

    # ---- granular path (the individual TaskEnv methods, batched) ------------------------------------------------
    def next_decision(self):
        d = torch.empty(self.B, dtype=torch.int64, device=self.device)
        t = torch.empty(self.B, dtype=torch.float64, device=self.device)
        check(lib().dcm_next_decision(self._h, _ptr(d), _ptr(t), self._stream()))
        return d, t

    def unique_group(self, deciders):
        d = self._dev(deciders, torch.int64)
        r = torch.empty(self.B, self.A, dtype=torch.int8, device=self.device)
        check(lib().dcm_unique_group(self._h, _ptr(d), _ptr(r), self._stream()))
        return r

    def set_clock(self, t):
        tt = self._dev(t, torch.float64).reshape(self.B)
        check(lib().dcm_set_clock(self._h, _ptr(tt), self._stream()))
        self._keep = [tt]

    def get_clock(self):
        t = torch.empty(self.B, dtype=torch.float64, device=self.device)
        check(lib().dcm_get_clock(self._h, _ptr(t), self._stream()))
        return t

    def task_update(self, want_newly=False):
        n = torch.zeros(self.B, self.T, dtype=torch.uint8, device=self.device) if want_newly else None
        check(lib().dcm_task_update(self._h, _ptr(n), self._stream()))
        return n

    def agent_update(self):
        check(lib().dcm_agent_update(self._h, self._stream()))

    def apply_members(self, actions, members, n_members):
        a = self._dev(actions, torch.int32).reshape(self.B)
        m = self._dev(members, torch.int32).reshape(self.B, -1)
        n = self._dev(n_members, torch.int32).reshape(self.B)
        r = torch.zeros(self.B, dtype=torch.float64, device=self.device)
        check(lib().dcm_apply_members(self._h, _ptr(a), _ptr(m), m.shape[1], _ptr(n), _ptr(r), self._stream()))
        self._keep = [a, m, n]
        return r

    def build_obs(self, leaders):
        l = self._dev(leaders, torch.int32).reshape(self.B)
        check(lib().dcm_build_obs(self._h, _ptr(l), _ptr(self.agent_obs), _ptr(self.task_obs), _ptr(self.mask_u8), self._stream()))
        self._keep = [l]
        return self.agent_obs, self.task_obs, self.mask

    def check_finished(self):
        f = torch.empty(self.B, dtype=torch.uint8, device=self.device)
        check(lib().dcm_check_finished(self._h, _ptr(f), self._stream()))
        return f.view(torch.bool)

    def compute_metrics(self, per_element=False):
        """get_episode_reward + worker.py:103-108 now.  per_element=True also returns the task / agent sum_waiting_time arrays."""
        out = torch.empty(self.B, 8, dtype=torch.float64, device=self.device)
        tw = torch.zeros(self.B, self.T, dtype=torch.float64, device=self.device) if per_element else None
        aw = torch.zeros(self.B, self.A, dtype=torch.float64, device=self.device) if per_element else None
        check(lib().dcm_compute_metrics(self._h, _ptr(out), _ptr(tw), _ptr(aw), self._stream()))
        return (out, tw, aw) if per_element else out

    def execute_by_route(self, routes, route_len):
        """pre_set_route + execute_by_route (task_env.py:562-599).  routes [B,A,L] int32 actions, route_len [B,A]."""
        r = self._dev(routes, torch.int32).reshape(self.B, self.A, -1)
        n = self._dev(route_len, torch.int32).reshape(self.B, self.A)
        mk = torch.empty(self.B, dtype=torch.float64, device=self.device)
        check(lib().dcm_execute_by_route(self._h, _ptr(r), r.shape[2], _ptr(n), _ptr(mk), self._stream()))
        self._keep = [r, n]
        return mk

    # ---- inspection --------------------------------------------------------------------------------------------
    def env_flags(self):
        f = torch.empty(self.B, dtype=torch.int32, device=self.device)
        check(lib().dcm_env_flags(self._h, _ptr(f), self._stream()))
        return f

    def total_steps(self):
        out = C.c_uint64()
        check(lib().dcm_total_steps(self._h, C.byref(out)))
        return out.value

    def total_episodes(self):
        out = C.c_uint64()
        check(lib().dcm_total_episodes(self._h, C.byref(out)))
        return out.value

    def launch_count(self):
        return int(lib().dcm_launch_count(self._h))

    def algorithmic_bytes_per_step(self):
        return int(lib().dcm_algorithmic_bytes_per_step(self._h))

    def record_bytes(self):
        return int(lib().dcm_record_bytes(self._h))

    def export_raw(self):
        """Raw dynamic records as a [B, record_bytes] uint8 numpy array (synchronises)."""
        n = self.record_bytes()
        buf = torch.empty(self.B, n, dtype=torch.uint8, device=self.device)
        check(lib().dcm_export_state(self._h, _ptr(buf), self.B * n, self._stream()))
        return buf.cpu().numpy()

    def import_raw(self, raw):
        t = self._dev(raw, torch.uint8).reshape(self.B, self.record_bytes())
        check(lib().dcm_import_state(self._h, _ptr(t), t.numel(), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def export_state(self, envs=None):
        """Decode the records into flat per-env dicts (same field names as the reference's live state, SURVEY App. A)."""
        raw = self.export_raw()
        dur = self.get_instances()["dur"].cpu().numpy()
        return [decode_record(raw[b], self.layout, dur[b]) for b in (range(self.B) if envs is None else envs)]


def decode_record(rec: np.ndarray, L: dict, dur) -> dict:
    """One raw dynamic record and its env's task durations [T] -> dict of arrays: n_mem, members[T,MC] (-1 pad), mem_arr, status,
    feasible, finished, time_start, time_finish (time_start + duration once feasible, else 0; task_env.py:257), n_aband_task,
    node (-1 = depot), has_route, last_arrival, next_decision, travel_dist, assigned, returned, n_aband_agent, now, and the
    header fields."""
    A, T, MC, Tp, Ap = L["A"], L["T"], L["MC"], L["Tp"], L["Ap"]
    rec = np.ascontiguousarray(rec, dtype=np.uint8)

    def arr(off, dtype, count):
        return np.frombuffer(rec, dtype=dtype, count=count, offset=off)

    n_mem = arr(L["o_nmem"], np.uint8, Tp)[:T].astype(np.int32)
    mem = arr(L["o_mem"], np.uint8, MC * Tp).reshape(MC, Tp)[:, :T].T.astype(np.int32)
    marr = arr(L["o_arr"], np.float64, MC * Tp).reshape(MC, Tp)[:, :T].T.copy()
    slot = np.arange(MC)[None, :]
    valid = slot < n_mem[:, None]
    mem = np.where(valid, mem, -1)
    marr = np.where(valid, marr, 0.0)
    tflags = arr(L["o_tflags"], np.uint8, Tp)[:T]
    aflags = arr(L["o_aflags"], np.uint8, Ap)[:A]
    node = arr(L["o_anode"], np.uint8, Ap)[:A].astype(np.int32)
    node = np.where(node == 0xFF, -1, node)
    feasible = (tflags & 1).astype(np.uint8)
    time_start = arr(L["o_tstart"], np.float64, Tp)[:T].copy()
    hdr = np.frombuffer(rec, dtype=_HDR_DTYPE, count=1, offset=L["o_hdr"])[0]
    return dict(
        n_mem=n_mem, members=mem, mem_arr=marr,
        status=arr(L["o_status"], np.int8, Tp)[:T].astype(np.int32),
        feasible=feasible, finished=((tflags >> 1) & 1).astype(np.uint8),
        time_start=time_start, time_finish=np.where(feasible > 0, time_start + np.asarray(dur, np.float64), 0.0),
        n_aband_task=arr(L["o_tnab"], np.uint16, Tp)[:T].astype(np.int32),
        node=node, has_route=(aflags & 1).astype(np.uint8),
        last_arrival=arr(L["o_alast"], np.float64, Ap)[:A].copy(),
        next_decision=arr(L["o_and"], np.float64, Ap)[:A].copy(),
        travel_dist=arr(L["o_adist"], np.float64, Ap)[:A].copy(),
        assigned=((aflags >> 1) & 1).astype(np.uint8), returned=((aflags >> 2) & 1).astype(np.uint8),
        n_aband_agent=arr(L["o_anab"], np.uint16, Ap)[:A].astype(np.int32),
        now=float(hdr["now"]), pending=int(hdr["pending"]), group=int(hdr["group"]), n_steps=int(hdr["n_steps"]),
        episode=int(hdr["episode"]), leader=int(hdr["leader"]), flags=int(hdr["flags"]), instance=int(hdr["instance"]),
        total_steps=int(hdr["total_steps"]))
