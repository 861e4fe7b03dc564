"""oracle/oracle.py -- ctypes front end of the CPU checker (oracle/taskenv_oracle.c).

TEST INFRASTRUCTURE ONLY.  May be imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py; never by dcmrta_b200/.

`OracleEnv` mirrors the slice of the reference TaskEnv API the callers use
(/root/reference/env/task_env.py; worker.py:45-87) on top of the C restatement, and adds the
fused one-call-per-decision driver (`fused_reset` / `fused_step`) that the CUDA step kernel is
compared against.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB = None


def build(force: bool = False) -> Path:
    """Compile oracle/liboracle.so with gcc (seconds).  Building the checker is not using it."""
    so = _HERE / "liboracle.so"
    src = _HERE / "taskenv_oracle.c"
    if force or not so.exists() or so.stat().st_mtime < src.stat().st_mtime:
        subprocess.run(["make", "-C", str(_HERE), "-s", "-B", "liboracle.so"], check=True)
    return so


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        L = C.CDLL(str(build()))
        vp, i32, f64, u64, u32 = C.c_void_p, C.c_int, C.c_double, C.c_uint64, C.c_uint32
        P = C.POINTER
        sig = {
            "orc_create": (vp, [i32, i32, vp, vp, vp, vp, f64, f64, f64]),
            "orc_destroy": (None, [vp]),
            "orc_clear_decisions": (None, [vp]),
            "orc_set_max_wait": (None, [vp, f64]),
            "orc_set_now": (None, [vp, f64]),
            "orc_get_now": (f64, [vp]),
            "orc_set_finished": (None, [vp, i32]),
            "orc_next_decision": (i32, [vp, vp, P(f64)]),
            "orc_get_unique_group": (i32, [vp, vp, i32, vp, vp]),
            "orc_task_update": (i32, [vp, vp]),
            "orc_agent_update": (None, [vp]),
            "orc_agent_step": (f64, [vp, i32, i32]),
            "orc_vacancy": (i32, [vp, i32, i32]),
            "orc_step_members": (f64, [vp, vp, i32, i32]),
            "orc_mask": (None, [vp, vp]),
            "orc_agent_status": (None, [vp, i32, vp]),
            "orc_task_status": (None, [vp, i32, vp]),
            "orc_check_finished": (i32, [vp]),
            "orc_calculate_waiting_time": (None, [vp]),
            "orc_episode_metrics": (None, [vp, vp, vp]),
            "orc_pre_set_route": (None, [vp, i32, vp, i32]),
            "orc_execute_by_route": (f64, [vp]),
            "orc_export": (None, [vp, i32] + [vp] * 18),
            "orc_route_len": (i32, [vp, i32]),
            "orc_route": (None, [vp, i32, vp, vp]),
            "orc_agent_scalars": (None, [vp, vp, vp]),
            "orc_philox": (None, [vp, vp, vp]),
            "orc_np_sum": (f64, [vp, i32]),
            "orc_seed": (None, [vp, u64, u64, u32]),
            "orc_fused_reset": (i32, [vp, i32]),
            "orc_policy_action": (i32, [vp, i32]),
            "orc_fused_step": (i32, [vp, i32, vp, i32, i32, P(f64), P(i32), P(i32), vp, P(i32)]),
            "orc_leader": (i32, [vp]),
            "orc_done": (i32, [vp]),
            "orc_stuck": (i32, [vp]),
            "orc_pending": (u64, [vp]),
            "orc_current_group": (u64, [vp]),
            "orc_nsteps": (C.c_long, [vp]),
            "orc_rollout_bench": (C.c_long, [vp, i32, C.c_long, u64, vp]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _LIB = L
    return _LIB


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


METRIC_NAMES = ("reward", "success_rate", "makespan", "time_cost", "waiting_time", "travel_dist", "efficiency", "n_steps")


class OracleEnv:
    """One environment instance held by the C oracle."""

    def __init__(self, task_xy, depot_xy, req, dur, velocity=0.2, max_wait=10.0, max_time=100.0):
        self.task_xy = np.ascontiguousarray(task_xy, dtype=np.float64).reshape(-1, 2)
        self.depot_xy = np.ascontiguousarray(depot_xy, dtype=np.float64).reshape(2)
        self.req = np.ascontiguousarray(req, dtype=np.int32).reshape(-1)
        self.dur = np.ascontiguousarray(dur, dtype=np.float64).reshape(-1)
        self.T = self.task_xy.shape[0]
        self.A = None
        self._h = None
        self._args = (velocity, max_wait, max_time)

    @classmethod
    def make(cls, A, task_xy, depot_xy, req, dur, velocity=0.2, max_wait=10.0, max_time=100.0):
        self = cls(task_xy, depot_xy, req, dur, velocity, max_wait, max_time)
        self.A = int(A)
        self._h = lib().orc_create(self.A, self.T, _p(self.task_xy), _p(self.depot_xy), _p(self.req), _p(self.dur),
                                   velocity, max_wait, max_time)
        if not self._h:
            raise ValueError("orc_create failed (bad A/T)")
        return self

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_destroy(self._h)
            self._h = None

    # ---- reference-shaped API -------------------------------------------------
    tasks_num = property(lambda s: s.T)
    agents_num = property(lambda s: s.A)

    @property
    def current_time(self):
        return lib().orc_get_now(self._h)

    @current_time.setter
    def current_time(self, t):
        lib().orc_set_now(self._h, float(t))

    def set_max_wait(self, w):
        lib().orc_set_max_wait(self._h, float(w))

    def clear_decisions(self):
        lib().orc_clear_decisions(self._h)

    def next_decision(self):
        ids = np.zeros(64, np.int32)
        t = C.c_double()
        n = lib().orc_next_decision(self._h, _p(ids), C.byref(t))
        return ids[:n].copy(), t.value

    def get_unique_group(self, ids):
        ids = np.ascontiguousarray(ids, np.int32)
        out = np.zeros(max(len(ids), 1), np.int32)
        sizes = np.zeros(max(len(ids), 1), np.int32)
        ng = lib().orc_get_unique_group(self._h, _p(ids), len(ids), _p(out), _p(sizes))
        groups, o = [], 0
        for g in range(ng):
            groups.append(out[o:o + sizes[g]].tolist())
            o += sizes[g]
        return groups

    def task_update(self):
        newly = np.zeros(self.T, np.int32)
        n = lib().orc_task_update(self._h, _p(newly))
        return newly[:n].tolist()

    def agent_update(self):
        lib().orc_agent_update(self._h)

    def agent_step(self, agent_id, action):
        return lib().orc_agent_step(self._h, int(agent_id), int(action))

    def vacancy(self, action, group_len):
        return lib().orc_vacancy(self._h, int(action), int(group_len))

    def step_members(self, members, action):
        m = np.ascontiguousarray(members, np.int32)
        return lib().orc_step_members(self._h, _p(m), len(m), int(action))

    def mask(self):
        m = np.zeros(self.T + 1, np.uint8)
        lib().orc_mask(self._h, _p(m))
        return m

    def agent_status(self, leader):
        out = np.zeros((self.A, 6), np.float64)
        lib().orc_agent_status(self._h, int(leader), _p(out))
        return out

    def task_status(self, leader):
        out = np.zeros((self.T + 1, 5), np.float64)
        lib().orc_task_status(self._h, int(leader), _p(out))
        return out

    def check_finished(self):
        return bool(lib().orc_check_finished(self._h))

    def episode_metrics(self):
        out = np.zeros(8, np.float64)
        fin = np.zeros(self.T, np.uint8)
        lib().orc_episode_metrics(self._h, _p(out), _p(fin))
        return dict(zip(METRIC_NAMES, out.tolist())), fin

    def pre_set_route(self, routes, agent_id):
        r = np.ascontiguousarray(routes, np.int32)
        lib().orc_pre_set_route(self._h, int(agent_id), _p(r), len(r))

    def execute_by_route(self):
        return lib().orc_execute_by_route(self._h)

    def export(self, MC=None):
        MC = int(MC or self.A)
        T, A = self.T, self.A
        d = dict(
            n_mem=np.zeros(T, np.int32), members=np.zeros((T, MC), np.int32), mem_arr=np.zeros((T, MC), np.float64),
            status=np.zeros(T, np.int32), feasible=np.zeros(T, np.uint8), finished=np.zeros(T, np.uint8),
            time_start=np.zeros(T, np.float64), time_finish=np.zeros(T, np.float64), n_aband_task=np.zeros(T, np.int32),
            node=np.zeros(A, np.int32), has_route=np.zeros(A, np.uint8), last_arrival=np.zeros(A, np.float64),
            next_decision=np.zeros(A, np.float64), travel_dist=np.zeros(A, np.float64), assigned=np.zeros(A, np.uint8),
            returned=np.zeros(A, np.uint8), n_aband_agent=np.zeros(A, np.int32), now_finished=np.zeros(2, np.float64))
        lib().orc_export(self._h, MC, *[_p(v) for v in d.values()])
        d["now"] = d["now_finished"][0]
        d["env_finished"] = bool(d.pop("now_finished")[1])
        return d

    def routes(self):
        out = []
        for a in range(self.A):
            n = lib().orc_route_len(self._h, a)
            r = np.zeros(max(n, 1), np.int32)
            t = np.zeros(max(n, 1), np.float64)
            lib().orc_route(self._h, a, _p(r), _p(t))
            out.append((r[:n].copy(), t[:n].copy()))
        return out

    def agent_scalars(self):
        """-> (agent sum_waiting_time [A], task sum_waiting_time [T]) as the last calculate_waiting_time (task_env.py:344-364) left them"""
        aw, tw = np.zeros(self.A, np.float64), np.zeros(self.T, np.float64)
        lib().orc_agent_scalars(self._h, _p(aw), _p(tw))
        return aw, tw

    # ---- fused driver ---------------------------------------------------------
    def seed(self, seed, gid=0, episode=0):
        lib().orc_seed(self._h, int(seed), int(gid), int(episode))

    def fused_reset(self, leader=-1):
        return lib().orc_fused_reset(self._h, int(leader))

    def policy_action(self, policy):
        return lib().orc_policy_action(self._h, int(policy))

    def fused_step(self, action, followers=None, next_leader=-1):
        """-> (rc, reward, done, used_action, members)"""
        r, d, ua, nm = C.c_double(), C.c_int(), C.c_int(), C.c_int()
        mem = np.zeros(64, np.int32)
        if followers is None:
            fp, nf = None, 0
        else:
            f = np.ascontiguousarray(followers, np.int32)
            fp, nf = _p(f), len(f)
        rc = lib().orc_fused_step(self._h, int(action), fp, nf, int(next_leader), C.byref(r), C.byref(d), C.byref(ua),
                                  _p(mem), C.byref(nm))
        return rc, r.value, bool(d.value), ua.value, mem[:nm.value].tolist()

    leader = property(lambda s: lib().orc_leader(s._h))
    done = property(lambda s: bool(lib().orc_done(s._h)))
    stuck = property(lambda s: bool(lib().orc_stuck(s._h)))
    pending = property(lambda s: int(lib().orc_pending(s._h)))
    n_steps = property(lambda s: int(lib().orc_nsteps(s._h)))

    def current_group(self):
        """bitmask of the group that decides now: the pending agents at the lexicographically smallest location (task_env.py:291-298)"""
        return int(lib().orc_current_group(self._h))

    def rollout_bench(self, policy, min_steps, seed=0):
        return int(lib().orc_rollout_bench(self._h, int(policy), int(min_steps), int(seed), None))


def philox(ctr, key):
    c = np.ascontiguousarray(ctr, np.uint32)
    k = np.ascontiguousarray(key, np.uint32)
    o = np.zeros(4, np.uint32)
    lib().orc_philox(_p(c), _p(k), _p(o))
    return o


def np_sum(a):
    """the oracle's restatement of np.add.reduce on a float64 vector (pairwise summation)"""
    a = np.ascontiguousarray(a, np.float64)
    return lib().orc_np_sum(_p(a), len(a))


def synthetic_instance(A, T, M, seed, max_duration=5.0, random_duration=False):
    """Host-side synthetic instance with the generator's distributions (task_env.py:66-71): depot, task xy ~ U[0,1)^2,
    requirement ~ U{1..M}, duration = max_duration (or U(0,max_duration) like the bundled pickles)."""
    rng = np.random.default_rng(seed)
    depot = rng.random(2)
    xy = rng.random((T, 2))
    req = rng.integers(1, M + 1, T).astype(np.int32)
    dur = rng.random(T) * max_duration if random_duration else np.full(T, float(max_duration))
    return dict(A=A, task_xy=xy, depot_xy=depot, req=req, dur=dur)
