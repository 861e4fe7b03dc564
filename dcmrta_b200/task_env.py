"""dcmrta_b200/task_env.py -- drop-in replacement of the reference class `TaskEnv` (env/task_env.py:8-623).

Same constructor, methods, attributes and return conventions as the reference, so that the reference's callers
(worker.py:45-87 / :114-235, RL_test.py:34-48, baselines/CTAS-D.py:60-80, TestSetGenerator.py:17-51) run unchanged:

    from dcmrta_b200.task_env import TaskEnv          # instead of: from env.task_env import TaskEnv

Every simulation method is one launch of the corresponding batched CUDA op on a batch of ONE env (the granular part of
include/dcmrta.h); there is no CPU simulation code here.  Host-side work is limited to what the reference also does on
the host outside the simulator proper: drawing the instance with the reference's RNG call order (task_env.py:57-71),
drawing followers with `random_choice` (task_env.py:331), and presenting device state as the dict-of-dicts the callers
index (`agent_dic[i]['returned']`, `get_matrix(task_dic, 'time_start')`, ...).  For throughput use BatchedTaskEnv; this
class exists for API compatibility and costs a kernel launch + a device->host read per call.

Not provided (out of scope, SURVEY.md 2 rows 3-4): plotting / gif / trajectory / process_map, get_grouped_tasks,
reactive_planning=True.
"""
from __future__ import annotations

import copy

import numpy as np
import torch

from .batched_env import BatchedTaskEnv, decode_record

_STATIC_TASK_KEYS = ("ID", "requirements", "location", "time", "cost", "efficiency")
_AGENT_HOST_KEYS = ("current_action_index", "pre_set_route", "cost", "abilities", "velocity", "working_condition", "trajectory", "angle")


def generate_instance(agents_range, tasks_range, max_coalition_size, max_duration, rng=None):
    """generate_env (task_env.py:57-71): the same draws in the same order as the reference, so that a given seed yields the
    same instance.  rng: np.random.Generator, or None for the global NumPy state (task_env.py:36-48).
    Returns (A, task_xy[T,2], depot_xy[2], req[T], dur[T], cost[A,1])."""
    rint = (lambda lo, hi, size=None: rng.integers(lo, hi, size)) if rng is not None else (lambda lo, hi, size=None: np.random.randint(lo, hi, size))
    rval = (lambda r, c: rng.random((r, c))) if rng is not None else (lambda r, c: np.random.rand(r, c))
    tasks_num = rint(tasks_range[0], tasks_range[1] + 1) if type(tasks_range) is tuple else tasks_range
    agents_num = rint(agents_range[0], agents_range[1] + 1) if type(agents_range) is tuple else agents_range
    depot = rval(1, 2)
    cost_ini = rval(int(agents_num), 1)
    tasks_loc = rval(int(tasks_num), 2)
    tasks_time = np.ones(int(tasks_num)) * max_duration
    req = rint(1, max_coalition_size + 1, int(tasks_num))
    return int(agents_num), tasks_loc, depot[0], np.asarray(req).reshape(-1), tasks_time, cost_ini


class _Row:
    """dict-like view of one task / agent / the depot: reads come from the decoded device state, writes to host-only keys."""

    def __init__(self, env, kind, idx):
        self._env, self._kind, self._idx = env, kind, idx

    def __getitem__(self, key):
        return self._env._get(self._kind, self._idx, key)

    def __setitem__(self, key, value):
        self._env._set(self._kind, self._idx, key, value)

    def get(self, key, default=None):
        try:
            return self[key]
        except KeyError:
            return default

    def update(self, **kw):
        for k, v in kw.items():
            self[k] = v

    def keys(self):
        return self._env._keys(self._kind)

    def __contains__(self, key):
        return key in self.keys()

    def items(self):
        return [(k, self[k]) for k in self.keys()]


class _Table(dict):
    """task_dic / agent_dic: id -> _Row (a real dict, so len(), .values(), .keys(), `in` behave as in the reference)."""


class TaskEnv:
    def __init__(self, agents_range=(10, 10), tasks_range=(10, 10), traits_dim=1, max_coalition_size=3, max_duration=5,
                 seed=None, plot_figure=False, device=0):
        self.rng = None
        self.agents_range = agents_range
        self.tasks_range = tasks_range
        self.max_coalition_size = max_coalition_size
        self.max_duration = max_duration
        self.plot_figure = plot_figure
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.traits_dim = traits_dim
        if traits_dim != 1:
            raise NotImplementedError("traits_dim != 1 does not work in the reference either (task_env.py:71, :254)")
        self._device = device
        self._be = None
        self._cache = None
        self._install(*self._generate_instance())
        self.dt = 0.1
        self._max_waiting_time = 10
        self.finished = False
        self.force_wait = True
        self.reactive_planning = False
        self.visible_length = 0
        self._sync_params()

    # ---- reference RNG helpers (task_env.py:36-55) ---------------------------------------------------------------
    def random_int(self, low, high, size=None):
        return self.rng.integers(low, high, size) if self.rng is not None else np.random.randint(low, high, size)

    def random_value(self, row, col):
        return self.rng.random((row, col)) if self.rng is not None else np.random.rand(row, col)

    def random_choice(self, a, size=None, replace=True):
        return self.rng.choice(a, size, replace) if self.rng is not None else np.random.choice(a, size, replace)

    def _generate_instance(self):
        return generate_instance(self.agents_range, self.tasks_range, self.max_coalition_size, self.max_duration, self.rng)

    # ---- instance / device handle --------------------------------------------------------------------------------
    def _install(self, A, task_xy, depot_xy, req, dur, cost=None):
        T = int(np.asarray(task_xy).shape[0])
        M = 8                                              # member slots (DCM_MAX_M): routes / masked actions may exceed the requirements
        if int(np.max(req)) > M:
            raise ValueError(f"requirements above {M} are not supported (the reference uses max_coalition_size = 5)")
        if self._be is None or (self._be.A, self._be.T, self._be.M) != (A, T, M):
            if self._be is not None:
                self._be.close()
            self._be = BatchedTaskEnv(1, A, T, M=M, device=self._device)
        self._xy = np.ascontiguousarray(task_xy, np.float64).reshape(T, 2)
        self._depot_xy = np.ascontiguousarray(depot_xy, np.float64).reshape(2)
        self._req = np.ascontiguousarray(req, np.int64).reshape(T)
        self._dur = np.ascontiguousarray(dur, np.float64).reshape(T)
        self._cost = np.zeros((A, 1)) if cost is None else np.asarray(cost, np.float64).reshape(A, 1)
        self._be.load_instances(self._xy[None], self._depot_xy[None], self._req[None].astype(np.int32), self._dur[None])
        self.tasks_num, self.agents_num = T, A
        self.coalition_matrix = np.zeros((A, T))
        self._routes = [[] for _ in range(A)]
        self._arrivals = [[] for _ in range(A)]
        self._host = [dict(current_action_index=0, pre_set_route=None, working_condition=0, trajectory=[], angle=0) for _ in range(A)]
        self._abandoned = [[] for _ in range(T)]
        self._agent_wait = np.zeros(A)
        self._task_wait = np.zeros(T)
        self.task_dic = _Table((j, _Row(self, "task", j)) for j in range(T))
        self.agent_dic = _Table((i, _Row(self, "agent", i)) for i in range(A))
        self.depot = _Row(self, "depot", -1)
        self._be.reset()                                  # clear_decisions on the device (granular ops ignore the fused path's slot bookkeeping)
        self._cache = None

    def _sync_params(self):
        if self._be is not None:
            self._be.set_params(0.2, float(self._max_waiting_time), 100.0)

    @property
    def max_waiting_time(self):
        return self._max_waiting_time

    @max_waiting_time.setter
    def max_waiting_time(self, w):
        self._max_waiting_time = w
        self._sync_params()

    @property
    def current_time(self):
        return float(self._be.get_clock()[0])

    @current_time.setter
    def current_time(self, t):                             # worker.py:49 writes the clock from outside
        self._be.set_clock(np.array([float(t)]))
        self._cache = None

    # ---- reset / clear (task_env.py:116-140) -----------------------------------------------------------------------
    def reset(self, test_env=None, seed=None):
        self.rng = np.random.default_rng(seed) if seed is not None else None
        if test_env is not None:
            tasks, agents, depot = test_env
            T, A = len(tasks), len(agents)
            xy = np.array([np.asarray(tasks[j]["location"], np.float64) for j in range(T)])
            req = np.array([int(np.asarray(tasks[j]["requirements"]).reshape(-1)[0]) for j in range(T)])
            dur = np.array([float(np.asarray(tasks[j]["time"]).reshape(-1)[0]) for j in range(T)])
            dep = np.asarray(depot["location"], np.float64)
            self._install(A, xy, dep, req, dur)
        else:
            self.current_time = 0
        self.finished = False

    def clear_decisions(self):
        self._be.reset()
        A, T = self.agents_num, self.tasks_num
        self._routes = [[] for _ in range(A)]
        self._arrivals = [[] for _ in range(A)]
        for h in self._host:
            h.update(current_action_index=0, pre_set_route=None, working_condition=0, trajectory=[], angle=0)
        self._abandoned = [[] for _ in range(T)]
        self._agent_wait = np.zeros(A)
        self._task_wait = np.zeros(T)
        self.finished = False
        self._cache = None

    # ---- dict views -------------------------------------------------------------------------------------------------
    def _state(self):
        if self._cache is None:
            self._cache = decode_record(self._be.export_raw()[0], self._be.layout, self._dur)
        return self._cache

    def _keys(self, kind):
        if kind == "task":
            return ["ID", "requirements", "members", "cost", "location", "feasible_assignment", "finished", "time_start", "time_finish",
                    "status", "time", "sum_waiting_time", "efficiency", "abandoned_agent"]
        if kind == "agent":
            return ["ID", "abilities", "location", "next_location", "route", "arrival_time", "cost", "travel_time", "velocity", "next_decision",
                    "depot", "travel_dist", "sum_waiting_time", "current_action_index", "working_condition", "trajectory", "angle", "returned",
                    "assigned", "pre_set_route"]
        return ["location", "members", "ID"]

    def _get(self, kind, i, key):
        s = self._state()
        if kind == "depot":
            if key == "location":
                return self._depot_xy
            if key == "ID":
                return -1
            if key == "members":
                return [a for a in range(self.agents_num) if s["has_route"][a] and s["node"][a] == -1]
            raise KeyError(key)
        if kind == "task":
            if key == "ID":
                return i
            if key == "requirements":
                return np.array([self._req[i]])
            if key == "status":
                return np.array([int(s["status"][i])])
            if key == "members":
                return [int(m) for m in s["members"][i, :s["n_mem"][i]]]
            if key == "location":
                return self._xy[i]
            if key == "feasible_assignment":
                return bool(s["feasible"][i])
            if key == "finished":
                return bool(s["finished"][i])
            if key == "time_start":
                return float(s["time_start"][i]) if s["feasible"][i] else 0
            if key == "time_finish":
                return float(s["time_finish"][i]) if s["feasible"][i] else 0
            if key == "time":
                return float(self._dur[i])
            if key == "sum_waiting_time":
                return float(self._task_wait[i])
            if key == "abandoned_agent":
                return [-1] * int(s["n_aband_task"][i])        # only its length is meaningful (ids are not kept on the device)
            if key in ("cost",):
                return []
            if key == "efficiency":
                return 0
            raise KeyError(key)
        # agent
        if key == "ID":
            return i
        if key in _AGENT_HOST_KEYS and key in self._host[i]:
            return self._host[i][key]
        if key == "location" or key == "next_location":
            n = int(s["node"][i])
            return self._depot_xy if n < 0 else self._xy[n]
        if key == "depot":
            return self._depot_xy
        if key == "route":
            return self._routes[i]
        if key == "arrival_time":
            return self._arrivals[i]
        if key == "next_decision":
            return float(s["next_decision"][i])
        if key == "travel_dist":
            return float(s["travel_dist"][i])
        if key == "travel_time":
            return float(self._host[i].get("travel_time", 0))
        if key == "returned":
            return bool(s["returned"][i])
        if key == "assigned":
            return bool(s["assigned"][i])
        if key == "sum_waiting_time":
            return float(self._agent_wait[i])
        if key == "velocity":
            return 0.2
        if key == "abilities":
            return np.ones(1)
        if key == "cost":
            return self._cost[i]
        raise KeyError(key)

    def _set(self, kind, i, key, value):
        if kind == "agent" and key in _AGENT_HOST_KEYS:
            self._host[i][key] = value
            return
        raise KeyError(f"'{key}' is device state and cannot be assigned through the dict view")

    @staticmethod
    def get_matrix(dictionary, key):
        return [value[key] for value in dictionary.values()]

    # ---- simulator methods ------------------------------------------------------------------------------------------
    def next_decision(self):                               # task_env.py:283-289
        d, t = self._be.next_decision()
        mask, t = int(d[0]) & 0xFFFFFFFFFFFFFFFF, float(t[0])
        ids = np.array([i for i in range(self.agents_num) if (mask >> i) & 1], dtype=np.int64)
        return (ids if len(ids) else []), t

    def get_unique_group(self, agents):                    # task_env.py:291-298
        agents = np.asarray(agents, dtype=np.int64)
        mask = 0
        for a in agents:
            mask |= 1 << int(a)
        rank = self._be.unique_group(np.array([mask], dtype=np.uint64).view(np.int64)).cpu().numpy()[0]
        ng = int(rank.max()) + 1 if len(agents) else 0
        return [[int(a) for a in agents if rank[a] == g] for g in range(ng)]

    def task_update(self):                                 # task_env.py:245-281
        before = self._state()
        newly = self._be.task_update(want_newly=True).cpu().numpy()[0]
        self._cache = None
        after = self._state()
        for j in range(self.tasks_num):                    # keep the host copy of abandoned_agent ids in step (members that vanished)
            gone = [int(m) for m in before["members"][j, :before["n_mem"][j]] if m not in after["members"][j, :after["n_mem"][j]]]
            self._abandoned[j] += gone
        return [int(j) for j in np.flatnonzero(newly)]

    def agent_update(self):                                # task_env.py:207-243
        self._be.agent_update()
        self._cache = None

    def agent_step(self, agent_id, task_id):               # task_env.py:300-324 ; returns -travel_time
        now = self.current_time
        r = self._be.apply_members(np.array([int(task_id)]), np.array([[int(agent_id)]]), np.array([1]))
        self._cache = None
        r = float(r[0])
        self._routes[int(agent_id)].append(int(task_id) - 1)
        self._arrivals[int(agent_id)].append(now - r)
        self._host[int(agent_id)]["travel_time"] = -r
        return r

    def step(self, group, leader_id, action, current_action_index=0):        # task_env.py:326-342
        s = self._state()
        vacancy = int(s["status"][action - 1]) if 0 <= action - 1 < self.tasks_num else len(group)
        group.remove(leader_id)
        available_agents = len(group)
        if vacancy > 1:
            followers = self.random_choice(group, np.minimum(vacancy - 1, available_agents), False).tolist()
            for follower in followers:
                group.remove(follower)
            members = [leader_id] + followers
        else:
            members = [leader_id]
        r = float(self._be.apply_members(np.array([int(action)]), np.array([members]), np.array([len(members)]))[0])
        self._cache = None
        after = self._state()
        for m in members:
            self._routes[m].append(int(action) - 1)
            self._arrivals[m].append(float(after["last_arrival"][m]))
            self._host[m]["current_action_index"] = current_action_index
        return group, r

    def get_unfinished_tasks(self):                        # task_env.py:196-200
        return [not bool(m) for m in self.get_unfinished_task_mask()]

    def get_unfinished_task_mask(self):                    # task_env.py:192-194 (task bits only; the caller prepends the depot bit)
        self._be.build_obs(np.array([0]))
        return self._be.mask_u8[0, 1:].cpu().numpy().astype(bool)

    def _leader_of(self, agent):
        return int(agent["ID"])

    def get_current_agent_status(self, agent):             # task_env.py:165-180 -> [A,6]; fp32-exact values (the caller casts, worker.py:62)
        self._be.build_obs(np.array([self._leader_of(agent)]))
        return self._be.agent_obs[0].cpu().numpy().astype(np.float64)

    def get_current_task_status(self, agent):              # task_env.py:182-190 -> [T+1,5]
        self._be.build_obs(np.array([self._leader_of(agent)]))
        return self._be.task_obs[0].cpu().numpy().astype(np.float64)

    def check_finished(self):                              # task_env.py:366-373 (moves the clock when nobody can decide)
        f = bool(self._be.check_finished()[0])
        self._cache = None
        return f

    def calculate_waiting_time(self):                      # task_env.py:344-364
        _, tw, aw = self._be.compute_metrics(per_element=True)
        self._task_wait, self._agent_wait = tw[0].cpu().numpy(), aw[0].cpu().numpy()
        self._cache = None

    def get_episode_reward(self, max_time=100):            # task_env.py:420-425
        m, tw, aw = self._be.compute_metrics(per_element=True)
        self._task_wait, self._agent_wait = tw[0].cpu().numpy(), aw[0].cpu().numpy()
        self._cache = None
        finished_tasks = self.get_matrix(self.task_dic, "finished")
        return float(m[0, 0]), finished_tasks

    def get_arrival_time(self, agent_id, task_id):         # task_env.py:202-205
        r = self._routes[agent_id]
        idx = max(k for k, x in enumerate(r) if x == task_id)
        return float(self._arrivals[agent_id][idx])

    # ---- preset routes (task_env.py:562-599) --------------------------------------------------------------------------
    def pre_set_route(self, routes, agent_id):
        h = self._host[agent_id]
        if not h["pre_set_route"]:
            h["pre_set_route"] = list(routes)
        else:
            h["pre_set_route"] += list(routes)

    def execute_by_route(self, path="./", method=0, plot_figure=False):
        if self.reactive_planning:
            raise NotImplementedError("reactive_planning=True is out of scope")
        self.plot_figure = plot_figure
        self.max_waiting_time = 100                        # task_env.py:564
        A = self.agents_num
        routes = [list(self._host[a]["pre_set_route"] or []) for a in range(A)]
        L = max(1, max(len(r) for r in routes))
        arr = np.zeros((1, A, L), np.int32)
        ln = np.zeros((1, A), np.int32)
        for a, r in enumerate(routes):
            arr[0, a, :len(r)] = r
            ln[0, a] = len(r)
        mk = float(self._be.execute_by_route(arr, ln)[0])
        for a in range(A):
            self._host[a]["pre_set_route"] = []
        self._cache = None
        flags = int(self._be.env_flags()[0])
        if flags & 0xF0:
            raise RuntimeError(f"device reported contract violation bits {flags & 0xF0:#x} while executing preset routes")
        self.finished = bool(flags & 2)
        print(mk)                                          # task_env.py:591
        return mk

    # ---- copying / pickling (worker.py:33, :116; TestSetGenerator.py:18; RL_test.py:35) ----------------------------------------
    def __copy__(self):                                    # shallow copy shares the dicts in the reference; here it shares the device env
        new = object.__new__(type(self))
        new.__dict__.update(self.__dict__)
        return new

    def __deepcopy__(self, memo):
        new = object.__new__(type(self))
        for k, v in self.__dict__.items():
            if k in ("_be", "task_dic", "agent_dic", "depot", "_cache"):
                continue
            new.__dict__[k] = copy.deepcopy(v, memo)
        new._be = None
        new._cache = None
        raw = self._be.export_raw()
        new._be = BatchedTaskEnv(1, self._be.A, self._be.T, M=self._be.M, device=self._device)
        new._be.load_instances(self._xy[None], self._depot_xy[None], self._req[None].astype(np.int32), self._dur[None])
        new._be.import_raw(raw)
        new._sync_params()
        new.task_dic = _Table((j, _Row(new, "task", j)) for j in range(self.tasks_num))
        new.agent_dic = _Table((i, _Row(new, "agent", i)) for i in range(self.agents_num))
        new.depot = _Row(new, "depot", -1)
        return new

    def __getstate__(self):
        d = {k: v for k, v in self.__dict__.items() if k not in ("_be", "task_dic", "agent_dic", "depot", "_cache")}
        d["_raw"] = self._be.export_raw()
        d["_shape"] = (self._be.A, self._be.T, self._be.M)
        return d

    def __setstate__(self, d):
        if "task_dic" in d and "_raw" not in d:            # a pickle written by the REFERENCE class (RL_test.py:35): import the instance
            self.__dict__.update({k: v for k, v in d.items() if k not in ("task_dic", "agent_dic", "depot")})
            self._device, self._be, self._cache = 0, None, None
            self.max_coalition_size = d.get("max_coalition_size", d.get("coalition_size", 5))
            self._max_waiting_time = d.get("max_waiting_time", 10)
            self.__dict__.pop("max_waiting_time", None)
            self.reactive_planning = d.get("reactive_planning", False)
            self.finished = False
            self.rng = None
            self.reset((d["task_dic"], d["agent_dic"], d["depot"]))
            return
        raw, (A, T, M) = d.pop("_raw"), d.pop("_shape")
        self.__dict__.update(d)
        self._cache = None
        self._be = BatchedTaskEnv(1, A, T, M=M, device=self._device)
        self._be.load_instances(self._xy[None], self._depot_xy[None], self._req[None].astype(np.int32), self._dur[None])
        self._be.import_raw(raw)
        self._sync_params()
        self.task_dic = _Table((j, _Row(self, "task", j)) for j in range(T))
        self.agent_dic = _Table((i, _Row(self, "agent", i)) for i in range(A))
        self.depot = _Row(self, "depot", -1)

    # ---- out of scope ---------------------------------------------------------------------------------------------------
    def _unsupported(self, *a, **k):
        raise NotImplementedError("plotting / trajectories / OR-Tools grouping are outside the step path (SURVEY.md 2, rows 3-4)")

    plot_animation = generate_traj = stack_trajectory = process_map = get_grouped_tasks = _unsupported
