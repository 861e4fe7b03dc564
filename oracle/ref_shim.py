"""oracle/ref_shim.py -- import the REAL reference TaskEnv (a read-only checkout of the original project, found at
$DCMRTA_REFERENCE).  TEST INFRASTRUCTURE ONLY: the tests do not use it; the oracle/make_*golden.py generators record
tests/golden/ from the reference through it.

Shims (SURVEY.md App. B): (1) stub matplotlib, which env/task_env.py:2-5 imports at module top and this image
lacks; (2) remap the pickles' `__main__.TaskEnv` to env.task_env.TaskEnv; (3) normalise an unpickled env
exactly as RL_test.py:34-44 does.  The reference sources are not modified or copied.
"""
from __future__ import annotations

import ctypes
import io
import os
import pickle
import sys
import types
import warnings
from pathlib import Path

import numpy as np

REF_ROOT = Path(os.environ.get("DCMRTA_REFERENCE", "/root/reference"))
TESTSET = REF_ROOT / "testSet_20A_50T_CONDET"
MAX_TIME = 100          # parameters.py:19
COALITION_SIZE = 5      # parameters.py:18


def available() -> bool:
    return (REF_ROOT / "env" / "task_env.py").exists()


def _stub_matplotlib():
    if "matplotlib" in sys.modules and not isinstance(sys.modules["matplotlib"], types.ModuleType):
        return
    try:
        import matplotlib  # noqa: F401
        return
    except Exception:
        pass
    names = ["matplotlib", "matplotlib.pyplot", "matplotlib.patches", "matplotlib.animation", "matplotlib.offsetbox"]
    for n in names:
        sys.modules.setdefault(n, types.ModuleType(n))
    sys.modules["matplotlib.animation"].FuncAnimation = object
    sys.modules["matplotlib.offsetbox"].OffsetImage = object
    sys.modules["matplotlib.offsetbox"].AnnotationBbox = object
    sys.modules["matplotlib"].patches = sys.modules["matplotlib.patches"]
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]


_TASKENV = None


def ref_taskenv_class():
    """The reference class object (env/task_env.py:8)."""
    global _TASKENV
    if _TASKENV is None:
        if not available():
            raise RuntimeError(f"reference tree not found at {REF_ROOT}")
        _stub_matplotlib()
        # load the module under a private name so it cannot collide with any package called `env`
        import importlib.util
        spec = importlib.util.spec_from_file_location("_dcmrta_reference_task_env", REF_ROOT / "env" / "task_env.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _TASKENV = mod.TaskEnv
    return _TASKENV


class _Unpickler(pickle.Unpickler):
    def find_class(self, module, name):
        if name == "TaskEnv":
            return ref_taskenv_class()
        return super().find_class(module, name)


def load_pickle(i: int, max_waiting_time: float = 10):
    """RL_test.py:34-44: unpickle env_i, normalise it, return the reference TaskEnv ready for an episode."""
    warnings.filterwarnings("ignore", category=DeprecationWarning)
    with open(TESTSET / f"env_{i}.pkl", "rb") as f:
        env = _Unpickler(io.BytesIO(f.read())).load()
    env.max_waiting_time = max_waiting_time          # RL_test.py:39
    env.reactive_planning = False                    # RL_test.py:40
    env.reset((env.task_dic, env.agent_dic, env.depot))   # RL_test.py:41-42
    env.clear_decisions()                            # RL_test.py:43
    env.force_waiting = True
    return env


def instance_arrays(env):
    """Static instance data of a reference env as flat arrays (the layout dcm_load_instances takes)."""
    T, A = env.tasks_num, env.agents_num
    xy = np.array([np.asarray(env.task_dic[j]["location"], np.float64) for j in range(T)])
    req = np.array([int(np.asarray(env.task_dic[j]["requirements"]).reshape(-1)[0]) for j in range(T)], np.int32)
    dur = np.array([float(np.asarray(env.task_dic[j]["time"]).reshape(-1)[0]) for j in range(T)], np.float64)
    depot = np.asarray(env.depot["location"], np.float64).copy()
    return dict(A=A, task_xy=xy, depot_xy=depot, req=req, dur=dur)


def canonical_state(env, MC: int = 8):
    """Live state of a reference env in the canonical flat form shared with OracleEnv.export / the GPU export."""
    T, A = env.tasks_num, env.agents_num
    d = dict(
        n_mem=np.zeros(T, np.int32), members=np.full((T, MC), -1, np.int32), mem_arr=np.zeros((T, MC), np.float64),
        status=np.zeros(T, np.int32), feasible=np.zeros(T, np.uint8), finished=np.zeros(T, np.uint8),
        time_start=np.zeros(T, np.float64), time_finish=np.zeros(T, np.float64), n_aband_task=np.zeros(T, np.int32),
        node=np.zeros(A, np.int32), has_route=np.zeros(A, np.uint8), last_arrival=np.zeros(A, np.float64),
        next_decision=np.zeros(A, np.float64), travel_dist=np.zeros(A, np.float64), assigned=np.zeros(A, np.uint8),
        returned=np.zeros(A, np.uint8), n_aband_agent=np.zeros(A, np.int32))
    for j in range(T):
        t = env.task_dic[j]
        mem = list(t["members"])
        assert len(mem) <= MC, "member list longer than the canonical capacity"
        d["n_mem"][j] = len(mem)
        for k, m in enumerate(mem):
            d["members"][j, k] = m
            d["mem_arr"][j, k] = env.get_arrival_time(m, j)
        d["status"][j] = int(np.asarray(t["status"]).reshape(-1)[0])
        d["feasible"][j] = bool(t["feasible_assignment"])
        d["finished"][j] = bool(t["finished"])
        d["time_start"][j] = float(t["time_start"])
        d["time_finish"][j] = float(t["time_finish"])
        d["n_aband_task"][j] = len(t["abandoned_agent"])
        for m in t["abandoned_agent"]:
            d["n_aband_agent"][int(m)] += 1
    for i in range(A):
        a = env.agent_dic[i]
        d["has_route"][i] = len(a["route"]) > 0
        d["node"][i] = a["route"][-1] if a["route"] else -1
        d["last_arrival"][i] = float(a["arrival_time"][-1]) if a["arrival_time"] else 0.0
        d["next_decision"][i] = float(a["next_decision"])
        d["travel_dist"][i] = float(a["travel_dist"])
        d["assigned"][i] = bool(a["assigned"])
        d["returned"][i] = bool(a["returned"])
    d["now"] = float(env.current_time)
    d["env_finished"] = bool(env.finished)
    return d


_libm = ctypes.CDLL("libm.so.6")
_libm.fma.restype = ctypes.c_double
_libm.fma.argtypes = [ctypes.c_double] * 3


def _fma(a, b, c):
    return _libm.fma(a, b, c)          # Python 3.12 has no math.fma


def greedy_nearest(mask, task_rows64):
    """Benchmark policy (ii) of SURVEY.md 8(d): argmin squared distance over unmasked tasks, depot only if none."""
    open_tasks = np.flatnonzero(~mask[1:].astype(bool))
    if len(open_tasks) == 0:
        return 0
    dx = task_rows64[1 + open_tasks, 3]
    dy = task_rows64[1 + open_tasks, 4]
    d2 = np.array([_fma(float(y), float(y), float(x) * float(x)) for x, y in zip(dx, dy)])
    return int(open_tasks[int(np.argmin(d2))]) + 1


def run_reference_episode(env, policy, seed: int, on_decision=None, max_time=MAX_TIME, leader_fn=None, on_slot=None):
    """The loop of worker.py:45-87 around the REAL reference env, with the attention policy replaced by
    `policy` in {"random", "greedy"} -- or a callable (env, leader, mask_u8, k) -> action for scripted fixtures -- and every
    random draw recorded.  leader_fn(group, k) -> leader replaces the random leader choice; on_slot(env, groups) is called
    after get_unique_group (quirk fixtures record how many location groups a slot had).

    on_decision(env, leader, mask_u8[T+1], agent_obs_f64[A,6], task_obs_f64[T+1,5]) is called when the obs are built
    (before the action is applied).  Returns (trace, reward, finished_tasks)."""
    rng = np.random.default_rng(seed)
    trace = dict(leader=[], action=[], followers=[], now=[], reward=[])
    drawn = []

    def recording_choice(a, size=None, replace=True):
        out = rng.choice(a, size, replace) if len(a) else np.array([], dtype=np.int64)
        drawn.append(np.asarray(out).reshape(-1).tolist())
        return out

    env.random_choice = recording_choice                      # looked up through self (task_env.py:331)
    idx = 0
    empty_slots = 0
    while not env.finished and env.current_time < max_time:    # worker.py:45
        ids, t = env.next_decision()
        # Nobody can decide and the episode is not finished: one such slot is normal (it marks agents as returned), after a second
        # in a row the state can no longer change and the reference loop would spin forever.  The oracle and the CUDA path stop
        # there and flag the env STUCK (DESIGN.md 2); so does this driver.
        empty_slots = empty_slots + 1 if len(ids) == 0 else 0
        if empty_slots >= 3:
            break
        groups = env.get_unique_group(ids)
        if on_slot is not None:
            on_slot(env, groups)
        env.current_time = t
        env.task_update()
        env.agent_update()
        for group in groups:
            while len(group) > 0:
                leader = int(leader_fn(group, idx)) if leader_fn is not None else int(rng.choice(group))   # worker.py:54 (np.random.choice there)
                agent = env.agent_dic[leader]
                assert not agent["returned"], "reference would spin forever (worker.py:56)"
                m = env.get_unfinished_task_mask()            # worker.py:57-61
                m = np.insert(m, 0, False) if np.sum(m) == env.tasks_num else np.insert(m, 0, True)
                ag = np.asarray(env.get_current_agent_status(agent), np.float64)
                tk = np.asarray(env.get_current_task_status(agent), np.float64)
                mask = m.astype(np.uint8)
                if on_decision is not None:
                    on_decision(env, leader, mask, ag, tk)
                if callable(policy):
                    action = int(policy(env, leader, mask, idx))
                elif policy == "random":
                    action = int(rng.choice(np.flatnonzero(mask == 0)))
                else:
                    action = greedy_nearest(mask, tk)
                drawn.clear()
                now = float(env.current_time)
                group, r = env.step(group, leader, action, idx)   # worker.py:73
                env.task_update()
                env.agent_update()
                trace["leader"].append(leader)
                trace["action"].append(action)
                trace["followers"].append(drawn[0] if drawn else [])
                trace["now"].append(now)
                trace["reward"].append(float(r))
                idx += 1
        env.finished = env.check_finished()                   # worker.py:85
    reward, finished_tasks = env.get_episode_reward(max_time)  # worker.py:87
    return trace, float(reward), np.asarray(finished_tasks, bool)


def reference_metrics(env, finished_tasks):
    """worker.py:103-108."""
    return dict(
        success_rate=float(np.sum(finished_tasks) / len(finished_tasks)),
        makespan=float(env.current_time),
        time_cost=float(np.nanmean(env.get_matrix(env.task_dic, "time_start"))),
        waiting_time=float(np.mean(env.get_matrix(env.agent_dic, "sum_waiting_time"))),
        travel_dist=float(np.sum(env.get_matrix(env.agent_dic, "travel_dist"))),
        efficiency=float(np.mean(env.get_matrix(env.task_dic, "sum_waiting_time"))))


def ctasd_routes(i: int):
    """baselines/CTAS-D.py:10-46: per-agent node lists of env_i/results.yaml, first node dropped; [0] routes skipped."""
    import yaml
    d = TESTSET / f"env_{i}"
    with open(d / "planner_param.yaml") as f:
        p = yaml.safe_load(f)
    num_veh = p["vehNum"] if p["flagSolver"] == "TEAMPLANNER_DET" else p["vehNumPerType"][0]
    with open(d / "results.yaml") as f:
        data = yaml.safe_load(f)
    if "vehicle" not in data:
        return None
    nodes = []
    for v in range(num_veh):
        key = "vv" + str(v + 1)
        if key not in data["vehicle"]:
            continue
        nodes.append(data["vehicle"][key]["node"])
    routes = {}
    for a, r in enumerate(nodes):
        if r == [0]:
            continue
        routes[a] = list(r)[1:]
    return routes
