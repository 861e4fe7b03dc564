"""Shared test helpers: golden loaders and trace replay drivers (tests only)."""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np

GOLD = Path(__file__).resolve().parent / "golden"
METRIC_KEYS = ("reward", "success_rate", "makespan", "time_cost", "waiting_time", "travel_dist", "efficiency", "n_steps")


def pickle_instances():
    z = np.load(GOLD / "instances_20A_50T.npz")
    return [dict(A=int(z["A"]), task_xy=z["task_xy"][i], depot_xy=z["depot_xy"][i], req=z["req"][i], dur=z["dur"][i])
            for i in range(z["task_xy"].shape[0])]


class Traces:
    """Flat trace arrays + offsets -> per-episode views."""

    def __init__(self, path):
        self.z = np.load(path)
        self.names = [str(n) for n in self.z["names"]]
        self.off = self.z["offsets"]

    def __len__(self):
        return len(self.names)

    def episode(self, i):
        s, e = int(self.off[i]), int(self.off[i + 1])
        ep = {k: self.z[k][s:e] for k in ("leader", "action", "nfol", "followers", "now", "reward", "dig_obs", "dig_state")}
        ep["metrics"] = self.z["metrics"][i]
        ep["final_digest"] = int(self.z["final_digest"][i])
        ep["name"] = self.names[i]
        return ep

    def followers(self, ep, k):
        return [int(x) for x in ep["followers"][k, :int(ep["nfol"][k])]]


def pickle_traces():
    t = Traces(GOLD / "traces_pickles.npz")
    t.finished = t.z["finished"]
    return t


def sweep_traces():
    return Traces(GOLD / "traces_sweep.npz")


def sweep_instance(tr: Traces, name: str):
    shape, s, _ = name.split("/")
    A, T = (int(x) for x in shape.split("x"))
    g = lambda k: tr.z[f"inst/{shape}/{s}/{k}"]
    return dict(A=A, task_xy=g("task_xy"), depot_xy=g("depot_xy"), req=g("req"), dur=g("dur"))


def ctasd():
    return json.load(open(GOLD / "ctasd.json"))


def full_dump():
    return np.load(GOLD / "full_dump.npz")


def quirk_traces():
    """tests/golden/quirks.npz (oracle/make_quirk_golden.py): hand-built and searched small fixtures, one quirk of SURVEY App. A each."""
    t = Traces(GOLD / "quirks.npz")
    t.census_keys = [str(k) for k in t.z["census_keys"]]
    return t


def quirk_instance(tr: Traces, name: str):
    g = lambda k: tr.z[f"inst/{name}/{k}"]
    return dict(A=int(g("A")), task_xy=g("task_xy"), depot_xy=g("depot_xy"), req=g("req").astype(np.int32), dur=g("dur"))


def quirk_census(tr: Traces, name: str):
    return dict(zip(tr.census_keys, (int(x) for x in tr.z[f"census/{name}"])))


# ---- the supported shape range (include/dcmrta.h: 1 <= A <= 64, 1 <= T <= 254, 1 <= M <= 8) -------------------------------------
# Shapes at which the CUDA path changes code path, shared by tests/test_gpu_shape_envelope.py (CUDA against the oracle) and
# tests/test_shape_envelope_oracle.py (the same trajectories on the oracle alone, so the census below cannot become vacuous).
class EnvelopeShape:
    """A, T, M, batch size B, the in-kernel policy, the decisions a test plays (`steps`; `ia_steps` for the individual-agent
    protocol, None where it is not run) and the census events (envelope_census) its sampled trajectories must reach."""

    def __init__(self, A, T, M, B, policy, steps, ia_steps, reaches, census):
        self.A, self.T, self.M, self.B, self.policy, self.steps, self.ia_steps = A, T, M, B, policy, steps, ia_steps
        self.reaches, self.census = reaches, tuple(census)
        self.seed = 100 + A + 7 * T + 11 * M

    @property
    def name(self):
        return f"{self.A}A_{self.T}T_{self.M}M_B{self.B}_{self.policy}"

    @property
    def random_duration(self):
        return self.policy == "greedy"

    def sample(self):
        """env 0, the last env, and the first and last env of the last (partial) tile of 32 envs"""
        return sorted({0, min(31, self.B - 1), 32 * ((self.B - 1) // 32), self.B - 1})

    def first_gid(self):
        return 1000 * self.A + self.T


ENVELOPE_SHAPES = [
    EnvelopeShape(1, 1, 1, 33, "random", 40, None, "the smallest instance; a second tile holding one env", ["leader_last", "task_last", "full_coalition"]),
    EnvelopeShape(2, 3, 3, 100, "random", 60, None, "requirements above A: episodes end by the clock cap or stuck",
                  ["leader_last", "task_last", "give_up", "clock_cap_or_stuck"]),
    EnvelopeShape(7, 63, 2, 100, "greedy", 240, 300, "A < 8; ragged agent chunk; T just below a word", ["leader_last", "task_last", "full_coalition"]),
    EnvelopeShape(24, 64, 8, 100, "random", 280, None, "last shape with the next_decision scratch; word 0 full; 8-member coalitions",
                  ["leader_last", "task_last", "task_63", "full_coalition"]),
    EnvelopeShape(25, 65, 8, 100, "greedy", 420, None, "first shape without the scratch; TW = 2 with one bit in word 1",
                  ["leader_last", "task_last", "task_64", "full_coalition"]),
    EnvelopeShape(32, 128, 4, 100, "random", 500, None, "ANB = 32; TW = 2 full", ["leader_last", "task_last", "task_63", "task_64", "task_127", "full_coalition"]),
    EnvelopeShape(33, 129, 5, 100, "greedy", 600, 1100, "ANB = 64; TW = 4",
                  ["leader_last", "task_last", "task_63", "task_64", "task_127", "task_128", "full_coalition", "depot16"]),
    EnvelopeShape(20, 55, 5, 100, "random", 270, None, "largest T of the k_obs_tile path at A = 20 (228 kB of shared memory per SM)", ["leader_last", "task_last"]),
    EnvelopeShape(20, 56, 5, 100, "random", 270, None, "smallest T of the chunked k_obs path at A = 20 (228 kB of shared memory per SM)", ["leader_last", "task_last"]),
    EnvelopeShape(64, 249, 3, 100, "greedy", 450, None, "agent bit 63; the first T whose metric sums split twice",
                  ["leader_last", "task_last", "task_63", "task_64", "task_127", "task_128", "full_coalition", "depot16"]),
    EnvelopeShape(64, 254, 8, 100, "random", 800, 650, "the largest shape",
                  ["leader_last", "task_last", "task_63", "task_64", "task_127", "task_128", "full_coalition", "wait16", "clock_cap"]),
    EnvelopeShape(64, 254, 8, 1, "greedy", 600, None, "the largest shape in a batch of one", ["leader_last", "task_last", "full_coalition"]),
]


def envelope_shape(name):
    return next(s for s in ENVELOPE_SHAPES if s.name == name)


def device_instance(A, T, M, seed, gid, instance=0, max_duration=5.0, random_duration=False):
    """The instance dcm_generate draws for global env `gid` (dcm_kernels.cu t_generate): Philox counter (gid_lo, gid_hi, instance,
    0x80000000 + 2 j + {0, 1}) for task j and 0xFFFFFFFF for the depot, key = seed, uniforms of 53 bits."""
    from oracle.oracle import philox
    key = [seed & 0xFFFFFFFF, seed >> 32]
    g = [gid & 0xFFFFFFFF, gid >> 32, instance]
    u01 = lambda hi, lo: float(((int(hi) >> 5) << 26) | (int(lo) >> 6)) * (1.0 / 9007199254740992.0)
    xy, req, dur = np.empty((T, 2)), np.empty(T, np.int32), np.full(T, float(max_duration))
    for j in range(T):
        a, b = philox(g + [0x80000000 + 2 * j], key), philox(g + [0x80000001 + 2 * j], key)
        xy[j] = u01(a[0], a[1]), u01(a[2], a[3])
        req[j] = 1 + ((int(b[0]) * M) >> 32)
        if random_duration:
            dur[j] = u01(b[1], b[2]) * max_duration
    a = philox(g + [0xFFFFFFFF], key)
    return dict(A=A, task_xy=xy, depot_xy=np.array([u01(a[0], a[1]), u01(a[2], a[3])]), req=req, dur=dur)


# ---- preset routes (dcm_execute_by_route), shared by tests/test_routes_oracle.py and tests/test_gpu_routes.py ------------------------
ROUTE_FAMILIES = ("coalition", "short", "partial", "noisy")
ROUTE_MAX_LEN = 255                     # dcm_execute_by_route: rstride <= 255
ROUTE_MAX_DURATION = 0.5                # task durations of the route instances: short enough that 64 agents finish 254 tasks under the clock


def route_family(b):
    return ROUTE_FAMILIES[b % len(ROUTE_FAMILIES)]


def make_routes(seed, inst, A, M, family):
    """Preset routes of one env (lists of actions, 0 = depot, j + 1 = task j), seeded.  The tasks are handed out in one sweep of the
    unit square (six vertical strips, up one and down the next), so no two agents wait for each other in opposite orders and the
    hops are short enough for 64 agents to finish 254 tasks under the clock cap:
      coalition  each task to min(req, A) distinct agents drawn at random, appended to their routes;
      short      one agent fewer than req (at least one): members wait, give up after W = 100 and run into the 200-unit clock;
      partial    as coalition, but about a tenth of the tasks are never routed: once every agent is home the episode is stuck;
      noisy      as coalition, plus re-visits, a depot entry in the middle of some routes, empty routes and one route padded with
                 re-visits of its own tasks to one more entry than any other route of the env.
    Each task lies on the routes of at most M distinct agents, so no member list overflows and the oracle compares exactly."""
    rng = np.random.default_rng(seed)
    xy, req = np.asarray(inst["task_xy"]), inst["req"]
    strip = np.minimum((xy[:, 0] * 6).astype(int), 5)
    R = [[] for _ in range(A)]
    for j in np.lexsort((np.where(strip % 2 == 0, xy[:, 1], -xy[:, 1]), strip)):
        if family == "partial" and rng.random() < 0.1:
            continue
        k = min(int(req[j]), A, M)
        if family == "short":
            k = max(k - 1, 1)
        for a in rng.choice(A, k, replace=False):
            R[a].append(int(j) + 1)
    if family == "noisy":
        for a in range(A):
            u = rng.random()
            if u < 0.15:
                R[a] = []                                                    # an empty route: straight home
            elif u < 0.45 and R[a]:
                R[a].insert(int(rng.integers(len(R[a]) + 1)), R[a][int(rng.integers(len(R[a])))])   # re-visit one of its tasks
            elif u < 0.65 and len(R[a]) > 1:
                R[a].insert(int(rng.integers(1, len(R[a]))), 0)               # home in the middle: the rest is never played
        full = [a for a in range(A) if any(R[a])]
        if full:
            a = full[int(rng.integers(len(full)))]
            own = [x for x in R[a] if x]
            L = min(max(len(r) for r in R) + 1, ROUTE_MAX_LEN)
            while len(R[a]) < L:
                R[a].append(own[int(rng.integers(len(own)))])
    return [r[:ROUTE_MAX_LEN] for r in R]


def pack_routes(routes_per_env, A, L=None):
    """list over envs of per-agent routes -> routes [B, A, L] int32 (zero padded), route_len [B, A] int32"""
    L = L or max(1, max(len(r) for R in routes_per_env for r in R))
    out = np.zeros((len(routes_per_env), A, L), np.int32)
    n = np.zeros((len(routes_per_env), A), np.int32)
    for b, R in enumerate(routes_per_env):
        for a, r in enumerate(R):
            out[b, a, :len(r)] = r
            n[b, a] = len(r)
    return out, n


def route_oracle(A, inst, R, velocity=0.2):
    """the oracle after execute_by_route of routes R on instance inst -> (OracleEnv, makespan)"""
    from oracle.oracle import OracleEnv
    o = OracleEnv.make(A, inst["task_xy"], inst["depot_xy"], inst["req"], inst["dur"], velocity=velocity)
    for a, r in enumerate(R):
        if len(r):
            o.pre_set_route(np.asarray(r, np.int32), a)
    return o, o.execute_by_route()


def route_census(ev, o, A, T, M, R):
    """Add to the set `ev` what one execute_by_route episode reached on the oracle `o` (routes R)."""
    s = o.export(M)
    ev.add("finished" if s["env_finished"] else ("stuck" if o.stuck else "clock_cap"))
    if (s["n_mem"] == M).any():
        ev.add("full_coalition")
    if s["n_aband_task"].any():
        ev.add("give_up")
    played = [r for r, _ in o.routes()]
    for j, key in ((T - 1, "task_last"), (63, "task_63"), (64, "task_64"), (127, "task_127"), (128, "task_128")):
        if j < T and any((p == j).any() for p in played):
            ev.add(key)
    if (played[A - 1] >= 0).any():
        ev.add("agent_last")                                          # the last agent (bit A - 1) moved to a task
    if any((np.diff(t) < 0).any() for _, t in o.routes()):
        ev.add("clock_back")                                          # a re-visit of an ended task: next_decision in the past, the clock goes back
    return ev


def route_census_needs(shape):
    """what the route batches of a shape must reach: with M = 1 every task starts on arrival (no wait, no give-up, and one task cannot
    take 200 units), and A < M agents cannot fill M slots"""
    need = {"finished", "stuck", "task_last", "agent_last"} | \
        {key for j, key in ((63, "task_63"), (64, "task_64"), (127, "task_127"), (128, "task_128")) if j < shape.T}
    if shape.M > 1:
        need |= {"clock_cap", "give_up"}
    if shape.A >= shape.M:
        need.add("full_coalition")
    if shape.A > 1 and shape.B >= 100:                                # one to ten envs in a hundred re-visit a task after it ended
        need.add("clock_back")
    return need


def route_batch_sizes(shape):
    """the batch sizes tests/test_gpu_routes.py plays a shape at: its own B, one env, and one env past a tile of 32"""
    return sorted({shape.B, 1, 33})


def route_seed(shape, b):
    return 1000 * shape.seed + b


def envelope_census(ev, o, A, T, M, leader, used_action, done=False, env=None):
    """Add to the set `ev` what one decision of the oracle reached.  `o` is the OracleEnv after the decision, `leader` the agent that
    decided and `used_action` its action (0 = depot, j + 1 = task j); `env` the OracleEnv whose episode ended (`done`), for its cause."""
    if leader == A - 1:
        ev.add("leader_last")
    for j, key in ((T - 1, "task_last"), (63, "task_63"), (64, "task_64"), (127, "task_127"), (128, "task_128")):
        if j < T and used_action == j + 1:
            ev.add(key)
    s = o.export(M)
    if (s["n_mem"] == M).any():
        ev.add("full_coalition")
    waiting = (s["n_mem"] > 0) & (s["feasible"] == 0)
    if any(waiting[w:w + 64].sum() > 16 for w in range(0, T, 64)):
        ev.add("wait16")                                              # a second SCR_TMP chunk of the waiting-coalition scan
    if ((s["has_route"] > 0) & (s["node"] < 0) & (s["returned"] == 0)).sum() > 16 and (s["feasible"] > 0).all():
        ev.add("depot16")                                             # ... and of the depot-return scan, which runs once all tasks are feasible
    if s["n_aband_task"].any():
        ev.add("give_up")
    if done:
        e = env if env is not None else o
        if e.stuck:
            ev.add("stuck")
            ev.add("clock_cap_or_stuck")
        elif not e.export(M)["env_finished"]:
            ev.add("clock_cap")
            ev.add("clock_cap_or_stuck")
    return ev


class EnvelopeOracle:
    """One sampled env of an envelope shape on the CPU reference, restarted as an auto-reset handle restarts it: the oracle's
    leader-follower driver (protocol "LF") or the individual-agent loop of tests/ia_oracle.py ("IA"), with the Philox draws of
    (seed, gid, episode): the shape's seed and global ids unless `seed` and `first_gid` (the global id of env 0) are given."""

    def __init__(self, shape, b, inst, protocol="LF", seed=None, first_gid=None):
        from oracle.oracle import OracleEnv
        self.shape, self.protocol = shape, protocol
        self.seed = shape.seed if seed is None else seed
        self.gid = (shape.first_gid() if first_gid is None else first_gid) + b
        if protocol == "IA":
            from ia_oracle import IAOracle
            self.o = IAOracle(shape.A, inst["task_xy"], inst["depot_xy"], inst["req"], inst["dur"])
            self.env = self.o.env
        else:
            self.o = self.env = OracleEnv.make(shape.A, inst["task_xy"], inst["depot_xy"], inst["req"], inst["dur"])
        self.episodes, self.last_metrics, self.first_end, self.census = 0, None, None, set()
        self._restart()

    def _restart(self, leader=-1):
        self.o.seed(self.seed, gid=self.gid, episode=self.episodes)
        self.o.reset() if self.protocol == "IA" else self.o.fused_reset(leader)

    @property
    def leader(self):
        return self.o.leader

    def step(self):
        """one decision of the shape's built-in policy -> (reward, done, used_action); restarts a finished episode"""
        code = -1 if self.shape.policy == "random" else -2
        leader = self.o.leader
        if self.protocol == "IA":
            r, d, ua, _ = self.o.step(code)
        else:
            rc, r, d, ua, _ = self.o.fused_step(code)
            assert rc == 0, (self.shape.name, self.gid, rc)
        s = self.shape
        envelope_census(self.census, self.env, s.A, s.T, s.M, leader, ua, d, self.o)
        if d:
            if self.first_end is None:
                self.first_end = (bool(self.o.export(s.M)["env_finished"]), bool(self.o.stuck))
            self.last_metrics = np.array([self.o.episode_metrics()[0][k] for k in METRIC_KEYS])
            self.episodes += 1
            self._restart()
        return r, d, ua


# ---- caller-supplied actions (DCM_POLICY_EXTERNAL), shared by tests/test_external_actions_oracle.py (the oracle alone) and
# tests/test_gpu_external_actions.py (CUDA against the oracle).  The kernel plays any action in [0, T] it is given, as
# TaskEnv.step does (task_env.py:326-342): masked ones too.  A masked task has status <= 0, so its vacancy moves the leader alone.
EXTERNAL_EVENTS = ("join_running", "join_finished", "join_satisfied", "clock_back", "revisit_feasible", "depot_masked",
                   "inject_want_ge2", "follower_last")
EXT_DEPOT, EXT_REVISIT, EXT_JOIN = 0.04, 0.10, 0.30     # cumulative probabilities of the three masked kinds; the rest is a legal action


def external_words(seed, gid, k):
    """four uniform words of decision k of global env gid: Philox counter (gid_lo, gid_hi, 0xE0000000, k), key = seed, a region the
    env's own draws (episode numbers) never reach"""
    from oracle.oracle import philox
    return [int(x) for x in philox([gid & 0xFFFFFFFF, gid >> 32, 0xE0000000, k], [seed & 0xFFFFFFFF, seed >> 32])]


def inject_followers_at(k):
    """the decisions on which the leader-follower tests draw the followers themselves (the others leave them to the Philox stream)"""
    return k % 3 == 1


def external_steps(shape, protocol="LF"):
    """decisions the external-action tests play at a shape: enough for every env of the batch to end episodes and reach the census"""
    steps = shape.steps if protocol == "LF" else shape.ia_steps
    return min(steps, 200)


def external_census_needs(shape, protocol="LF"):
    """what the external-action trajectories of a shape must reach (external census events, over all envs of the batch).  With one
    agent nobody else can be on a masked task and nothing can send the clock back"""
    need = set()
    if shape.A >= 2:
        need |= {"join_running", "join_finished", "clock_back", "depot_masked"}
    return need


class ExternalOracle(EnvelopeOracle):
    """EnvelopeOracle played by caller-supplied actions.  decide(k) draws decision k of this env from external_words: a masked depot, a
    re-visit of a feasible task the leader is a member of, a masked task with fewer than M members (running, finished, or waiting
    with status <= 0), else a legal action; and, under leader-follower on the decisions inject_followers_at names, the followers (a
    random subset of the current group of the size step() draws, in random order).  The draw depends on (seed, gid, k) and on the
    state only, so the oracle-only test and the GPU test play the same trajectories.  `ext_census` collects EXTERNAL_EVENTS."""

    def __init__(self, shape, b, inst, protocol="LF"):
        super().__init__(shape, b, inst, protocol)
        self.ext_census, self.max_joined = set(), 0

    def choose(self, k):
        """-> (action, kind) of decision k: kind is "legal" or the census event the masked action reaches"""
        s = self.shape
        T, M = s.T, s.M
        w = external_words(s.seed, self.gid, k)
        mask, L, u = self.env.mask(), self.o.leader, w[0] / 2.0 ** 32
        kind, action = "legal", None
        if u < EXT_DEPOT:
            if mask[0]:
                kind, action = "depot_masked", 0
        elif u < EXT_JOIN:
            st = self.env.export(M)
            own = (st["members"] == L).any(1)
            feas, fin = st["feasible"] > 0, st["finished"] > 0
            if u < EXT_REVISIT:
                js = np.flatnonzero(feas & own)
                if len(js):
                    kind, action = "revisit_feasible", int(js[pick_word(w[1], len(js))]) + 1
            else:
                free = (mask[1:] > 0) & (st["n_mem"] < M) & ~own
                cats = [(n, np.flatnonzero(m)) for n, m in (("join_running", free & feas & ~fin), ("join_finished", free & feas & fin),
                                                            ("join_satisfied", free & ~feas & (st["status"] <= 0))) if m.any()]
                if cats:
                    kind, js = cats[pick_word(w[1], len(cats))]
                    action = int(js[pick_word(w[2], len(js))]) + 1
        if action is None:
            legal = np.flatnonzero(mask == 0)
            action = int(legal[pick_word(w[3], len(legal))])
        return action, kind

    def want(self, action):
        """-> (number of followers step() draws for `action`, the current group without the leader as a bitmask)"""
        g = self.o.current_group() & ~(1 << self.o.leader)
        vac = int(self.env.export(self.shape.M)["status"][action - 1]) if action else 0
        return (min(vac - 1, bin(g).count("1")) if vac > 1 else 0), g

    def draw_followers(self, k, action, fstride):
        """-> (followers row [fstride] int32, -1 padded, for dcm_step; followers list for the oracle, None for the depot)"""
        row = np.full(fstride, -1, np.int32)
        if action == 0:
            return row, None
        want, g = self.want(action)
        ids = [i for i in range(self.shape.A) if g >> i & 1]
        fol = [int(x) for x in np.random.default_rng((self.shape.seed, self.gid, k)).permutation(ids)[:want]]
        row[:want] = fol
        return row, fol

    def decide(self, k, fstride=0, inject=None):
        """-> (action, followers row or None, followers list or None, kind) of decision k; followers under leader-follower on the
        decisions inject_followers_at names (or as `inject` says)"""
        action, kind = self.choose(k)
        if self.protocol == "LF" and (inject_followers_at(k) if inject is None else inject):
            return (action, *self.draw_followers(k, action, fstride), kind)
        return action, None, None, kind

    def apply(self, action, followers=None, next_leader=-1, kind="legal", restart_leader=-1):
        """the decision on the oracle -> (reward, done, used_action); the census; restarts a finished episode (with `restart_leader`
        injected when >= 0)"""
        s, before = self.shape, self.o.current_time
        if self.protocol == "IA":
            r, d, ua, _ = self.o.step(action)
        else:
            rc, r, d, ua, _ = self.o.fused_step(action, followers, next_leader)
            assert rc == 0, (s.name, self.gid, rc)
        if kind != "legal":
            self.ext_census.add(kind)
        if kind.startswith("join_"):
            self.max_joined = max(self.max_joined, int(self.env.export(s.M)["n_mem"][action - 1]))
        if not d and self.o.current_time < before:
            self.ext_census.add("clock_back")
        if followers:
            if len(followers) >= 2:
                self.ext_census.add("inject_want_ge2")
            if s.A - 1 in followers:
                self.ext_census.add("follower_last")
        if d:
            self.last_metrics = np.array([self.o.episode_metrics()[0][k] for k in METRIC_KEYS])
            self.episodes += 1
            self._restart(restart_leader)
        return r, d, ua


def pick_word(word, n):
    """uniform integer in [0, n) from a 32-bit word, as the RNG contract draws (DESIGN.md 5)"""
    return (int(word) * n) >> 32
