"""The reference's individual-agent test loop, worker.py:159-198 `Worker.run_test_IS` (RL_test.py METHOD = 'IA'), restated on top of the
C oracle's per-method calls (oracle/oracle.py `OracleEnv`: next_decision, task_update, agent_update, agent_step, check_finished, mask,
observations) -- the CPU reference the IA tests compare the fused CUDA step with (tests only).

    while not env.finished and env.current_time < max_time:              # worker.py:163
        decision_agents, t = env.next_decision(); env.current_time = t
        env.task_update(); env.agent_update()
        for agent_id in decision_agents:                                 # ascending ids
            if not agent_dic[agent_id]['returned']:
                action = policy(observation of agent_id); env.agent_step(agent_id, action)
                env.task_update(); env.agent_update()
        env.finished = env.check_finished()

One `step()` is one individual decision, so the loop is unrolled decision by decision.  A loop that could only spin (two slots in a row in
which nobody decides) is stopped and flagged `stuck`, as the oracle's leader-follower driver and the CUDA path do.  The built-in policies
follow the RNG contract of DESIGN.md 5 (random: word 0 of block 0 of the decision) and the greedy-nearest rule of the in-kernel policy.
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np

from oracle import canon
from oracle.oracle import OracleEnv, philox


class IAOracle:
    def __init__(self, A, task_xy, depot_xy, req, dur, max_time=100.0):
        self.env = OracleEnv.make(A, task_xy, depot_xy, req, dur, max_time=max_time)
        self.task_xy = np.asarray(task_xy, np.float64).reshape(-1, 2)
        self.depot_xy = np.asarray(depot_xy, np.float64).reshape(2)
        self.A, self.T, self.max_time = int(A), self.task_xy.shape[0], float(max_time)
        self.seed(0)
        self.reset()

    def seed(self, seed, gid=0, episode=0):
        self._seed, self._gid, self._episode = int(seed), int(gid), int(episode)

    # ---- the loop ---------------------------------------------------------------------------------------------------
    def reset(self):
        """clear_decisions + the first slot; returns the first agent to act (-1 if the episode is over at once)."""
        self.env.clear_decisions()
        self.finished, self.done, self.stuck, self.n_steps, self.queue = False, False, False, 0, []
        self._first = True
        self._advance()
        return self.leader

    def _advance(self):
        empty = 0
        while True:
            if not self._first:
                self.finished = self.env.check_finished()                 # end of the slot
            self._first = False
            if self.finished or not self.env.current_time < self.max_time:      # worker.py:163
                self.done, self.queue = True, []
                return
            ids, t = self.env.next_decision()
            self.env.current_time = t
            self.env.task_update()
            self.env.agent_update()
            self.queue = [int(i) for i in ids]
            self._skip_returned()
            if self.queue:
                return
            empty += 1
            if empty >= 2:                                                # nothing can change any more
                self.done, self.stuck, self.queue = True, True, []
                return

    def _skip_returned(self):
        while self.queue and self.env.export()["returned"][self.queue[0]]:
            self.queue.pop(0)

    @property
    def leader(self):
        return self.queue[0] if self.queue else -1

    @property
    def pending(self):
        """bitmask of the deciders of the current slot that have not acted yet (the acting agent included)"""
        return sum(1 << i for i in self.queue)

    @property
    def current_time(self):
        return self.env.current_time

    def step(self, action):
        """agent_step of the acting agent (action 0..T, or -1 random / -2 greedy-nearest), then task_update + agent_update and, once the
        slot's deciders are exhausted, the slot boundary.  -> (reward, done, used_action, mover)"""
        assert not self.done
        a = self.leader
        if action < 0:
            action = self.policy_action(-action)
        reward = self.env.agent_step(a, action)                           # worker.py:186
        self.env.task_update()
        self.env.agent_update()
        self.n_steps += 1
        self.queue.pop(0)
        self._skip_returned()
        if not self.queue:
            self._advance()
        return reward, self.done, action, a

    # ---- what the policy sees, and the built-in policies ----------------------------------------------------------------
    def mask(self):
        return self.env.mask()

    def agent_status(self, agent):
        return self.env.agent_status(agent)

    def task_status(self, agent):
        return self.env.task_status(agent)

    def export(self, MC=canon.MC_CANON):
        return self.env.export(MC)

    def position(self, agent):
        node = int(self.env.export()["node"][agent])
        return self.depot_xy if node < 0 else self.task_xy[node]

    def policy_action(self, policy):
        mask = self.env.mask()
        if policy == 2:               # nearest unmasked task by fma(dy, dy, dx * dx) in fp64, first on ties; the depot if none
            lx, ly = self.position(self.leader)
            best, bd = 0, None
            for j in range(self.T):
                if mask[1 + j]:
                    continue
                dx, dy = float(self.task_xy[j, 0] - lx), float(self.task_xy[j, 1] - ly)
                d2 = float(Fraction(dy) * Fraction(dy) + Fraction(dx * dx))  # one rounding: fma
                if best == 0 or d2 < bd:
                    best, bd = j + 1, d2
            return best
        legal = np.flatnonzero(mask == 0)
        s, g = self._seed, self._gid
        word = int(philox([g & 0xFFFFFFFF, g >> 32, self._episode, (self.n_steps * 8) & 0xFFFFFFFF], [s & 0xFFFFFFFF, s >> 32])[0])
        return int(legal[(word * len(legal)) >> 32])

    def episode_metrics(self):
        """get_episode_reward + perf_metrics (worker.py:103-108) and the number of individual decisions."""
        m, fin = self.env.episode_metrics()
        m["n_steps"] = float(self.n_steps)
        return m, fin
