"""dcmrta_b200/rollout.py -- batched rollout loop: the device-resident replacement of the Ray CPU workers
(reference worker.py:41-112 `Worker.run_episode`, :200-235 `baseline_test`, runner.py:32-71).

One `BatchedRollout.run` plays one episode in EVERY env of a `BatchedTaskEnv`: per decision one batched policy forward over
the B observations the step kernels wrote, on-device sampling (or argmax), one `dcm_step`.  Nothing crosses PCIe inside the
loop except a done-flag poll every `check_every` decisions (the reference moves every observation to the device and every
action back, worker.py:62-73).  The 7 used slots of the reference's 9-slot episode buffer (worker.py:42, :77-83) live in
preallocated device tensors; the env writes each observation straight into its slot (`set_output_buffers`), so there is no
copy between "observation" and "experience".

Reward and advantage follow worker.py:87-101: the episode reward is -makespan (task_env.py:424), the advantage of every
decision of an episode is reward - greedy-baseline reward of the same instance (GAMMA = 1, parameters.py:6).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

from .batched_env import BatchedTaskEnv
from .policy import greedy_actions, sample_actions


@dataclass
class Episodes:
    """Result of one batched rollout.  L = decisions actually played (max over envs)."""
    reward: torch.Tensor        # [B] f64   -makespan (get_episode_reward, task_env.py:420-425); -current_time where the horizon cut the episode
    metrics: torch.Tensor       # [B,8] f64 reward, success_rate, makespan, time_cost, waiting_time, travel_dist, efficiency, decisions
    ended: torch.Tensor         # [B] bool  False = cut by the buffer horizon before the env was done
    length: int
    # experience (None when record=False); index [t, b]
    agent_obs: torch.Tensor | None = None   # [L,B,A,6]  f32
    task_obs: torch.Tensor | None = None    # [L,B,T+1,5] f32
    mask: torch.Tensor | None = None        # [L,B,T+1]  u8 (1 = forbidden)
    action: torch.Tensor | None = None      # [L,B]      i32
    leader: torch.Tensor | None = None      # [L,B]      i32  (agent id, buffer slot 5 of the reference)
    active: torch.Tensor | None = None      # [L,B]      bool: env b took its t-th decision
    logp: torch.Tensor | None = None        # [L,B,T+1]  f32 log-probabilities of every decision (run(keep_logp=True) only)
    forwarded: int = 0                      # env rows the policy was called on, summed over the decisions (B * length without compaction)


class BatchedRollout:
    def __init__(self, env: BatchedTaskEnv, horizon: int, record: bool = True, check_every: int = 16):
        self.env, self.horizon, self.record, self.check_every = env, int(horizon), bool(record), int(check_every)
        B, A, T, dev = env.B, env.A, env.T, env.device
        L = self.horizon + 1 if record else 2                       # without recording two slots are ping-ponged
        self.agent_obs = torch.zeros(L, B, A, 6, dtype=torch.float32, device=dev)
        self.task_obs = torch.zeros(L, B, T + 1, 5, dtype=torch.float32, device=dev)
        self.mask = torch.zeros(L, B, T + 1, dtype=torch.uint8, device=dev)
        self.action = torch.zeros(self.horizon, B, dtype=torch.int32, device=dev) if record else None
        self.leader = torch.zeros(self.horizon, B, dtype=torch.int32, device=dev) if record else None
        self.active = torch.zeros(self.horizon, B, dtype=torch.bool, device=dev) if record else None

    def _slot(self, t):
        return t if self.record else t & 1

    def _forward_net(self, net, amp):
        """The module the decision loop calls.  amp = "fused": policy_fused.FusedPolicy.  amp = True: a bf16 SHADOW COPY of `net` (weights refreshed here, at the start of every run), fed
        bf16 observations -- not autocast, which keeps LayerNorm in fp32 and casts around every op (14.0 ms per forward of 8,192 envs,
        32 % of it LayerNorm; profiles/r09_policy_forward_profile.txt).  The update always runs on the fp32 network."""
        if not amp:
            return net
        if amp == "fused":
            # the same parameters behind the inference path of policy_fused.py: bf16 GEMMs + one sm_100a kernel for everything between
            # two GEMMs (include/dcmrta_policy.h); re-laid-out weights refreshed here, into buffers that keep their addresses
            from .policy_fused import FusedPolicy
            fused = self.__dict__.setdefault("_fused", {})
            if id(net) not in fused:
                fused[id(net)] = FusedPolicy(net)
            return fused[id(net)].refresh()
        import copy
        shadows = self.__dict__.setdefault("_shadows", {})           # one per network object (the trainer alternates policy and baseline)
        if id(net) not in shadows:
            shadows[id(net)] = copy.deepcopy(net).to(torch.bfloat16).eval()
        shadow = shadows[id(net)]
        with torch.no_grad():
            torch._foreach_copy_(list(shadow.parameters()), list(net.parameters()))
        return shadow

    @staticmethod
    def _logp(fnet, amp, tasks, agents, mask):
        if amp == "fused":
            return fnet(tasks, agents, mask)                         # fp32 observations in (the embedding kernel reads them), fp32 logp out
        if amp:
            return fnet(tasks.to(torch.bfloat16), agents.to(torch.bfloat16), mask).float()
        return fnet(tasks, agents, mask)

    @torch.no_grad()
    def run(self, net, mode: str = "sample", generator: torch.Generator | None = None, amp: bool | str = False, replay: dict | None = None,
            keep_logp: bool = False, sampler: tuple | None = None) -> Episodes:
        """Play one episode per env with `net` (sampling: worker.py:70; greedy: worker.py:222).  The env must not auto-reset.

        sampler=(seed, stream): sample with the Philox kernel (policy_fused.sample, DESIGN.md 5) instead of torch.multinomial on `generator`:
        the action of env b at decision t is a function of (seed, global env id, stream, t) and of its own log-probabilities alone.

        replay (tests: pins this loop to a recorded reference episode): the draws the reference made OUTSIDE the env, injected instead of
        drawn here -- "leader" [L+1,B] int32 (np.random.choice(group), worker.py:54; -1 where the env is done), "followers" [L,B,F] int32
        (-1 padded, task_env.py:331) and, optionally, "action" [L,B] int32 (Categorical.sample, worker.py:70; without it `mode` picks)."""
        env = self.env
        assert not env.auto_reset, "rollouts use one episode per env: create the env with auto_reset=False"
        was_training = net.training
        net.eval()
        fnet = self._forward_net(net, amp)
        s = self._slot(0)
        env.set_output_buffers(self.agent_obs[s], self.task_obs[s], self.mask[s])
        env.reset(leaders=replay["leader"][0] if replay else None)
        horizon = min(self.horizon, replay["followers"].shape[0]) if replay else self.horizon
        draw = None
        if sampler is not None:
            assert mode == "sample" and generator is None, "sampler= replaces the torch generator of a sampled rollout"
            from .policy_fused import draw_tensor, sample
            draw = draw_tensor(int(sampler[0]), int(sampler[1]), 0, env.device)
        logps = [] if keep_logp else None
        t = 0
        while t < horizon:
            s = self._slot(t)
            logp = self._logp(fnet, amp, self.task_obs[s], self.agent_obs[s], self.mask[s].view(torch.bool))
            if keep_logp:
                logps.append(logp.float().clone())
            if replay is not None and "action" in replay:
                act = torch.where(env.done, torch.zeros_like(replay["action"][t]), replay["action"][t]).to(torch.int32)
            elif draw is not None:
                draw[3].fill_(t)                                     # the decision word: Episodes.action[t]
                act = sample(logp.float(), self.mask[s], draw, first_gid=env.first_gid)
            else:
                act = sample_actions(logp.float(), generator) if mode == "sample" else greedy_actions(logp)
            if self.record:
                self.action[t].copy_(act)
                self.leader[t].copy_(env.leader)
                torch.logical_not(env.done, out=self.active[t])
            n = self._slot(t + 1)
            env.set_output_buffers(self.agent_obs[n], self.task_obs[n], self.mask[n])
            if not self.record:                                      # an env that is done keeps a valid (stale) row in both slots
                self.mask[n].copy_(self.mask[s])
            if replay is not None:
                env.step(act, followers=replay["followers"][t], next_leaders=replay["leader"][t + 1])
            else:
                env.step(act)
            t += 1
            if t % self.check_every == 0 and bool(env.done.all()):
                break
        ended = env.done.clone()
        metrics = env.episode_metrics()
        if not bool(ended.all()):
            # Episodes cut by the buffer horizon: scored like the reference scores an episode cut at MAX_TIME (worker.py:45, :87 ->
            # get_episode_reward = -current_time, task_env.py:420-425), from the state they stopped in -- never dropped from training.
            live = env.compute_metrics()
            metrics = torch.where(ended.unsqueeze(1), metrics, live)
        reward = metrics[:, 0].clone()
        if was_training:
            net.train()
        ep = Episodes(reward=reward, metrics=metrics, ended=ended, length=t, forwarded=t * env.B)
        if self.record:
            ep.agent_obs, ep.task_obs, ep.mask = self.agent_obs[:t], self.task_obs[:t], self.mask[:t]
            ep.action, ep.leader, ep.active = self.action[:t], self.leader[:t], self.active[:t]
        if keep_logp:
            ep.logp = torch.stack(logps) if logps else None
        return ep


def sub_batch_sizes(B: int, fractions) -> list:
    """Rows per policy forward the graphed loop is captured at, ascending: the whole batch and ceil(f B) for every fraction 0 < f < 1."""
    return sorted({int(B)} | {max(1, math.ceil(B * f - 1e-9)) for f in fractions if 0 < f < 1})


def rows_for(sizes, n_live: int) -> int:
    """The smallest captured size that holds n_live envs."""
    return min(r for r in sizes if r >= n_live)


class GraphedRollout(BatchedRollout):
    """BatchedRollout whose decision loop -- policy forward, sampling, experience recording, dcm_step -- is captured ONCE in a CUDA graph
    of `unroll` decisions and replayed: the loop issues hundreds of small kernels per decision, and at a few thousand envs the eager
    version is bound by their launches, not by the GPU (DESIGN.md 9).  dcm_step is asynchronous on the caller's stream and synchronises
    nothing, so it is captured like any other kernel launch (its fork to the episode stream and the join become graph edges).

    The env writes each observation into one of two fixed ping-pong slots (graph nodes have fixed addresses); a captured index_copy_
    files it into the episode buffer at a decision counter that lives on the device.  `unroll` is even: the env alternates two
    ended-episode counters from pass to pass, and a replay must leave that parity where the capture found it.  Sampling uses the default
    CUDA generator (graph-safe Philox offsets; seed it with torch.cuda.manual_seed) or, with run(sampler=(seed, stream)), the Philox kernel
    of policy_fused.sample, which reads its draw words from a device tensor: they are set at the start of a run and the decision word is
    bumped inside the graph, and a compacted forward passes its index list, so every env draws what the eager loop would draw for it.

    `fractions`: forward only the envs that are still playing.  Episodes of one batch end at different decisions (20A/50T: 120 +- 9, the
    longest of 8,192 near 150), so late in a rollout most rows of a full-batch forward belong to finished envs.  For every fraction f < 1
    the loop is also captured with the policy called on ceil(f B) gathered rows -- an index list of the live envs, padded with one finished
    env (whose action the step ignores), rebuilt at the done-flag poll that already synchronises every `check_every` decisions -- and each
    replay picks the smallest capture that holds the live envs.  Envs only ever finish between two polls, so the list stays valid."""

    def __init__(self, env: BatchedTaskEnv, horizon: int, record: bool = True, check_every: int = 16, unroll: int = 8,
                 fractions: tuple = (1.0,)):
        assert unroll >= 2 and unroll % 2 == 0
        horizon = -(-int(horizon) // unroll) * unroll                # whole replays
        super().__init__(env, horizon, record, check_every)
        B, A, T, dev = env.B, env.A, env.T, env.device
        self.unroll = unroll
        self.pp = [(torch.zeros(B, A, 6, dtype=torch.float32, device=dev), torch.zeros(B, T + 1, 5, dtype=torch.float32, device=dev),
                    torch.ones(B, T + 1, dtype=torch.uint8, device=dev)) for _ in range(2)]
        self.t_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.sizes = sub_batch_sizes(B, fractions)                                                           # rows per forward, ascending
        self.live = {n: torch.zeros(n, dtype=torch.int64, device=dev) for n in self.sizes if n < B}            # the index lists
        self.draw = torch.zeros(4, dtype=torch.int32, device=dev)                                             # run(sampler=...): the draw words
        self._graphs = {}

    def _act(self, logp, mask, mode, philox, idx=None):
        if mode != "sample":
            return greedy_actions(logp)
        if philox:
            from .policy_fused import sample
            return sample(logp.float(), mask, self.draw, idx, self.env.first_gid)
        return sample_actions(logp.float())

    def _decision(self, net, mode, amp, s, rows=None, philox=False):
        env = self.env
        a, k, m = self.pp[s]
        if rows is None or rows == env.B:
            logp = self._logp(net, amp, k, a, m.view(torch.bool))
            act = self._act(logp, m, mode, philox)
        else:
            idx = self.live[rows]
            ms = m.index_select(0, idx)
            logp = self._logp(net, amp, k.index_select(0, idx), a.index_select(0, idx), ms.view(torch.bool))
            sub = self._act(logp, ms, mode, philox, idx)
            # Envs off the list are done and the step ignores their action -- except in the warm-up before the capture, where the list is
            # arbitrary: give them their first legal action there too (a forbidden depot move would send the whole team home, end the
            # episode and advance the env's Philox episode index, so the recorded rollout would no longer replay on a fresh env).
            act = torch.argmax((m == 0).int(), 1).to(torch.int32).index_copy_(0, idx, sub)
        if self.record:
            self.agent_obs.index_copy_(0, self.t_dev, a.unsqueeze(0)); self.task_obs.index_copy_(0, self.t_dev, k.unsqueeze(0))
            self.mask.index_copy_(0, self.t_dev, m.unsqueeze(0)); self.action.index_copy_(0, self.t_dev, act.unsqueeze(0))
            self.leader.index_copy_(0, self.t_dev, env.leader.unsqueeze(0))
            self.active.index_copy_(0, self.t_dev, torch.logical_not(env.done).unsqueeze(0))
        env.set_output_buffers(*self.pp[1 - s])
        env.step(act)
        self.t_dev.add_(1)
        if philox:
            self.draw[3:].add_(1)

    def _graph(self, net, mode, amp, rows=None, philox=False):
        """net: the module the loop calls (the bf16 shadow / FusedPolicy when amp); its parameters keep their addresses, so refreshing them
        between replays is all an update of the policy needs.  rows: policy rows per decision (None = every env).  philox: sample with
        the Philox kernel (its launch holds the env's first global id)."""
        rows = self.env.B if rows is None else rows
        key = (id(net), mode, amp, rows, self.env.first_gid if philox else None)
        if key not in self._graphs:
            env = self.env
            if rows < env.B:
                self.live[rows].copy_(torch.arange(rows, device=env.device))     # any valid list for the warm-up
            side = torch.cuda.Stream(device=env.device)
            side.wait_stream(torch.cuda.current_stream(env.device))
            with torch.cuda.stream(side):                            # warm-up off the capture: allocator, cuBLAS handles, the env's one-time setup
                env.set_output_buffers(*self.pp[0])
                env.reset()
                self.t_dev.zero_()
                for u in range(2):
                    self._decision(net, mode, amp, u % 2, rows, philox)
            torch.cuda.current_stream(env.device).wait_stream(side)
            g = torch.cuda.CUDAGraph()
            self.t_dev.zero_()
            with torch.cuda.graph(g):
                for u in range(self.unroll):
                    self._decision(net, mode, amp, u % 2, rows, philox)
            self._graphs[key] = g
        return self._graphs[key]

    @torch.no_grad()
    def run(self, net, mode: str = "sample", generator=None, amp: bool | str = False, replay=None, keep_logp: bool = False,
            sampler: tuple | None = None) -> Episodes:
        assert replay is None and not keep_logp and generator is None, \
            "the graphed loop draws from the default CUDA generator or from sampler=(seed, stream), and replays nothing"
        philox = sampler is not None
        assert not philox or mode == "sample"
        env = self.env
        assert not env.auto_reset
        was_training = net.training
        net.eval()
        fnet = self._forward_net(net, amp)
        # all captured before the episode starts (a warm-up resets the env), the full batch FIRST: the policy's workspaces are allocated by
        # the largest forward and only sliced by the smaller ones, so no capture ever holds a buffer that a later one replaced
        graphs = {n: self._graph(fnet, mode, amp, n, philox) for n in sorted(self.sizes, reverse=True)}
        env.set_output_buffers(*self.pp[0])
        env.reset()
        self.t_dev.zero_()
        if philox:
            from .policy_fused import draw_tensor
            self.draw.copy_(draw_tensor(int(sampler[0]), int(sampler[1]), 0, env.device))
        t, rows, forwarded = 0, env.B, 0
        while t < self.horizon:
            graphs[rows].replay()
            t += self.unroll
            forwarded += rows * self.unroll
            if t % self.check_every < self.unroll:
                alive = torch.logical_not(env.done)
                n = int(alive.sum())                                 # the loop's only host synchronisation
                if n == 0:
                    break
                rows = rows_for(self.sizes, n)
                if rows < env.B:                                     # the live envs, then one finished env repeated
                    idx = self.live[rows]
                    idx.copy_(env.done.nonzero()[:1, 0].expand(rows))
                    idx[:n] = alive.nonzero().squeeze(1)
        ended = env.done.clone()
        metrics = env.episode_metrics()
        if not bool(ended.all()):
            live = env.compute_metrics()                             # horizon cut: scored -current_time (see BatchedRollout.run)
            metrics = torch.where(ended.unsqueeze(1), metrics, live)
        if was_training:
            net.train()
        ep = Episodes(reward=metrics[:, 0].clone(), metrics=metrics, ended=ended, length=t, forwarded=forwarded)
        if self.record:
            ep.agent_obs, ep.task_obs, ep.mask = self.agent_obs[:t], self.task_obs[:t], self.mask[:t]
            ep.action, ep.leader, ep.active = self.action[:t], self.leader[:t], self.active[:t]
        return ep


def clone_instances(src: BatchedTaskEnv, dst: BatchedTaskEnv) -> None:
    """copy.deepcopy(self.env) of worker.py:33 for a batch: the baseline env plays the same instances."""
    inst = src.get_instances()
    dst.load_instances(inst["task_xy"], inst["depot_xy"], inst["req"], inst["dur"])
