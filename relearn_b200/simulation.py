"""Rollouts and the training loop: Steps + TakeAlignedSteps + write_experience + StepsSummary + train_parallel
(src/simulation).

`rollout()` is one collection period of `train_parallel` (src/simulation/train.rs:108-158) with one GPU lane per
reference worker thread; `train_device()` is the loop around it (train.rs:68-186): collect -> log the merged
StepsSummary -> `batch_update`, with the reference's log ids.
"""
from __future__ import annotations

import ctypes as C
import math
import time
from dataclasses import dataclass

import numpy as np

from . import _lib as L
from .envs import BatchedEnv
from .runtime import Context, DeviceBuffer


@dataclass
class HistoryDataBound:
    """src/agents/buffers/mod.rs:25-113"""

    min_steps: int = 0
    slack_steps: int = 0

    @staticmethod
    def with_default_slack(min_steps: int) -> "HistoryDataBound":
        return HistoryDataBound(min_steps, min(max(min_steps // 100, 5), 1000))

    def max(self, other: "HistoryDataBound") -> "HistoryDataBound":
        return HistoryDataBound(max(self.min_steps, other.min_steps), max(self.slack_steps, other.slack_steps))

    def divide(self, n: int) -> "HistoryDataBound":
        return HistoryDataBound(-(-self.min_steps // n), self.slack_steps)


@dataclass
class ActorSpec:
    """Agent::actor(mode) flattened for the rollout kernel (src/agents/mod.rs:48-114)."""

    kind: int = L.RL_ACTOR_RANDOM
    net: object = None                 # modules.Mlp
    actions: np.ndarray | None = None  # [T, E] u8, REPLAY_ACTIONS
    table: object = None               # agents.TabularQ
    exploration_rate: float = 0.0
    training: bool = True
    lanes_per_env: int = 0
    seq_net: object = None             # modules.GruLinear / LstmLinear (recurrent CATEGORICAL_POLICY / EPS_GREEDY_Q)
    ucb: object = None                 # agents.UCB1Agent
    inner_kind: int = L.RL_INNER_RANDOM  # RESETTING_META: the inner agent (L.RL_INNER_*)
    bts: object = None                 # agents.BetaThompsonSamplingAgent
    num_samples: int = 0               # RESETTING_META with the Thompson-sampling inner agent: Beta draws per arm (1 .. 1024)


class Trajectory:
    """Device-resident history buffer for all lanes (the batched analogue of VecBuffer, vec.rs:15)."""

    def __init__(self, env: BatchedEnv, step_capacity: int):
        self.env, self.ctx, self._lib = env, env.ctx, env.ctx._lib
        h = C.c_void_p()
        L.check(self._lib.rl_traj_create(env.handle, step_capacity, C.byref(h)), self.ctx.handle)
        self.handle = h
        self.step_capacity = step_capacity

    def close(self):
        if self.handle and self.ctx.handle:
            self._lib.rl_traj_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def view(self) -> L.TrajView:
        v = L.TrajView()
        L.check(self._lib.rl_traj_view_of(self.handle, C.byref(v)), self.ctx.handle)
        return v

    def to_host(self) -> dict:
        """Read the whole buffer back: obs/next_obs [T, E, F], action/reward/succ [T, E], lane_len [E]."""
        v = self.view()
        T, E, F = v.step_capacity, v.num_lanes, v.num_features
        rd = self.ctx.read
        return {
            "obs": rd(v.obs, (T, F, E), np.float32).transpose(0, 2, 1).copy(),
            "next_obs": rd(v.next_obs, (T, F, E), np.float32).transpose(0, 2, 1).copy(),
            "action": rd(v.action, (T, E), np.uint8),
            "reward": rd(v.reward, (T, E), np.float32),
            "succ": rd(v.succ, (T, E), np.uint8),
            "lane_len": rd(v.lane_len, (E,), np.uint32),
            "num_steps": int(v.num_steps),
        }

    def load(self, obs, action, reward, succ, next_obs=None):
        """Fill from host arrays obs [T, E, F], action/reward/succ [T, E] (parity entry point)."""
        T, E, F = obs.shape
        bufs = [self.ctx.to_device(np.ascontiguousarray(np.asarray(obs, np.float32).transpose(0, 2, 1))),
                self.ctx.to_device(np.asarray(action, np.uint8)),
                self.ctx.to_device(np.asarray(reward, np.float32)),
                self.ctx.to_device(np.asarray(succ, np.uint8))]
        nb = None
        if next_obs is not None:
            nb = self.ctx.to_device(np.ascontiguousarray(np.asarray(next_obs, np.float32).transpose(0, 2, 1)))
        L.check(self._lib.rl_traj_load(self.handle, T, bufs[0].c, bufs[1].c, bufs[2].c, bufs[3].c,
                                       nb.c if nb else None), self.ctx.handle)
        self.ctx.synchronize()
        for b in bufs + ([nb] if nb else []):
            b.free()


def rollout(env: BatchedEnv, actor: ActorSpec, bound: HistoryDataBound, traj: Trajectory, want_summary: bool = True):
    """One period of experience for every lane.  Returns StepsSummary (or None)."""
    lib = env.ctx._lib
    cfg = L.ActorCfg()
    cfg.kind = actor.kind
    cfg.net = actor.net.handle if actor.net is not None else None
    keep = None
    if actor.actions is not None:
        if isinstance(actor.actions, DeviceBuffer):
            cfg.actions_dev = actor.actions.c
        else:
            keep = env.ctx.to_device(np.ascontiguousarray(actor.actions, np.uint8))
            cfg.actions_dev = keep.c
    cfg.table = actor.table.handle if actor.table is not None else None
    cfg.exploration_rate = actor.exploration_rate
    cfg.training = 1 if actor.training else 0
    cfg.lanes_per_env = actor.lanes_per_env
    cfg.seq_net = actor.seq_net.handle if actor.seq_net is not None else None
    cfg.ucb = actor.ucb.handle if actor.ucb is not None else None
    cfg.inner_kind = actor.inner_kind
    cfg.bts = actor.bts.handle if actor.bts is not None else None
    cfg.num_samples = actor.num_samples
    summ = L.StepsSummary() if want_summary else None
    L.check(lib.rl_rollout(env.handle, C.byref(cfg), L.Bound(bound.min_steps, bound.slack_steps), traj.handle,
                           C.byref(summ) if want_summary else None), env.ctx.handle)
    if keep is not None:
        env.ctx.synchronize()
        keep.free()
    return summ


# ------------------------------------------------------------------------------------------------
# train_parallel / train_serial over device lanes (src/simulation/train.rs:15-186)
# ------------------------------------------------------------------------------------------------
@dataclass
class TrainParallelConfig:
    """train.rs:51-60.  `num_threads` is the number of reference worker threads = device lanes (it must equal the
    env's lane count: a lane IS a worker, with its own buffer and its own noise streams)."""

    num_periods: int = 1
    num_threads: int = 1
    min_worker_steps: int = 0


def _log_summary(summary, logger, collect_s: float) -> None:
    """The `sim/*` block of train_parallel (train.rs:160-178)."""
    sim = logger.with_scope("sim")
    ep = sim.with_scope("ep")
    num_episodes = int(summary.episode_length.count)
    if num_episodes > 0:
        fbk = ep.with_scope("fbk").with_scope("reward")  # RewardSummary::log -> OnlineMeanVariance::log (stats.rs:48-69)
        fbk.log_scalar("mean", summary.episode_reward.mean)
        fbk.log_scalar("stddev", math.sqrt(summary.episode_reward.variance()))
        ep.log_scalar("length_mean", summary.episode_length.mean)
        ep.log_scalar("length_stddev", math.sqrt(summary.episode_length.variance()))
    ep.log_counter_increment("count", num_episodes)
    step = sim.with_scope("step")
    if summary.step_reward.count > 0:
        fbk = step.with_scope("fbk").with_scope("reward")
        fbk.log_scalar("mean", summary.step_reward.mean)
        fbk.log_scalar("stddev", math.sqrt(summary.step_reward.variance()))
    step.log_counter_increment("count", int(summary.step_reward.count))
    sim.log_duration("time", collect_s)


def train_device(agent, env: BatchedEnv, config: TrainParallelConfig, logger=None, on_period=None) -> None:
    """`train_parallel` (train.rs:68-186) with the worker threads as device lanes.

    Per period: `worker_update_size = agent.min_update_size().divide(num_threads).max(min_worker_steps)` (train.rs:111-118),
    one fused rollout collects that much experience on every lane with `agent.actor(Training)` -- created once per period,
    so the policy / table / exploration rate is frozen while the period runs, as in the reference --, the lanes'
    StepsSummaries arrive merged (Chan et al., train.rs:153-156) and are logged under `sim/...`, then
    `agent.batch_update(buffers)` runs and `agent_update/{time,count}` are logged.

    `agent` is any of the package's batch-update agents: `ActorCriticAgent` (trajectory buffer), `DqnAgent` (replay
    rings, one per lane, appended every period), `TabularQ` (one shared table with `num_replicas = 1`, or one per lane).
    `on_period(period_index, summary)` is an optional hook (e.g. checkpointing, early stopping when it returns True)."""
    from .logging import NullLogger

    if config.num_threads != env.num_envs:
        raise ValueError(f"num_threads ({config.num_threads}) must equal the env's lane count ({env.num_envs}): one lane per worker")
    logger = logger if logger is not None else NullLogger()
    replay = None
    traj, traj_cap = None, -1
    try:
        for period in range(config.num_periods):
            collect_start = time.perf_counter()
            bound = agent.min_update_size().divide(config.num_threads).max(HistoryDataBound(config.min_worker_steps, 0))
            cap = bound.min_steps + bound.slack_steps
            if traj is None or cap > traj_cap:
                if traj is not None:
                    traj.close()
                traj, traj_cap = Trajectory(env, cap), cap
            summary = rollout(env, agent.actor(), bound, traj, want_summary=True)
            update_start = time.perf_counter()
            _log_summary(summary, logger, update_start - collect_start)
            if hasattr(agent, "buffer") and getattr(agent, "uses_replay", False):
                if replay is None:
                    replay = agent.buffer()
                replay.write_experience(traj)
                agent.batch_update(replay, _ScopeDict(logger))
            else:
                agent.batch_update(traj, _ScopeDict(logger))
            env.ctx.synchronize()
            upd = logger.with_scope("agent_update")
            upd.log_duration("time", time.perf_counter() - update_start)
            upd.log_counter_increment("count", 1)
            if on_period is not None and on_period(period, summary):
                break
    finally:
        if traj is not None:
            traj.close()
        if replay is not None:
            replay.close()
    logger.flush()


def train_serial(agent, env: BatchedEnv, num_periods: int, logger=None) -> None:
    """`train_serial` (train.rs:15-49): the same loop with the full `min_update_size` on every lane (one lane = the
    reference's single thread)."""
    from .logging import NullLogger

    logger = logger if logger is not None else NullLogger()
    traj = None
    try:
        for _ in range(num_periods):
            bound = agent.min_update_size()
            cap = bound.min_steps + bound.slack_steps
            if traj is None or traj.step_capacity < cap:
                if traj is not None:
                    traj.close()
                traj = Trajectory(env, cap)
            rollout(env, agent.actor(), bound, traj, want_summary=False)
            agent.batch_update(traj, _ScopeDict(logger))
    finally:
        if traj is not None:
            traj.close()
    logger.flush()


class _ScopeDict(dict):
    """The agents' update methods log into a dict (`logger[name] = value`); this forwards every item to a StatsLogger
    as a scalar (durations for `*time`), keeping the dict interface the tests use."""

    def __init__(self, logger):
        super().__init__()
        self._logger = logger

    def __setitem__(self, key, value):
        super().__setitem__(key, value)
        try:
            v = float(value)
        except (TypeError, ValueError):
            return
        if key.endswith("time"):
            self._logger.log_duration(key, v)
        else:
            self._logger.log_scalar(key, v)

    def update(self, other=(), **kw):
        for k, v in dict(other, **kw).items():
            self[k] = v


def pack_history(traj: Trajectory) -> dict:
    """LazyHistoryFeatures (src/torch/agents/features.rs:70-215) of the stored episodes, built on the device by
    `rl_pack_history` and read back: packed observation features [N, F], extended observation features [N + M, F] with
    their is_invalid flags, actions (i64), rewards, and the batch sizes of the two PackedStructures."""
    ctx, lib = traj.ctx, traj.ctx._lib
    v = traj.view()
    T, E, F = int(v.step_capacity), int(v.num_lanes), int(v.num_features)
    cap = max(T * E, 1)
    obs, ext, inv = ctx.alloc(cap * F * 4), ctx.alloc(2 * cap * F * 4), ctx.alloc(2 * cap)
    act, rew = ctx.alloc(cap * 8), ctx.alloc(cap * 4)
    bs, ebs = ctx.alloc((T + 1) * 8), ctx.alloc((T + 2) * 8)
    info = L.PackedInfo()
    L.check(lib.rl_pack_history(traj.handle, obs.c, ext.c, inv.c, act.c, rew.c, bs.c, ebs.c, C.byref(info)), ctx.handle)
    N, M, Lmax = int(info.num_steps), int(info.num_episodes), int(info.max_len)
    out = {
        "num_steps": N, "num_episodes": M, "max_len": Lmax,
        "obs": obs.download((N, F), np.float32), "ext_obs": ext.download((N + M, F), np.float32),
        "ext_invalid": inv.download((N + M,), np.uint8).astype(bool), "action": act.download((N,), np.int64),
        "reward": rew.download((N,), np.float32), "batch_sizes": bs.download((Lmax,), np.int64),
        "ext_batch_sizes": ebs.download((Lmax + 1 if M else 0,), np.int64),
    }
    for b in (obs, ext, inv, act, rew, bs, ebs):
        b.free()
    return out
