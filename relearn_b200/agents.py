"""Finite-space agents (src/agents): tabular Q-learning, UCB1 and Beta Thompson sampling; the neural agents (ActorCritic / TRPO / PPO, DQN) live
in `torch_agents.py`."""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L
from .runtime import Context
from .simulation import ActorSpec, Trajectory


class TabularQ:
    """BaseTabularQLearningAgent (src/agents/tabular.rs:84-232).

    `num_replicas = 1` over an env with E > 1 lanes is the reference under `train_parallel`: every lane (worker) acts
    from the one shared table, frozen while a period runs, and `batch_update` folds the lanes' buffers into it one after
    the other in lane order (tabular.rs:197-207) -- bit-identical to the reference's sequential fold.
    `num_replicas = E` trains E INDEPENDENT agents, one table per lane, each seeing only its own lane's data: replicas
    for sweeps, not a faster way to train one agent (sample efficiency per table is that of a single worker)."""

    def __init__(self, ctx: Context, num_replicas: int, num_observations: int, num_actions: int,
                 discount_factor: float, exploration_rate: float = 0.2):
        self.ctx, self._lib = ctx, ctx._lib
        self.shape = (num_replicas, num_observations, num_actions)
        self.exploration_rate = exploration_rate
        h = C.c_void_p()
        L.check(self._lib.rl_tabq_create(ctx.handle, num_replicas, num_observations, num_actions, discount_factor,
                                         C.byref(h)), ctx.handle)
        self.handle = h

    def close(self):
        if self.handle and self.ctx.handle:
            self._lib.rl_tabq_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def actor(self, training: bool = True) -> ActorSpec:
        """Agent::actor(mode) (tabular.rs:148-156)."""
        return ActorSpec(kind=L.RL_ACTOR_TABULAR_EPS_GREEDY, table=self, exploration_rate=self.exploration_rate,
                         training=training)

    def update(self, traj: Trajectory, logger=None):
        """BatchUpdate::batch_update (tabular.rs:197-207)."""
        L.check(self._lib.rl_tabq_update(self.handle, traj.handle), self.ctx.handle)

    batch_update = update

    def min_update_size(self):
        """tabular.rs:190-195: one step (the training loop's min_worker_steps sets the period)."""
        from .simulation import HistoryDataBound

        return HistoryDataBound(1, 0)

    def get_table(self):
        q = np.empty(self.shape, np.float64)
        c = np.empty(self.shape, np.uint64)
        L.check(self._lib.rl_tabq_get_table(self.handle, q.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p)),
                self.ctx.handle)
        return q, c

    def set_table(self, q, counts):
        q = np.ascontiguousarray(q, np.float64)
        c = np.ascontiguousarray(counts, np.uint64)
        L.check(self._lib.rl_tabq_set_table(self.handle, q.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p)),
                self.ctx.handle)


@dataclass
class UCB1AgentConfig:
    """ucb.rs:20-40: `exploration_rate` scales the confidence interval (0.2 after Audibert and Munos)."""

    exploration_rate: float = 0.2

    def build_agent(self, env, num_replicas: int = 1) -> "UCB1Agent":
        """BuildAgent::build_agent (ucb.rs:42-76): tables sized by the env's finite observation / action spaces, rewards
        scaled by its feedback range.  `num_replicas`: 1 = one agent shared by every lane (train_parallel), env.num_envs =
        one independent agent per lane."""
        st = env.structure
        if st.num_observations <= 0:
            raise ValueError("UCB1 needs a finite observation space")
        return UCB1Agent(env.ctx, num_replicas, st.num_observations, st.num_actions, (st.reward_lo, st.reward_hi),
                         self.exploration_rate)


class UCB1Agent:
    """BaseUCB1Agent (src/agents/bandits/ucb.rs:78-243): UCB1 (Auer 2002) applied independently to each state."""

    def __init__(self, ctx: Context, num_replicas: int, num_observations: int, num_actions: int, reward_range,
                 exploration_rate: float = 0.2):
        self.ctx, self._lib = ctx, ctx._lib
        self.shape = (num_replicas, num_observations, num_actions)
        self.exploration_rate = exploration_rate
        h = C.c_void_p()
        L.check(self._lib.rl_ucb1_create(ctx.handle, num_replicas, num_observations, num_actions, float(reward_range[0]),
                                         float(reward_range[1]), exploration_rate, C.byref(h)), ctx.handle)
        self.handle = h

    def close(self):
        if self.handle and self.ctx.handle:
            self._lib.rl_ucb1_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def actor(self, training: bool = True) -> ActorSpec:
        """Agent::actor(mode) (ucb.rs:162-171): Training maximises the upper confidence bound, Evaluation the count."""
        return ActorSpec(kind=L.RL_ACTOR_UCB1, ucb=self, training=training)

    def update(self, traj: Trajectory, logger=None):
        """BatchUpdate::batch_update (ucb.rs:186-199)."""
        L.check(self._lib.rl_ucb1_update(self.handle, traj.handle), self.ctx.handle)

    batch_update = update

    def min_update_size(self):
        """ucb.rs:179-184."""
        from .simulation import HistoryDataBound

        return HistoryDataBound(1, 0)

    def get_tables(self):
        """(state_action_mean_reward f64 [R, S, A], state_action_count u64 [R, S, A], state_visit_count u64 [R, S])."""
        m = np.empty(self.shape, np.float64)
        c = np.empty(self.shape, np.uint64)
        v = np.empty(self.shape[:2], np.uint64)
        L.check(self._lib.rl_ucb1_get_tables(self.handle, m.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p),
                                             v.ctypes.data_as(C.c_void_p)), self.ctx.handle)
        return m, c, v

    def set_tables(self, mean, count, visits):
        m = np.ascontiguousarray(mean, np.float64)
        c = np.ascontiguousarray(count, np.uint64)
        v = np.ascontiguousarray(visits, np.uint64)
        L.check(self._lib.rl_ucb1_set_tables(self.handle, m.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p),
                                             v.ctypes.data_as(C.c_void_p)), self.ctx.handle)


@dataclass
class BetaThompsonSamplingAgentConfig:
    """BetaThompsonSamplingAgentConfig (src/agents/bandits/thompson_sampling.rs:20-39): `num_samples` Beta draws are summed
    per action (1 is plain Thompson sampling; rl2-bandits' "OTS" row uses 10)."""

    num_samples: int = 1

    def build_agent(self, env, num_replicas: int = 1) -> "BetaThompsonSamplingAgent":
        """BuildAgent::build_agent (thompson_sampling.rs:41-75): counts sized by the env's finite observation / action
        spaces, the reward threshold halfway through its feedback range.  `num_replicas`: 1 = one agent shared by every
        lane (train_parallel), env.num_envs = one independent agent per lane."""
        st = env.structure
        if st.num_observations <= 0:
            raise ValueError("Thompson sampling needs a finite observation space")
        return BetaThompsonSamplingAgent(env.ctx, num_replicas, st.num_observations, st.num_actions,
                                         (st.reward_lo, st.reward_hi), self.num_samples)


class BetaThompsonSamplingAgent:
    """BaseBetaThompsonSamplingAgent (src/agents/bandits/thompson_sampling.rs:84-212): a Beta posterior over each state-action
    pair's chance of a reward above the threshold.  The device draws Beta samples with its own sampler (DESIGN section 5):
    exact in distribution, not the reference's bit stream."""

    def __init__(self, ctx: Context, num_replicas: int, num_observations: int, num_actions: int, reward_range,
                 num_samples: int = 1):
        self.ctx, self._lib = ctx, ctx._lib
        self.shape = (num_replicas, num_observations, num_actions)
        self.num_samples = num_samples
        h = C.c_void_p()
        L.check(self._lib.rl_bts_create(ctx.handle, num_replicas, num_observations, num_actions, float(reward_range[0]),
                                        float(reward_range[1]), int(num_samples), C.byref(h)), ctx.handle)
        self.handle = h

    def close(self):
        if self.handle and self.ctx.handle:
            self._lib.rl_bts_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def actor(self, training: bool = True) -> ActorSpec:
        """Agent::actor(mode) (thompson_sampling.rs:139-147): Training samples, Evaluation takes the posterior mean."""
        return ActorSpec(kind=L.RL_ACTOR_BETA_THOMPSON, bts=self, training=training)

    def update(self, traj: Trajectory, logger=None):
        """BatchUpdate::batch_update (thompson_sampling.rs:166-177)."""
        L.check(self._lib.rl_bts_update(self.handle, traj.handle), self.ctx.handle)

    batch_update = update

    def min_update_size(self):
        """thompson_sampling.rs:159-164."""
        from .simulation import HistoryDataBound

        return HistoryDataBound(1, 0)

    def get_counts(self):
        """(low reward count u64 [R, S, A], high reward count u64 [R, S, A])."""
        lo = np.empty(self.shape, np.uint64)
        hi = np.empty(self.shape, np.uint64)
        L.check(self._lib.rl_bts_get_counts(self.handle, lo.ctypes.data_as(C.c_void_p), hi.ctypes.data_as(C.c_void_p)),
                self.ctx.handle)
        return lo, hi

    def set_counts(self, low, high):
        lo = np.ascontiguousarray(low, np.uint64)
        hi = np.ascontiguousarray(high, np.uint64)
        L.check(self._lib.rl_bts_set_counts(self.handle, lo.ctypes.data_as(C.c_void_p), hi.ctypes.data_as(C.c_void_p)),
                self.ctx.handle)


@dataclass
class RandomAgentConfig:
    """RandomAgentConfig (src/agents/random.rs): acts uniformly at random and never learns.  Here only as the inner agent of
    `ResettingMetaAgentConfig`."""


@dataclass
class TabularQLearningAgentConfig:
    """TabularQLearningAgentConfig (src/agents/tabular.rs:43-51).  Here only as the inner agent of
    `ResettingMetaAgentConfig`; `TabularQ` is the standalone agent.  `build_agent` in the reference ignores
    `initial_action_count` and `initial_action_value` and starts every table from value 0 and count 0
    (tabular.rs:61-77,97-111); the fields are kept, with no effect, so that configs read the same as the reference's."""

    exploration_rate: float = 0.2
    initial_action_count: int = 0
    initial_action_value: float = 0.0


@dataclass
class ResettingMetaAgentConfig:
    """ResettingMetaAgentConfig (src/agents/meta.rs:16-70): lifts a bandit agent onto the bandit meta-env.  The inner agent
    is rebuilt at the start of every trial and learns online within it.  `agent_config` is a `RandomAgentConfig`, a
    `TabularQLearningAgentConfig`, a `UCB1AgentConfig` or a `BetaThompsonSamplingAgentConfig`."""

    agent_config: object = field(default_factory=UCB1AgentConfig)

    def build_agent(self, env) -> "ResettingMetaAgent":
        """BuildAgent::build_agent (meta.rs:72-100): checks the inner agent can be built on the inner env structure (one
        observation, the meta-env's actions, its reward range)."""
        from .envs import MetaEnv

        if not isinstance(env.config, MetaEnv):
            raise ValueError("ResettingMetaAgent needs a meta environment (MetaEnv)")
        c = self.agent_config
        if isinstance(c, RandomAgentConfig):
            inner, rate = L.RL_INNER_RANDOM, 0.0
        elif isinstance(c, TabularQLearningAgentConfig):
            inner, rate = L.RL_INNER_TABULAR_Q, float(c.exploration_rate)
        elif isinstance(c, UCB1AgentConfig):
            st = env.structure
            width = st.reward_hi - st.reward_lo
            if not math.isfinite(width) or not width > 0.0:  # BuildAgentError::UnboundedReward (ucb.rs:112-117)
                raise ValueError("UCB1 needs a bounded reward range")
            inner, rate = L.RL_INNER_UCB1, float(c.exploration_rate)
        elif isinstance(c, BetaThompsonSamplingAgentConfig):
            if not 1 <= int(c.num_samples) <= 1024:
                raise ValueError("Thompson sampling needs num_samples in 1 .. 1024")
            return ResettingMetaAgent(L.RL_INNER_BETA_THOMPSON, 0.0, int(c.num_samples))
        else:
            raise ValueError(f"ResettingMetaAgent has no device inner agent for {type(c).__name__}")
        return ResettingMetaAgent(inner, rate)


class ResettingMetaAgent:
    """ResettingMetaAgent (src/agents/meta.rs:102-227).  All its learning happens inside the rollout: each lane rebuilds the
    inner agent at every trial start and folds each pull into it as the next meta observation reports it.  There is
    nothing to update between rollouts."""

    def __init__(self, inner_kind: int, exploration_rate: float, num_samples: int = 1):
        self.inner_kind = inner_kind
        self.exploration_rate = exploration_rate
        self.num_samples = num_samples

    def actor(self, training: bool = True) -> ActorSpec:
        """Agent::actor (meta.rs:103-106): the mode is ignored; the inner agent always acts in training mode."""
        return ActorSpec(kind=L.RL_ACTOR_RESETTING_META, inner_kind=self.inner_kind, exploration_rate=self.exploration_rate,
                         training=training, num_samples=self.num_samples)

    def min_update_size(self):
        """HistoryDataBound::empty (meta.rs:211-213)."""
        from .simulation import HistoryDataBound

        return HistoryDataBound(0, 0)

    def batch_update(self, traj: Trajectory, logger=None):
        """No updates at the meta level (meta.rs:215-226)."""

    update = batch_update
