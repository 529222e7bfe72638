"""Neural agents on the hot path: ActorCriticAgent with a TRPO policy and a ValuesOpt critic.

Mirrors `src/torch/agents` (actor_critic.rs, policies/trpo.rs, critics/opt.rs, critics/mod.rs) and
`src/torch/optimizers` (conjugate_gradient.rs, coptimizer.rs): same config names and defaults, same
log keys, same error behaviour (a failed trust-region step restores the parameters and is reported,
NaN raises).  All tensor work runs in the CUDA library; there is no torch on this path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L
from .envs import BatchedEnv
from .modules import GruLinearConfig, LstmLinearConfig, Mlp, MlpConfig, SeqLinear
from .runtime import Context, DeviceBuffer
from .simulation import ActorSpec, HistoryDataBound, Trajectory


class OptimizerStepError(RuntimeError):
    """src/torch/optimizers/mod.rs:80-94"""

    KINDS = {L.RL_STEP_NAN_LOSS: "NaNLoss", L.RL_STEP_NAN_CONSTRAINT: "NaNConstraint",
             L.RL_STEP_LOSS_NOT_IMPROVING: "LossNotImproving", L.RL_STEP_CONSTRAINT_VIOLATED: "ConstraintViolated"}

    def __init__(self, status: int):
        super().__init__(self.KINDS.get(status, str(status)))
        self.status = status
        self.kind = self.KINDS.get(status, str(status))


@dataclass
class ConjugateGradientOptimizerConfig:
    """conjugate_gradient.rs:41-64"""

    iterations: int = 10
    max_backtracks: int = 15
    backtrack_ratio: float = 0.8
    hpv_reg_coeff: float = 1e-5
    accept_violation: bool = False


@dataclass
class AdamConfig:
    """coptimizer.rs:136-168 (eps is libtorch's default)."""

    learning_rate: float = 1e-3
    beta1: float = 0.9
    beta2: float = 0.999
    weight_decay: float = 0.0
    eps: float = 1e-8


class Adam:
    def __init__(self, mlp: Mlp, cfg: AdamConfig):
        self.ctx, self._lib, self.mlp = mlp.ctx, mlp.ctx._lib, mlp
        c = L.AdamCfg(cfg.learning_rate, cfg.beta1, cfg.beta2, cfg.weight_decay, cfg.eps)
        h = C.c_void_p()
        create = self._lib.rl_adam_create_seq if isinstance(mlp, SeqLinear) else self._lib.rl_adam_create
        L.check(create(mlp.handle, C.byref(c), C.byref(h)), self.ctx.handle)
        self.handle = h

    def close(self):
        if self.handle and self.ctx.handle:
            self._lib.rl_adam_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class TrpoConfig:
    """policies/trpo.rs:17-59"""

    policy_fn_config: object = field(default_factory=MlpConfig)  # MlpConfig | GruLinearConfig | LstmLinearConfig
    optimizer_config: ConjugateGradientOptimizerConfig = field(default_factory=ConjugateGradientOptimizerConfig)
    max_policy_step_kl: float = 0.01

    def build_policy(self, ctx: Context, in_dim: int, out_dim: int) -> "Trpo":
        return Trpo(self.policy_fn_config.build_module(ctx, in_dim, out_dim), self)


class Trpo:
    """Policy (policies/mod.rs:21-53) with the TRPO update (trpo.rs:97-164)."""

    def __init__(self, policy_fn: Mlp, cfg: TrpoConfig):
        self.policy_fn, self.cfg = policy_fn, cfg
        self.ctx, self._lib = policy_fn.ctx, policy_fn.ctx._lib

    @property
    def recurrent(self) -> bool:
        return isinstance(self.policy_fn, SeqLinear)

    def actor(self, lanes_per_env: int = 0) -> ActorSpec:
        """Policy::actor -> PolicyActor (policies/actor.rs)."""
        if self.recurrent:
            return ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=self.policy_fn)
        return ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=self.policy_fn, lanes_per_env=lanes_per_env)

    def _c_cfg(self) -> L.TrpoCfg:
        o = self.cfg.optimizer_config
        return L.TrpoCfg(self.cfg.max_policy_step_kl, o.iterations, o.max_backtracks, o.backtrack_ratio,
                         o.hpv_reg_coeff, 1 if o.accept_violation else 0)

    def update(self, traj: Trajectory, advantages: DeviceBuffer, logger: dict | None = None) -> int:
        """Returns the step status (RL_OK or RL_STEP_*).  NaN statuses raise like the reference's panic
        (trpo.rs:154-159); the others are warnings there and are returned here."""
        stats = L.TrpoStats()
        cfg = self._c_cfg()
        fn = self._lib.rl_trpo_update_seq if self.recurrent else self._lib.rl_trpo_update
        status = L.check(fn(traj.handle, advantages.c, self.policy_fn.handle, C.byref(cfg), C.byref(stats)), self.ctx.handle)
        if logger is not None:
            logger.update({
                "entropy": stats.entropy, "step_size": stats.step_size, "loss_initial": stats.loss_initial,
                "loss_final": stats.loss_final, "constraint_val_final": stats.constraint_val_final,
                "num_backtracks": stats.num_backtracks, "step_scale": stats.step_scale,
                "cg_iterations": stats.cg_iterations, "num_steps": stats.num_steps,
                "policy/update_time": stats.policy_update_ms * 1e-3, "status": status,
            })
        if status in (L.RL_STEP_NAN_LOSS, L.RL_STEP_NAN_CONSTRAINT):
            raise OptimizerStepError(status)
        return status

    def probe(self, traj: Trajectory, advantages: DeviceBuffer, vector: np.ndarray | None = None) -> dict:
        """loss / kl / entropy / flat gradient / Fisher-vector product at the current parameters."""
        P = self.policy_fn.num_params
        loss, kl, ent = C.c_double(), C.c_double(), C.c_double()
        grad = np.zeros(P, np.float32)
        fvp = np.zeros(P, np.float32)
        vec = np.ascontiguousarray(vector, np.float32) if vector is not None else None
        fn = self._lib.rl_trpo_probe_seq if self.recurrent else self._lib.rl_trpo_probe
        L.check(fn(traj.handle, advantages.c, self.policy_fn.handle,
                                        vec.ctypes.data_as(C.c_void_p) if vec is not None else None,
                                        self.cfg.optimizer_config.hpv_reg_coeff, C.byref(loss), C.byref(kl),
                                        C.byref(ent), grad.ctypes.data_as(C.c_void_p),
                                        fvp.ctypes.data_as(C.c_void_p) if vec is not None else None), self.ctx.handle)
        return {"loss": loss.value, "kl": kl.value, "entropy": ent.value, "grad": grad, "fvp": fvp}


@dataclass
class PpoConfig:
    """policies/ppo.rs:14-41"""

    policy_fn_config: object = field(default_factory=MlpConfig)  # MlpConfig | GruLinearConfig | LstmLinearConfig
    optimizer_config: AdamConfig = field(default_factory=AdamConfig)
    opt_steps_per_update: int = 10
    clip_distance: float = 0.2

    def build_policy(self, ctx: Context, in_dim: int, out_dim: int) -> "Ppo":
        return Ppo(self.policy_fn_config.build_module(ctx, in_dim, out_dim), self)


class _AdamPolicy:
    def __init__(self, policy_fn: Mlp, cfg):
        self.policy_fn, self.cfg = policy_fn, cfg
        self.ctx, self._lib = policy_fn.ctx, policy_fn.ctx._lib
        self.optimizer = Adam(policy_fn, cfg.optimizer_config)

    @property
    def recurrent(self) -> bool:
        return isinstance(self.policy_fn, SeqLinear)

    def actor(self, lanes_per_env: int = 0) -> ActorSpec:
        if self.recurrent:
            return ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=self.policy_fn)
        return ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=self.policy_fn, lanes_per_env=lanes_per_env)

    def _log(self, stats, logger):
        if logger is not None:
            logger.update({"entropy": stats.entropy, "loss_first": stats.loss_first, "loss_last": stats.loss_last,
                           "num_steps": stats.num_steps, "policy/update_time": stats.update_ms * 1e-3, "status": L.RL_OK})


class Ppo(_AdamPolicy):
    """Policy with the clipped-surrogate PPO update (ppo.rs:97-147)."""

    def update(self, traj: Trajectory, advantages: DeviceBuffer, logger: dict | None = None) -> int:
        stats = L.PolicyOptStats()
        cfg = L.PpoCfg(self.cfg.opt_steps_per_update, self.cfg.clip_distance)
        fn = self._lib.rl_ppo_update_seq if self.recurrent else self._lib.rl_ppo_update
        L.check(fn(traj.handle, advantages.c, self.policy_fn.handle, self.optimizer.handle, C.byref(cfg), C.byref(stats)),
                self.ctx.handle)
        self._log(stats, logger)
        return L.RL_OK


@dataclass
class ReinforceConfig:
    """policies/reinforce.rs:10-16"""

    policy_fn_config: object = field(default_factory=MlpConfig)  # MlpConfig | GruLinearConfig | LstmLinearConfig
    optimizer_config: AdamConfig = field(default_factory=AdamConfig)

    def build_policy(self, ctx: Context, in_dim: int, out_dim: int) -> "Reinforce":
        return Reinforce(self.policy_fn_config.build_module(ctx, in_dim, out_dim), self)


class Reinforce(_AdamPolicy):
    """Policy with the REINFORCE policy-gradient update (reinforce.rs:64-89)."""

    def update(self, traj: Trajectory, advantages: DeviceBuffer, logger: dict | None = None) -> int:
        stats = L.PolicyOptStats()
        fn = self._lib.rl_reinforce_update_seq if self.recurrent else self._lib.rl_reinforce_update
        L.check(fn(traj.handle, advantages.c, self.policy_fn.handle, self.optimizer.handle, C.byref(stats)), self.ctx.handle)
        self._log(stats, logger)
        return L.RL_OK


@dataclass
class ValuesOptConfig:
    """critics/opt.rs:14-50: GAE(lambda 0.95) advantages, reward-to-go targets, 80 Adam steps, gamma <= 0.99."""

    state_value_fn_config: object = field(default_factory=MlpConfig)  # MlpConfig | GruLinearConfig | LstmLinearConfig
    optimizer_config: AdamConfig = field(default_factory=AdamConfig)
    gae_lambda: float = 0.95          # AdvantageFn::Gae { lambda } (critics/mod.rs:78)
    opt_steps_per_update: int = 80
    max_discount_factor: float = 0.99

    def build_critic(self, ctx: Context, in_dim: int, discount_factor: float) -> "ValuesOpt":
        return ValuesOpt(ctx, self, in_dim, discount_factor)


class ValuesOpt:
    """Critic (critics/mod.rs:20-40) using a gradient-optimized state value function (opt.rs:81-127)."""

    def __init__(self, ctx: Context, cfg: ValuesOptConfig, in_dim: int, discount_factor: float):
        self.ctx, self._lib, self.cfg = ctx, ctx._lib, cfg
        self.state_value_fn = cfg.state_value_fn_config.build_module(ctx, in_dim, 1)
        self.recurrent = isinstance(self.state_value_fn, SeqLinear)
        self.optimizer = Adam(self.state_value_fn, cfg.optimizer_config)
        self.discount_factor = np.float32(min(cfg.max_discount_factor, discount_factor))  # opt.rs:73
        self._adv = self._rtg = None

    def _buffers(self, traj: Trajectory):
        n = traj.step_capacity * traj.env.num_envs * 4
        if self._adv is None or self._adv.nbytes < n:
            self._adv, self._rtg = self.ctx.alloc(n), self.ctx.alloc(n)
        return self._adv, self._rtg

    def advantages(self, traj: Trajectory) -> DeviceBuffer:
        """Critic::advantages: GAE; also leaves the reward-to-go targets of this batch in `self._rtg`."""
        adv, rtg = self._buffers(traj)
        gae = self._lib.rl_gae_seq if self.recurrent else self._lib.rl_gae
        L.check(gae(traj.handle, self.state_value_fn.handle, self.discount_factor, np.float32(self.cfg.gae_lambda), adv.c,
                    rtg.c), self.ctx.handle)
        return adv

    def probe(self, traj: Trajectory, kernel: int = L.RL_PASS_KERNEL_TCGEN05) -> dict:
        """One full-batch pass at the current parameters: mean MSE against the reward-to-go targets and its flat
        gradient, by the tcgen05 kernel (what `update` runs) or the FP32-pipe kernel (diagnostics / parity)."""
        adv, rtg = self._buffers(traj)
        L.check(self._lib.rl_gae(traj.handle, None, self.discount_factor, np.float32(self.cfg.gae_lambda), None, rtg.c),
                self.ctx.handle)
        loss = C.c_double()
        grad = np.zeros(self.state_value_fn.num_params, np.float32)
        L.check(self._lib.rl_value_probe(traj.handle, rtg.c, self.state_value_fn.handle, kernel, C.byref(loss),
                                         grad.ctypes.data_as(C.c_void_p)), self.ctx.handle)
        return {"loss": loss.value, "grad": grad}

    def update(self, traj: Trajectory, logger: dict | None = None):
        """Critic::update: targets = reward-to-go (no_grad), then n Adam steps on the MSE."""
        adv, rtg = self._buffers(traj)
        L.check(self._lib.rl_gae(traj.handle, None, self.discount_factor, np.float32(self.cfg.gae_lambda), None, rtg.c),
                self.ctx.handle)
        stats = L.OptStats()
        upd = self._lib.rl_value_update_seq if self.recurrent else self._lib.rl_value_update
        L.check(upd(traj.handle, rtg.c, self.state_value_fn.handle, self.optimizer.handle, self.cfg.opt_steps_per_update,
                    C.byref(stats)), self.ctx.handle)
        if logger is not None:
            logger.update({"critic/loss": stats.loss_last, "critic/loss_first": stats.loss_first,
                           "critic/update_time": stats.update_ms * 1e-3})
        return stats


@dataclass
class ActorCriticConfig:
    """actor_critic.rs:20-46"""

    policy_config: object = field(default_factory=TrpoConfig)  # TrpoConfig | PpoConfig | ReinforceConfig
    critic_config: ValuesOptConfig = field(default_factory=ValuesOptConfig)
    min_batch_size: HistoryDataBound = field(default_factory=lambda: HistoryDataBound(10_000, 100))

    def build_agent(self, env: BatchedEnv) -> "ActorCriticAgent":
        return ActorCriticAgent(env, self)


class ActorCriticAgent:
    """Agent + BatchUpdate (actor_critic.rs:100-211) over a batched env on one GPU."""

    def __init__(self, env: BatchedEnv, cfg: ActorCriticConfig):
        self.env, self.cfg, self.ctx = env, cfg, env.ctx
        self.policy = cfg.policy_config.build_policy(env.ctx, env.num_features, env.num_actions)
        self.critic = cfg.critic_config.build_critic(env.ctx, env.num_features, env.discount_factor)

    def actor(self, lanes_per_env: int = 0) -> ActorSpec:
        return self.policy.actor(lanes_per_env)

    def min_update_size(self) -> HistoryDataBound:
        return self.cfg.min_batch_size

    def buffer(self, bound: HistoryDataBound) -> Trajectory:
        return Trajectory(self.env, bound.min_steps + bound.slack_steps)

    def batch_update(self, traj: Trajectory, logger: dict | None = None) -> int:
        """actor_critic.rs:176-211: advantages -> policy update -> critic update."""
        adv = self.critic.advantages(traj)
        status = self.policy.update(traj, adv, logger)
        self.critic.update(traj, logger)
        return status


# ------------------------------------------------------------------------------------------------
# DQN (src/torch/agents/dqn.rs, schedules.rs; src/agents/buffers/replay.rs)
# ------------------------------------------------------------------------------------------------
class ReplayBuffer:
    """One ReplayBuffer (replay.rs:11-126) per lane, resident in HBM."""

    def __init__(self, env: BatchedEnv, capacity_per_lane: int):
        self.env, self.ctx, self._lib = env, env.ctx, env.ctx._lib
        self.capacity = int(capacity_per_lane)
        h = C.c_void_p()
        L.check(self._lib.rl_replay_create(env.handle, self.capacity, C.byref(h)), self.ctx.handle)
        self.handle = h

    def close(self):
        if self.handle and self.ctx.handle:
            self._lib.rl_replay_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def write_experience(self, traj: Trajectory):
        """WriteExperience::write_experience of every lane (raises RL_ERR_BUFFER_FULL like
        WriteExperienceError::Full)."""
        L.check(self._lib.rl_replay_append(self.handle, traj.handle), self.ctx.handle)

    def stats(self) -> L.ReplayStats:
        s = L.ReplayStats()
        L.check(self._lib.rl_replay_stats_of(self.handle, C.byref(s)), self.ctx.handle)
        return s

    def total_step_count(self) -> int:
        return int(self.stats().total_step_count)

    def read_lane(self, lane: int) -> dict:
        """Stored steps of one lane, oldest first, and its episode lengths (parity read-back)."""
        F, n = self.env.num_features, self.capacity
        obs, nobs = np.zeros((n, F), np.float32), np.zeros((n, F), np.float32)
        act, succ = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        rew = np.zeros(n, np.float32)
        eps = np.zeros(n, np.uint64)
        s = L.ReplayStats()
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        L.check(self._lib.rl_replay_read_lane(self.handle, lane, n, p(obs), p(act), p(rew), p(succ), p(nobs), p(eps),
                                              C.byref(s)), self.ctx.handle)
        k = int(s.num_steps)
        return {"obs": obs[:k], "next_obs": nobs[:k], "action": act[:k], "reward": rew[:k], "succ": succ[:k],
                "episode_len": eps[:int(s.num_episodes)].astype(np.int64), "total_step_count": int(s.total_step_count)}

    def sample_seq(self, cfg: "L.DqnCfg", q: SeqLinear | None, draw_index: int) -> dict:
        """The same sample_minibatch as padded sequences for a recurrent Q-network, read back to the host: planes
        [L][.][B] with one episode per column (draw order), succ RL_PAD past each episode, targets [L][B]."""
        v, tgt = L.TrajView(), C.c_void_p()
        L.check(self._lib.rl_replay_sample_seq(self.handle, C.byref(cfg), q.handle if q is not None else None, draw_index,
                                               C.byref(v), C.byref(tgt)), self.ctx.handle)
        B, T, F = int(v.num_lanes), int(v.step_capacity), int(v.num_features)
        rd = self.ctx.read
        return {"num_steps": int(v.num_steps), "num_episodes": B, "max_len": T,
                "lane_len": rd(v.lane_len, (B,), np.uint32).astype(np.int64),
                "obs": rd(v.obs, (T, F, B), np.float32).transpose(0, 2, 1).copy(),
                "next_obs": rd(v.next_obs, (T, F, B), np.float32).transpose(0, 2, 1).copy(),
                "action": rd(v.action, (T, B), np.uint8), "reward": rd(v.reward, (T, B), np.float32),
                "succ": rd(v.succ, (T, B), np.uint8), "target": rd(tgt.value, (T, B), np.float32)}

    def sample(self, cfg: "L.DqnCfg", q: Mlp | None, draw_index: int) -> dict:
        """One sample_minibatch (dqn.rs:280-314), read back to the host."""
        v = L.MinibatchView()
        L.check(self._lib.rl_replay_sample(self.handle, C.byref(cfg), q.handle if q is not None else None, draw_index,
                                           C.byref(v)), self.ctx.handle)
        M, cap, F = int(v.num_steps), int(v.capacity), self.env.num_features
        rd = self.ctx.read
        return {"num_steps": M, "num_episodes": int(v.num_episodes),
                "obs": rd(v.obs, (F, cap), np.float32)[:, :M].T.copy(), "action": rd(v.action, (cap,), np.uint8)[:M],
                "target": rd(v.target, (cap,), np.float32)[:M], "succ": rd(v.succ, (cap,), np.uint8)}


@dataclass
class ExplorationRateSchedule:
    """schedules.rs:7-45 (LinearAnnealed; a constant schedule has start == end)."""

    start: float = 1.0
    end: float = 0.1
    period: int = 10_000_000

    def exploration_rate(self, global_steps: int, training: bool = True) -> float:
        return float(L.lib().rl_exploration_rate(self.start, self.end, self.period, global_steps, 1 if training else 0))


@dataclass
class DataCollectionSchedule:
    """schedules.rs:51-68: FirstRest{first, rest}; Constant is first == rest."""

    first: int = 1_000_000
    rest: int = 100_000

    def update_size(self, global_steps: int) -> HistoryDataBound:
        return HistoryDataBound.with_default_slack(self.first if global_steps < self.first else self.rest)


@dataclass
class DqnConfig:
    """dqn.rs:26-72"""

    action_value_fn_config: MlpConfig | GruLinearConfig | LstmLinearConfig = field(default_factory=MlpConfig)
    optimizer_config: AdamConfig = field(default_factory=AdamConfig)
    target_one_step_td: bool = False          # StepValueTarget::RewardToGo is the default
    exploration_rate: ExplorationRateSchedule = field(default_factory=ExplorationRateSchedule)
    minibatch_steps: int = 100_000
    opt_steps_per_update: int = 50
    buffer_capacity: int = 10_000_000         # per buffer (= per lane)
    update_size: DataCollectionSchedule = field(default_factory=DataCollectionSchedule)
    sample_seed: int = 0

    def build_agent(self, env: BatchedEnv) -> "DqnAgent":
        return DqnAgent(env, self)


class DqnAgent:
    """Agent + BatchUpdate (dqn.rs:186-337) over a batched env on one GPU; every lane is one worker with
    its own ReplayBuffer."""

    uses_replay = True  # train_device appends every period's trajectory to the replay rings before batch_update

    def __init__(self, env: BatchedEnv, cfg: DqnConfig):
        self.env, self.cfg, self.ctx, self._lib = env, cfg, env.ctx, env.ctx._lib
        self.action_value_fn = cfg.action_value_fn_config.build_module(env.ctx, env.num_features, env.num_actions)
        self.optimizer = Adam(self.action_value_fn, cfg.optimizer_config)
        self.discount_factor = np.float32(env.discount_factor)  # dqn.rs:178
        self.global_steps = 0

    @property
    def recurrent(self) -> bool:
        return isinstance(self.action_value_fn, SeqLinear)

    def actor(self, training: bool = True) -> ActorSpec:
        """Agent::actor(mode): epsilon is fixed from global_steps at actor creation (dqn.rs:202-212)."""
        eps = self.cfg.exploration_rate.exploration_rate(self.global_steps, training)
        if self.recurrent:
            return ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, seq_net=self.action_value_fn, exploration_rate=eps, training=training)
        return ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, net=self.action_value_fn, exploration_rate=eps, training=training)

    def buffer(self) -> ReplayBuffer:
        return ReplayBuffer(self.env, self.cfg.buffer_capacity)

    def min_update_size(self) -> HistoryDataBound:
        return self.cfg.update_size.update_size(self.global_steps)

    def c_cfg(self, minibatch_steps: int | None = None) -> L.DqnCfg:
        world = max(self.ctx.world_size, 1)
        mb = minibatch_steps if minibatch_steps is not None else -(-self.cfg.minibatch_steps // world)
        return L.DqnCfg(mb, self.cfg.opt_steps_per_update, 1 if self.cfg.target_one_step_td else 0,
                        float(self.discount_factor), self.cfg.sample_seed)

    def batch_update(self, buffer: ReplayBuffer, logger: dict | None = None):
        """dqn.rs:263-337"""
        if logger is not None:
            logger["exploration_rate"] = self.cfg.exploration_rate.exploration_rate(self.global_steps, True)
        self.global_steps = buffer.total_step_count()
        stats = L.OptStats()
        cfg = self.c_cfg()
        update = self._lib.rl_dqn_update_seq if self.recurrent else self._lib.rl_dqn_update
        L.check(update(buffer.handle, self.action_value_fn.handle, self.optimizer.handle, C.byref(cfg), C.byref(stats)),
                self.ctx.handle)
        if logger is not None:
            logger.update({"loss": stats.loss_last, "loss_first": stats.loss_first, "minibatch_steps": stats.num_steps,
                           "agent_update/time": stats.update_ms * 1e-3})
        return stats
