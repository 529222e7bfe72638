"""ctypes binding of ``librelearn_b200.so`` (the C ABI declared in ``include/relearn_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no fallback:
if the shared object is missing this module raises, and every compute entry point returns
``RL_ERR_CUDA`` when no GPU is present.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librelearn_b200.so")

RL_OK = 0
RL_ERR_INVALID_ARG, RL_ERR_CUDA, RL_ERR_UNSUPPORTED, RL_ERR_OOM, RL_ERR_NCCL, RL_ERR_BUFFER_FULL = 1, 2, 3, 4, 5, 6
RL_STEP_NAN_LOSS, RL_STEP_NAN_CONSTRAINT, RL_STEP_LOSS_NOT_IMPROVING, RL_STEP_CONSTRAINT_VIOLATED = 16, 17, 18, 19
RL_CONTINUE, RL_TERMINATE, RL_INTERRUPT, RL_PAD = 0, 1, 2, 255
RL_LANES_TENSOR_CORE = 128  # rl_actor_cfg.lanes_per_env: the tensor-core rollout kernel (K2t)
RL_LANES_WARP_SPECIALIZED = 160  # the warp-specialised rollout kernel K2q (bit-identical to lanes_per_env 8)
RL_ENV_CARTPOLE, RL_ENV_CHAIN, RL_ENV_MEMORY_GAME, RL_ENV_BANDIT_META, RL_ENV_PARTITION_GAME = 0, 1, 2, 3, 4
RL_NOISE_PHILOX, RL_NOISE_REPLAY = 0, 1
RL_SPACE_INTERVAL, RL_SPACE_INDEX, RL_SPACE_BOOLEAN, RL_SPACE_OPTION_INDEX = 0, 1, 2, 3
RL_ACT_IDENTITY, RL_ACT_RELU, RL_ACT_SIGMOID, RL_ACT_TANH = 0, 1, 2, 3
(RL_ACTOR_REPLAY_ACTIONS, RL_ACTOR_RANDOM, RL_ACTOR_CATEGORICAL_POLICY, RL_ACTOR_EPS_GREEDY_Q,
 RL_ACTOR_TABULAR_EPS_GREEDY, RL_ACTOR_UCB1, RL_ACTOR_RESETTING_META, RL_ACTOR_BETA_THOMPSON) = range(8)
# rl_actor_cfg.inner_kind of RL_ACTOR_RESETTING_META
RL_INNER_RANDOM, RL_INNER_TABULAR_Q, RL_INNER_UCB1, RL_INNER_BETA_THOMPSON = 0, 1, 2, 3
RL_STREAM_ENV_STEP, RL_STREAM_ENV_RESET, RL_STREAM_ACTOR, RL_STREAM_SAMPLER = 0, 1, 2, 3
RL_NCCL_UNIQUE_ID_BYTES = 128
RL_PASS_KERNEL_FFMA, RL_PASS_KERNEL_TCGEN05 = 0, 1

vp = C.c_void_p


class CartPoleCfg(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "gravity", "mass_cart", "mass_pole", "length_half_pole", "friction_cart", "friction_pole", "time_step",
        "action_force", "max_pos", "max_angle", "discount_factor")] + [("max_steps_per_episode", C.c_uint64),
                                                                        ("step_limit_visible", C.c_uint64)]


class ChainCfg(C.Structure):
    _fields_ = [("size", C.c_uint64), ("discount_factor", C.c_double)]


class MemoryCfg(C.Structure):
    _fields_ = [("num_actions", C.c_uint64), ("history_len", C.c_uint64)]


class BanditMetaCfg(C.Structure):
    _fields_ = [("num_arms", C.c_uint64), ("episodes_per_trial", C.c_uint64), ("distribution", C.c_uint64)]


class EnvStructure(C.Structure):
    _fields_ = [("num_features", C.c_int32), ("num_actions", C.c_int32), ("num_observations", C.c_int32),
                ("reward_lo", C.c_double), ("reward_hi", C.c_double), ("discount_factor", C.c_double)]


class StepOut(C.Structure):
    _fields_ = [("obs", vp), ("reward", vp), ("succ", vp), ("next_obs", vp)]


class ActorCfg(C.Structure):
    _fields_ = [("kind", C.c_int32), ("net", vp), ("actions_dev", vp), ("table", vp),
                ("exploration_rate", C.c_double), ("training", C.c_int32), ("lanes_per_env", C.c_int32),
                ("seq_net", vp), ("ucb", vp), ("inner_kind", C.c_int32), ("bts", vp), ("num_samples", C.c_int32)]


class PackedInfo(C.Structure):
    _fields_ = [("num_steps", C.c_uint64), ("num_episodes", C.c_uint64), ("max_len", C.c_uint64)]


class Bound(C.Structure):
    _fields_ = [("min_steps", C.c_uint64), ("slack_steps", C.c_uint64)]


class MeanVar(C.Structure):
    _fields_ = [("mean", C.c_double), ("squared_residual_sum", C.c_double), ("count", C.c_uint64)]

    def variance(self):
        return self.squared_residual_sum / self.count if self.count else None


class StepsSummary(C.Structure):
    _fields_ = [("step_reward", MeanVar), ("episode_reward", MeanVar), ("episode_length", MeanVar),
                ("num_stored_steps", C.c_uint64), ("num_stored_episodes", C.c_uint64)]


class TrajView(C.Structure):
    _fields_ = [("num_lanes", C.c_uint64), ("step_capacity", C.c_uint64), ("num_features", C.c_uint64),
                ("obs", vp), ("action", vp), ("reward", vp), ("succ", vp), ("next_obs", vp), ("lane_len", vp),
                ("num_steps", C.c_uint64)]


class TrpoCfg(C.Structure):
    _fields_ = [("max_policy_step_kl", C.c_double), ("cg_iterations", C.c_uint64), ("max_backtracks", C.c_uint64),
                ("backtrack_ratio", C.c_double), ("hpv_reg_coeff", C.c_double), ("accept_violation", C.c_int32)]


class TrpoStats(C.Structure):
    _fields_ = [("entropy", C.c_double), ("step_size", C.c_double), ("loss_initial", C.c_double),
                ("loss_final", C.c_double), ("constraint_val_final", C.c_double), ("step_scale", C.c_double),
                ("num_backtracks", C.c_int64), ("cg_iterations", C.c_int64), ("num_steps", C.c_uint64),
                ("policy_update_ms", C.c_float)]


class AdamCfg(C.Structure):
    _fields_ = [("learning_rate", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double),
                ("weight_decay", C.c_double), ("eps", C.c_double)]


class OptStats(C.Structure):
    _fields_ = [("loss_first", C.c_double), ("loss_last", C.c_double), ("num_steps", C.c_uint64),
                ("opt_steps", C.c_uint64), ("update_ms", C.c_float)]


class PpoCfg(C.Structure):
    _fields_ = [("opt_steps_per_update", C.c_uint64), ("clip_distance", C.c_double)]


class PolicyOptStats(C.Structure):
    _fields_ = [("entropy", C.c_double), ("loss_first", C.c_double), ("loss_last", C.c_double),
                ("num_steps", C.c_uint64), ("opt_steps", C.c_uint64), ("update_ms", C.c_float)]


class ReplayStats(C.Structure):
    _fields_ = [("num_steps", C.c_uint64), ("num_episodes", C.c_uint64), ("total_step_count", C.c_uint64)]


class DqnCfg(C.Structure):
    _fields_ = [("minibatch_steps", C.c_uint64), ("opt_steps_per_update", C.c_int32),
                ("target_one_step_td", C.c_int32), ("discount_factor", C.c_float), ("sample_seed", C.c_uint64)]


class MinibatchView(C.Structure):
    _fields_ = [("num_steps", C.c_uint64), ("num_episodes", C.c_uint64), ("capacity", C.c_uint64),
                ("obs", vp), ("action", vp), ("target", vp), ("succ", vp)]


P = C.POINTER
st = C.c_int32

# name -> (restype, argtypes); mirrors include/relearn_b200.h one to one
SIGNATURES = {
    "rl_ctx_create": (st, [C.c_int32, vp, P(vp)]),
    "rl_ctx_destroy": (st, [vp]),
    "rl_ctx_synchronize": (st, [vp]),
    "rl_last_error": (C.c_char_p, [vp]),
    "rl_status_str": (C.c_char_p, [st]),
    "rl_version": (C.c_uint32, []),
    "rl_device_count": (C.c_int32, []),
    "rl_ctx_launch_count": (C.c_uint64, [vp]),
    "rl_ctx_device_info": (st, [vp, P(C.c_int32), P(C.c_int32), P(C.c_int32), P(C.c_uint64)]),
    "rl_event_create": (st, [vp, P(vp)]),
    "rl_event_destroy": (st, [vp]),
    "rl_event_record": (st, [vp]),
    "rl_event_elapsed_ms": (st, [vp, vp, P(C.c_float)]),
    "rl_probe_fp32_tflops": (st, [vp, P(C.c_double)]),
    "rl_malloc": (st, [vp, C.c_size_t, P(vp)]),
    "rl_free": (st, [vp, vp]),
    "rl_memcpy_h2d": (st, [vp, vp, vp, C.c_size_t]),
    "rl_memcpy_d2h": (st, [vp, vp, vp, C.c_size_t]),
    "rl_memset": (st, [vp, vp, C.c_int32, C.c_size_t]),
    "rl_malloc_host": (st, [vp, C.c_size_t, P(vp)]),
    "rl_free_host": (st, [vp, vp]),
    "rl_nccl_unique_id": (st, [vp]),
    "rl_ctx_comm_init": (st, [vp, vp, C.c_int32, C.c_int32]),
    "rl_ctx_comm_info": (st, [vp, P(C.c_int32), P(C.c_int32)]),
    "rl_ctx_comm_peer_info": (st, [vp, P(C.c_int32), P(C.c_int32)]),
    "rl_ctx_allreduce_f64": (st, [vp, vp, C.c_size_t]),
    "rl_cartpole_cfg_default": (None, [P(CartPoleCfg), C.c_uint64]),
    "rl_chain_cfg_default": (None, [P(ChainCfg)]),
    "rl_env_create": (st, [vp, C.c_int32, vp, C.c_uint64, C.c_uint64, C.c_uint64, P(vp)]),
    "rl_env_destroy": (st, [vp]),
    "rl_env_structure_of": (st, [vp, P(EnvStructure)]),
    "rl_env_set_noise_replay": (st, [vp, vp, vp, C.c_uint64]),
    "rl_env_set_noise_philox": (st, [vp, C.c_uint64, C.c_uint32]),
    "rl_philox_slot": (C.c_uint64, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int32, C.c_uint32]),
    "rl_env_reset_all": (st, [vp]),
    "rl_env_step": (st, [vp, vp, P(StepOut)]),
    "rl_env_observation": (st, [vp, P(vp)]),
    "rl_env_get_state": (st, [vp, vp, vp]),
    "rl_env_set_state": (st, [vp, vp, vp]),
    "rl_encode_features": (st, [vp, C.c_int32, C.c_uint64, vp, C.c_uint64, vp]),
    "rl_mlp_create": (st, [vp, C.c_int32, P(C.c_int32), C.c_int32, C.c_int32, C.c_int32, P(vp)]),
    "rl_mlp_destroy": (st, [vp]),
    "rl_mlp_num_params": (st, [vp, P(C.c_uint64)]),
    "rl_mlp_set_weights": (st, [vp, vp, C.c_uint64]),
    "rl_mlp_set_weights_async": (st, [vp, vp, C.c_uint64]),
    "rl_mlp_get_weights": (st, [vp, vp, C.c_uint64]),
    "rl_mlp_forward": (st, [vp, vp, C.c_uint64, vp]),
    "rl_grunet_create": (st, [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, P(vp)]),
    "rl_lstmnet_create": (st, [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, P(vp)]),
    "rl_grunet_destroy": (st, [vp]),
    "rl_grunet_num_params": (st, [vp, P(C.c_uint64)]),
    "rl_grunet_set_weights": (st, [vp, vp, C.c_uint64]),
    "rl_grunet_get_weights": (st, [vp, vp, C.c_uint64]),
    "rl_grunet_seq_forward": (st, [vp, vp, vp]),
    "rl_traj_create": (st, [vp, C.c_uint64, P(vp)]),
    "rl_traj_destroy": (st, [vp]),
    "rl_traj_view_of": (st, [vp, P(TrajView)]),
    "rl_traj_load": (st, [vp, C.c_uint64, vp, vp, vp, vp, vp]),
    "rl_rollout": (st, [vp, P(ActorCfg), Bound, vp, P(StepsSummary)]),
    "rl_discounted_cumsum": (st, [vp, vp, vp, C.c_uint64, C.c_uint64, C.c_float, vp]),
    "rl_discounted_cumsum_packed": (st, [vp, vp, C.c_uint64, P(C.c_uint64), C.c_uint64, C.c_float]),
    "rl_gae": (st, [vp, vp, C.c_float, C.c_float, vp, vp]),
    "rl_trpo_cfg_default": (None, [P(TrpoCfg)]),
    "rl_trpo_update": (st, [vp, vp, vp, P(TrpoCfg), P(TrpoStats)]),
    "rl_trpo_probe": (st, [vp, vp, vp, vp, C.c_double, P(C.c_double), P(C.c_double), P(C.c_double), vp, vp]),
    "rl_adam_cfg_default": (None, [P(AdamCfg)]),
    "rl_adam_create": (st, [vp, P(AdamCfg), P(vp)]),
    "rl_adam_destroy": (st, [vp]),
    "rl_value_update": (st, [vp, vp, vp, vp, C.c_int32, P(OptStats)]),
    "rl_value_probe": (st, [vp, vp, vp, C.c_int32, P(C.c_double), vp]),
    "rl_pass_kernel_select": (st, [C.c_int32]),
    "rl_trpo_update_seq": (st, [vp, vp, vp, P(TrpoCfg), P(TrpoStats)]),
    "rl_trpo_probe_seq": (st, [vp, vp, vp, vp, C.c_double, P(C.c_double), P(C.c_double), P(C.c_double), vp, vp]),
    "rl_adam_create_seq": (st, [vp, P(AdamCfg), P(vp)]),
    "rl_value_update_seq": (st, [vp, vp, vp, vp, C.c_int32, P(OptStats)]),
    "rl_gae_seq": (st, [vp, vp, C.c_float, C.c_float, vp, vp]),
    "rl_ppo_cfg_default": (None, [P(PpoCfg)]),
    "rl_ppo_update": (st, [vp, vp, vp, vp, P(PpoCfg), P(PolicyOptStats)]),
    "rl_reinforce_update": (st, [vp, vp, vp, vp, P(PolicyOptStats)]),
    "rl_ppo_update_seq": (st, [vp, vp, vp, vp, P(PpoCfg), P(PolicyOptStats)]),
    "rl_reinforce_update_seq": (st, [vp, vp, vp, vp, P(PolicyOptStats)]),
    "rl_pack_history": (st, [vp, vp, vp, vp, vp, vp, vp, vp, P(PackedInfo)]),
    "rl_tabq_create": (st, [vp, C.c_uint64, C.c_int32, C.c_int32, C.c_double, P(vp)]),
    "rl_tabq_destroy": (st, [vp]),
    "rl_tabq_update": (st, [vp, vp]),
    "rl_tabq_get_table": (st, [vp, vp, vp]),
    "rl_tabq_set_table": (st, [vp, vp, vp]),
    "rl_ucb1_create": (st, [vp, C.c_uint64, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double, P(vp)]),
    "rl_ucb1_destroy": (st, [vp]),
    "rl_ucb1_update": (st, [vp, vp]),
    "rl_ucb1_get_tables": (st, [vp, vp, vp, vp]),
    "rl_ucb1_set_tables": (st, [vp, vp, vp, vp]),
    "rl_bts_create": (st, [vp, C.c_uint64, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_int32, P(vp)]),
    "rl_bts_destroy": (st, [vp]),
    "rl_bts_update": (st, [vp, vp]),
    "rl_bts_get_counts": (st, [vp, vp, vp]),
    "rl_bts_set_counts": (st, [vp, vp, vp]),
    "rl_replay_create": (st, [vp, C.c_uint64, P(vp)]),
    "rl_replay_destroy": (st, [vp]),
    "rl_replay_append": (st, [vp, vp]),
    "rl_replay_stats_of": (st, [vp, P(ReplayStats)]),
    "rl_replay_sample": (st, [vp, P(DqnCfg), vp, C.c_uint32, P(MinibatchView)]),
    "rl_replay_read_lane": (st, [vp, C.c_uint64, C.c_uint64, vp, vp, vp, vp, vp, vp, P(ReplayStats)]),
    "rl_dqn_update": (st, [vp, vp, vp, P(DqnCfg), P(OptStats)]),
    "rl_dqn_update_seq": (st, [vp, vp, vp, P(DqnCfg), P(OptStats)]),
    "rl_replay_sample_seq": (st, [vp, P(DqnCfg), vp, C.c_uint32, P(TrajView), P(vp)]),
    "rl_dqn_probe_seq": (st, [vp, P(DqnCfg), vp, C.c_uint32, P(C.c_double), P(C.c_float)]),
    "rl_exploration_rate": (C.c_double, [C.c_double, C.c_double, C.c_uint64, C.c_uint64, C.c_int32]),
}

_lib = None


class RelearnB200Error(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"relearn_b200 status {status}: {message}")
        self.status = status
        self.message = message


def lib() -> C.CDLL:
    """Load the CUDA library.  Raises if it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RelearnB200Error(
                RL_ERR_CUDA,
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(relearn_b200 has no CPU fallback)",
            )
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here = header/library drift
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status: int, ctx=None) -> int:
    """Raise on hard errors; RL_STEP_* statuses are returned to the caller."""
    if status == RL_OK or status >= RL_STEP_NAN_LOSS:
        return status
    msg = lib().rl_last_error(ctx)
    raise RelearnB200Error(status, msg.decode() if msg else lib().rl_status_str(status).decode())
