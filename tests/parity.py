"""Shared GPU-vs-oracle comparison helpers (used by tests/ and __graft_entry__.smoke())."""
from __future__ import annotations

import ctypes as C

import numpy as np

import oracle as O
import relearn_b200 as R
from relearn_b200 import _lib as L


def oracle_cfg_for(config) -> O.EnvCfg:
    """Translate a relearn_b200 env config into the oracle's config struct."""
    if isinstance(config, R.CartPoleConfig):
        c = O.cartpole_cfg(config.max_steps_per_episode)
        for k in ("gravity", "mass_cart", "mass_pole", "length_half_pole", "friction_cart", "friction_pole",
                  "time_step", "action_force", "max_pos", "max_angle", "discount_factor"):
            setattr(c, k, getattr(config, k))
        c.step_limit_visible = int(config.step_limit_visible)
        return c
    if isinstance(config, R.Chain):
        return O.chain_cfg(config.size, config.discount_factor)
    if isinstance(config, R.MemoryGame):
        return O.memory_cfg(config.num_actions, config.history_len)
    if isinstance(config, R.MetaEnv):
        dist = O.BANDIT_ONE_HOT if isinstance(config.env_distribution, R.OneHotBandits) else O.BANDIT_UNIFORM_BERNOULLI
        return O.bandit_meta_cfg(config.env_distribution.num_arms, config.episodes_per_trial, dist)
    if isinstance(config, R.PartitionGame):
        return O.partition_cfg()
    raise TypeError(config)


def oracle_rollout(config, E, min_steps, slack, *, actor_kind, actions=None, params=None, hidden=128,
                   env_words=None, actor_words=None, philox_seed=None, lane_offset=0, t0=0,
                   exploration_rate=0.0, q_tables=None, training=True):
    """Run E oracle lanes.  Returns dict of arrays shaped like Trajectory.to_host() plus summary."""
    ocfg = oracle_cfg_for(config)
    env0 = O.make_env(ocfg)
    F = O.lib().ro_env_num_features(C.byref(env0))
    A = O.lib().ro_env_num_actions(C.byref(env0))
    cap = max(min_steps + slack, 1)
    out = {
        "obs": np.zeros((cap, E, F), np.float32), "next_obs": np.zeros((cap, E, F), np.float32),
        "action": np.zeros((cap, E), np.uint8), "reward": np.zeros((cap, E), np.float32),
        "succ": np.full((cap, E), L.RL_PAD, np.uint8), "lane_len": np.zeros(E, np.uint32),
        "n_taken": np.zeros(E, np.uint32),
    }
    total = O.Summary()
    for e in range(E):
        if actor_kind == O.ACTOR_REPLAY:
            actor, _keep = O.replay_actor(actions[:, e])
        elif actor_kind in (O.ACTOR_POLICY, O.ACTOR_EPS_GREEDY_Q):
            actor = O.policy_actor(params, F, hidden, A, kind=actor_kind, exploration_rate=exploration_rate)
        elif actor_kind == O.ACTOR_TABULAR:
            actor = O.Actor()
            actor.kind = O.ACTOR_TABULAR
            qt = np.ascontiguousarray(q_tables[e], np.float64)
            actor.q_table = qt.ctypes.data_as(C.POINTER(C.c_double))
            actor.n_obs, actor.n_act = qt.shape
            actor.exploration_rate = exploration_rate
            actor.training = 1 if training else 0
        else:
            actor = O.Actor()
            actor.kind = O.ACTOR_RANDOM
        if philox_seed is not None:
            rng_env = O.PhiloxRng(philox_seed, lane_offset + e, t0)
            rng_actor = None
        else:
            rng_env = O.ScriptRng(env_words[e] if env_words is not None else np.zeros(0, np.uint32))
            rng_actor = O.ScriptRng(actor_words[e] if actor_words is not None else np.zeros(0, np.uint32))
        r = O.rollout_lane(ocfg, actor, min_steps, slack, rng_env, rng_actor, t0=t0)
        n = r["n"]
        out["lane_len"][e] = n
        out["n_taken"][e] = r["n_taken"]
        out["obs"][:n, e] = r["obs"][:n]
        out["action"][:n, e] = r["action"][:n]
        out["reward"][:n, e] = r["reward"][:n]
        out["succ"][:n, e] = r["succ"][:n]
        intr = r["succ"][:n] == L.RL_INTERRUPT
        out["next_obs"][:n, e][intr] = r["next_obs"][:n][intr]
        O.lib().ro_summary_merge(C.byref(total), C.byref(r["summary"]))
    out["summary"] = total
    out["F"], out["A"] = F, A
    return out


def compare_traj(gpu: dict, ref: dict, *, obs_rtol=0.0, obs_atol=0.0, what=""):
    """Compare Trajectory.to_host() with oracle_rollout() output over the valid slots."""
    np.testing.assert_array_equal(gpu["lane_len"], ref["lane_len"], err_msg=f"{what}: lane lengths")
    T = ref["succ"].shape[0]
    g_succ = gpu["succ"][:T]
    np.testing.assert_array_equal(g_succ, ref["succ"], err_msg=f"{what}: successor codes")
    valid = ref["succ"] != L.RL_PAD
    np.testing.assert_array_equal(gpu["action"][:T][valid], ref["action"][valid], err_msg=f"{what}: actions")
    np.testing.assert_array_equal(gpu["reward"][:T][valid], ref["reward"][valid], err_msg=f"{what}: rewards")
    if obs_rtol == 0.0 and obs_atol == 0.0:
        np.testing.assert_array_equal(gpu["obs"][:T][valid], ref["obs"][valid], err_msg=f"{what}: observations")
    else:
        np.testing.assert_allclose(gpu["obs"][:T][valid], ref["obs"][valid], rtol=obs_rtol, atol=obs_atol,
                                   err_msg=f"{what}: observations")
    intr = ref["succ"] == L.RL_INTERRUPT
    if intr.any():
        if obs_rtol == 0.0 and obs_atol == 0.0:
            np.testing.assert_array_equal(gpu["next_obs"][:T][intr], ref["next_obs"][intr],
                                          err_msg=f"{what}: interrupt observations")
        else:
            np.testing.assert_allclose(gpu["next_obs"][:T][intr], ref["next_obs"][intr], rtol=obs_rtol, atol=obs_atol,
                                       err_msg=f"{what}: interrupt observations")


def compare_summary(gpu_summary: L.StepsSummary, ref: O.Summary, rtol=1e-9):
    for name in ("step_reward", "episode_reward", "episode_length"):
        g, r = getattr(gpu_summary, name), getattr(ref, name)
        assert g.count == r.count, (name, g.count, r.count)
        if r.count:
            np.testing.assert_allclose(g.mean, r.mean, rtol=rtol, atol=1e-12, err_msg=name)
            np.testing.assert_allclose(g.squared_residual_sum, r.m2, rtol=1e-6, atol=1e-6 * max(1.0, r.count),
                                       err_msg=name)


def random_words(rng: np.random.Generator, E: int, n: int) -> np.ndarray:
    return rng.integers(0, 2**32, size=(E, n), dtype=np.uint64).astype(np.uint32)


def mlp_forward_any(params, F, hidden, A, x, activation="relu"):
    """Mlp::forward (mlp.rs:139-151): the C oracle for one ReLU hidden layer, numpy (f64 accumulation, rounded to f32) for
    `hidden_sizes` with several entries or another activation."""
    if isinstance(hidden, (int, np.integer)) and activation == "relu":
        return O.mlp_forward(params, F, hidden, A, x)
    sizes = [hidden] if isinstance(hidden, (int, np.integer)) else list(hidden)
    act = {"relu": lambda v: np.maximum(v, 0.0), "tanh": np.tanh, "sigmoid": lambda v: 1.0 / (1.0 + np.exp(-v)),
           "identity": lambda v: v}[activation]
    h = np.asarray(x, np.float64).reshape(-1, F)
    o, prev = 0, F
    for li, width in enumerate(sizes + [A]):
        w = np.asarray(params[o:o + width * prev], np.float64).reshape(width, prev); o += width * prev
        b = np.asarray(params[o:o + width], np.float64); o += width
        h = h @ w.T + b
        if li < len(sizes):
            h = act(h)
        prev = width
    return h.astype(np.float32)


def check_policy_consistency(host: dict, params, hidden, A, actor_words, atol=2e-6, activation="relu"):
    """Every sampled action must be the inverse-CDF choice of the oracle's softmax for the observation the kernel
    recorded, unless the uniform lies within `atol` of a CDF boundary (rounding near-tie)."""
    T, E, F = host["obs"].shape
    near_ties = 0
    checked = 0
    for e in range(E):
        n = int(host["lane_len"][e])
        # the dropped dangling step also consumed a uniform: n_taken = n or n + 1; index by step
        logits = mlp_forward_any(params, F, hidden, A, host["obs"][:n, e], activation)
        m = logits.max(axis=1, keepdims=True)
        lse = m + np.log(np.exp(logits - m).sum(axis=1, keepdims=True))
        p = np.exp(logits - lse)
        cdf = np.cumsum(p, axis=1)
        u = (actor_words[e, :n] >> 8).astype(np.float32) * np.float32(2.0**-24)
        expect = (u[:, None] >= cdf).sum(axis=1).clip(max=A - 1)
        got = host["action"][:n, e]
        bad = np.nonzero(expect != got)[0]
        for i in bad:
            if np.min(np.abs(cdf[i] - u[i])) < atol:
                near_ties += 1
            else:
                raise AssertionError(f"lane {e} step {i}: action {got[i]} != expected {expect[i]} (u={u[i]}, cdf={cdf[i]})")
        checked += n
    return checked, near_ties


def check_eps_greedy_consistency(host: dict, params, hidden, A, eps, *, actor_words=None, philox=None, activation="relu"):
    """DqnActor (dqn.rs:360-379) on every stored step: the lane's actor stream is walked in order -- `actor_words[e]` for
    replayed noise, or `philox = (seed, lane_offset, t0)` with the step index set per step -- and decides with
    Bernoulli(eps) whether the step explores.  An exploring action must equal the uniform draw over A; any other must be
    the first argmax of the module's outputs for the recorded observation, unless the two outputs lie within
    1e-5 * max(1, |z|) of each other (rounding near-tie).  Returns (steps checked, near-ties)."""
    assert (actor_words is None) != (philox is None)
    lib = O.lib()
    T, E, F = host["obs"].shape
    near_ties = 0
    checked = 0
    for e in range(E):
        n = int(host["lane_len"][e])
        rng = O.ScriptRng(actor_words[e]) if philox is None else O.PhiloxRng(philox[0], philox[1] + e, philox[2])
        q = mlp_forward_any(params, F, hidden, A, host["obs"][:n, e], activation) if n else None
        for i in range(n):
            if philox is not None:
                lib.ro_rng_set_step(rng.ref, philox[2] + i)
            got = int(host["action"][i, e])
            if lib.ro_gen_bool(rng.ref, O.STREAM_ACTOR, eps):
                want = int(lib.ro_gen_range(rng.ref, O.STREAM_ACTOR, A))
                if got != want:
                    raise AssertionError(f"lane {e} step {i}: exploring action {got} != drawn {want}")
                continue
            z = q[i]
            best = int(np.argmax(z))
            if got != best:
                if got < A and abs(float(z[got]) - float(z[best])) < 1e-5 * max(1.0, float(np.abs(z).max())):
                    near_ties += 1
                else:
                    raise AssertionError(f"lane {e} step {i}: greedy action {got} != argmax {best} (q={z})")
        checked += n
    return checked, near_ties


def smoke_check():
    """Small fused CartPole rollout with replayed actions and noise, compared with the oracle."""
    ctx = R.Context(0)
    rng = np.random.default_rng(0)
    E, T = 64, 48
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(20))
    env = R.build_env(ctx, cfg, E, seed=1)
    words = random_words(rng, E, 8 * T)
    env.set_noise_replay(words, None)
    actions = rng.integers(0, 2, size=(T, E), dtype=np.uint8)
    traj = R.Trajectory(env, T)
    n0 = ctx.launch_count
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_REPLAY_ACTIONS, actions=actions), R.HistoryDataBound(T, 0), traj)
    assert ctx.launch_count - n0 >= 2  # the rollout kernel and rollout_finalize_kernel
    host = traj.to_host()
    ref = oracle_rollout(cfg, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=actions, env_words=words)
    compare_traj(host, ref, obs_rtol=1e-6, obs_atol=1e-7, what="smoke")
    compare_summary(summ, ref["summary"])
    # policy-driven rollout in production (Philox) mode
    params = R.init_params(rng, 5, 128, 2)
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    env.set_noise_philox(7, 0)
    n1 = ctx.launch_count
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net), R.HistoryDataBound(T, 0), traj)
    assert summ.step_reward.count == E * T
    assert ctx.launch_count - n1 >= 1  # K2q, which sums the statistics itself
    ctx.close()
