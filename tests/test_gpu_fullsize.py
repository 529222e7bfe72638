"""Full-size checks (BASELINE.json configurations) through size-independent properties: at these sizes the oracle
would take minutes, so the CUDA path is checked against invariants, exact recurrences evaluated by numpy on the
read-back arrays, linearity/symmetry of the operators, and cross-checks between independent kernels."""
import ctypes as C

import numpy as np
import pytest

import relearn_b200 as R
from relearn_b200 import _lib as L

pytestmark = pytest.mark.gpu

CARTPOLE = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
CONT, TERM, INTR, PAD = L.RL_CONTINUE, L.RL_TERMINATE, L.RL_INTERRUPT, L.RL_PAD


@pytest.fixture(scope="module")
def trpo_batch(ctx):
    """configs[1] cartpole-trpo: 4096 envs x 256 steps = 1 048 576 env-steps, MLP 5-128-2 policy."""
    E, T = 4096, 256
    env = R.build_env(ctx, CARTPOLE, E, seed=77)
    agent = R.ActorCriticConfig().build_agent(env)
    rng = np.random.default_rng(0)
    params = R.init_params(rng, 5, 128, 2)
    agent.policy.policy_fn.set_weights(params)
    agent.critic.state_value_fn.set_weights(R.init_params(rng, 5, 128, 1))
    traj = R.Trajectory(env, T)
    summ = R.rollout(env, agent.actor(), R.HistoryDataBound(T, 0), traj)
    return env, agent, traj, summ, traj.to_host(), params


def test_rollout_invariants_at_bench_size(ctx, trpo_batch):
    """envs/testing.rs check_structured_env at full size + the episode protocol of steps.rs / step_limit.rs."""
    env, agent, traj, summ, host, _ = trpo_batch
    E, T = 4096, 256
    succ, obs, lane_len = host["succ"], host["obs"], host["lane_len"].astype(np.int64)
    valid = succ != PAD
    # every lane took T steps, dropped the dangling one unless it ended an episode
    assert ((lane_len == T) | (lane_len == T - 1)).all()
    assert valid.sum() == lane_len.sum() == summ.num_stored_steps == host["num_steps"]
    assert (valid == (np.arange(T)[:, None] < lane_len[None, :])).all()
    assert np.isin(succ[valid], [CONT, TERM, INTR]).all()
    assert (host["reward"][valid] == 1.0).all() and np.isin(host["action"][valid], [0, 1]).all()
    # observation space: |x| <= 2.4, |theta| <= 12 deg, remaining in (0, 1]
    assert (np.abs(obs[..., 0][valid]) <= 2.4).all() and (np.abs(obs[..., 2][valid]) <= np.float32(np.deg2rad(12.0))).all()
    rem = obs[..., 4]
    assert (rem[valid] > 0).all() and (rem[valid] <= 1).all()
    # remaining counts down by 1/500 inside an episode and restarts at 1 after an episode end
    prev_done = np.vstack([np.ones((1, E), bool), succ[:-1] != CONT])
    steps_left = np.rint(rem.astype(np.float64) * 500).astype(np.int64)
    assert (steps_left[valid & prev_done] == 500).all()
    cont = valid[1:] & ~prev_done[1:]
    assert (steps_left[1:][cont] == steps_left[:-1][cont] - 1).all()
    # an episode is Interrupted exactly when it used its last remaining step, or is the lane's final stored step
    last = np.zeros_like(valid)
    last[lane_len - 1, np.arange(E)] = True
    intr = succ == INTR
    assert (intr <= ((steps_left == 1) | last)).all()
    # summary == host-side recount
    ends = valid & (succ != CONT)
    assert summ.num_stored_episodes == ends.sum()
    assert summ.step_reward.count == E * T and abs(summ.step_reward.mean - 1.0) < 1e-12


def test_fused_rollout_equals_unfused_steps_at_bench_size(ctx, trpo_batch):
    """K2c (fused, 8 threads per env) against K1 (one launch per step) on the same Philox noise and the fused
    kernel's own actions: 1 M observations must agree exactly (both evaluate the same f64 step)."""
    env, agent, traj, summ, host, _ = trpo_batch
    E, T = 4096, 256
    env2 = R.build_env(ctx, CARTPOLE, E, seed=77)
    obs = env2.reset_all()
    for t in range(T):
        stored = host["lane_len"] > t
        np.testing.assert_array_equal(obs[stored], host["obs"][t][stored], err_msg=f"step {t}")
        out = env2.step(host["action"][t])
        keep = host["lane_len"] > t + 1  # the last stored step may have been rewritten to Interrupt
        np.testing.assert_array_equal(out["succ"][keep], host["succ"][t][keep])
        obs = out["obs"]


def test_rollout_is_deterministic_and_shard_invariant_at_bench_size(ctx, trpo_batch):
    env, agent, traj, summ, host, params = trpo_batch
    halves = []
    for off in (0, 2048):
        e = R.build_env(ctx, CARTPOLE, 2048, seed=77, lane_offset=off)
        net = R.Mlp(ctx, 5, [128], 2)
        net.set_weights(params)
        tr = R.Trajectory(e, 256)
        R.rollout(e, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net), R.HistoryDataBound(256, 0), tr)
        halves.append(tr.to_host())
    for k in ("obs", "action", "succ"):
        np.testing.assert_array_equal(np.concatenate([halves[0][k], halves[1][k]], axis=1), host[k])


def test_gae_and_cumsum_recurrences_at_1m_steps(ctx, trpo_batch):
    """packed.rs:336 / critics/mod.rs:158-199 checked exactly by numpy on the whole [256, 4096] arrays:
    y_t = x_t + fl(d * y_{t+1}) inside an episode, y_t = x_t at its last step."""
    env, agent, traj, summ, host, _ = trpo_batch
    E, T = 4096, 256
    succ, valid = host["succ"], host["succ"] != PAD
    gamma, lam = np.float32(0.99), np.float32(0.95)
    adv_d, rtg_d = ctx.alloc(T * E * 4), ctx.alloc(T * E * 4)
    L.check(ctx._lib.rl_gae(traj.handle, agent.critic.state_value_fn.handle, gamma, lam, adv_d.c, rtg_d.c), ctx.handle)
    adv, rtg = adv_d.download((T, E), np.float32), rtg_d.download((T, E), np.float32)
    r = host["reward"]
    nxt = np.vstack([rtg[1:], np.zeros((1, E), np.float32)])
    carry = np.where(succ == CONT, nxt, np.float32(0))
    np.testing.assert_array_equal(rtg[valid], (r + carry * gamma)[valid])
    # advantages: delta_t + fl(lambda*gamma) * A_{t+1}; recover delta and check it against V from an independent forward
    v = agent.critic.state_value_fn.forward(host["obs"].reshape(-1, 5)).reshape(T, E)
    vn = agent.critic.state_value_fn.forward(host["next_obs"].reshape(-1, 5)).reshape(T, E)
    v_next = np.where(succ == CONT, np.vstack([v[1:], np.zeros((1, E), np.float32)]), np.where(succ == INTR, vn, np.float32(0)))
    delta = (r + gamma * v_next) - v
    gl = np.float32(lam * gamma)
    a_next = np.where(succ == CONT, np.vstack([adv[1:], np.zeros((1, E), np.float32)]), np.float32(0))
    np.testing.assert_allclose(adv[valid], (delta + a_next * gl)[valid], rtol=2e-5, atol=2e-5)
    # linearity of the scan: cumsum(a x + y) = a cumsum(x) + cumsum(y)
    rng = np.random.default_rng(1)
    x, y = rng.normal(size=(T, E)).astype(np.float32), rng.normal(size=(T, E)).astype(np.float32)
    def scan(z):
        zd, od = ctx.to_device(z), ctx.alloc(T * E * 4)
        L.check(ctx._lib.rl_discounted_cumsum(ctx.handle, zd.c, C.c_void_p(traj.view().succ), T, E, gamma, od.c), ctx.handle)
        return od.download((T, E), np.float32)
    lhs, rhs = scan(np.float32(2.5) * x + y), np.float32(2.5) * scan(x) + scan(y)
    np.testing.assert_allclose(lhs[valid], rhs[valid], rtol=1e-4, atol=1e-4)


def test_trpo_operator_properties_and_step_at_1m_steps(ctx, trpo_batch):
    """Fisher-vector product: linear, symmetric, positive definite (with the 1e-5 regulariser); the full step
    satisfies conjugate_gradient.rs:218 (loss down, KL <= 0.01) and moves against the gradient -- at N = 1 048 576."""
    env, agent, traj, summ, host, params = trpo_batch
    E, T = 4096, 256
    agent.policy.policy_fn.set_weights(params)
    adv = agent.critic.advantages(traj)
    rng = np.random.default_rng(5)
    P_ = agent.policy.policy_fn.num_params
    u, v = rng.normal(size=P_).astype(np.float32), rng.normal(size=P_).astype(np.float32)
    fu, fv = agent.policy.probe(traj, adv, u), agent.policy.probe(traj, adv, v)
    fuv = agent.policy.probe(traj, adv, (2 * u - 3 * v).astype(np.float32))
    np.testing.assert_allclose(fuv["fvp"], 2 * fu["fvp"] - 3 * fv["fvp"], rtol=2e-4, atol=2e-6)
    np.testing.assert_allclose(np.dot(u.astype(np.float64), fv["fvp"]), np.dot(v.astype(np.float64), fu["fvp"]), rtol=1e-4)
    assert np.dot(u.astype(np.float64), fu["fvp"]) > 0 and np.dot(v.astype(np.float64), fv["fvp"]) > 0
    assert abs(fu["kl"]) < 1e-7  # KL(p0 || p) at theta0
    g = fu["grad"].astype(np.float64)
    net = agent.policy.policy_fn
    log = {}
    status = agent.policy.update(traj, adv, log)
    assert status == L.RL_OK and log["num_steps"] == host["num_steps"]
    assert log["loss_final"] < log["loss_initial"] and 0 <= log["constraint_val_final"] <= 0.01
    assert 0 <= log["num_backtracks"] < 15 and log["cg_iterations"] == 10
    delta = net.get_weights().astype(np.float64) - params
    assert np.dot(delta, g) < 0  # a descent direction of the loss


def test_replay_and_sampler_invariants_at_dqn_size(ctx):
    """configs[2] cartpole-dqn: 65 536 envs, per-lane rings; bookkeeping and sampled minibatches satisfy the
    ReplayBuffer / sample_minibatch contracts (replay.rs:74-126, dqn.rs:280-297) at full size."""
    E, cap = 65536, 96
    env = R.build_env(ctx, CARTPOLE, E, seed=4)
    agent = R.DqnConfig(buffer_capacity=cap, minibatch_steps=100_000, sample_seed=9).build_agent(env)
    agent.action_value_fn.set_weights(R.init_params(np.random.default_rng(2), 5, 128, 2))
    rb = agent.buffer()
    bound = R.HistoryDataBound(40, 5)
    traj = R.Trajectory(env, 45)
    total_stored = 0
    for period in range(4):  # 4 x ~42 steps into rings of 96: the later periods evict
        s = R.rollout(env, agent.actor(), bound, traj)
        rb.write_experience(traj)
        total_stored += s.num_stored_steps
    st = rb.stats()
    assert st.total_step_count == total_stored and st.num_steps <= E * cap and st.num_episodes > E
    for lane in (0, 1, 4095, 65535):
        d = rb.read_lane(lane)
        n = len(d["succ"])
        assert 0 < n <= cap and d["episode_len"].sum() == n
        ends = np.cumsum(d["episode_len"]) - 1
        assert (d["succ"][ends] != CONT).all() and (np.delete(d["succ"], ends) == CONT).all()
    mb = rb.sample(agent.c_cfg(), None, 0)
    M = mb["num_steps"]
    assert 100_000 <= M < 100_000 + cap and mb["num_episodes"] > 0
    assert (mb["succ"][:M] == 0).all() and (mb["succ"][M:] == PAD).all()
    # reward-to-go targets of all-ones rewards: within an episode they follow y_t = 1 + gamma * y_{t+1}, and every
    # target is one of the partial sums G_k = sum_{i<k} gamma^i evaluated in the same f32 recurrence
    gk = np.zeros(cap + 1, np.float32)
    for k in range(1, cap + 1):
        gk[k] = np.float32(1.0) + gk[k - 1] * np.float32(agent.discount_factor)
    assert np.isin(mb["target"], gk[1:]).all()
    stats = agent.batch_update(rb, {})
    assert stats.opt_steps == 50 and np.isfinite(stats.loss_last) and stats.loss_last < stats.loss_first


def test_tensor_core_rollout_at_65536_envs(ctx):
    """configs[2] / configs[4] size: 65 536 envs on the tensor-core rollout kernel (K2t, what `lanes_per_env = 0` picks
    there).  (i) the episode protocol invariants; (ii) K1 (one launch per step) replaying K2t's actions on the same
    Philox noise reproduces all 4.2 M observations and successor codes exactly -- K2t only differs from the FP32-pipe
    kernels in how the logits are rounded, never in the dynamics; (iii) two half-size shards with lane offsets equal
    the full run bit for bit (tile position does not enter the arithmetic)."""
    E, T = 65536, 64
    params = R.init_params(np.random.default_rng(1), 5, 128, 2)
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)

    def run(n, off, lanes):
        env = R.build_env(ctx, CARTPOLE, n, seed=78, lane_offset=off)
        tr = R.Trajectory(env, T)
        summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=lanes),
                         R.HistoryDataBound(T, 0), tr)
        host = tr.to_host()
        tr.close()
        env.close()
        return host, summ

    host, summ = run(E, 0, 0)
    explicit, _ = run(E, 0, L.RL_LANES_TENSOR_CORE)
    for k in ("obs", "action", "succ", "lane_len"):
        np.testing.assert_array_equal(host[k], explicit[k], err_msg=f"auto selection is not K2t at E = {E}: {k}")
    succ, lane_len = host["succ"], host["lane_len"].astype(np.int64)
    valid = succ != PAD
    assert ((lane_len == T) | (lane_len == T - 1)).all()
    assert valid.sum() == lane_len.sum() == summ.num_stored_steps
    assert (valid == (np.arange(T)[:, None] < lane_len[None, :])).all()
    assert (host["reward"][valid] == 1.0).all() and np.isin(host["action"][valid], [0, 1]).all()
    assert summ.num_stored_episodes == (valid & (succ != CONT)).sum()
    assert summ.step_reward.count == E * T
    # both actions occur with a random-init policy, and episodes end
    assert 0.3 < host["action"][valid].mean() < 0.7 and (succ == TERM).sum() > E
    # (ii)
    env2 = R.build_env(ctx, CARTPOLE, E, seed=78)
    obs = env2.reset_all()
    for t in range(T):
        stored = host["lane_len"] > t
        np.testing.assert_array_equal(obs[stored], host["obs"][t][stored], err_msg=f"step {t}")
        out = env2.step(host["action"][t])
        keep = host["lane_len"] > t + 1
        np.testing.assert_array_equal(out["succ"][keep], host["succ"][t][keep])
        obs = out["obs"]
    env2.close()
    # (iii)
    a, _ = run(E // 2, 0, 0)
    b, _ = run(E // 2, E // 2, 0)
    for k in ("obs", "action", "succ"):
        np.testing.assert_array_equal(np.concatenate([a[k], b[k]], axis=1), host[k])


# ------------------------------------------------------------------------------------------------
# Full-size runs against the ORACLE itself (not a sibling kernel): the oracle regenerates the Philox noise per lane,
# so a sample of lanes of the BASELINE-size runs is replayed through it in milliseconds.
# ------------------------------------------------------------------------------------------------
def _check_lanes_against_oracle(host, lanes, T, seed, params, what):
    import oracle as O
    from tests import parity as P

    lib = L.lib()
    for lane in lanes:
        sub = {k: np.ascontiguousarray(host[k][:, lane:lane + 1]) for k in ("obs", "next_obs", "action", "reward", "succ")}
        sub["lane_len"] = host["lane_len"][lane:lane + 1].copy()
        ref = P.oracle_rollout(CARTPOLE, 1, T, 0, actor_kind=O.ACTOR_REPLAY, actions=sub["action"].copy(), philox_seed=seed,
                               lane_offset=int(lane), t0=0)
        # CartPole observations to 1e-6: the device polynomial sin/cos differs from glibc's by <= 1 ulp of f64
        P.compare_traj(sub, ref, obs_rtol=1e-6, obs_atol=1e-7, what=f"{what} lane {lane}")
        awords = np.array([[lib.rl_philox_slot(seed, int(lane), i, 2, 0) & 0xFFFFFFFF for i in range(T)]], dtype=np.uint64).astype(np.uint32)
        checked, near = P.check_policy_consistency(sub, params, 128, 2, awords)
        assert checked == int(sub["lane_len"][0]) and near <= 1, (what, lane, near)


def test_bench_size_rollout_lanes_against_the_oracle(ctx, trpo_batch):
    """configs[1] at its full size (E = 4096, T = 256, the kernel `lanes_per_env = 0` picks = K2q): 64 evenly spaced lanes
    replayed through the CPU oracle -- successor codes, lane lengths, rewards exactly, observations to 1e-6, and every
    action the inverse-CDF choice of the oracle's softmax under the step's Philox uniform."""
    env, agent, traj, summ, host, params = trpo_batch
    _check_lanes_against_oracle(host, np.linspace(0, 4095, 64).astype(int), 256, 77, params, "K2q E=4096")


def test_tensor_core_rollout_lanes_against_the_oracle(ctx):
    """configs[2] size (E = 65 536 on K2t): 64 evenly spaced lanes replayed through the CPU oracle."""
    E, T, seed = 65536, 64, 79
    params = R.init_params(np.random.default_rng(3), 5, 128, 2)
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    env = R.build_env(ctx, CARTPOLE, E, seed=seed)
    env.set_noise_philox(seed, 0)
    tr = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=L.RL_LANES_TENSOR_CORE),
              R.HistoryDataBound(T, 0), tr)
    host = tr.to_host()
    tr.close()
    env.close()
    _check_lanes_against_oracle(host, np.linspace(0, E - 1, 64).astype(int), T, seed, params, "K2t E=65536")


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def test_trpo_and_critic_update_at_1m_steps_against_the_f64_oracle(ctx, trpo_batch):
    """One TRPO step (trpo.rs:97-164: CG, step size, line search) and one 80-step Adam critic update (opt.rs:100-127) on
    the whole 1 048 576-step batch, against oracle/tensor_oracle.py run in f64 on the same batch (CPU, tens of seconds).
    hpv_reg_coeff = 0.1 keeps ten f32 CG iterations well conditioned (tests/test_gpu_update.py explains why the
    reference's own 1e-5 is not): the parameter delta must agree with f64 to 1e-4 relative (north_star's 1e-5 class; the
    small-batch tests show torch's own f32 run at 0.6e-5 .. 3e-5), decisions and log values to 1e-5."""
    torch = pytest.importorskip("torch")
    import oracle as O
    from oracle import tensor_oracle as TO

    env, agent, traj, summ, host, params = trpo_batch
    E, T = 4096, 256
    valid = host["succ"] != PAD
    rng = np.random.default_rng(21)
    vparams = R.init_params(rng, 5, 128, 1)
    critic = R.ValuesOpt(ctx, R.ValuesOptConfig(), 5, 0.99)  # fresh Adam state
    critic.state_value_fn.set_weights(vparams)
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    adv_d = critic.advantages(traj)
    adv = adv_d.download((T, E), np.float32)
    reg = 0.1
    policy = R.Trpo(net, R.TrpoConfig(optimizer_config=R.ConjugateGradientOptimizerConfig(hpv_reg_coeff=reg)))
    log = {}
    status = policy.update(traj, adv_d, log)
    new = net.get_weights()
    obs, act, a = host["obs"][valid], host["action"][valid], adv[valid]
    new64, log64 = TO.trpo_update(params, 5, 128, 2, obs, act, a, cfg=TO.CgConfig(hpv_reg_coeff=reg), dtype=torch.float64)
    d, d64 = new - params, new64 - params.astype(np.float64)
    print(f"N={int(valid.sum())} TRPO: status {status}, backtracks {log['num_backtracks']}/{log64['num_backtracks']}, "
          f"step_size {log['step_size']:.6e}/{log64['step_size']:.6e}, delta rel err vs f64 {_rel(d, d64):.2e}")
    assert status == L.RL_OK and log64["error"] is None and log["num_steps"] == int(valid.sum())
    # (f32 CG can cross the residual tolerance one iteration apart from f64: conjugate_gradient.rs:125-179 stops on r.r < tol)
    assert log["num_backtracks"] == log64["num_backtracks"] and abs(log["cg_iterations"] - log64["cg_iterations"]) <= 1
    np.testing.assert_allclose(log["entropy"], log64["entropy"], rtol=1e-5)
    np.testing.assert_allclose(log["step_size"], log64["step_size"], rtol=1e-4)
    np.testing.assert_allclose(log["loss_initial"], log64["loss_initial"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(log["loss_final"], log64["loss_final"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(log["constraint_val_final"], log64["constraint_val_final"], rtol=1e-4, atol=1e-8)
    assert _rel(d, d64) <= 1e-4
    # critic: 80 Adam steps on mse(V(obs), reward-to-go)
    steps = 80
    stats = critic.update(traj)
    vnew = critic.state_value_fn.get_weights()
    rtg = np.zeros((T, E), np.float32)
    for e in range(E):
        n = int(host["lane_len"][e])
        rtg[:n, e] = O.discounted_cumsum_lane(host["reward"][:n, e], host["succ"][:n, e], np.float32(0.99))
    vnew64, losses64, _ = TO.value_update(vparams, 5, 128, obs, rtg[valid], n_steps=steps, dtype=torch.float64)
    dv, dv64 = vnew - vparams, vnew64 - vparams.astype(np.float64)
    print(f"critic: loss first/last {stats.loss_first:.6f}/{stats.loss_last:.6f} vs f64 {losses64[0]:.6f}/{losses64[-1]:.6f}, "
          f"delta rel err vs f64 {_rel(dv, dv64):.2e}")
    assert stats.num_steps == int(valid.sum()) and stats.opt_steps == steps
    np.testing.assert_allclose(stats.loss_first, losses64[0], rtol=1e-5)
    np.testing.assert_allclose(stats.loss_last, losses64[-1], rtol=1e-4)
    assert _rel(dv, dv64) <= 2e-4
