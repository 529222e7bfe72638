"""GPU parity: environment dynamics, unfused step kernels and fused rollouts vs the CPU oracle."""
import numpy as np
import pytest

import oracle as O
import relearn_b200 as R
from relearn_b200 import _lib as L
from tests import parity as P

pytestmark = pytest.mark.gpu

CARTPOLE = R.CartPoleConfig().wrap(R.VisibleStepLimit(25))
INT_ENVS = [
    pytest.param(R.Chain(), id="chain"),
    pytest.param(R.Chain(size=9, discount_factor=0.9), id="chain9"),
    pytest.param(R.MemoryGame(2, 1), id="memory-2-1"),
    pytest.param(R.MemoryGame(4, 3), id="memory-4-3"),
    pytest.param(R.MetaEnv(R.UniformBernoulliBandits(2), 3), id="bandit-2x3"),
    pytest.param(R.MetaEnv(R.UniformBernoulliBandits(10), 7), id="bandit-10x7"),
    pytest.param(R.MetaEnv(R.OneHotBandits(3), 4), id="onehot-3x4"),
    pytest.param(R.MetaEnv(R.OneHotBandits(2), 10), id="onehot-2x10"),
    pytest.param(R.PartitionGame(), id="partition"),
]


def _unfused_vs_oracle(ctx, cfg, E, T, rng, exact):
    """Drive rl_env_step with scripted actions; the oracle lane consumes the same word stream."""
    env = R.build_env(ctx, cfg, E, seed=3)
    A = env.num_actions
    words = P.random_words(rng, E, 24 * T + 64)
    env.set_noise_replay(words, None)
    actions = rng.integers(0, A, size=(T, E), dtype=np.uint8)
    ref = P.oracle_rollout(cfg, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=actions, env_words=words)
    obs = env.reset_all()
    for t in range(T):
        live = ref["n_taken"] > t  # every lane takes exactly T steps
        assert live.all()
        # the observation acted on at step t (before finalize the oracle stored it at obs[t])
        stored = ref["lane_len"] > t
        if exact:
            np.testing.assert_array_equal(obs[stored], ref["obs"][t][stored])
        else:
            np.testing.assert_allclose(obs[stored], ref["obs"][t][stored], rtol=1e-6, atol=1e-7)
        out = env.step(actions[t])
        # successor codes: finalize may have rewritten the oracle's last stored step to Interrupt
        unchanged = ref["lane_len"] > t + 1
        np.testing.assert_array_equal(out["succ"][unchanged], ref["succ"][t][unchanged])
        np.testing.assert_array_equal(out["reward"][stored], ref["reward"][t][stored])
        obs = out["obs"]
    env.close()


@pytest.mark.parametrize("cfg", INT_ENVS)
def test_unfused_step_integer_envs_bit_exact(ctx, cfg):
    _unfused_vs_oracle(ctx, cfg, E=97, T=40, rng=np.random.default_rng(11), exact=True)


def test_unfused_step_cartpole(ctx):
    _unfused_vs_oracle(ctx, CARTPOLE, E=300, T=60, rng=np.random.default_rng(12), exact=False)


def test_cartpole_single_step_map_f64(ctx):
    """Single-step map from random oracle states: f64 state within 1e-12 rel (sincos is the only
    non-bit-identical primitive), successor codes and flags exact."""
    import ctypes as C

    rng = np.random.default_rng(5)
    E = 4096
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
    env = R.build_env(ctx, cfg, E, seed=0)
    st = np.stack([rng.uniform(-2.3, 2.3, E), rng.uniform(-2, 2, E), rng.uniform(-0.2, 0.2, E), rng.uniform(-2, 2, E)])
    meta = (rng.integers(2, 500, E).astype(np.uint32) | (rng.integers(0, 2, E).astype(np.uint32) << 31))
    env.set_state(st, meta)
    env.set_noise_replay(P.random_words(rng, E, 16), None)
    actions = rng.integers(0, 2, E).astype(np.uint8)
    out = env.step(actions)
    f64, u32 = env.get_state()
    oenv = O.make_env(P.oracle_cfg_for(cfg))
    lib = O.lib()
    n_cont = 0
    for e in range(E):
        s = O.State()
        s.x, s.xd, s.th, s.thd = st[:, e]
        s.flag = int(meta[e] >> 31)
        s.steps_remaining = int(meta[e] & 0x7FFFFFFF)
        rew = C.c_double()
        rng_o = O.ScriptRng(np.zeros(4, np.uint32))
        succ = lib.ro_env_step(C.byref(oenv), C.byref(s), int(actions[e]), rng_o.ref, C.byref(rew))
        assert succ == out["succ"][e], e
        if succ == O.CONTINUE:
            n_cont += 1
            got = f64[:, e]
            np.testing.assert_allclose(got, [s.x, s.xd, s.th, s.thd], rtol=1e-12, atol=1e-15)
            assert int(u32[e] >> 31) == s.flag
            assert int(u32[e] & 0x7FFFFFFF) == s.steps_remaining
    assert n_cont > E // 2
    env.close()


@pytest.mark.parametrize("cfg", INT_ENVS)
@pytest.mark.parametrize("slack", [0, 5])
def test_fused_rollout_replay_integer_envs_bit_exact(ctx, cfg, slack):
    rng = np.random.default_rng(21)
    E, T = 130, 37
    env = R.build_env(ctx, cfg, E, seed=3)
    words = P.random_words(rng, E, 24 * (T + slack) + 64)
    env.set_noise_replay(words, None)
    actions = rng.integers(0, env.num_actions, size=(T + slack, E), dtype=np.uint8)
    traj = R.Trajectory(env, T + slack)
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_REPLAY_ACTIONS, actions=actions), R.HistoryDataBound(T, slack), traj)
    ref = P.oracle_rollout(cfg, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=actions, env_words=words)
    P.compare_traj(traj.to_host(), ref, what="fused replay")
    P.compare_summary(summ, ref["summary"])
    assert summ.num_stored_steps == int(ref["lane_len"].sum())


@pytest.mark.parametrize("slack", [0, 7])
def test_fused_rollout_replay_cartpole(ctx, slack):
    rng = np.random.default_rng(22)
    E, T = 257, 64
    env = R.build_env(ctx, CARTPOLE, E, seed=3)
    words = P.random_words(rng, E, 8 * (T + slack) + 64)
    env.set_noise_replay(words, None)
    actions = rng.integers(0, 2, size=(T + slack, E), dtype=np.uint8)
    traj = R.Trajectory(env, T + slack)
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_REPLAY_ACTIONS, actions=actions), R.HistoryDataBound(T, slack), traj)
    ref = P.oracle_rollout(CARTPOLE, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=actions, env_words=words)
    P.compare_traj(traj.to_host(), ref, obs_rtol=1e-6, obs_atol=1e-7, what="fused cartpole replay")
    P.compare_summary(summ, ref["summary"])


@pytest.mark.parametrize("cfg", INT_ENVS)
def test_fused_rollout_philox_random_actor_bit_exact(ctx, cfg):
    """Production noise: the oracle regenerates the Philox slots and must reproduce the rollout exactly."""
    E, T, seed, off = 150, 33, 0xC0FFEE, 1000
    env = R.build_env(ctx, cfg, E, seed=seed, lane_offset=off)
    env.set_noise_philox(seed, 17)
    traj = R.Trajectory(env, T + 3)
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_RANDOM), R.HistoryDataBound(T, 3), traj)
    ref = P.oracle_rollout(cfg, E, T, 3, actor_kind=O.ACTOR_RANDOM, philox_seed=seed, lane_offset=off, t0=17)
    P.compare_traj(traj.to_host(), ref, what="philox random")
    P.compare_summary(summ, ref["summary"])


def test_philox_slot_matches_oracle():
    lib, olib = L.lib(), O.lib()
    rng = np.random.default_rng(0)
    for _ in range(200):
        seed, lane = int(rng.integers(0, 2**63)), int(rng.integers(0, 2**40))
        t, stream, draw = int(rng.integers(0, 2**32)), int(rng.integers(0, 3)), int(rng.integers(0, 9))
        assert lib.rl_philox_slot(seed, lane, t, stream, draw) == olib.ro_philox_slot(seed, lane, t, stream, draw)


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32, L.RL_LANES_TENSOR_CORE])
def test_fused_rollout_policy_cartpole_consistent(ctx, lanes):
    """Categorical policy inside the step kernel: every action is the inverse-CDF choice for the recorded
    observation (near-ties within 2e-6 of a CDF edge are tolerated and counted), and the dynamics given those
    actions match the oracle."""
    rng = np.random.default_rng(30 + lanes)
    E, T = 96, 50
    env = R.build_env(ctx, CARTPOLE, E, seed=3)
    ewords = P.random_words(rng, E, 8 * T + 64)
    awords = P.random_words(rng, E, 8 * T + 64)
    env.set_noise_replay(ewords, awords)
    params = R.init_params(rng, 5, 128, 2) * 3.0
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=lanes),
              R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    checked, near = P.check_policy_consistency(host, params, 128, 2, awords)
    assert checked > E * (T - 2) and near <= 3
    # replaying the kernel's own actions through the oracle reproduces the trajectory
    acts = host["action"].copy()
    ref = P.oracle_rollout(CARTPOLE, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=acts, env_words=ewords)
    P.compare_traj(host, ref, obs_rtol=1e-6, obs_atol=1e-7, what=f"policy lanes={lanes}")


def test_eps_greedy_q_actor_chain(ctx):
    rng = np.random.default_rng(50)
    cfg = R.Chain()
    E, T, eps = 80, 30, 0.3
    env = R.build_env(ctx, cfg, E, seed=3)
    ewords = P.random_words(rng, E, 16 * T)
    awords = P.random_words(rng, E, 16 * T)
    env.set_noise_replay(ewords, awords)
    params = R.init_params(rng, 5, 128, 2)
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, net=net, exploration_rate=eps), R.HistoryDataBound(T, 0), traj)
    ref = P.oracle_rollout(cfg, E, T, 0, actor_kind=O.ACTOR_EPS_GREEDY_Q, params=params, env_words=ewords,
                           actor_words=awords, exploration_rate=eps)
    P.compare_traj(traj.to_host(), ref, what="eps-greedy chain")


def test_rollout_lane_sharding_invariance(ctx):
    """Philox noise is keyed by the global lane id: two half-size shards equal one full-size env."""
    cfg, seed, E, T = R.Chain(), 99, 64, 25
    def run(n, off):
        env = R.build_env(ctx, cfg, n, seed=seed, lane_offset=off)
        traj = R.Trajectory(env, T)
        R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_RANDOM), R.HistoryDataBound(T, 0), traj)
        return traj.to_host()
    full, a, b = run(E, 0), run(E // 2, 0), run(E // 2, E // 2)
    for k in ("obs", "action", "reward", "succ"):
        np.testing.assert_array_equal(full[k][:, : E // 2], a[k])
        np.testing.assert_array_equal(full[k][:, E // 2 :], b[k])


def test_actor_file_roundtrip_reproduces_rollout(ctx, tmp_path):
    """A policy written in the reference's actor format (serde TensorDef in CBOR, examples/cartpole-trpo.rs:69-75) and
    read back drives bit-identical rollouts."""
    import relearn_b200 as R
    from relearn_b200 import _lib as L

    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
    params = R.init_params(np.random.default_rng(5), 5, 128, 2)
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    path = str(tmp_path / "actor.cbor")
    R.save_actor(path, net.get_weights())
    loaded = R.load_actor(path)
    net2 = R.Mlp(ctx, loaded["in_dim"], loaded["hidden_sizes"], loaded["out_dim"])
    net2.set_weights(loaded["params"])
    hosts = []
    for n in (net, net2):
        env = R.build_env(ctx, cfg, 256, seed=9)
        traj = R.Trajectory(env, 64)
        R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=n), R.HistoryDataBound(64, 0), traj)
        hosts.append(traj.to_host())
    for k in ("obs", "action", "reward", "succ"):
        assert np.array_equal(hosts[0][k], hosts[1][k]), k


LATENT = R.CartPoleConfig().wrap(R.LatentStepLimit(9))


def test_latent_step_limit_unfused_and_fused(ctx):
    """LatentStepLimit (step_limit.rs:13-90): same interruption after the limit as VisibleStepLimit, but the observation
    keeps CartPole's four features.  Unfused steps and the fused replay rollout against the oracle (limit 9 so that
    Interrupt, Terminate and resets all occur)."""
    env = R.build_env(ctx, LATENT, 8, seed=1)
    assert env.num_features == 4 and env.num_actions == 2
    env.close()
    _unfused_vs_oracle(ctx, LATENT, E=200, T=40, rng=np.random.default_rng(51), exact=False)
    rng = np.random.default_rng(52)
    E, T, slack = 193, 48, 5
    env = R.build_env(ctx, LATENT, E, seed=3)
    words = P.random_words(rng, E, 8 * (T + slack) + 64)
    env.set_noise_replay(words, None)
    actions = rng.integers(0, 2, size=(T + slack, E), dtype=np.uint8)
    traj = R.Trajectory(env, T + slack)
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_REPLAY_ACTIONS, actions=actions), R.HistoryDataBound(T, slack), traj)
    ref = P.oracle_rollout(LATENT, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=actions, env_words=words)
    host = traj.to_host()
    assert host["obs"].shape[-1] == 4 and (host["succ"] == L.RL_INTERRUPT).any() and (host["succ"] == L.RL_TERMINATE).any()
    P.compare_traj(host, ref, obs_rtol=1e-6, obs_atol=1e-7, what="fused cartpole latent limit")
    P.compare_summary(summ, ref["summary"])


@pytest.mark.parametrize("lanes", [1, 8, L.RL_LANES_TENSOR_CORE])
def test_latent_step_limit_policy_rollout(ctx, lanes):
    """A 4-feature policy (MLP 4 -> 128 -> 2) inside the fused step kernel under the latent limit."""
    rng = np.random.default_rng(60 + lanes)
    E, T = 96, 40
    env = R.build_env(ctx, LATENT, E, seed=3)
    ewords, awords = P.random_words(rng, E, 8 * T + 64), P.random_words(rng, E, 8 * T + 64)
    env.set_noise_replay(ewords, awords)
    params = R.init_params(rng, 4, 128, 2) * 3.0
    net = R.Mlp(ctx, 4, [128], 2)
    net.set_weights(params)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=lanes), R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    checked, near = P.check_policy_consistency(host, params, 128, 2, awords)
    assert checked > E * (T - 2) and near <= 3
    ref = P.oracle_rollout(LATENT, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), env_words=ewords)
    P.compare_traj(host, ref, obs_rtol=1e-6, obs_atol=1e-7, what=f"latent policy lanes={lanes}")


# ------------------------------------------------------------------------------------------------
# K2t: the tensor-core rollout (hidden layer of the policy on tcgen05, 128-env tiles)
# ------------------------------------------------------------------------------------------------
SHORT = R.CartPoleConfig().wrap(R.VisibleStepLimit(23))


@pytest.mark.parametrize("E,T,slack", [(300, 60, 7), (128, 31, 0), (1, 17, 3), (1031, 40, 5)])
def test_tc_rollout_policy_replay_ragged(ctx, E, T, slack):
    """K2t on env counts that do not fill its 128-env tiles, with slack (ragged lane lengths), Interrupts (limit 23),
    Terminates and resets: actions are the inverse-CDF choices of the oracle's softmax for the recorded observations,
    and the oracle reproduces the whole trajectory (dangling-step finalisation included) from those actions."""
    rng = np.random.default_rng(70 + E)
    env = R.build_env(ctx, SHORT, E, seed=3)
    nw = 8 * (T + slack) + 64
    ewords, awords = P.random_words(rng, E, nw), P.random_words(rng, E, nw)
    env.set_noise_replay(ewords, awords)
    params = R.init_params(rng, 5, 128, 2) * 3.0
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    traj = R.Trajectory(env, T + slack)
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=L.RL_LANES_TENSOR_CORE),
                     R.HistoryDataBound(T, slack), traj)
    host = traj.to_host()
    checked, near = P.check_policy_consistency(host, params, 128, 2, awords)
    assert checked >= E * (T - 1) and near <= 3
    # the action slot of a dropped dangling step keeps the action that was taken, so the oracle can replay it
    acts = host["action"][: T + slack].copy()
    ref = P.oracle_rollout(SHORT, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=acts, env_words=ewords)
    P.compare_traj(host, ref, obs_rtol=1e-6, obs_atol=1e-7, what=f"K2t E={E}")
    assert summ.num_stored_steps == int(host["lane_len"].sum())
    assert E < 100 or ((host["succ"] == L.RL_INTERRUPT).any() and (host["succ"] == L.RL_TERMINATE).any())


def test_tc_rollout_equals_fp32_rollout_philox(ctx):
    """Production (Philox) noise: K2t and the FP32-pipe kernel (K2c, one thread per env) see the same noise and differ
    only in the rounding of the logits, so lanes agree bit for bit except where a uniform fell within rounding of the
    CDF edge -- and there the first difference must be that action, with identical observations up to it."""
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
    E, T = 4096, 96
    params = R.init_params(np.random.default_rng(81), 5, 128, 2) * 2.0
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    hosts, summs = [], []
    for lanes in (1, L.RL_LANES_TENSOR_CORE):
        env = R.build_env(ctx, cfg, E, seed=11, lane_offset=5000)
        env.set_noise_philox(11, 3)
        traj = R.Trajectory(env, T)
        summs.append(R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=lanes),
                               R.HistoryDataBound(T, 0), traj))
        hosts.append(traj.to_host())
        env.close()
    a, b = hosts
    same = (a["action"] == b["action"]).all(axis=0) & (a["succ"] == b["succ"]).all(axis=0) & \
        (a["obs"] == b["obs"]).all(axis=(0, 2))
    assert same.mean() >= 0.995, same.mean()
    for e in np.nonzero(~same)[0]:
        t = int(np.argmax(a["action"][:, e] != b["action"][:, e]))
        assert a["action"][t, e] != b["action"][t, e]
        np.testing.assert_array_equal(a["obs"][: t + 1, e], b["obs"][: t + 1, e])
    assert summs[0].step_reward.count == summs[1].step_reward.count == E * T
    if same.all():
        assert summs[0].episode_length.count == summs[1].episode_length.count


def test_tc_rollout_eps_greedy_cartpole(ctx):
    """DqnActor (dqn.rs:360-379) on K2t: exploration draws replayed, greedy choice = argmax of the oracle's Q values
    unless the two values are within rounding of each other."""
    rng = np.random.default_rng(90)
    E, T, eps = 200, 40, 0.25
    ewords, awords = P.random_words(rng, E, 8 * T + 64), P.random_words(rng, E, 8 * T + 64)
    params = R.init_params(rng, 5, 128, 2) * 2.0
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    hosts = []
    for lanes in (1, L.RL_LANES_TENSOR_CORE):
        env = R.build_env(ctx, SHORT, E, seed=3)
        env.set_noise_replay(ewords, awords)
        traj = R.Trajectory(env, T)
        R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, net=net, exploration_rate=eps, lanes_per_env=lanes),
                  R.HistoryDataBound(T, 0), traj)
        hosts.append(traj.to_host())
    a, b = hosts
    differing = 0
    for e in range(E):
        n = int(a["lane_len"][e])
        if np.array_equal(a["action"][:n, e], b["action"][:n, e]) and b["lane_len"][e] == n:
            np.testing.assert_array_equal(a["obs"][:n, e], b["obs"][:n, e])
            continue
        differing += 1
        t = int(np.argmax(a["action"][:, e] != b["action"][:, e]))
        q = O.mlp_forward(params, 5, 128, 2, b["obs"][t : t + 1, e])[0]
        assert abs(q[1] - q[0]) < 1e-5 * max(1.0, abs(q).max()), (e, t, q)
    assert differing <= 2
    ref = P.oracle_rollout(SHORT, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=b["action"].copy(), env_words=ewords)
    P.compare_traj(b, ref, obs_rtol=1e-6, obs_atol=1e-7, what="K2t eps-greedy")


@pytest.mark.parametrize("cfg", [pytest.param(R.PartitionGame(), id="partition-23f"), pytest.param(R.MemoryGame(4, 3), id="memory-7f")])
def test_fused_rollout_policy_other_envs_consistent(ctx, cfg):
    """The generic fused kernel (K2a) with a categorical MLP policy on envs with wider observations / more actions:
    every action is the inverse-CDF choice of the oracle's softmax for the recorded observation, and replaying the
    actions through the oracle reproduces the trajectory bit for bit."""
    rng = np.random.default_rng(95)
    E, T = 90, 30
    env = R.build_env(ctx, cfg, E, seed=3)
    F, A = env.num_features, env.num_actions
    W = 24 * T + 64  # PartitionGame draws ten words per step
    ewords, awords = P.random_words(rng, E, W), P.random_words(rng, E, W)
    env.set_noise_replay(ewords, awords)
    params = R.init_params(rng, F, 64, A) * 3.0
    net = R.Mlp(ctx, F, [64], A)
    net.set_weights(params)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net), R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    checked, near = P.check_policy_consistency(host, params, 64, A, awords)
    assert checked > E * (T - 2) and near <= 3
    ref = P.oracle_rollout(cfg, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), env_words=ewords)
    P.compare_traj(host, ref, what=f"policy on {cfg}")


@pytest.mark.parametrize("E,T,slack,limit,visible", [(4096, 64, 0, 500, True), (1000, 70, 9, 20, True), (37, 45, 3, 15, False),
                                                     (16, 33, 0, 500, True), (300, 50, 2, 0, False),
                                                     # a ragged last CTA with each count of policy warps (148 SMs: 1 at
                                                     # E = 37, 2 .. 6 at 1001 .. 3401, 7 at 4096, 8 at 4700)
                                                     (1001, 36, 4, 11, True), (1501, 40, 0, 13, False), (2367, 30, 6, 9, True),
                                                     (2901, 34, 2, 0, False), (3401, 28, 3, 17, False),
                                                     (2400, 40, 5, 20, True), (4700, 33, 0, 15, False), (4736, 21, 2, 9, True),
                                                     (5000, 20, 3, 9, True), (9472, 12, 0, 500, True),  # two waves
                                                     (12000, 12, 2, 9, True)])  # past two waves, ragged last CTA
def test_warp_specialized_rollout_is_bit_identical_to_k2c(ctx, E, T, slack, limit, visible):
    """K2q, the warp-specialised kernel `RL_LANES_WARP_SPECIALIZED` runs (policy and dynamics of an env on different warps,
    hand-off through named barriers; 1 to 8 policy warps per CTA by size), performs the same
    operations on the same operands as K2c with 8 threads per env: under Philox noise every stored byte, the lane
    lengths and the summary must be identical -- ragged last CTA, slack, step-limit Interrupts, latent limit (F = 4),
    resets, dangling steps."""
    wrap = R.VisibleStepLimit(limit) if visible else R.LatentStepLimit(limit)
    cfg = R.CartPoleConfig().wrap(wrap) if limit else R.CartPoleConfig()  # limit 0: the bare env, episodes end by Terminate only
    F = 5 if visible else 4
    params = R.init_params(np.random.default_rng(E), F, 128, 2) * 2.0
    net = R.Mlp(ctx, F, [128], 2)
    net.set_weights(params)

    def run(lanes, periods=2):
        env = R.build_env(ctx, cfg, E, seed=21, lane_offset=5)
        traj = R.Trajectory(env, T + slack)
        out = []
        for _ in range(periods):  # the second period starts from the advanced Philox step counter
            summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=lanes),
                             R.HistoryDataBound(T, slack), traj)
            out.append((traj.to_host(), summ))
        return out

    for (ws, sw), (gk, sg) in zip(run(L.RL_LANES_WARP_SPECIALIZED), run(8)):
        for k in ("lane_len", "succ"):
            np.testing.assert_array_equal(ws[k], gk[k], err_msg=k)
        valid = gk["succ"] != L.RL_PAD  # slots past a lane's last step are never written by either kernel
        for k in ("action", "reward", "obs"):
            np.testing.assert_array_equal(ws[k][valid], gk[k][valid], err_msg=k)
        intr = gk["succ"] == L.RL_INTERRUPT
        assert intr.any() or limit >= T or limit == 0
        np.testing.assert_array_equal(ws["next_obs"][intr], gk["next_obs"][intr])
        assert ws["num_steps"] == gk["num_steps"]
        for name in ("step_reward", "episode_reward", "episode_length"):
            a, b = getattr(sw, name), getattr(sg, name)
            assert (a.mean, a.squared_residual_sum, a.count) == (b.mean, b.squared_residual_sum, b.count), name
        assert (sw.num_stored_steps, sw.num_stored_episodes) == (sg.num_stored_steps, sg.num_stored_episodes)


def test_warp_specialized_rollout_rejects_replayed_noise(ctx):
    env = R.build_env(ctx, CARTPOLE, 32, seed=1)
    env.set_noise_replay(P.random_words(np.random.default_rng(0), 32, 256), P.random_words(np.random.default_rng(1), 32, 256))
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(R.init_params(np.random.default_rng(2), 5, 128, 2))
    traj = R.Trajectory(env, 8)
    with pytest.raises(Exception):
        R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=L.RL_LANES_WARP_SPECIALIZED),
                  R.HistoryDataBound(8, 0), traj)


def test_set_weights_async_from_pinned_memory(ctx):
    """rl_mlp_set_weights_async: the stream-ordered weight refresh (no host round trip) gives the rollout the same
    weights as the synchronous copy, and refuses pageable memory."""
    rng = np.random.default_rng(5)
    params = R.init_params(rng, 5, 128, 2)
    net_a, net_b = R.Mlp(ctx, 5, [128], 2), R.Mlp(ctx, 5, [128], 2)
    net_a.set_weights(params)
    pinned = ctx.pinned_array((params.size,), np.float32)
    pinned[:] = params
    net_b.set_weights_async(pinned)
    outs = []
    for net in (net_a, net_b):
        env = R.build_env(ctx, CARTPOLE, 300, seed=4)
        traj = R.Trajectory(env, 40)
        R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net), R.HistoryDataBound(40, 0), traj)
        outs.append(traj.to_host())
    for k in ("obs", "action", "succ", "lane_len"):
        np.testing.assert_array_equal(outs[0][k], outs[1][k])
    np.testing.assert_array_equal(net_b.get_weights(), params)
    with pytest.raises(L.RelearnB200Error):
        net_b.set_weights_async(np.ascontiguousarray(params))  # pageable


def test_warp_specialized_rollout_against_the_oracle(ctx):
    """K2q (200 envs: one policy warp per CTA) directly against the CPU oracle under production noise: (i) replaying its actions through the oracle, which
    regenerates the Philox reset draws itself, reproduces the trajectory (Terminate / Interrupt codes, lane lengths and
    summary exactly, CartPole observations to 1e-6: sin/cos differ from glibc by <= 1 ulp); (ii) every action is the
    inverse-CDF choice of the oracle's softmax for the recorded observation and the step's Philox uniform."""
    E, T, slack, seed, off, t0 = 200, 60, 4, 0xBEEF, 77, 9
    params = R.init_params(np.random.default_rng(8), 5, 128, 2) * 2.0
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(params)
    env = R.build_env(ctx, CARTPOLE, E, seed=seed, lane_offset=off)
    env.set_noise_philox(seed, t0)
    traj = R.Trajectory(env, T + slack)
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=L.RL_LANES_WARP_SPECIALIZED),
                     R.HistoryDataBound(T, slack), traj)
    host = traj.to_host()
    ref = P.oracle_rollout(CARTPOLE, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), philox_seed=seed,
                           lane_offset=off, t0=t0)
    P.compare_traj(host, ref, obs_rtol=1e-6, obs_atol=1e-7, what="K2q vs oracle")
    P.compare_summary(summ, ref["summary"])
    lib = L.lib()
    awords = np.array([[lib.rl_philox_slot(seed, off + e, t0 + i, 2, 0) & 0xFFFFFFFF for i in range(T + slack)] for e in range(E)],
                      dtype=np.uint64).astype(np.uint32)
    checked, near = P.check_policy_consistency(host, params, 128, 2, awords)
    assert checked == int(host["lane_len"].sum()) and near <= 3
    assert (host["succ"] == L.RL_INTERRUPT).any() and (host["succ"] == L.RL_TERMINATE).any()
