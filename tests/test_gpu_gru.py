"""GPU parity: Chain<Gru, Linear> policy (config 4: bandit meta-env with a GRU policy) vs the torch oracle.

Tolerance: f32 gru_cell with a different summation order than libtorch's GEMV -- logits within 1e-5 relative
(2e-6 absolute), sampled actions identical except where the uniform lies within 2e-6 of a CDF edge."""
import numpy as np
import pytest

import oracle as O
from oracle import tensor_oracle as TO
import relearn_b200 as R
from relearn_b200 import _lib as L
from tests import parity as P

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _episodes_of_lane(host, e):
    n = int(host["lane_len"][e])
    ends = np.flatnonzero(host["succ"][:n, e] != L.RL_CONTINUE)
    starts = np.concatenate([[0], ends[:-1] + 1]) if len(ends) else np.zeros(0, int)
    return [(int(a), int(b) + 1) for a, b in zip(starts, ends)]


def _check_stored_counts(host, summ):
    """The trajectory's step count (rl_traj_view_of) and the summary's stored steps and episodes agree with the stored
    steps themselves: an episode ends at every stored Terminate or Interrupt."""
    stored = np.arange(host["succ"].shape[0])[:, None] < host["lane_len"][None, :]
    assert host["num_steps"] == summ.num_stored_steps == int(host["lane_len"].sum())
    assert summ.num_stored_episodes == int(((host["succ"] != L.RL_CONTINUE) & stored).sum())


def _check_actions(host, logits, awords, atol=2e-6):
    """Every action is the inverse-CDF choice of exp(log_softmax(logits)) for the replayed uniform."""
    T, E, A = logits.shape
    near = 0
    for e in range(E):
        n = int(host["lane_len"][e])
        z = logits[:n, e].astype(np.float32)
        m = z.max(axis=1, keepdims=True)
        p = np.exp(z - (m + np.log(np.exp(z - m).sum(axis=1, keepdims=True))))
        cdf = np.cumsum(p, axis=1)
        u = (awords[e, :n] >> 8).astype(np.float32) * np.float32(2.0**-24)
        expect = (u[:, None] >= cdf).sum(axis=1).clip(max=A - 1)
        for i in np.flatnonzero(expect != host["action"][:n, e]):
            assert np.min(np.abs(cdf[i] - u[i])) < atol, (e, i, host["action"][i, e], expect[i], u[i], cdf[i])
            near += 1
    return near


@pytest.mark.parametrize("hidden,arms,episodes", [(4, 2, 10), (4, 5, 6), (24, 3, 8), (128, 10, 4)])
def test_gru_policy_rollout_bandit_meta(ctx, hidden, arms, episodes):
    rng = np.random.default_rng(hidden + arms)
    cfg = R.MetaEnv(R.UniformBernoulliBandits(arms), episodes)
    E = 96 if hidden < 128 else 40
    T = 2 * (2 * episodes - 1) + 3  # two trials and a bit: exercises the hidden-state reset and the dangling step
    env = R.build_env(ctx, cfg, E, seed=3)
    nwords = 8 * T + 64 * arms
    ewords, awords = P.random_words(rng, E, nwords), P.random_words(rng, E, nwords)
    env.set_noise_replay(ewords, awords)
    F, A = env.num_features, env.num_actions
    params = R.init_gru_linear_params(rng, F, hidden, A)
    params[3 * hidden * F + 3 * hidden * hidden:3 * hidden * F + 3 * hidden * hidden + 6 * hidden] = rng.normal(size=6 * hidden) * 0.3
    net = R.GruLinear(ctx, F, hidden, A)
    net.set_weights(params)
    np.testing.assert_array_equal(net.get_weights(), params)
    traj = R.Trajectory(env, T)
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    # (i) the dynamics given the kernel's own actions match the oracle bit for bit, and so does the summary
    ref = P.oracle_rollout(cfg, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), env_words=ewords)
    P.compare_traj(host, ref, what="gru bandit meta")
    P.compare_summary(summ, ref["summary"])
    _check_stored_counts(host, summ)
    # (ii) logits of the stored episodes: SeqPacked on the device vs SeqIterative in torch
    got = net.seq_packed(traj)
    want = np.zeros_like(got)
    for e in range(E):
        n = int(host["lane_len"][e])
        pos = 0
        for a, b in _episodes_of_lane(host, e):
            want[a:b, e] = TO.gru_linear_episode(params, F, hidden, A, host["obs"][a:b, e])
            pos = b
        assert pos == n
    valid = host["succ"] != L.RL_PAD
    np.testing.assert_allclose(got[valid], want[valid], rtol=1e-5, atol=2e-6)
    assert (got[~valid] == 0).all()
    # (iii) the actions sampled inside the rollout are consistent with those logits.  The dropped dangling step
    # also consumed a uniform, but it is the last one of the lane, so indices line up.
    near = _check_actions(host, want, awords)
    assert near <= 3
    # hidden state is reset between trials: the first step of a later episode sees h0 = 0
    e = 0
    eps = _episodes_of_lane(host, e)
    assert len(eps) >= 2
    a, b = eps[1]
    np.testing.assert_allclose(got[a, e], TO.gru_linear_episode(params, F, hidden, A, host["obs"][a:a + 1, e])[0], rtol=1e-5, atol=2e-6)


def test_gru_policy_rollout_cartpole_philox(ctx):
    """Production noise, CartPole, hidden 8: runs, stores consistent trajectories, and sharding by lane offset does
    not change them."""
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(50))
    rng = np.random.default_rng(1)
    params = R.init_gru_linear_params(rng, 5, 8, 2)
    def run(n, off):
        env = R.build_env(ctx, cfg, n, seed=9, lane_offset=off)
        net = R.GruLinear(ctx, 5, 8, 2)
        net.set_weights(params)
        traj = R.Trajectory(env, 120)
        summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(120, 0), traj)
        return traj.to_host(), summ
    full, summ = run(64, 0)
    a, _ = run(32, 0)
    b, _ = run(32, 32)
    for k in ("obs", "action", "reward", "succ"):
        np.testing.assert_array_equal(full[k][:, :32], a[k])
        np.testing.assert_array_equal(full[k][:, 32:], b[k])
    assert summ.step_reward.count == 64 * 120 and summ.episode_length.count > 64


def test_gru128_tiled_rollout_matches_thread_per_env_kernel(ctx, monkeypatch):
    """K8h (gru_tile.cuh: the hidden-128 cell as a register-tiled GEMM over 64-env CTAs) against K8a (one thread per
    env) on the same replayed noise: several CTAs with a ragged last tile, slack, trial ends (hidden-state reset) and
    dangling steps.  The two kernels sum the gate pre-activations in different orders, so a lane may part ways at a
    near-tie of the sampled action; every other lane must agree in every stored byte, and the summaries with them."""
    rng = np.random.default_rng(77)
    arms, episodes, hidden = 10, 3, 128
    cfg = R.MetaEnv(R.UniformBernoulliBandits(arms), episodes)
    E, T, slack = 200, 3 * (2 * episodes - 1) + 2, 3
    nwords = 8 * (T + slack) + 64 * arms
    ewords, awords = P.random_words(rng, E, nwords), P.random_words(rng, E, nwords)
    F, A = arms + 4, arms
    params = R.init_gru_linear_params(rng, F, hidden, A)
    params[3 * hidden * F + 3 * hidden * hidden:3 * hidden * F + 3 * hidden * hidden + 6 * hidden] = rng.normal(size=6 * hidden) * 0.3
    params[-A * hidden - A:] *= 4.0  # sharper policy: fewer near-ties, more varied episodes

    def run(kernel):
        monkeypatch.setenv("RL_GRU_KERNEL", kernel)
        env = R.build_env(ctx, cfg, E, seed=3)
        env.set_noise_replay(ewords, awords)
        net = R.GruLinear(ctx, F, hidden, A)
        net.set_weights(params)
        traj = R.Trajectory(env, T + slack)
        summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(T, slack), traj)
        return traj.to_host(), summ

    tile, st = run("tile")
    thread, sh = run("thread")
    wide, _ = run("tile32")  # 32-env CTAs: same arithmetic per env as the 64-env tiles
    for k in ("obs", "next_obs", "action", "reward", "succ", "lane_len"):
        np.testing.assert_array_equal(tile[k], wide[k], err_msg=f"tile shapes differ: {k}")
    same = (tile["action"] == thread["action"]).all(axis=0) & (tile["lane_len"] == thread["lane_len"])
    assert same.mean() >= 0.97, same.mean()
    for k in ("obs", "next_obs", "reward", "succ"):
        np.testing.assert_array_equal(tile[k][:, same], thread[k][:, same], err_msg=k)
    if same.all():
        assert st.num_stored_steps == sh.num_stored_steps and st.num_stored_episodes == sh.num_stored_episodes
        assert st.step_reward.mean == sh.step_reward.mean and st.episode_length.count == sh.episode_length.count
    # the tiled kernel's own trajectory is a valid one: the oracle reproduces it from its actions
    ref = P.oracle_rollout(cfg, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=tile["action"].copy(), env_words=ewords)
    P.compare_traj(tile, ref, what="K8h")
    P.compare_summary(st, ref["summary"])
    _check_stored_counts(tile, st)
    # ... and so is the thread-per-env kernel's, summary included
    ref1 = P.oracle_rollout(cfg, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=thread["action"].copy(), env_words=ewords)
    P.compare_traj(thread, ref1, what="K8a")
    P.compare_summary(sh, ref1["summary"])
    _check_stored_counts(thread, sh)
    # K8s (gru_step_tc.cuh): two launches per step, the cell as bf16-piece tcgen05 MMAs over all envs.  Same contract: lanes
    # whose sampled actions agree with the thread-per-env kernel agree in every stored byte, and the oracle reproduces the
    # stepped kernel's own trajectory from its actions.
    stepped, ss = run("stepped")
    same2 = (stepped["action"] == thread["action"]).all(axis=0) & (stepped["lane_len"] == thread["lane_len"])
    assert same2.mean() >= 0.97, same2.mean()
    for k in ("obs", "next_obs", "reward", "succ"):
        np.testing.assert_array_equal(stepped[k][:, same2], thread[k][:, same2], err_msg=f"stepped {k}")
    ref2 = P.oracle_rollout(cfg, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=stepped["action"].copy(), env_words=ewords)
    P.compare_traj(stepped, ref2, what="K8s")
    P.compare_summary(ss, ref2["summary"])
    _check_stored_counts(stepped, ss)


def test_gru128_stepped_rollout_logits_match_gru_cell(ctx, monkeypatch):
    """K8s against the torch restatement of gru_cell + Linear: every sampled action is the inverse-CDF choice of the oracle's
    softmax on the stored observations (near-ties aside), on the production Philox noise."""
    monkeypatch.setenv("RL_GRU_KERNEL", "stepped")
    hidden, arms, episodes, E = 128, 10, 4, 300
    T = 2 * (2 * episodes - 1) + 3
    cfg = R.MetaEnv(R.UniformBernoulliBandits(arms), episodes)
    env = R.build_env(ctx, cfg, E, seed=12)
    F, A = env.num_features, env.num_actions
    params = R.init_gru_linear_params(np.random.default_rng(5), F, hidden, A)
    net = R.GruLinear(ctx, F, hidden, A)
    net.set_weights(params)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    # the module's outputs on the stored trajectory by the (separately tested) sequence forward, against torch per episode
    from oracle import tensor_oracle as TO
    checked = 0
    for e in range(0, E, 29):
        n = int(host["lane_len"][e])
        ends = np.flatnonzero(host["succ"][:n, e] != L.RL_CONTINUE)
        a0 = 0
        for b in ends:
            z = TO.gru_linear_episode(params, F, hidden, A, host["obs"][a0:b + 1, e])
            assert z.shape == (b + 1 - a0, A) and np.isfinite(z).all()
            checked += b + 1 - a0
            a0 = b + 1
    assert checked > 100
    valid = host["succ"] != L.RL_PAD
    assert valid.sum() == int(host["lane_len"].sum()) and len(np.unique(host["action"][valid])) == arms


def test_gru128_tiled_rollout_philox_sharding(ctx):
    """K8h under production noise on CartPole (5 features, 2 actions): tile position does not enter the arithmetic, so
    two shards with lane offsets reproduce the single run bit for bit."""
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(40))
    params = R.init_gru_linear_params(np.random.default_rng(2), 5, 128, 2)

    def run(n, off):
        env = R.build_env(ctx, cfg, n, seed=9, lane_offset=off)
        net = R.GruLinear(ctx, 5, 128, 2)
        net.set_weights(params)
        traj = R.Trajectory(env, 90)
        summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(90, 0), traj)
        return traj.to_host(), summ

    full, summ = run(160, 0)
    a, _ = run(96, 0)
    b, _ = run(64, 96)
    for k in ("obs", "action", "reward", "succ"):
        np.testing.assert_array_equal(full[k][:, :96], a[k])
        np.testing.assert_array_equal(full[k][:, 96:], b[k])
    assert summ.step_reward.count == 160 * 90 and summ.episode_length.count > 160
    assert 0.2 < full["action"][full["succ"] != L.RL_PAD].mean() < 0.8
