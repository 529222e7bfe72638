"""GPU parity: Chain<Lstm, Linear> (rl_lstmnet_create) through every recurrent path -- the rollout with the categorical
policy and with the epsilon-greedy actor, the SeqPacked forward, the TRPO / critic passes (K9 at hidden <= 8, K10 above),
GAE and the recurrent DQN update -- against the torch restatement in tests/lstm_oracle.py.

Tolerances are those of the GRU tests (test_gpu_gru.py, test_gpu_gru_update.py, test_gpu_dqn_seq.py): the env side and
explored actions bit-exact, outputs within 1e-5 relative (2e-6 absolute), sampled actions the inverse-CDF choice except
near-ties, losses / gradients / Fisher-vector products within 1e-5 of f64 autograd."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
import relearn_b200 as R
from relearn_b200 import _lib as L
from tests import parity as P
from tests.test_gpu_dqn import _fill, _oracle_minibatch
from tests.test_gpu_dqn_seq import _actor_draws, _rtg
from tests.test_gpu_gru import _check_actions, _check_stored_counts, _episodes_of_lane

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from tests import lstm_oracle as LO  # noqa: E402

CONT, INTR, PAD = L.RL_CONTINUE, L.RL_INTERRUPT, L.RL_PAD


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) /
                 max(np.linalg.norm(np.asarray(b, np.float64)), 1e-300))


def _params(rng, F, H, A, bias_scale=0.3, head_scale=1.0, input_scale=1.0, head_bias=True):
    p = R.init_lstm_linear_params(rng, F, H, A).astype(np.float32)
    p[:4 * H * F] *= input_scale
    o = 4 * H * F + 4 * H * H
    p[o:o + 8 * H] = rng.normal(size=8 * H) * bias_scale
    p[-A * H - A:] *= head_scale
    if not head_bias:
        p[-A:] = 0.0
    return p


def _env_cfg(kind, arms=2):
    if kind == "bandit":
        return R.MetaEnv(R.UniformBernoulliBandits(arms), 6)
    if kind == "memory":
        return R.MemoryGame(3, 4)
    return R.CartPoleConfig().wrap(R.VisibleStepLimit(12))


# ------------------------------------------------------------------------------------------------
# Rollout (K8a) and the SeqPacked forward (K8b / K10)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,hidden,arms", [("bandit", 4, 2), ("bandit", 3, 5), ("bandit", 8, 3), ("bandit", 24, 3),
                                              ("bandit", 128, 10), ("memory", 8, 0), ("cartpole", 8, 0), ("memory", 128, 0)])
def test_lstm_policy_rollout(ctx, kind, hidden, arms):
    rng = np.random.default_rng(hidden + arms)
    cfg = _env_cfg(kind, arms)
    E, T = (96 if hidden < 128 else 40), 25
    env = R.build_env(ctx, cfg, E, seed=3)
    nwords = 16 * T + 64 * max(arms, 1)
    ewords, awords = P.random_words(rng, E, nwords), P.random_words(rng, E, nwords)
    env.set_noise_replay(ewords, awords)
    F, A = env.num_features, env.num_actions
    params = _params(rng, F, hidden, A)
    net = R.LstmLinear(ctx, F, hidden, A)
    assert net.num_params == R.lstm_linear_num_params(F, hidden, A)
    net.set_weights(params)
    np.testing.assert_array_equal(net.get_weights(), params)
    traj = R.Trajectory(env, T)
    summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    # the dynamics given the kernel's own actions match the oracle bit for bit, and so does the summary
    ref = P.oracle_rollout(cfg, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), env_words=ewords)
    P.compare_traj(host, ref, what=f"lstm {kind} {hidden}")
    P.compare_summary(summ, ref["summary"])
    _check_stored_counts(host, summ)
    # the outputs on the stored episodes: SeqPacked on the device vs the iterated lstm_cell in torch
    got = net.seq_packed(traj)
    want = np.zeros_like(got)
    for e in range(E):
        for a, b in _episodes_of_lane(host, e):
            want[a:b, e] = LO.lstm_linear_episode(params, F, hidden, A, host["obs"][a:b, e])
    valid = host["succ"] != PAD
    np.testing.assert_allclose(got[valid], want[valid], rtol=1e-5, atol=2e-6)
    assert (got[~valid] == 0).all()
    # the actions sampled inside the rollout are the inverse-CDF choices on those outputs
    assert _check_actions(host, want, awords) <= 3
    assert (host["succ"][valid] != CONT).sum() > E  # several episodes per lane: (h, c) were reset


@pytest.mark.parametrize("hidden", [8, 128])
def test_lstm_rollout_philox_sharding(ctx, hidden):
    """Production noise: two shards of lanes (lane_offset) reproduce the full run."""
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(40))
    params = _params(np.random.default_rng(1), 5, hidden, 2)

    def run(n, off):
        env = R.build_env(ctx, cfg, n, seed=9, lane_offset=off)
        net = R.LstmLinear(ctx, 5, hidden, 2)
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


@pytest.mark.parametrize("hidden", [24, 128])
def test_lstm_seq_forward_thread_kernel_matches_gemm_form(ctx, monkeypatch, hidden):
    """K8b<128> (RL_GRU_KERNEL=thread) and K10's forward on the same trajectory, and both against the oracle; the
    successor outputs of interrupted steps are checked through GAE below."""
    rng = np.random.default_rng(hidden)
    env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(3), 4), 64, seed=5)
    F, A = env.num_features, env.num_actions
    params = _params(rng, F, hidden, A)
    net = R.LstmLinear(ctx, F, hidden, A)
    net.set_weights(params)
    traj = R.Trajectory(env, 20)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(20, 0), traj)
    host = traj.to_host()
    big = net.seq_packed(traj)
    monkeypatch.setenv("RL_GRU_KERNEL", "thread")
    thread = net.seq_packed(traj)
    valid = host["succ"] != PAD
    np.testing.assert_allclose(thread[valid], big[valid], rtol=1e-5, atol=2e-6)
    for e in range(0, 64, 7):
        for a, b in _episodes_of_lane(host, e):
            np.testing.assert_allclose(big[a:b, e], LO.lstm_linear_episode(params, F, hidden, A, host["obs"][a:b, e]), rtol=1e-5, atol=2e-6)


# ------------------------------------------------------------------------------------------------
# Epsilon-greedy actor of a recurrent Q-network
# ------------------------------------------------------------------------------------------------
def _restate_eps_greedy(host, params, F, H, A, explore, drawn, *, advance_always=False, tie_rtol=1e-5):
    """Explored steps take the drawn action; greedy steps the first argmax of Q in f64.  (h, c) start at zero in every
    episode and are NOT advanced on an explored step (DqnActor::act returns before step).  Returns (greedy, mismatches,
    near-ties)."""
    T, E = host["action"].shape
    w_ih, w_hh, b_ih, b_hh, lw, lb = [t.to(torch.float64) for t in LO.unflatten_lstm_linear(params, F, H, A)]
    h = torch.zeros(E, H, dtype=torch.float64)
    c = torch.zeros_like(h)
    lens = host["lane_len"].astype(np.int64)
    greedy = mism = near = 0
    for t in range(int(lens.max(initial=0))):
        valid = t < lens
        hn, cn = torch.lstm_cell(torch.tensor(host["obs"][t], dtype=torch.float64), (h, c), w_ih, w_hh, b_ih, b_hh)
        z = torch.nn.functional.linear(torch.relu(hn), lw, lb).numpy()
        got = host["action"][t].astype(np.int64)
        ex = explore[t] & valid
        assert (got[ex] == drawn[t][ex]).all(), f"step {t}: an explored action differs from the drawn one"
        g = valid & ~explore[t]
        best = z.argmax(axis=1)
        for e in np.flatnonzero(g & (got != best)):
            if abs(z[e, got[e]] - z[e, best[e]]) < tie_rtol * max(1.0, float(np.abs(z[e]).max())):
                near += 1
            else:
                mism += 1
        greedy += int(g.sum())
        keep = torch.tensor(explore[t] & (not advance_always))[:, None]
        h, c = torch.where(keep, h, hn), torch.where(keep, c, cn)
        done = torch.tensor(host["succ"][t] != CONT)[:, None]
        h, c = torch.where(done, torch.zeros_like(h), h), torch.where(done, torch.zeros_like(c), c)
    return greedy, mism, near


@pytest.mark.parametrize("kind,hidden", [("memory", 4), ("bandit", 8), ("bandit", 128)])
def test_eps_greedy_lstm_rollout(ctx, kind, hidden):
    cfg = R.MemoryGame(4, 3) if kind == "memory" else R.MetaEnv(R.UniformBernoulliBandits(2 if hidden < 128 else 10), 6)
    E, T, eps = (96 if hidden < 128 else 64), 30, 0.3
    for attempt in range(6):
        rng = np.random.default_rng(hidden + 101 * attempt)
        env = R.build_env(ctx, cfg, E, seed=hidden + attempt)
        nwords = 16 * T + 64 * env.num_actions
        ewords, awords = P.random_words(rng, E, nwords), P.random_words(rng, E, nwords)
        env.set_noise_replay(ewords, awords)
        F, A = env.num_features, env.num_actions
        params = _params(rng, F, hidden, A, head_scale=3.0, input_scale=3.0, head_bias=False)
        net = R.LstmLinear(ctx, F, hidden, A)
        net.set_weights(params)
        traj = R.Trajectory(env, T)
        summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, seq_net=net, exploration_rate=eps), R.HistoryDataBound(T - 2, 2), traj)
        host = traj.to_host()
        ref = P.oracle_rollout(cfg, E, T - 2, 2, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), env_words=ewords)
        P.compare_traj(host, ref, what=f"eps-greedy LSTM {hidden}")
        P.compare_summary(summ, ref["summary"])
        explore, drawn = _actor_draws(host, A, eps, actor_words=awords)
        greedy, mism, near = _restate_eps_greedy(host, params, F, hidden, A, explore, drawn)
        print(f"{kind} h={hidden} attempt {attempt}: greedy {greedy}, explored {int(explore.sum())}, near-ties {near}")
        assert greedy > 0 and explore.any() and mism == 0 and near <= 3
        # the restatement that advances (h, c) on every step must disagree somewhere for the case to exercise the hold
        if _restate_eps_greedy(host, params, F, hidden, A, explore, drawn, advance_always=True)[1] > 0:
            return
    raise AssertionError("no case exercised the state held on explored steps")


# ------------------------------------------------------------------------------------------------
# TRPO, critic and GAE
# ------------------------------------------------------------------------------------------------
def _collect(ctx, hidden, arms, episodes, E, T, seed, scale=1.0, activation="relu"):
    rng = np.random.default_rng(seed)
    cfg = R.MetaEnv(R.UniformBernoulliBandits(arms), episodes)
    env = R.build_env(ctx, cfg, E, seed=seed)
    F, A = env.num_features, env.num_actions
    params = _params(rng, F, hidden, A, bias_scale=0.2)
    params[:-A * hidden - A] *= scale
    net = R.LstmLinear(ctx, F, hidden, A, activation)
    net.set_weights(params)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    spans = [(e, a, b) for e in range(E) for a, b in _episodes_of_lane(host, e)]
    assert sum(b - a for _, a, b in spans) == int((host["succ"] != PAD).sum())
    return env, traj, net, params, host, spans


def _per_episode(x, spans):
    return [x[a:b, e] for e, a, b in spans]


@pytest.mark.parametrize("hidden,arms,episodes,activation", [(4, 2, 10, "relu"), (8, 5, 4, "tanh"), (3, 3, 6, "relu"),
                                                             (24, 3, 4, "tanh"), (128, 10, 4, "relu")])
def test_lstm_trpo_probe_loss_grad_fvp(ctx, hidden, arms, episodes, activation):
    E, T = (80 if hidden <= 24 else 45), 2 * (2 * episodes - 1) + 5
    env, traj, net, params, host, spans = _collect(ctx, hidden, arms, episodes, E, T, seed=hidden + arms, scale=1.5,
                                                   activation=activation)
    F, A = env.num_features, env.num_actions
    rng = np.random.default_rng(2)
    adv = rng.normal(size=(T, E)).astype(np.float32)
    vec = rng.normal(size=net.num_params).astype(np.float32)
    got = R.Trpo(net, R.TrpoConfig()).probe(traj, ctx.to_device(adv), vec)
    eps, acts, advs = _per_episode(host["obs"], spans), _per_episode(host["action"], spans), _per_episode(adv, spans)
    loss64, kl64, ent64, g64, hv64 = LO.seq_policy_loss_kl_grad_fvp(params, F, hidden, A, eps, acts, advs, vec, 1e-5,
                                                                    torch.float64, activation)
    print(f"episodes={len(spans)} grad rel err {_rel(got['grad'], g64):.2e}, fvp rel err {_rel(got['fvp'], hv64):.2e}")
    assert abs(got["loss"] - loss64) <= 1e-6 * max(1.0, abs(loss64))
    assert abs(got["kl"]) <= 1e-7 and abs(kl64) <= 1e-12
    assert abs(got["entropy"] - ent64) <= 1e-6
    assert _rel(got["grad"], g64) <= 1e-5
    assert _rel(got["fvp"], hv64) <= 1e-5


@pytest.mark.parametrize("hidden,arms,episodes", [(4, 2, 10), (8, 4, 5), (128, 10, 3)])
def test_lstm_trpo_update_matches_f64(ctx, hidden, arms, episodes):
    E, T = (96 if hidden <= 8 else 40), 2 * (2 * episodes - 1) + 3
    env, traj, net, params, host, spans = _collect(ctx, hidden, arms, episodes, E, T, seed=7 + hidden, scale=1.5)
    F, A = env.num_features, env.num_actions
    adv = np.random.default_rng(11).normal(size=(T, E)).astype(np.float32)
    reg = 0.1
    policy = R.Trpo(net, R.TrpoConfig(optimizer_config=R.ConjugateGradientOptimizerConfig(hpv_reg_coeff=reg)))
    log = {}
    status = policy.update(traj, ctx.to_device(adv), log)
    new = net.get_weights()
    eps, acts, advs = _per_episode(host["obs"], spans), _per_episode(host["action"], spans), _per_episode(adv, spans)
    from oracle import tensor_oracle as TO
    ocfg = TO.CgConfig(hpv_reg_coeff=reg)
    new64, log64 = LO.seq_trpo_update(params, F, hidden, A, eps, acts, advs, cfg=ocfg, dtype=torch.float64)
    new32, log32 = LO.seq_trpo_update(params, F, hidden, A, eps, acts, advs, cfg=ocfg, dtype=torch.float32)
    d, d64, d32 = new - params, new64 - params.astype(np.float64), new32 - params
    print(f"status={status} backtracks {log['num_backtracks']}/{log64['num_backtracks']}; delta rel err kernel "
          f"{_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}")
    assert status == L.RL_OK and log64["error"] is None
    assert log["num_steps"] == sum(b - a for _, a, b in spans)
    assert log["num_backtracks"] == log64["num_backtracks"]
    np.testing.assert_allclose(log["entropy"], log64["entropy"], rtol=1e-5)
    np.testing.assert_allclose(log["step_size"], log64["step_size"], rtol=2e-5)
    np.testing.assert_allclose(log["loss_initial"], log64["loss_initial"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(log["loss_final"], log64["loss_final"], rtol=1e-5, atol=1e-7)
    assert _rel(d, d64) <= max(2e-5, 1.25 * _rel(d32, d64)) and _rel(d, d64) <= 1e-4


@pytest.mark.parametrize("hidden,arms,episodes,E,steps", [(4, 2, 6, 72, 20), (24, 3, 4, 48, 8), (128, 10, 4, 40, 6)])
def test_lstm_gae_and_value_update(ctx, hidden, arms, episodes, E, steps):
    """ValuesOpt<Chain<Lstm, Linear>>: GAE over SeqPacked values (an interrupted trial bootstraps from one more step of the
    same sequence) and Adam steps on the reward-to-go targets."""
    T = 2 * (2 * episodes - 1) + 4
    env, traj, net, params, host, spans = _collect(ctx, hidden, arms, episodes, E, T, seed=21)
    F = env.num_features
    vparams = _params(np.random.default_rng(5), F, hidden, 1, bias_scale=0.2)
    critic = R.ValuesOpt(ctx, R.ValuesOptConfig(state_value_fn_config=R.LstmLinearConfig(hidden_dim=hidden),
                                                opt_steps_per_update=steps), F, env.discount_factor)
    assert isinstance(critic.state_value_fn, R.LstmLinear)
    critic.state_value_fn.set_weights(vparams)
    gamma, lam = critic.discount_factor, np.float32(0.95)
    adv = critic.advantages(traj).download((T, E), np.float32)
    v = np.zeros((T, E), np.float32)
    vn = np.zeros((T, E), np.float32)
    n_intr = 0
    for e, a, b in spans:
        obs = host["obs"][a:b, e]
        if host["succ"][b - 1, e] == INTR:
            out = LO.lstm_linear_episode(vparams, F, hidden, 1, np.concatenate([obs, host["next_obs"][b - 1:b, e]]))[:, 0]
            v[a:b, e], vn[b - 1, e] = out[:-1], out[-1]
            n_intr += 1
        else:
            v[a:b, e] = LO.lstm_linear_episode(vparams, F, hidden, 1, obs)[:, 0]
    assert n_intr > E
    for e in range(E):
        n = int(host["lane_len"][e])
        ref = O.gae_lane(host["reward"][:n, e], v[:n, e], vn[:n, e], host["succ"][:n, e], gamma, lam)
        np.testing.assert_allclose(adv[:n, e], ref, rtol=2e-5, atol=2e-6)
    stats = critic.update(traj)
    new = critic.state_value_fn.get_weights()
    rtg = np.zeros((T, E), np.float32)
    for e in range(E):
        n = int(host["lane_len"][e])
        rtg[:n, e] = O.discounted_cumsum_lane(host["reward"][:n, e], host["succ"][:n, e], gamma)
    eps, tg = _per_episode(host["obs"], spans), _per_episode(rtg, spans)
    new64, losses64 = LO.seq_value_update(vparams, F, hidden, eps, tg, n_steps=steps, dtype=torch.float64)
    new32, _ = LO.seq_value_update(vparams, F, hidden, eps, tg, n_steps=steps, dtype=torch.float32)
    d, d64, d32 = new - vparams, new64 - vparams.astype(np.float64), new32 - vparams
    print(f"LSTM critic delta rel err kernel {_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}")
    assert stats.opt_steps == steps and stats.num_steps == sum(b - a for _, a, b in spans)
    np.testing.assert_allclose(stats.loss_first, losses64[0], rtol=1e-5)
    np.testing.assert_allclose(stats.loss_last, losses64[-1], rtol=1e-4)
    assert _rel(d, d64) <= max(2e-4, 4 * _rel(d32, d64) + 1e-5)


def test_lstm_gemm_formulation_serves_the_small_modules_too():
    """K10 against the oracle on the modules K9 normally serves: the probe, update and critic tests above in a child process
    with RL_SEQ_FORCE_BIG=1 (the switch is read once per process), the Q-loss probe below included."""
    if os.environ.get("RL_SEQ_FORCE_BIG") == "1":
        pytest.skip("already the forced run")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RL_SEQ_FORCE_BIG="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_lstm.py"), "-x", "-q", "-m", "gpu",
                        "-k", "(probe or update_matches or gae_and_value) and not 128 and not 24 and not 32"],
                       capture_output=True, text=True, env=env, cwd=root, timeout=1200)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and " passed" in r.stdout


# ------------------------------------------------------------------------------------------------
# Recurrent DQN
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def filled(ctx):
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(15))
    E = 48
    env, rb, _ = _fill(ctx, cfg, 15, E, 120, R.HistoryDataBound(30, 6), periods=6, seed=33)
    lanes = [rb.read_lane(e) for e in range(E)]
    return env, rb, lanes


def _td_targets(params, F, H, A, eps, g):
    ext = [np.concatenate([e["obs"], e["next_obs"][None]]) if e["last_succ"] == INTR else e["obs"] for e in eps]
    out = []
    for ep, q in zip(eps, LO.seq_q_values(params, F, H, A, ext)):
        n = len(ep["reward"])
        m = q.max(axis=1)
        nxt = np.zeros(n)
        nxt[:-1] = m[1:n]
        if ep["last_succ"] == INTR:
            nxt[-1] = m[n]
        out.append(ep["reward"].astype(np.float64) + float(np.float32(g)) * nxt)
    return out


@pytest.mark.parametrize("hidden", [4, 8, 32, 128])
@pytest.mark.parametrize("td", [False, True])
def test_lstm_qloss_probe_matches_f64(ctx, filled, hidden, td):
    env, rb, lanes = filled
    F, A = 5, 2
    params = _params(np.random.default_rng(100 + hidden), F, hidden, A, head_scale=2.0)
    q = R.LstmLinear(ctx, F, hidden, A)
    q.set_weights(params)
    seed, di, minibatch, g = 9, 4, 700, 0.99
    cfg = L.DqnCfg(minibatch, 1, 1 if td else 0, np.float32(g), seed)
    loss, grad = C.c_double(), np.zeros(q.num_params, np.float32)
    L.check(ctx._lib.rl_dqn_probe_seq(rb.handle, C.byref(cfg), q.handle, di, C.byref(loss), grad.ctypes.data_as(C.POINTER(C.c_float))),
            ctx.handle)
    eps = _oracle_minibatch(lanes, seed, di, minibatch)
    got_t = rb.sample_seq(cfg, q, di)["target"]
    tg32 = [got_t[:len(e["action"]), b] for b, e in enumerate(eps)]
    if td:  # the one-step TD targets come from the module's SeqPacked forward on the successor observations
        for a, b in zip(tg32, _td_targets(params, F, hidden, A, eps, g)):
            np.testing.assert_allclose(a, b, rtol=1e-5, atol=1e-6)
    else:
        for a, ep in zip(tg32, eps):
            np.testing.assert_array_equal(a, _rtg(ep, g))
    obs, acts = [e["obs"] for e in eps], [e["action"] for e in eps]
    loss64, g64 = LO.seq_q_loss_grad(params, F, hidden, A, obs, acts, tg32)
    print(f"h={hidden} td={td}: loss {loss.value:.8f} vs {loss64:.8f}; grad rel err {_rel(grad, g64):.2e}")
    assert abs(loss.value - loss64) <= 1e-6 * max(1.0, abs(loss64))
    assert _rel(grad, g64) <= 1e-5


def _oracle_seq_dqn(params, F, H, A, minibatches, g, dtype, lr=1e-3):
    from oracle import tensor_oracle as TO
    prm = LO.seq_params(params, F, H, A, dtype)
    opt = TO.Adam112(prm, lr)
    for eps in minibatches:
        q = LO.lstm_linear_forward(prm, TO.EpisodeBatch([e["obs"] for e in eps], dtype))
        act = torch.tensor(np.concatenate([e["action"] for e in eps]), dtype=torch.int64).unsqueeze(-1)
        tgt = torch.tensor(np.concatenate([_rtg(e, g) for e in eps]), dtype=dtype)
        loss = torch.nn.functional.mse_loss(q.gather(-1, act).squeeze(-1), tgt)
        opt.step(torch.autograd.grad(loss, prm))
    return TO.flatten_tensors([p.detach() for p in prm]).numpy().copy()


_DRAWS = {}


@pytest.mark.parametrize("hidden", [8, 32])
def test_lstm_dqn_update_seq_matches_oracle(ctx, filled, hidden):
    """opt_steps x {sequence sample, Q-loss with BPTT, Adam} against the torch loop on the same episodes."""
    env, rb, lanes = filled
    F, A = 5, 2
    params = _params(np.random.default_rng(7 + hidden), F, hidden, A)
    steps, minibatch, seed = 5, 500, 321
    agent = R.DqnConfig(action_value_fn_config=R.LstmLinearConfig(hidden_dim=hidden), minibatch_steps=minibatch,
                        opt_steps_per_update=steps, sample_seed=seed, buffer_capacity=120).build_agent(env)
    agent.action_value_fn.set_weights(params)
    assert isinstance(agent.action_value_fn, R.LstmLinear) and agent.actor().seq_net is agent.action_value_fn
    # the buffer's draw counter advances by one per optimizer step, over every update on it
    base = _DRAWS.get(id(rb), 0)
    _DRAWS[id(rb)] = base + steps
    stats = agent.batch_update(rb, {})
    new = agent.action_value_fn.get_weights()
    mbs = [_oracle_minibatch(lanes, seed, base + s, minibatch) for s in range(steps)]
    g = float(agent.discount_factor)
    new64 = _oracle_seq_dqn(params, F, hidden, A, mbs, g, torch.float64)
    new32 = _oracle_seq_dqn(params, F, hidden, A, mbs, g, torch.float32)
    d, d64, d32 = new - params, new64 - params.astype(np.float64), new32 - params
    print(f"seq dqn LSTM h={hidden}: delta rel err kernel {_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}")
    assert stats.opt_steps == steps and stats.num_steps == sum(len(e["action"]) for e in mbs[-1])
    assert _rel(d, d64) <= max(2e-4, 4 * _rel(d32, d64) + 1e-5)


# ------------------------------------------------------------------------------------------------
# Learning and status codes
# ------------------------------------------------------------------------------------------------
def test_dqn_lstm_learns_memory_game(ctx):
    """MemoryGame(2, 4): the reward depends on the first observation of the episode, which only a recurrent Q-network can
    keep; with an LSTM the greedy mean final reward reaches 0.9 under the GRU test's schedule (test_gpu_dqn_seq.py)."""
    E = 2048
    env = R.build_env(ctx, R.MemoryGame(2, 4), E, seed=6)
    agent = R.DqnConfig(action_value_fn_config=R.LstmLinearConfig(hidden_dim=8), minibatch_steps=20_000, opt_steps_per_update=40,
                        buffer_capacity=200, optimizer_config=R.AdamConfig(learning_rate=3e-3),
                        exploration_rate=R.ExplorationRateSchedule(1.0, 0.1, 150_000),
                        update_size=R.DataCollectionSchedule(10 * E, 10 * E), sample_seed=2).build_agent(env)
    agent.action_value_fn.set_weights(R.init_lstm_linear_params(np.random.default_rng(0), env.num_features, 8, 2))
    rb = agent.buffer()
    means = []
    for period in range(20):
        bound = agent.min_update_size().divide(E)
        traj = R.Trajectory(env, bound.min_steps + bound.slack_steps)
        R.rollout(env, agent.actor(training=True), bound, traj)
        rb.write_experience(traj)
        agent.batch_update(rb, {})
        ev = R.Trajectory(env, 25)
        summ = R.rollout(env, agent.actor(training=False), R.HistoryDataBound(25, 0), ev)
        means.append(summ.episode_reward.mean)
        traj.close(); ev.close()
    print("greedy mean episode reward, LSTM:", [round(x, 3) for x in means])
    assert max(means[-3:]) >= 0.9


def test_lstm_actor_critic_learns_bandits(ctx):
    """TRPO with an LSTM policy and an LSTM critic on 2-armed Bernoulli bandit trials raises the mean per-step reward."""
    arms, episodes, E, hidden = 2, 10, 2048, 8
    T = 2 * episodes - 1
    env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(arms), episodes), E, seed=4)
    lcfg = R.LstmLinearConfig(hidden_dim=hidden)
    agent = R.ActorCriticConfig(policy_config=R.TrpoConfig(policy_fn_config=lcfg),
                                critic_config=R.ValuesOptConfig(state_value_fn_config=lcfg, opt_steps_per_update=20)
                                ).build_agent(env)
    rng = np.random.default_rng(0)
    agent.policy.policy_fn.set_weights(R.init_lstm_linear_params(rng, env.num_features, hidden, arms))
    agent.critic.state_value_fn.set_weights(R.init_lstm_linear_params(rng, env.num_features, hidden, 1))
    traj = R.Trajectory(env, T)
    means = []
    for period in range(25):
        summ = R.rollout(env, agent.actor(), R.HistoryDataBound(T, 0), traj)
        means.append(summ.step_reward.mean)
        agent.batch_update(traj, {})
    print("mean step reward per period:", [round(x, 4) for x in means])
    assert np.mean(means[-3:]) > np.mean(means[:3]) * 1.08


def test_lstm_status_codes(ctx):
    lib = ctx._lib
    h = C.c_void_p()
    for args in [(6, 0, 2), (6, 129, 2), (0, 4, 2), (37, 4, 2), (6, 4, 0), (6, 4, 33)]:
        assert lib.rl_lstmnet_create(ctx.handle, *args, L.RL_ACT_RELU, C.byref(h)) == L.RL_ERR_INVALID_ARG, args
    net = R.LstmLinear(ctx, 6, 4, 2)
    assert net.num_params == R.lstm_linear_num_params(6, 4, 2) == 4 * 4 * 10 + 32 + 8 + 2
    bad = np.zeros(net.num_params - 1, np.float32)
    assert lib.rl_grunet_set_weights(net.handle, bad.ctypes.data_as(C.c_void_p), bad.size) == L.RL_ERR_INVALID_ARG
    assert lib.rl_grunet_get_weights(net.handle, bad.ctypes.data_as(C.c_void_p), bad.size) == L.RL_ERR_INVALID_ARG
    # an optimizer built for a GRU of the same shape belongs to another module
    env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(2), 3), 16, seed=1)
    traj = R.Trajectory(env, 8)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(8, 0), traj)
    critic = R.LstmLinear(ctx, 6, 4, 1)
    gru = R.GruLinear(ctx, 6, 4, 1)
    tg = ctx.to_device(np.zeros((8, 16), np.float32))
    stats = L.OptStats()
    assert lib.rl_value_update_seq(traj.handle, tg.c, critic.handle, R.Adam(gru, R.AdamConfig()).handle, 2, C.byref(stats)) == L.RL_ERR_INVALID_ARG
    assert lib.rl_value_update_seq(traj.handle, tg.c, critic.handle, R.Adam(critic, R.AdamConfig()).handle, 2, C.byref(stats)) == L.RL_OK
