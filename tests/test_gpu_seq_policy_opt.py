"""GPU parity and behaviour of the PPO and REINFORCE updates through a recurrent policy (Chain<Gru, Linear>,
Chain<Lstm, Linear>): rl_ppo_update_seq / rl_reinforce_update_seq, Ppo / Reinforce with a GruLinearConfig or
LstmLinearConfig policy, against the torch-CPU restatement in f64 (tests/seq_policy_oracle.py).

Trajectories are rolled out by the recurrent categorical actor on the bandit meta-env, so batches hold interrupted
episodes; the head of more than 16 outputs runs on a synthetic trajectory (Trajectory.load).  Shapes: K9 (one thread per
lane) at GRU 6-4-2 (its compile-time instance), GRU hidden 3 and 8, LSTM hidden 4 and 8; K10 (tiled GEMMs) at hidden 24
(FP32 pipe) and 128 (the GRU's per-step GEMMs on tcgen05).

Tolerances are those of test_gpu_update.py's MLP PPO / REINFORCE tests: PPO entropy within 1e-5 relative, first loss
within 1e-5, last loss within 1e-4, parameter delta within max(2e-4, 4x the torch-f32 run's own distance from f64 + 1e-5);
REINFORCE entropy and loss within 1e-5, delta within max(2e-3, 4x torch-f32's + 1e-5)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import relearn_b200 as R
from relearn_b200 import _lib as L

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from tests import seq_policy_oracle as SPO  # noqa: E402
from tests.test_gpu_gru_update import _collect as _collect_gru, _per_episode  # noqa: E402
from tests.test_gpu_lstm import _collect as _collect_lstm  # noqa: E402
from tests.test_gpu_seq_update_tiling import _load, _params as _synthetic_params, _planes  # noqa: E402

CONT, PAD = L.RL_CONTINUE, L.RL_PAD

# (cell, hidden, arms, episodes per trial, activation); hidden <= 8: K9, above: K10
SHAPES = [
    pytest.param("gru", 4, 2, 10, "relu", id="gru4"),       # config 4: the <6, 4, 2> compile-time instance
    pytest.param("gru", 3, 3, 6, "tanh", id="gru3"),
    pytest.param("gru", 8, 5, 4, "tanh", id="gru8"),
    pytest.param("lstm", 4, 2, 10, "relu", id="lstm4"),
    pytest.param("lstm", 8, 4, 5, "tanh", id="lstm8"),
    pytest.param("gru", 24, 3, 4, "tanh", id="gru24"),
    pytest.param("lstm", 24, 3, 4, "relu", id="lstm24"),
    pytest.param("gru", 128, 10, 3, "relu", id="gru128"),
    pytest.param("lstm", 128, 10, 3, "relu", id="lstm128"),
]
# (clip distance, Adam steps, learning rate, advantage signal).  The small clip runs with larger steps on advantages that
# favour action 0, so that the ratio leaves [1 - eps, 1 + eps] on a clear share of the samples: on noise alone the small
# bandit policies hardly move (at 0.05 / 25 steps / 1e-3, 0.1 % of GRU 6-4-2's samples were clipped at the last step).
CLIPS = [pytest.param(0.2, 10, 1e-3, 0.0, id="clip0.2"), pytest.param(0.05, 25, 1e-2, 1.0, id="clip0.05")]


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) /
                 max(np.linalg.norm(np.asarray(b, np.float64)), 1e-300))


def _batch(ctx, cell, hidden, arms, episodes, activation, seed, signal=0.0):
    """A rollout of the policy itself (two trials per lane and an interrupted third), advantages ~ N(0, 1) + `signal` where
    the action was 0 and - `signal` elsewhere."""
    E, T = (80 if hidden <= 24 else 40), 2 * (2 * episodes - 1) + 3
    collect = _collect_gru if cell == "gru" else _collect_lstm
    env, traj, net, params, host, spans = collect(ctx, hidden, arms, episodes, E, T, seed=seed, scale=1.5, activation=activation)
    adv = (np.random.default_rng(seed + 100).normal(size=(T, E)) + signal * np.where(host["action"] == 0, 1, -1)).astype(np.float32)
    eps, acts, advs = _per_episode(host["obs"], spans), _per_episode(host["action"], spans), _per_episode(adv, spans)
    return dict(env=env, traj=traj, net=net, params=params, F=env.num_features, A=env.num_actions, adv=adv,
                oracle_args=(eps, acts, advs), num_steps=sum(b - a for _, a, b in spans))


def _oracle(kind, cell, b, hidden, activation, dtype, **kw):
    fn = SPO.seq_ppo_update if kind == "ppo" else SPO.seq_reinforce_update
    return fn(*SPO.CELLS[cell], b["params"], b["F"], hidden, b["A"], *b["oracle_args"], dtype=dtype, activation=activation, **kw)


@pytest.mark.parametrize("clip,steps,lr,signal", CLIPS)
@pytest.mark.parametrize("cell,hidden,arms,episodes,activation", SHAPES)
def test_seq_ppo_update_matches_f64(ctx, cell, hidden, arms, episodes, activation, clip, steps, lr, signal):
    """Ppo::update (ppo.rs:97-147) through BPTT: no_grad behaviour log-probabilities, then `steps` Adam steps on the clipped
    surrogate.  The small clip puts a clear share of the samples on the clipped branch, whose gradient is zero."""
    b = _batch(ctx, cell, hidden, arms, episodes, activation, seed=hidden + arms + steps, signal=signal)
    cfg = R.PpoConfig(opt_steps_per_update=steps, clip_distance=clip, optimizer_config=R.AdamConfig(learning_rate=lr))
    policy = R.Ppo(b["net"], cfg)
    log = {}
    policy.update(b["traj"], ctx.to_device(b["adv"]), log)
    new = b["net"].get_weights()
    kw = dict(opt_steps=steps, clip_distance=clip, lr=lr)
    new64, l64, ent64, share64 = _oracle("ppo", cell, b, hidden, activation, torch.float64, **kw)
    new32, _, _, _ = _oracle("ppo", cell, b, hidden, activation, torch.float32, **kw)
    p = b["params"]
    d, d64, d32 = new - p, new64 - p.astype(np.float64), new32 - p
    print(f"{cell}{hidden} clip {clip}: delta rel err kernel {_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}; loss "
          f"{log['loss_first']:.6f}->{log['loss_last']:.6f} vs {l64[0]:.6f}->{l64[-1]:.6f}; clipped share at the last step "
          f"{share64[-1]:.3f}")
    if clip < 0.1:
        assert share64[-1] >= 0.1
    assert log["num_steps"] == b["num_steps"]
    np.testing.assert_allclose(log["entropy"], ent64, rtol=1e-5)
    np.testing.assert_allclose(log["loss_first"], l64[0], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(log["loss_last"], l64[-1], rtol=1e-4, atol=1e-6)
    assert _rel(d, d64) <= max(2e-4, 4 * _rel(d32, d64) + 1e-5)


@pytest.mark.parametrize("cell,hidden,arms,episodes,activation", SHAPES)
def test_seq_reinforce_update_matches_f64(ctx, cell, hidden, arms, episodes, activation):
    """Reinforce::update (reinforce.rs:64-89) through BPTT: one Adam step on -(log_probs * advantages).mean(), with the
    entropy of that evaluation logged."""
    b = _batch(ctx, cell, hidden, arms, episodes, activation, seed=31 + hidden + arms)
    policy = R.Reinforce(b["net"], R.ReinforceConfig())
    log = {}
    policy.update(b["traj"], ctx.to_device(b["adv"]), log)
    new = b["net"].get_weights()
    new64, l64, ent64 = _oracle("reinforce", cell, b, hidden, activation, torch.float64)
    new32, _, _ = _oracle("reinforce", cell, b, hidden, activation, torch.float32)
    p = b["params"]
    d, d64, d32 = new - p, new64 - p.astype(np.float64), new32 - p
    print(f"{cell}{hidden}: delta rel err kernel {_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}")
    assert log["num_steps"] == b["num_steps"]
    np.testing.assert_allclose(log["entropy"], ent64, rtol=1e-5)
    np.testing.assert_allclose(log["loss_first"], l64, rtol=1e-5, atol=1e-7)
    # the first Adam step moves every parameter by ~lr * sign(g): parameters with a gradient near 0 dominate the error
    assert _rel(d, d64) <= max(2e-3, 4 * _rel(d32, d64) + 1e-5)


def test_seq_policy_gemm_formulation_serves_the_small_modules_too():
    """K10 against the oracle on the modules K9 normally serves: the PPO and REINFORCE cases above in a child process with
    RL_SEQ_FORCE_BIG=1 (the switch is read once per process)."""
    if os.environ.get("RL_SEQ_FORCE_BIG") == "1":
        pytest.skip("already the forced run")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RL_SEQ_FORCE_BIG="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_seq_policy_opt.py"), "-x", "-q", "-m",
                        "gpu", "-k", "(ppo_update_matches or reinforce_update_matches) and not 128 and not 24"],
                       capture_output=True, text=True, env=env, cwd=root, timeout=1200)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and "15 passed" in r.stdout


def _spans(succ):
    """(lane, start, end) of every episode in [T, E] successor codes with a PAD tail."""
    out = []
    for e in range(succ.shape[1]):
        n = int((succ[:, e] != PAD).sum())
        start = 0
        for t in np.flatnonzero(succ[:n, e] != CONT):
            out.append((e, start, int(t) + 1))
            start = int(t) + 1
    return out


@pytest.mark.parametrize("cell", ["gru", "lstm"])
def test_seq_ppo_wide_head_matches_f64(ctx, cell):
    """A head of 20 outputs, K10's HEAD_MAXA = 32 instance of big_head_kernel, on a synthetic trajectory (the bandit
    meta-env stops at 16 arms): episodes of length 1, lanes of one episode over all T steps, PAD tails, empty lanes."""
    E, T, F, H, A, steps, clip = 300, 30, 8, 24, 20, 10, 0.2
    pl = _planes(41, E, T, F, A)
    env, traj = _load(ctx, pl, E, T, F)
    params = _synthetic_params(cell, 43, F, H, A)
    net = (R.GruLinear if cell == "gru" else R.LstmLinear)(ctx, F, H, A)
    net.set_weights(params)
    log = {}
    R.Ppo(net, R.PpoConfig(opt_steps_per_update=steps, clip_distance=clip)).update(traj, ctx.to_device(pl["adv"]), log)
    new = net.get_weights()
    spans = _spans(pl["succ"])
    oargs = (_per_episode(pl["obs"], spans), _per_episode(pl["action"], spans), _per_episode(pl["adv"], spans))
    run = lambda dtype: SPO.seq_ppo_update(*SPO.CELLS[cell], params, F, H, A, *oargs, opt_steps=steps, clip_distance=clip, dtype=dtype)
    new64, l64, ent64, _ = run(torch.float64)
    new32, _, _, _ = run(torch.float32)
    d, d64, d32 = new - params, new64 - params.astype(np.float64), new32 - params
    print(f"{cell} A={A}: delta rel err kernel {_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}")
    assert log["num_steps"] == int((pl["succ"] != PAD).sum()) == sum(b - a for _, a, b in spans)
    np.testing.assert_allclose(log["entropy"], ent64, rtol=1e-5)
    np.testing.assert_allclose(log["loss_first"], l64[0], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(log["loss_last"], l64[-1], rtol=1e-4, atol=1e-6)
    assert _rel(d, d64) <= max(2e-4, 4 * _rel(d32, d64) + 1e-5)


@pytest.mark.parametrize("cell,hidden", [("gru", 4), ("lstm", 24)])
def test_seq_ppo_zero_opt_steps(ctx, cell, hidden):
    """opt_steps_per_update = 0: the parameters stay as they are and the behaviour policy's entropy is still reported, as
    the Mlp driver does."""
    b = _batch(ctx, cell, hidden, 2, 6, "relu", seed=5)
    log = {}
    R.Ppo(b["net"], R.PpoConfig(opt_steps_per_update=0)).update(b["traj"], ctx.to_device(b["adv"]), log)
    np.testing.assert_array_equal(b["net"].get_weights(), b["params"])
    _, _, ent64, _ = _oracle("ppo", cell, b, hidden, "relu", torch.float64, opt_steps=0)
    assert log["num_steps"] == b["num_steps"] and log["loss_first"] == 0.0 == log["loss_last"]
    np.testing.assert_allclose(log["entropy"], ent64, rtol=1e-5)


def test_seq_policy_opt_status_codes(ctx):
    lib = ctx._lib
    F, H, A, E, T = 6, 4, 2, 16, 8
    env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(2), 3), E, seed=1)
    net = R.GruLinear(ctx, F, H, A)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(T, 0), traj)
    adv = ctx.to_device(np.zeros((T, E), np.float32))
    opt = R.Adam(net, R.AdamConfig())
    stats = L.PolicyOptStats()

    def ppo(traj_h, adv_c, net_h, opt_h, cfg=L.PpoCfg(2, 0.2)):
        return lib.rl_ppo_update_seq(traj_h, adv_c, net_h, opt_h, C.byref(cfg) if cfg is not None else None, C.byref(stats))

    def reinforce(traj_h, adv_c, net_h, opt_h):
        return lib.rl_reinforce_update_seq(traj_h, adv_c, net_h, opt_h, C.byref(stats))

    ok = (traj.handle, adv.c, net.handle, opt.handle)
    ctx2 = R.Context(0)
    for fn in (ppo, reinforce):
        # NULL arguments
        for i in range(4):
            args = list(ok)
            args[i] = None
            assert fn(*args) == L.RL_ERR_INVALID_ARG, (fn.__name__, i)
        # an optimizer of another module of the same shape, and an Mlp's optimizer
        other = R.GruLinear(ctx, F, H, A)
        assert fn(traj.handle, adv.c, net.handle, R.Adam(other, R.AdamConfig()).handle) == L.RL_ERR_INVALID_ARG
        mlp = R.Mlp(ctx, F, [16], A)
        assert fn(traj.handle, adv.c, net.handle, R.Adam(mlp, R.AdamConfig()).handle) == L.RL_ERR_INVALID_ARG
        # a module of another context
        net2 = R.GruLinear(ctx2, F, H, A)
        assert fn(traj.handle, adv.c, net2.handle, R.Adam(net2, R.AdamConfig()).handle) == L.RL_ERR_INVALID_ARG
        # a feature count that does not match the trajectory's
        wide = R.GruLinear(ctx, F + 1, H, A)
        assert fn(traj.handle, adv.c, wide.handle, R.Adam(wide, R.AdamConfig()).handle) == L.RL_ERR_UNSUPPORTED
        assert fn(*ok) == L.RL_OK
    assert ppo(*ok, cfg=None) == L.RL_ERR_INVALID_ARG
    # an optimizer step count out of range
    assert ppo(*ok, cfg=L.PpoCfg(100_001, 0.2)) == L.RL_ERR_INVALID_ARG
    assert ppo(*ok, cfg=L.PpoCfg(2**32 + 2, 0.2)) == L.RL_ERR_INVALID_ARG
    assert ppo(*ok, cfg=L.PpoCfg(100_000, 0.2)) == L.RL_OK


# ------------------------------------------------------------------------------------------------
# Behaviour through ActorCriticConfig
# ------------------------------------------------------------------------------------------------
def _bandit_step_rewards(ctx, policy_config, critic_cell, hidden, periods):
    """Mean per-step reward of every period of an actor-critic agent on 2-armed Bernoulli bandit trials (10 episodes each),
    in the form of test_rl2_actor_critic_learns_bandits; the critic is of the policy's cell and size."""
    arms, episodes, E = 2, 10, 2048
    T = 2 * episodes - 1
    env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(arms), episodes), E, seed=4)
    agent = R.ActorCriticConfig(policy_config=policy_config,
                                critic_config=R.ValuesOptConfig(state_value_fn_config=critic_cell(hidden_dim=hidden),
                                                                opt_steps_per_update=20)).build_agent(env)
    assert agent.policy.recurrent and agent.actor().seq_net is agent.policy.policy_fn
    init = R.init_gru_linear_params if critic_cell is R.GruLinearConfig else R.init_lstm_linear_params
    rng = np.random.default_rng(0)
    agent.policy.policy_fn.set_weights(init(rng, env.num_features, hidden, arms))
    agent.critic.state_value_fn.set_weights(init(rng, env.num_features, hidden, 1))
    traj = R.Trajectory(env, T)
    means = []
    for period in range(periods):
        summ = R.rollout(env, agent.actor(), R.HistoryDataBound(T, 0), traj)
        means.append(summ.step_reward.mean)
        log = {}
        agent.batch_update(traj, log)
        assert set(log) >= {"entropy", "loss_first", "loss_last", "num_steps", "policy/update_time"}
    traj.close(); env.close()
    return means


@pytest.mark.parametrize("hidden", [8, 128])
def test_rl2_ppo_gru_learns_bandits(ctx, hidden):
    """PPO with a GRU policy and a GRU critic (hidden 128: the rl2-bandits.rs module size, served by K10 on the tensor cores)
    raises the mean per-step reward of the meta-episodes; random play earns 0.5 * (episodes / T) = 0.263.  Measured on a B200
    (1000 W): the mean of the last three periods over the first three was 1.15 at hidden 8 (0.262 -> 0.302) and 1.21 at
    hidden 128 (0.262 -> 0.317); the bar is 1.08, as for TRPO."""
    pc = R.PpoConfig(policy_fn_config=R.GruLinearConfig(hidden_dim=hidden), optimizer_config=R.AdamConfig(learning_rate=3e-3))
    means = _bandit_step_rewards(ctx, pc, R.GruLinearConfig, hidden, 25)
    print("PPO GRU", hidden, "mean step reward per period:", [round(x, 4) for x in means])
    assert np.mean(means[-3:]) > np.mean(means[:3]) * 1.08


def test_rl2_reinforce_lstm_learns_bandits(ctx):
    """REINFORCE with an LSTM policy and an LSTM critic raises the mean per-step reward of the meta-episodes.  One Adam step
    per period: at a learning rate of 0.01 over 25 periods the reward stayed at random play's 0.263; at 0.1 over 60 periods a
    B200 run (1000 W) went from 0.263 to 0.301 (1.15x) over the first and last three periods; the bar is 1.08."""
    pc = R.ReinforceConfig(policy_fn_config=R.LstmLinearConfig(hidden_dim=8), optimizer_config=R.AdamConfig(learning_rate=0.1))
    means = _bandit_step_rewards(ctx, pc, R.LstmLinearConfig, 8, 60)
    print("REINFORCE LSTM mean step reward per period:", [round(x, 4) for x in means])
    assert np.mean(means[-3:]) > np.mean(means[:3]) * 1.08


def test_ppo_gru_learns_memory_game(ctx):
    """MemoryGame(2, 4): the reward (+1 / -1) depends on the first observation of the episode, which a feed-forward policy
    never sees again, so it cannot beat random play's mean of 0 (the argument of test_dqn_gru_learns_memory_game).  PPO with
    a GRU policy and a GRU critic learns to recall it: on a B200 (1000 W) the mean episode reward of the stochastic policy
    went from 0.00 to 0.98 over the last three of 30 periods; the bar is 0.9."""
    E, T = 2048, 25
    env = R.build_env(ctx, R.MemoryGame(2, 4), E, seed=6)
    gcfg = R.GruLinearConfig(hidden_dim=8)
    agent = R.ActorCriticConfig(policy_config=R.PpoConfig(policy_fn_config=gcfg, optimizer_config=R.AdamConfig(learning_rate=3e-3)),
                                critic_config=R.ValuesOptConfig(state_value_fn_config=gcfg, opt_steps_per_update=20)).build_agent(env)
    rng = np.random.default_rng(0)
    agent.policy.policy_fn.set_weights(R.init_gru_linear_params(rng, env.num_features, 8, 2))
    agent.critic.state_value_fn.set_weights(R.init_gru_linear_params(rng, env.num_features, 8, 1))
    traj = R.Trajectory(env, T)
    means = []
    for period in range(30):
        summ = R.rollout(env, agent.actor(), R.HistoryDataBound(T, 0), traj)
        means.append(summ.episode_reward.mean)
        agent.batch_update(traj, {})
    traj.close(); env.close()
    print("PPO GRU memory game mean episode reward per period:", [round(x, 3) for x in means])
    assert np.mean(means[-3:]) >= 0.9
