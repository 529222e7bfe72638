"""GPU checks of the Beta Thompson-sampling agent (src/agents/bandits/thompson_sampling.rs): the actor inside the fused
rollout against tests/thompson_oracle.py on replayed and Philox noise, the fold of batch_update, the distribution of the
device's Beta draw, the inner agent of the resetting meta agent (the rl2-bandits TS / OTS rows), the training loop, and
the rejections."""
import math

import numpy as np
import pytest
from scipy import integrate, stats

import oracle as O
import relearn_b200 as R
from relearn_b200 import _lib as L
from tests import parity as P
from tests import thompson_oracle as TO

pytestmark = pytest.mark.gpu


def _obs_index(obs_row):
    return int(np.flatnonzero(obs_row)[-1]) if np.any(obs_row) else 0


def _random_counts(rng, R_, S, A):
    low = rng.integers(1, 40, size=(R_, S, A)).astype(np.uint64)
    high = rng.integers(1, 40, size=(R_, S, A)).astype(np.uint64)
    low[:, :, -1] = low[:, :, 0]   # exact ties between the first and the last action
    high[:, :, -1] = high[:, :, 0]
    return low, high


def _oracles(n, S, A, st, num_samples, low, high):
    out = []
    for r in range(n):
        o = TO.BetaThompsonOracle(S, A, (st.reward_lo, st.reward_hi), num_samples)
        o.low, o.high = low[r].copy(), high[r].copy()
        out.append(o)
    return out


def _check_actions(host, oracles, shared, training, rngs, philox_t0=None):
    """Every action is the oracle actor's choice for the recorded observation (counts are frozen during a rollout).  A
    disagreement is allowed only where the oracle's two largest sums agree to 1e-12 relative (device `log` against glibc
    `log`); the draws of every action are made either way, so the streams stay aligned."""
    lib = O.lib()
    near = 0
    for e in range(host["lane_len"].shape[0]):
        o = oracles[0 if shared else e]
        U = TO.uniform_of(rngs[e]) if training else None
        for t in range(int(host["lane_len"][e])):
            if philox_t0 is not None:
                lib.ro_rng_set_step(rngs[e].ref, philox_t0 + t)
            vals = o.values(_obs_index(host["obs"][t, e]), training, U)
            want, got = TO.last_argmax(vals), int(host["action"][t, e])
            if want != got:
                assert training and TO.near_tie(vals, 1e-12), (e, t, want, got, vals)
                near += 1
    assert near <= 2, near


def _check_fold(agent, host, oracles, shared):
    for e in range(host["lane_len"].shape[0]):
        o = oracles[0 if shared else e]
        for t in range(int(host["lane_len"][e])):
            o.step_update(_obs_index(host["obs"][t, e]), int(host["action"][t, e]), float(host["reward"][t, e]))
    gl, gh = agent.get_counts()
    for r in range(len(oracles)):
        np.testing.assert_array_equal(gl[r], oracles[r].low)
        np.testing.assert_array_equal(gh[r], oracles[r].high)


MODES = [("training-1", True, 1), ("training-10", True, 10), ("evaluation", False, 1)]


@pytest.mark.parametrize("cfg", [R.Chain(), R.MemoryGame(3, 2)], ids=["chain", "memory"])
@pytest.mark.parametrize("shared", [False, True], ids=["table-per-lane", "shared-table"])
@pytest.mark.parametrize("mode,training,num_samples", MODES, ids=[m[0] for m in MODES])
def test_bts_actor_and_update_match_the_oracle(ctx, cfg, shared, mode, training, num_samples):
    rng = np.random.default_rng(5)
    E, T = 48, 40
    env = R.build_env(ctx, cfg, E, seed=9)
    st = env.structure
    S, A = st.num_observations, st.num_actions
    reps = 1 if shared else E
    agent = R.BetaThompsonSamplingAgentConfig(num_samples).build_agent(env, num_replicas=reps)
    l0, h0 = agent.get_counts()
    assert (l0 == 1).all() and (h0 == 1).all()  # thompson_sampling.rs:104-105
    low, high = _random_counts(rng, reps, S, A)
    agent.set_counts(low, high)
    words = P.random_words(rng, E, 40 * T * A * num_samples)
    actor_words = P.random_words(rng, E, 40 * T * A * num_samples)
    env.set_noise_replay(words, actor_words)
    traj = R.Trajectory(env, T)
    R.rollout(env, agent.actor(training=training), R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    oracles = _oracles(reps, S, A, st, num_samples, low, high)
    _check_actions(host, oracles, shared, training, [O.ScriptRng(actor_words[e]) for e in range(E)])
    ref = P.oracle_rollout(cfg, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), env_words=words)
    P.compare_traj(host, ref, what=f"thompson {mode}")
    agent.update(traj)
    _check_fold(agent, host, oracles, shared)


@pytest.mark.parametrize("num_samples", [1, 10])
@pytest.mark.parametrize("cfg", [R.Chain(), R.MemoryGame(3, 2)], ids=["chain", "memory"])
def test_bts_philox_matches_the_oracle(ctx, cfg, num_samples):
    """Philox noise at a nonzero lane offset and step counter: the draws depend on (seed, global lane, step) only."""
    rng = np.random.default_rng(8)
    E, T, seed, off, t0 = 6, 30, 0xC0FFEE, 777, 11
    env = R.build_env(ctx, cfg, E, seed=seed, lane_offset=off)
    env.set_noise_philox(seed, t0)
    st = env.structure
    S, A = st.num_observations, st.num_actions
    agent = R.BetaThompsonSamplingAgentConfig(num_samples).build_agent(env, num_replicas=1)
    low, high = _random_counts(rng, 1, S, A)
    agent.set_counts(low, high)
    traj = R.Trajectory(env, T)
    summ = R.rollout(env, agent.actor(training=True), R.HistoryDataBound(T, 0), traj)
    host = traj.to_host()
    oracles = _oracles(1, S, A, st, num_samples, low, high)
    _check_actions(host, oracles, True, True, [O.PhiloxRng(seed, off + e, t0) for e in range(E)], philox_t0=t0)
    ref = P.oracle_rollout(cfg, E, T, 0, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), philox_seed=seed,
                           lane_offset=off, t0=t0)
    P.compare_traj(host, ref, what="thompson philox")
    P.compare_summary(summ, ref["summary"])
    agent.update(traj)
    _check_fold(agent, host, oracles, True)


def _action0_frequency(ctx, a0, b0, a1, b1, num_samples, seed):
    """One step on 2^20 Chain lanes, all in state 0, from one shared table: the share of lanes whose draw picked action 0."""
    E = 1 << 20
    env = R.build_env(ctx, R.Chain(), E, seed=seed)
    env.set_noise_philox(seed, 0)
    agent = R.BetaThompsonSamplingAgentConfig(num_samples).build_agent(env)
    low, high = agent.get_counts()
    high[0, 0] = [a0, a1]  # Beta(alpha = high, beta = low)
    low[0, 0] = [b0, b1]
    agent.set_counts(low, high)
    traj = R.Trajectory(env, 1)
    R.rollout(env, agent.actor(training=True), R.HistoryDataBound(1, 0), traj)
    acts = traj.to_host()["action"][0]
    return float(np.mean(acts == 0)), E


@pytest.mark.parametrize("a0,b0,a1,b1", [(2, 1, 1, 1), (5, 3, 4, 4), (400, 600, 410, 590)])
def test_bts_draw_distribution(ctx, a0, b0, a1, b1):
    """P(action 0) = P(X0 > X1) = integral of f0 * F1 (ties have probability 0 and would go to action 1)."""
    if (a0, b0, a1, b1) == (2, 1, 1, 1):
        p = 2.0 / 3.0
    else:
        f0, F1 = stats.beta(a0, b0).pdf, stats.beta(a1, b1).cdf
        p = integrate.quad(lambda x: f0(x) * F1(x), 0.0, 1.0, limit=200, points=[a0 / (a0 + b0)])[0]
    freq, n = _action0_frequency(ctx, a0, b0, a1, b1, 1, seed=31 + a0)
    sigma = math.sqrt(p * (1.0 - p) / n)
    print(f"Beta({a0},{b0}) vs Beta({a1},{b1}): device {freq:.5f}, exact {p:.5f}, sigma {sigma:.5f}")
    assert abs(freq - p) < 5 * sigma


def test_bts_draw_distribution_ten_samples(ctx):
    """num_samples = 10: P(sum of 10 Beta(5, 3) > sum of 10 Beta(4, 4)), estimated with scipy from 4 M pairs of sums."""
    a0, b0, a1, b1 = 5, 3, 4, 4
    rs = np.random.default_rng(2024)
    m, hits = 4_000_000, 0
    for _ in range(8):
        k = m // 8
        s0 = stats.beta(a0, b0).rvs(size=(k, 10), random_state=rs).sum(axis=1)
        s1 = stats.beta(a1, b1).rvs(size=(k, 10), random_state=rs).sum(axis=1)
        hits += int(np.count_nonzero(s0 > s1))
    p = hits / m
    freq, n = _action0_frequency(ctx, a0, b0, a1, b1, 10, seed=77)
    sigma = math.sqrt(p * (1.0 - p) / n + p * (1.0 - p) / m)
    print(f"10 samples: device {freq:.5f}, Monte Carlo {p:.5f}, sigma {sigma:.5f}")
    assert abs(freq - p) < 5 * sigma


# --- the inner agent of the resetting meta agent (rl2-bandits TS / OTS) ---------------------------------------------------
META = R.MetaEnv(R.UniformBernoulliBandits(5), 10)


def _trial_len(cfg):
    return 2 * cfg.episodes_per_trial - 1


@pytest.mark.parametrize("num_samples", [1, 10], ids=["ts", "ots"])
@pytest.mark.parametrize("noise", ["replay", "philox"])
def test_meta_thompson_matches_the_oracle(ctx, num_samples, noise):
    rng = np.random.default_rng(19)
    E = 48 if noise == "replay" else 16
    Lt = _trial_len(META)
    min_steps, slack = 3 * Lt + 2, Lt
    cap = min_steps + slack
    if noise == "replay":
        env = R.build_env(ctx, META, E, seed=3)
        env_words = P.random_words(rng, E, 40 * cap * 5 * num_samples)  # one words-per-lane count for both streams
        actor_words = P.random_words(rng, E, 40 * cap * 5 * num_samples)
        env.set_noise_replay(env_words, actor_words)
        check_kw, ref_kw = {"actor_words": actor_words}, {"env_words": env_words}
    else:
        seed, off, t0 = 0xFACE, 300, 4
        env = R.build_env(ctx, META, E, seed=seed, lane_offset=off)
        env.set_noise_philox(seed, t0)
        check_kw = ref_kw = {"philox_seed": seed, "lane_offset": off, "t0": t0}
    agent = R.ResettingMetaAgentConfig(R.BetaThompsonSamplingAgentConfig(num_samples)).build_agent(env)
    traj = R.Trajectory(env, cap)
    summ = R.rollout(env, agent.actor(), R.HistoryDataBound(min_steps, slack), traj)
    host = traj.to_host()
    near = TO.check_meta_actions(host, 5, num_samples, **check_kw)
    assert near <= 2, near
    ref = P.oracle_rollout(META, E, min_steps, slack, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), **ref_kw)
    P.compare_traj(host, ref, what=f"meta thompson {noise}")
    P.compare_summary(summ, ref["summary"])
    assert summ.num_stored_steps == int(ref["lane_len"].sum())


def _meta_trial_rewards(ctx, cfg, inner_cfg, E, trials, seed):
    Lt = _trial_len(cfg)
    env = R.build_env(ctx, cfg, E, seed=seed)
    env.set_noise_philox(seed, 0)
    traj = R.Trajectory(env, trials * Lt)
    summ = R.rollout(env, R.ResettingMetaAgentConfig(inner_cfg).build_agent(env).actor(), R.HistoryDataBound(trials * Lt, 0), traj)
    er = summ.episode_reward
    assert er.count == E * trials
    return er.mean, math.sqrt(er.variance() / er.count)


def test_meta_thompson_one_hot_bandits_learns(ctx):
    """MetaEnv<OneHotBandits(3)> with 20 pulls per trial: Thompson sampling earns clearly more than the random agent's 20 / 3."""
    cfg = R.MetaEnv(R.OneHotBandits(3), 20)
    ts = _meta_trial_rewards(ctx, cfg, R.BetaThompsonSamplingAgentConfig(1), 256, 4, 21)
    rnd = _meta_trial_rewards(ctx, cfg, R.RandomAgentConfig(), 256, 4, 21)
    print(f"one-hot 3 x 20: thompson {ts}, random {rnd}")
    assert ts[0] > 0.7 * (20 - 3)
    assert ts[0] > rnd[0] + 5.0


def test_meta_thompson_beats_eps_greedy_and_random(ctx):
    """k = 10, n = 100 over 20 480 trials: TS and OTS earn more than eps-greedy (0.2) and random by more than 5 standard
    errors, as the RL^2 paper's bandit table leads one to expect."""
    cfg = R.MetaEnv(R.UniformBernoulliBandits(10), 100)
    E, trials = 10240, 2
    rows = {name: _meta_trial_rewards(ctx, cfg, c, E, trials, 99) for name, c in [
        ("random", R.RandomAgentConfig()), ("eps-greedy", R.TabularQLearningAgentConfig(0.2)),
        ("ts", R.BetaThompsonSamplingAgentConfig(1)), ("ots", R.BetaThompsonSamplingAgentConfig(10))]}
    print(rows)
    for good in ("ts", "ots"):
        for base in ("random", "eps-greedy"):
            (mg, sg), (mb, sb) = rows[good], rows[base]
            assert mg - mb > 5 * math.hypot(sg, sb), (good, base, rows)


def test_train_device_with_a_shared_table(ctx):
    """train_parallel on Chain with one shared table: every stored step is folded in (the counts total the steps plus the
    (1, 1) start of every pair), and the evaluation actor takes the action of the highest posterior mean."""
    E, steps, periods = 64, 40, 5
    env = R.build_env(ctx, R.Chain(), E, seed=4)
    agent = R.BetaThompsonSamplingAgentConfig().build_agent(env)
    assert agent.min_update_size() == R.HistoryDataBound(1, 0)
    stored = []

    def on_period(i, summary):
        stored.append(summary.num_stored_steps)

    R.train_device(agent, env, R.TrainParallelConfig(num_periods=periods, num_threads=E, min_worker_steps=steps),
                   on_period=on_period)
    low, high = agent.get_counts()
    S, A = low.shape[1:]
    assert int(low.sum() + high.sum()) == sum(stored) + 2 * S * A
    traj = R.Trajectory(env, steps)
    R.rollout(env, agent.actor(training=False), R.HistoryDataBound(steps, 0), traj)
    acts = traj.to_host()["action"]
    mean0 = high[0, 0].astype(np.float64) / (high[0, 0] + low[0, 0]).astype(np.float64)
    assert (acts[0] == TO.last_argmax(list(mean0))).all()  # every lane starts in state 0
    agent.close()


def test_bts_rejections(ctx):
    cart = R.build_env(ctx, R.CartPoleConfig(), 8, seed=1)  # not a finite observation space
    with pytest.raises(ValueError):
        R.BetaThompsonSamplingAgentConfig().build_agent(cart)
    agent = R.BetaThompsonSamplingAgent(ctx, 1, 5, 2, (0.0, 10.0))
    traj = R.Trajectory(cart, 8)
    with pytest.raises(L.RelearnB200Error) as ex:
        R.rollout(cart, agent.actor(), R.HistoryDataBound(8, 0), traj)
    assert ex.value.status == L.RL_ERR_INVALID_ARG
    for n in (0, 1025):
        with pytest.raises(L.RelearnB200Error) as ex:
            R.BetaThompsonSamplingAgent(ctx, 1, 5, 2, (0.0, 10.0), num_samples=n)
        assert ex.value.status == L.RL_ERR_INVALID_ARG
    # a table shaped for Chain (5 x 2) on MemoryGame(3, 2), and a replica count that is neither 1 nor the lane count
    mem = R.build_env(ctx, R.MemoryGame(3, 2), 8, seed=1)
    chain = R.build_env(ctx, R.Chain(), 8, seed=1)
    for env, ag in ((mem, agent), (chain, R.BetaThompsonSamplingAgentConfig().build_agent(chain, num_replicas=3))):
        with pytest.raises(L.RelearnB200Error) as ex:
            R.rollout(env, ag.actor(), R.HistoryDataBound(8, 0), R.Trajectory(env, 8))
        assert ex.value.status == L.RL_ERR_INVALID_ARG
    # the inner agent: a meta env only, num_samples 1 .. 1024
    with pytest.raises(ValueError):
        R.ResettingMetaAgentConfig(R.BetaThompsonSamplingAgentConfig()).build_agent(chain)
    with pytest.raises(L.RelearnB200Error) as ex:
        R.rollout(chain, R.ActorSpec(kind=L.RL_ACTOR_RESETTING_META, inner_kind=L.RL_INNER_BETA_THOMPSON, num_samples=1),
                  R.HistoryDataBound(8, 0), R.Trajectory(chain, 8))
    assert ex.value.status == L.RL_ERR_UNSUPPORTED
    meta = R.build_env(ctx, META, 8, seed=1)
    for n in (0, 1025):
        with pytest.raises(ValueError):
            R.ResettingMetaAgentConfig(R.BetaThompsonSamplingAgentConfig(n)).build_agent(meta)
        with pytest.raises(L.RelearnB200Error) as ex:
            R.rollout(meta, R.ActorSpec(kind=L.RL_ACTOR_RESETTING_META, inner_kind=L.RL_INNER_BETA_THOMPSON, num_samples=n),
                      R.HistoryDataBound(8, 0), R.Trajectory(meta, 8))
        assert ex.value.status == L.RL_ERR_INVALID_ARG
