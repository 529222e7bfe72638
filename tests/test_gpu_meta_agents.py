"""GPU parity of the resetting meta agent (ResettingMetaAgent, src/agents/meta.rs:16-227; the rl2-bandits baselines) on the
bandit meta-env: whole trajectories against the oracle in REPLAY and Philox modes, lane sharding, the reference's own
behavioural test (`ucb_one_hot_bandits`, meta.rs:237-264), the baselines' ordering, and the rejections."""
import numpy as np
import pytest

import oracle as O
import relearn_b200 as R
from relearn_b200 import _lib as L
from tests import meta_oracle as M
from tests import parity as P

pytestmark = pytest.mark.gpu

# (id, inner agent config, oracle inner kind, exploration rate)
INNERS = [
    ("random", R.RandomAgentConfig(), M.INNER_RANDOM, 0.0),
    ("eps-greedy", R.TabularQLearningAgentConfig(0.2), M.INNER_TABULAR_Q, 0.2),
    ("greedy", R.TabularQLearningAgentConfig(0.0), M.INNER_TABULAR_Q, 0.0),
    ("ucb1", R.UCB1AgentConfig(0.2), M.INNER_UCB1, 0.2),
]
ENVS = [
    R.MetaEnv(R.UniformBernoulliBandits(10), 7),
    R.MetaEnv(R.UniformBernoulliBandits(2), 3),
    R.MetaEnv(R.OneHotBandits(3), 4),
]
ENV_IDS = ["bernoulli10x7", "bernoulli2x3", "onehot3x4"]


def _trial_len(cfg):
    return 2 * cfg.episodes_per_trial - 1


def _lanes(d: dict, lanes) -> dict:
    out = {k: (v[:, lanes] if isinstance(v, np.ndarray) and v.ndim >= 2 else v) for k, v in d.items()}
    out["lane_len"] = d["lane_len"][lanes]
    return out


def _check(host, summ, cfg, E, min_steps, slack, inner, rate, what, **noise):
    """Actions: recomputed by the oracle agent from the recorded observations and the lane's actor noise (UCB1: at most two
    near-ties, device `log` against glibc `log`).  Everything else: the oracle's rollout of those actions, bit for bit, and
    its summary."""
    actor_words, env_words = noise.pop("actor_words", None), noise.pop("env_words", None)
    near = M.check_actions(host, inner, cfg.env_distribution.num_arms, rate, actor_words=actor_words, **noise)
    assert near <= 2, (what, near)
    ref = P.oracle_rollout(cfg, E, min_steps, slack, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(),
                           env_words=env_words, **noise)
    P.compare_traj(host, ref, what=what)
    P.compare_summary(summ, ref["summary"])
    assert summ.num_stored_steps == int(ref["lane_len"].sum())
    return ref


@pytest.mark.parametrize("cfg", ENVS, ids=ENV_IDS)
@pytest.mark.parametrize("name,inner_cfg,inner,rate", INNERS, ids=[i[0] for i in INNERS])
@pytest.mark.parametrize("slack_trials", [0, 1], ids=["slack0", "slack1"])
def test_meta_agent_replay_matches_oracle(ctx, cfg, name, inner_cfg, inner, rate, slack_trials):
    rng = np.random.default_rng(17)
    E = 48
    Lt = _trial_len(cfg)
    min_steps, slack = 3 * Lt + 2, slack_trials * Lt  # several whole trials and a cut one
    cap = min_steps + slack
    env = R.build_env(ctx, cfg, E, seed=3)
    env_words, actor_words = P.random_words(rng, E, 40 * cap), P.random_words(rng, E, 40 * cap)
    env.set_noise_replay(env_words, actor_words)
    agent = R.ResettingMetaAgentConfig(inner_cfg).build_agent(env)
    traj = R.Trajectory(env, cap)
    summ = R.rollout(env, agent.actor(), R.HistoryDataBound(min_steps, slack), traj)
    host = traj.to_host()
    ref = _check(host, summ, cfg, E, min_steps, slack, inner, rate, f"{name} replay", env_words=env_words,
                 actor_words=actor_words)
    assert (ref["n_taken"] > Lt).all()


@pytest.mark.parametrize("name,inner_cfg,inner,rate", INNERS, ids=[i[0] for i in INNERS])
def test_meta_agent_philox_matches_oracle_and_sharding(ctx, name, inner_cfg, inner, rate):
    cfg = ENVS[0]
    E, seed, off, t0 = 64, 0xBEEF, 1000, 5
    Lt = _trial_len(cfg)
    min_steps, slack = 4 * Lt + 3, 2
    cap = min_steps + slack
    env = R.build_env(ctx, cfg, E, seed=seed, lane_offset=off)
    env.set_noise_philox(seed, t0)
    agent = R.ResettingMetaAgentConfig(inner_cfg).build_agent(env)
    traj = R.Trajectory(env, cap)
    summ = R.rollout(env, agent.actor(), R.HistoryDataBound(min_steps, slack), traj)
    host = traj.to_host()
    _check(host, summ, cfg, E, min_steps, slack, inner, rate, f"{name} philox", philox_seed=seed, lane_offset=off, t0=t0)
    # two envs over lanes [0, E/2) and [E/2, E) reproduce the full env's trajectories
    h = E // 2
    for lo in (0, h):
        part = R.build_env(ctx, cfg, h, seed=seed, lane_offset=off + lo)
        part.set_noise_philox(seed, t0)
        tp = R.Trajectory(part, cap)
        R.rollout(part, R.ResettingMetaAgentConfig(inner_cfg).build_agent(part).actor(), R.HistoryDataBound(min_steps, slack), tp)
        hp = tp.to_host()
        lanes = list(range(lo, lo + h))
        P.compare_traj(hp, _lanes(host, lanes), what=f"{name} shard {lo}")


def test_ucb_one_hot_bandits_learns(ctx):
    """meta.rs:237-264 (`ucb_one_hot_bandits`): UCB1 lifted onto MetaEnv<OneHotBandits(3)> with 20 episodes per trial earns
    more than 0.7 x (20 - 3) per trial, on the device and on the oracle."""
    cfg = R.MetaEnv(R.OneHotBandits(3), 20)
    E, steps, seed = 256, 1000, 21
    Lt = _trial_len(cfg)
    env = R.build_env(ctx, cfg, E, seed=seed)
    env.set_noise_philox(seed, 0)
    traj = R.Trajectory(env, steps)
    summ = R.rollout(env, R.ResettingMetaAgentConfig(R.UCB1AgentConfig()).build_agent(env).actor(),
                     R.HistoryDataBound(steps, 0), traj)
    ocfg = P.oracle_cfg_for(cfg)
    lanes = [M.rollout_lane(ocfg, M.INNER_UCB1, 0.2, steps, philox_seed=seed, lane=e) for e in range(8)]
    ref = np.concatenate([M.trial_rewards(r["succ"], r["reward"]) for r in lanes])
    # the summary's episodes are the whole trials: the cut last trial of a lane continues and is not counted
    assert summ.episode_reward.count == E * (steps // Lt) and ref.size == 8 * (steps // Lt)
    print(f"mean trial reward: device {summ.episode_reward.mean:.3f}, oracle {ref.mean():.3f}")
    assert summ.episode_reward.mean > 0.7 * (20 - 3)
    assert ref.mean() > 0.7 * (20 - 3)


def test_bernoulli_baselines_order(ctx):
    """UniformBernoulliBandits(10), 100 pulls per trial: random earns 50 per trial on average (within 4 sigma); eps-greedy
    and UCB1 earn clearly more."""
    cfg = R.MetaEnv(R.UniformBernoulliBandits(10), 100)
    E, m = 2048, 2
    Lt = _trial_len(cfg)
    env = R.build_env(ctx, cfg, E, seed=7)
    traj = R.Trajectory(env, m * Lt)
    means = {}
    for name, c in [("random", R.RandomAgentConfig()), ("eps-greedy", R.TabularQLearningAgentConfig(0.2)),
                    ("ucb1", R.UCB1AgentConfig(0.2))]:
        env.set_noise_philox(99, 0)
        summ = R.rollout(env, R.ResettingMetaAgentConfig(c).build_agent(env).actor(), R.HistoryDataBound(m * Lt, 0), traj)
        er = summ.episode_reward
        assert er.count == E * m and summ.num_stored_episodes == E * m
        means[name] = (er.mean, np.sqrt(er.variance() / er.count))
    print(means)
    mu, se = means["random"]
    assert abs(mu - 50.0) < 4 * se
    for name in ("eps-greedy", "ucb1"):
        assert means[name][0] > mu + 10.0, (name, means)


def test_meta_agent_rejections(ctx):
    for cfg in (R.CartPoleConfig(), R.Chain()):
        env = R.build_env(ctx, cfg, 8, seed=1)
        traj = R.Trajectory(env, 16)
        with pytest.raises(L.RelearnB200Error) as ex:
            R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_RESETTING_META, inner_kind=L.RL_INNER_UCB1), R.HistoryDataBound(16, 0), traj)
        assert ex.value.status == L.RL_ERR_UNSUPPORTED
        with pytest.raises(ValueError):
            R.ResettingMetaAgentConfig().build_agent(env)
    env = R.build_env(ctx, ENVS[0], 8, seed=1)
    traj = R.Trajectory(env, 16)
    for spec in (R.ActorSpec(kind=L.RL_ACTOR_RESETTING_META, inner_kind=3),
                 R.ActorSpec(kind=L.RL_ACTOR_RESETTING_META, inner_kind=-1),
                 R.ActorSpec(kind=L.RL_ACTOR_RESETTING_META, inner_kind=L.RL_INNER_RANDOM, lanes_per_env=8)):
        with pytest.raises(L.RelearnB200Error) as ex:
            R.rollout(env, spec, R.HistoryDataBound(16, 0), traj)
        assert ex.value.status == L.RL_ERR_INVALID_ARG
    with pytest.raises(ValueError):
        R.ResettingMetaAgentConfig(object()).build_agent(env)
    agent = R.ResettingMetaAgentConfig(R.TabularQLearningAgentConfig()).build_agent(env)
    assert agent.min_update_size() == R.HistoryDataBound(0, 0)
    assert agent.batch_update(traj) is None
