"""The tests' resetting meta agent oracle (tests/meta_oracle.py: ResettingMetaAgent, src/agents/meta.rs:146-198, acting on
the meta observation over the oracle's tabular Q and UCB1) against an independent restatement written here (plain Python
arithmetic on the env state), on replayed noise words, for the three inner agents; and its trajectory checker against the
oracle's own rollout of the same actions.  CPU only."""
import ctypes as C
import math

import numpy as np
import pytest

import oracle as O
from relearn_b200 import _lib as L
from tests import meta_oracle as M
from tests import parity as P


class PyMetaAgent:
    """meta.rs:146-198 with the inner agent built fresh (tabular.rs:61-111, ucb.rs:49-128, random.rs)."""

    def __init__(self, inner, k, rate):
        self.inner, self.k, self.rate = inner, k, rate

    def initial_state(self):
        if self.inner == M.INNER_UCB1:
            self.v, self.c, self.visits = [0.5] * self.k, [2] * self.k, 2 * self.k
        else:
            self.v, self.c, self.visits = [0.0] * self.k, [0] * self.k, 0

    def update(self, action, reward):
        if self.inner == M.INNER_TABULAR_Q:  # tabular.rs:159-179, successor Terminate
            self.c[action] += 1
            w = 1.0 / float(self.c[action])
            q = self.v[action] * (1.0 - w)
            self.v[action] = q + w * (reward + 0.0)
        elif self.inner == M.INNER_UCB1:  # ucb.rs:143-160, reward range (0, 1)
            scaled = (reward + -0.0) * (1.0 / 1.0)
            self.visits += 1
            self.c[action] += 1
            m = self.v[action]
            self.v[action] = m + (scaled - m) / float(self.c[action])

    def act(self, st, rng):
        if st.has_prev:
            self.update(int(st.prev_action), float(st.prev_reward))
        if st.inner_done:
            return 0
        lib = O.lib()
        if self.inner == M.INNER_RANDOM:
            return int(lib.ro_gen_range(rng.ref, O.STREAM_ACTOR, self.k))
        if self.inner == M.INNER_TABULAR_Q:
            if lib.ro_gen_f64(rng.ref, O.STREAM_ACTOR) < self.rate:
                return int(lib.ro_gen_range(rng.ref, O.STREAM_ACTOR, self.k))
            return int(np.argmax(self.v))  # first maximum
        lsv = 2.0 * math.log(float(self.visits))
        best, bv = 0, 0.0
        for i in range(self.k):
            u = math.sqrt(lsv / float(self.c[i])) * self.rate + self.v[i]
            if i == 0 or u >= bv:
                best, bv = i, u
        return best


def _python_lane(cfg, inner, rate, steps, env_words, actor_words):
    lib = O.lib()
    env = O.make_env(cfg)
    k = lib.ro_env_num_actions(C.byref(env))
    rng_env, rng_actor = O.ScriptRng(env_words), O.ScriptRng(actor_words)
    agent = PyMetaAgent(inner, k, rate)
    st = O.State()
    fresh = True
    actions, rewards, succs = [], [], []
    for _ in range(steps):
        if fresh:
            lib.ro_env_initial_state(C.byref(env), C.byref(st), rng_env.ref)
            agent.initial_state()
            fresh = False
        a = agent.act(st, rng_actor)
        r = C.c_double()
        sc = lib.ro_env_step(C.byref(env), C.byref(st), a, rng_env.ref, C.byref(r))
        fresh = sc != O.CONTINUE
        actions.append(a)
        rewards.append(np.float32(r.value))
        succs.append(sc)
    return np.array(actions, np.uint8), np.array(rewards, np.float32), np.array(succs, np.uint8)


@pytest.mark.parametrize("inner,rate", [(M.INNER_RANDOM, 0.0), (M.INNER_TABULAR_Q, 0.2), (M.INNER_TABULAR_Q, 0.0),
                                        (M.INNER_UCB1, 0.2)], ids=["random", "eps-greedy", "greedy", "ucb1"])
@pytest.mark.parametrize("arms,trial,dist", [(10, 7, O.BANDIT_UNIFORM_BERNOULLI), (3, 4, O.BANDIT_ONE_HOT)],
                         ids=["bernoulli10x7", "onehot3x4"])
def test_oracle_resetting_meta_matches_python_restatement(inner, rate, arms, trial, dist):
    rng = np.random.default_rng(11)
    cfg = O.bandit_meta_cfg(arms, trial, dist)
    steps = 5 * (2 * trial - 1) + 3  # several whole trials and a cut one
    for lane in range(6):
        ew = rng.integers(0, 2**32, size=16 * steps, dtype=np.uint64).astype(np.uint32)
        aw = rng.integers(0, 2**32, size=16 * steps, dtype=np.uint64).astype(np.uint32)
        res = M.rollout_lane(cfg, inner, rate, steps, env_words=ew, actor_words=aw)
        acts, rews, succ = _python_lane(cfg, inner, rate, steps, ew, aw)
        np.testing.assert_array_equal(res["action"], acts, err_msg=f"lane {lane}: actions")
        np.testing.assert_array_equal(res["reward"], rews, err_msg=f"lane {lane}: rewards")
        np.testing.assert_array_equal(res["succ"], succ, err_msg=f"lane {lane}: successors")
        # a trial is 2n - 1 meta steps: pull, reset, ..., pull (Interrupt)
        assert (np.flatnonzero(succ == L.RL_INTERRUPT) + 1 == np.arange(1, steps // (2 * trial - 1) + 1) * (2 * trial - 1)).all()


@pytest.mark.parametrize("inner,rate", [(M.INNER_RANDOM, 0.0), (M.INNER_TABULAR_Q, 0.2), (M.INNER_UCB1, 0.2)],
                         ids=["random", "eps-greedy", "ucb1"])
def test_check_actions_accepts_the_oracle_trajectory_and_rejects_a_change(inner, rate):
    """check_actions recomputes the actions of an oracle rollout (P.oracle_rollout with the online agent's actions) from
    its observations, and fails on a trajectory whose pulls were changed."""
    from relearn_b200 import envs as Renvs

    rng = np.random.default_rng(4)
    cfg = Renvs.MetaEnv(Renvs.UniformBernoulliBandits(5), 6)
    E, Lt = 8, 11
    steps = 3 * Lt + 4
    ew = rng.integers(0, 2**32, size=(E, 16 * steps), dtype=np.uint64).astype(np.uint32)
    aw = rng.integers(0, 2**32, size=(E, 16 * steps), dtype=np.uint64).astype(np.uint32)
    actions = np.stack([M.rollout_lane(P.oracle_cfg_for(cfg), inner, rate, steps, env_words=ew[e], actor_words=aw[e])["action"]
                        for e in range(E)], axis=1)
    host = P.oracle_rollout(cfg, E, steps, 0, actor_kind=O.ACTOR_REPLAY, actions=actions, env_words=ew)
    assert M.check_actions(host, inner, 5, rate, actor_words=aw) == 0
    bad = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in host.items()}
    pulls = np.flatnonzero(bad["obs"][:, 0, 0] == 0.0)  # every pull of lane 0 (UCB1 accepts a change at an exact tie)
    bad["action"][pulls, 0] = (bad["action"][pulls, 0] + 1) % 5
    with pytest.raises(AssertionError):
        M.check_actions(bad, inner, 5, rate, actor_words=aw)
