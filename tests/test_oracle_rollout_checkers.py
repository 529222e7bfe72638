"""The epsilon-greedy action checker (tests/parity.py: check_eps_greedy_consistency) on trajectories of the oracle's own
DqnActor (O.policy_actor(kind=O.ACTOR_EPS_GREEDY_Q)), on replayed and on Philox noise: it accepts them, and rejects one
altered exploring action, one altered greedy action and an exploration rate off by 0.05.  CPU only."""
import numpy as np
import pytest

import oracle as O
import relearn_b200 as R
from tests import parity as P

EPS = 0.3
SEED, LANE_OFFSET, T0 = 77, 40, 5
ENVS = [pytest.param(R.CartPoleConfig().wrap(R.VisibleStepLimit(23)), 5, id="cartpole"),
        pytest.param(R.MemoryGame(4, 3), 7, id="memory-4-3")]


def _oracle_trajectory(cfg, F, philox):
    """E lanes of the oracle's DqnActor (5-16-A ReLU) with slack; returns (host, params, A, checker noise keywords)."""
    rng = np.random.default_rng(3)
    A = O.lib().ro_env_num_actions(O.make_env(P.oracle_cfg_for(cfg)))
    params = R.init_params(rng, F, 16, A) * np.float32(3.0)
    E, T, slack = 8, 40, 6
    if philox:
        host = P.oracle_rollout(cfg, E, T, slack, actor_kind=O.ACTOR_EPS_GREEDY_Q, params=params, hidden=16, exploration_rate=EPS,
                                philox_seed=SEED, lane_offset=LANE_OFFSET, t0=T0)
        noise = dict(philox=(SEED, LANE_OFFSET, T0))
    else:
        W = 24 * (T + slack + 1) + 64
        ewords, awords = P.random_words(rng, E, W), P.random_words(rng, E, W)
        host = P.oracle_rollout(cfg, E, T, slack, actor_kind=O.ACTOR_EPS_GREEDY_Q, params=params, hidden=16, exploration_rate=EPS,
                                env_words=ewords, actor_words=awords)
        noise = dict(actor_words=awords)
    return host, params, A, noise


def _explores(noise, A, e, n):
    """Whether each of lane e's first n steps explores (the Bernoulli draw, and the uniform draw it is followed by)."""
    lib = O.lib()
    ph = noise.get("philox")
    rng = O.ScriptRng(noise["actor_words"][e]) if ph is None else O.PhiloxRng(ph[0], ph[1] + e, ph[2])
    out = []
    for i in range(n):
        if ph is not None:
            lib.ro_rng_set_step(rng.ref, ph[2] + i)
        x = bool(lib.ro_gen_bool(rng.ref, O.STREAM_ACTOR, EPS))
        if x:
            lib.ro_gen_range(rng.ref, O.STREAM_ACTOR, A)
        out.append(x)
    return np.array(out)


def _altered(host, i, e, A):
    bad = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in host.items()}
    bad["action"][i, e] = (bad["action"][i, e] + 1) % A
    return bad


@pytest.mark.parametrize("philox", [False, True], ids=["replay", "philox"])
@pytest.mark.parametrize("cfg,F", ENVS)
def test_eps_greedy_checker_accepts_the_oracle_and_rejects_changes(cfg, F, philox):
    host, params, A, noise = _oracle_trajectory(cfg, F, philox)
    checked, near = P.check_eps_greedy_consistency(host, params, 16, A, EPS, **noise)
    assert checked == int(host["lane_len"].sum()) and near == 0

    n = int(host["lane_len"][0])
    explores = _explores(noise, A, 0, n)
    assert explores.any() and not explores.all()
    for i in (int(np.flatnonzero(explores)[0]), int(np.flatnonzero(~explores)[0])):  # one exploring, one greedy step
        with pytest.raises(AssertionError):
            P.check_eps_greedy_consistency(_altered(host, i, 0, A), params, 16, A, EPS, **noise)
    with pytest.raises(AssertionError):
        P.check_eps_greedy_consistency(host, params, 16, A, EPS + 0.05, **noise)
