"""CPU checks of the Thompson-sampling test oracle (tests/thompson_oracle.py): its Beta sampler has the Beta distribution,
ends on exhausted replay words, and its agent's threshold, fold and evaluation choice agree with a plain restatement of
thompson_sampling.rs."""
import math

import numpy as np
import pytest
from scipy import stats

import oracle as O
from tests import thompson_oracle as TO


@pytest.mark.parametrize("alpha,beta", [(1, 1), (1, 7), (30, 2), (500, 700)])
def test_beta_sampler_has_the_beta_distribution(alpha, beta):
    words = np.random.default_rng(alpha * 1000 + beta).integers(0, 2**32, size=2_000_000, dtype=np.uint64).astype(np.uint32)
    rng = O.ScriptRng(words)
    U = TO.uniform_of(rng)
    draws = np.array([TO.beta_sample(U, float(alpha), float(beta)) for _ in range(20_000)])
    p = stats.kstest(draws, stats.beta(alpha, beta).cdf).pvalue
    assert p > 1e-3, p


def test_gamma_sampler_mean_and_variance():
    """Gamma(a) has mean a and variance a; 20 000 draws at a = 3 within 5 standard errors."""
    rng = O.ScriptRng(np.random.default_rng(5).integers(0, 2**32, size=1_000_000, dtype=np.uint64).astype(np.uint32))
    U = TO.uniform_of(rng)
    x = np.array([TO.gamma_sample(U, 3.0) for _ in range(20_000)])
    assert abs(x.mean() - 3.0) < 5 * math.sqrt(3.0 / x.size)
    assert abs(x.var() - 3.0) < 5 * math.sqrt((2 * 9.0 + 6 * 3.0) / x.size)  # Var of the sample variance: (2 a^2 + 6 a) / n


def test_exhausted_words_still_return():
    U = TO.uniform_of(O.ScriptRng(np.zeros(0, np.uint32)))
    assert TO.normal_sample(U) == 0.0  # u = v = -1: s = 2 rejects every try
    x = TO.beta_sample(U, 3.0, 5.0)    # Gamma falls through to z = 0, v = 1, u = 0 < 1: the result is d
    d3, d5 = 3.0 - 1.0 / 3.0, 5.0 - 1.0 / 3.0
    assert x == d3 / (d3 + d5)
    assert TO.beta_sample_sum(U, 1.0, 1.0, 10) == 5.0


def test_agent_matches_a_plain_restatement():
    rng = np.random.default_rng(11)
    S, A = 3, 4
    for lo, hi in [(0.0, 10.0), (-1.0, 1.0), (0.0, 1.0)]:
        o = TO.BetaThompsonOracle(S, A, (lo, hi), num_samples=2)
        assert o.threshold == (lo + hi) / 2.0
        assert (o.low == 1).all() and (o.high == 1).all()
        counts = {(s, a): [1, 1] for s in range(S) for a in range(A)}  # (low, high)
        thr = (lo + hi) / 2.0
        rewards = np.concatenate([rng.uniform(lo, hi, 300), np.full(20, thr), np.full(10, lo), np.full(10, hi)])
        for r in rewards:
            s, a = int(rng.integers(S)), int(rng.integers(A))
            o.step_update(s, a, float(r))
            counts[(s, a)][1 if r > thr else 0] += 1  # strictly above the threshold counts as high
        for (s, a), (low, high) in counts.items():
            assert (int(o.low[s, a]), int(o.high[s, a])) == (low, high)
        for s in range(S):
            means = [counts[(s, a)][1] / (counts[(s, a)][0] + counts[(s, a)][1]) for a in range(A)]
            want = max(a for a in range(A) if means[a] == max(means))
            assert o.act(s, training=False) == want
    # exact ties between the first and the last action go to the last
    o = TO.BetaThompsonOracle(1, 3, (0.0, 1.0))
    o.low[0] = [3, 9, 3]
    o.high[0] = [5, 1, 5]
    assert o.act(0, training=False) == 2
    # training: the action of the largest sum, draws in action order
    words = rng.integers(0, 2**32, size=4096, dtype=np.uint64).astype(np.uint32)
    o.num_samples = 3
    U1, U2 = TO.uniform_of(O.ScriptRng(words)), TO.uniform_of(O.ScriptRng(words))
    sums = [TO.beta_sample_sum(U1, float(h), float(lw), 3) for lw, h in zip(o.low[0], o.high[0])]
    assert o.act(0, training=True, U=U2) == TO.last_argmax(sums)
