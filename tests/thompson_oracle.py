"""CPU restatement of the Beta Thompson-sampling agent (src/agents/bandits/thompson_sampling.rs:84-212) for the tests.

The count tables, their (1, 1) start, the reward threshold, the fold and the evaluation argmax restate the reference.  The
Beta draw restates the device's own sampler (relearn_b200/csrc/beta.cuh, DESIGN section 5) operation for operation, in
Python floats (IEEE f64, every operation rounded on its own) with glibc `log` through `math.log`.  Uniforms are
rand's Standard f64 of a u64 actor-stream word (`ro_gen_f64`), so a `ScriptRng` or `PhiloxRng` of the oracle feeds the
same words the device's replayed or Philox noise does.

`check_meta_actions` recomputes the actions of the resetting meta agent (meta.rs:146-198) with this agent inside, the
way `tests/meta_oracle.check_actions` does for the other inner agents.
"""
from __future__ import annotations

import math

import numpy as np

import oracle as O
from tests import meta_oracle as MO


def uniform_of(rng):
    """U() over the actor stream of an oracle rng: (next_u64 >> 11) * 2^-53."""
    lib = O.lib()
    return lambda: lib.ro_gen_f64(rng.ref, O.STREAM_ACTOR)


def _log(x: float) -> float:
    return math.log(x) if x > 0.0 else -math.inf  # log(0) = -inf, as on the device


def normal_sample(U) -> float:
    """Marsaglia polar method; at most 64 tries, then 0."""
    for _ in range(64):
        u = 2.0 * U() - 1.0
        v = 2.0 * U() - 1.0
        s = u * u + v * v
        if 0.0 < s < 1.0:
            return u * math.sqrt(-2.0 * _log(s) / s)
    return 0.0


def gamma_sample(U, a: float) -> float:
    """Marsaglia-Tsang for a >= 1; a non-positive 1 + c z rejects before the uniform is drawn; at most 64 tries, then d."""
    d = a - 1.0 / 3.0
    c = 1.0 / math.sqrt(9.0 * d)
    for _ in range(64):
        z = normal_sample(U)
        b = 1.0 + c * z
        if not b > 0.0:
            continue
        v = b * b * b
        u = U()
        z2 = z * z
        if u < 1.0 - 0.0331 * (z2 * z2):
            return d * v
        if _log(u) < 0.5 * z2 + d - d * v + d * _log(v):
            return d * v
    return d


def beta_sample(U, alpha: float, beta: float) -> float:
    x = gamma_sample(U, alpha)
    y = gamma_sample(U, beta)
    return x / (x + y)


def beta_sample_sum(U, high: float, low: float, num_samples: int) -> float:
    """thompson_sampling.rs:195-202: the sequential sum from 0.0 of num_samples draws of Beta(alpha = high, beta = low)."""
    s = 0.0
    for _ in range(num_samples):
        s += beta_sample(U, high, low)
    return s


def last_argmax(vals) -> int:
    """argmax_by keeps the LAST maximal element (utils/iter/cmp.rs:58-76)."""
    best, bv = 0, vals[0]
    for k, v in enumerate(vals):
        if v >= bv:
            best, bv = k, v
    return best


class BetaThompsonOracle:
    """BaseBetaThompsonSamplingAgent + BaseBetaThompsonSamplingActor (thompson_sampling.rs:84-212)."""

    def __init__(self, num_observations: int, num_actions: int, reward_range, num_samples: int = 1):
        lo, hi = float(reward_range[0]), float(reward_range[1])
        self.threshold = (lo + hi) / 2.0  # :102-103
        self.num_samples = int(num_samples)
        self.low = np.ones((num_observations, num_actions), np.uint64)  # :104-105
        self.high = np.ones((num_observations, num_actions), np.uint64)

    def step_update(self, obs: int, action: int, reward: float):  # :126-136
        if float(reward) > self.threshold:
            self.high[obs, action] += np.uint64(1)
        else:
            self.low[obs, action] += np.uint64(1)

    def values(self, obs: int, training: bool, U=None):
        """Training (:195-202): one Beta sum per action, in action order; evaluation (:206-212): high / (high + low)."""
        if training:
            return [beta_sample_sum(U, float(h), float(lo), self.num_samples) for lo, h in zip(self.low[obs], self.high[obs])]
        return [float(h) / float(h + lo) for lo, h in zip(self.low[obs], self.high[obs])]

    def act(self, obs: int, training: bool = True, U=None) -> int:
        return last_argmax(self.values(obs, training, U))


def near_tie(vals, rtol: float) -> bool:
    top = sorted(vals)
    return abs(top[-1] - top[-2]) <= rtol * abs(top[-1])


def check_meta_actions(host: dict, num_arms: int, num_samples: int, reward_range=(0.0, 1.0), *, actor_words=None,
                       philox_seed=None, lane_offset: int = 0, t0: int = 0, tie_rtol: float = 1e-12) -> int:
    """Recompute every stored action of a resetting-meta trajectory whose inner agent is Thompson sampling.  Per meta step
    (meta.rs:159-198): fold the previous pull into the inner agent (observation 0), take action 0 without a draw at the end
    of an inner episode, otherwise act in training mode; a new agent at every trial end.  Where the device and the oracle
    disagree, the oracle's two largest sums must agree to `tie_rtol` relative (device `log` against glibc `log`); the walk
    follows the device.  Returns the number of such near-ties."""
    lib = O.lib()
    k = num_arms
    near = 0
    for e in range(host["lane_len"].shape[0]):
        rng = MO.actor_rng(e, actor_words, philox_seed, lane_offset, t0)
        U = uniform_of(rng)
        agent = BetaThompsonOracle(1, k, reward_range, num_samples)
        for t in range(int(host["lane_len"][e])):
            if philox_seed is not None:
                lib.ro_rng_set_step(rng.ref, t0 + t)
            obs = host["obs"][t, e]
            if obs[1] == 0.0:  # the previous inner step, successor Terminate (serial.rs:60-76)
                agent.step_update(0, int(np.argmax(obs[2:2 + k])), float(obs[2 + k]))
            vals = None
            if obs[0] == 1.0:  # inner episode done: some_element() = 0, no draw
                want = 0
            else:
                vals = agent.values(0, True, U)
                want = last_argmax(vals)
            got = int(host["action"][t, e])
            if want != got:
                assert vals is not None and near_tie(vals, tie_rtol), (e, t, want, got, vals)
                near += 1
            if host["succ"][t, e] != O.CONTINUE:
                agent = BetaThompsonOracle(1, k, reward_range, num_samples)
    return near
