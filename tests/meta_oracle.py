"""CPU restatement of the resetting meta agent (ResettingMetaAgent, src/agents/meta.rs:146-198) for the tests.

The inner agents are the oracle's: tabular Q-learning through `ro_tabq_step_update` / `ro_argmax_f64`
(tabular.rs:159-232) and UCB1 through `oracle.Ucb1Oracle` (ucb.rs:78-243, glibc `log` as Rust's `f64::ln` on Linux).
The meta agent acts on the meta observation's features (meta.rs:152-163,357-363):
[inner_done, prev_step is None, one-hot prev action (k), prev reward, episode_done].

Two uses:
- `check_actions` walks a device trajectory and recomputes every stored action from the recorded observations and the
  lane's actor noise.  With the env side replayed by the oracle from the device's actions (`P.oracle_rollout` with
  `ACTOR_REPLAY`), that pins the whole trajectory.
- `rollout_lane` runs the agent online against the oracle's env, for behavioural checks of the oracle itself.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

import oracle as O

INNER_RANDOM, INNER_TABULAR_Q, INNER_UCB1 = 0, 1, 2


class MetaAgentOracle:
    """ResettingMetaAgent over one inner agent (meta.rs:102-198)."""

    def __init__(self, inner: int, num_arms: int, exploration_rate: float, reward_range=(0.0, 1.0)):
        self.inner, self.k, self.rate, self.reward_range = inner, num_arms, float(exploration_rate), reward_range
        self.initial_state()

    def initial_state(self):
        """meta.rs:146-157: the inner agent is built anew; no builder draws (tabular.rs:61-77, ucb.rs:49-74, random.rs).
        BaseTabularQLearningAgent::new starts from zeros whatever initial_action_count / initial_action_value say
        (tabular.rs:97-111)."""
        if self.inner == INNER_TABULAR_Q:
            self.q = np.zeros((1, self.k), np.float64)
            self.counts = np.zeros((1, self.k), np.uint64)
            self.table = O.TabQ(1, self.k, 1.0, O._ptr(self.q, C.c_double), O._ptr(self.counts, C.c_uint64))
        elif self.inner == INNER_UCB1:
            self.ucb = O.Ucb1Oracle(1, self.k, self.reward_range, self.rate)

    def ucb_bounds(self):
        return self.ucb.ucb(0)

    def act(self, obs, rng) -> int:
        """meta.rs:159-198 on the observation row `obs` (F = k + 4 features), drawing from `rng` (actor stream)."""
        lib, k = O.lib(), self.k
        inner_done, has_prev = obs[0] == 1.0, obs[1] == 0.0
        if has_prev:
            # the previous inner step: observation 0, the meta observation's action and feedback, successor Terminate
            # (one-step inner episodes); SerialActorAgent::update applies it at once (serial.rs:60-76)
            action, reward = int(np.argmax(obs[2:2 + k])), float(obs[2 + k])
            if self.inner == INNER_TABULAR_Q:
                lib.ro_tabq_step_update(C.byref(self.table), 0, action, reward, 0, 0)
            elif self.inner == INNER_UCB1:
                self.ucb.step_update(0, action, reward)
        if inner_done:  # reset the inner actor state (nothing to reset) and return some_element() = 0, no draw
            return 0
        if self.inner == INNER_TABULAR_Q:  # tabular.rs:222-232: the f64 draw is made even when epsilon is 0
            if lib.ro_gen_f64(rng.ref, O.STREAM_ACTOR) < self.rate:
                return int(lib.ro_gen_range(rng.ref, O.STREAM_ACTOR, k))
            return int(lib.ro_argmax_f64(O._ptr(self.q, C.c_double), k))
        if self.inner == INNER_UCB1:  # training mode (SerialActorAgent::new, serial.rs:49)
            return self.ucb.act(0, True)
        return int(lib.ro_gen_range(rng.ref, O.STREAM_ACTOR, k))  # random.rs:71-72


def actor_rng(lane: int, actor_words=None, philox_seed=None, lane_offset: int = 0, t0: int = 0):
    if philox_seed is not None:
        return O.PhiloxRng(philox_seed, lane_offset + lane, t0)
    return O.ScriptRng(actor_words[lane] if actor_words is not None else np.zeros(0, np.uint32))


def check_actions(host: dict, inner: int, num_arms: int, rate: float, *, actor_words=None, philox_seed=None,
                  lane_offset: int = 0, t0: int = 0, tie_rtol: float = 1e-13) -> int:
    """Recompute every stored action of `host` (Trajectory.to_host()) with MetaAgentOracle from the recorded observations.
    A trial ends at every step whose successor is not Continue; the agent is rebuilt there.  UCB1 only: where the device
    and the oracle disagree, the two largest upper bounds must agree to `tie_rtol` relative (device `log` against glibc
    `log`); the walk then follows the device.  Returns the number of such near-ties."""
    lib = O.lib()
    E = host["lane_len"].shape[0]
    near = 0
    for e in range(E):
        rng = actor_rng(e, actor_words, philox_seed, lane_offset, t0)
        agent = MetaAgentOracle(inner, num_arms, rate)
        for t in range(int(host["lane_len"][e])):
            if philox_seed is not None:
                lib.ro_rng_set_step(rng.ref, t0 + t)
            want = agent.act(host["obs"][t, e], rng)
            got = int(host["action"][t, e])
            if want != got:
                vals = sorted(agent.ucb_bounds()) if inner == INNER_UCB1 else None
                assert vals is not None and abs(vals[-1] - vals[-2]) <= tie_rtol * abs(vals[-1]), (e, t, want, got, vals)
                near += 1
            if host["succ"][t, e] != O.CONTINUE:
                agent.initial_state()
    return near


def rollout_lane(cfg: O.EnvCfg, inner: int, rate: float, steps: int, *, env_words=None, actor_words=None,
                 philox_seed=None, lane: int = 0, t0: int = 0) -> dict:
    """`steps` meta steps of one lane from a fresh trial (Steps::step, steps.rs:113-168): actions, rewards and successor
    codes, with the env restated by the oracle."""
    lib = O.lib()
    env = O.make_env(cfg)
    k = lib.ro_env_num_actions(C.byref(env))
    F = lib.ro_env_num_features(C.byref(env))
    if philox_seed is not None:
        rng_env = rng_act = O.PhiloxRng(philox_seed, lane, t0)
    else:
        rng_env = O.ScriptRng(env_words if env_words is not None else np.zeros(0, np.uint32))
        rng_act = O.ScriptRng(actor_words if actor_words is not None else np.zeros(0, np.uint32))
    agent = MetaAgentOracle(inner, k, rate)
    st, obs = O.State(), np.zeros(F, np.float32)
    action, reward, succ = (np.zeros(steps, np.uint8), np.zeros(steps, np.float32), np.zeros(steps, np.uint8))
    fresh = True
    for i in range(steps):
        if philox_seed is not None:
            lib.ro_rng_set_step(rng_env.ref, t0 + i)
        if fresh:
            lib.ro_env_initial_state(C.byref(env), C.byref(st), rng_env.ref)
            agent.initial_state()
            fresh = False
        obs[:] = 0.0
        lib.ro_env_observe(C.byref(env), C.byref(st), O._ptr(obs, C.c_float))
        a = agent.act(obs, rng_act)
        r = C.c_double()
        sc = lib.ro_env_step(C.byref(env), C.byref(st), a, rng_env.ref, C.byref(r))
        fresh = sc != O.CONTINUE
        action[i], reward[i], succ[i] = a, r.value, sc
    return {"action": action, "reward": reward, "succ": succ}


def trial_rewards(succ: np.ndarray, reward: np.ndarray) -> np.ndarray:
    """Rewards of the completed trials (episodes ending in a non-Continue successor) of one lane."""
    out, cur = [], 0.0
    for r, s in zip(reward, succ):
        cur += float(r)
        if s != O.CONTINUE:
            out.append(cur)
            cur = 0.0
    return np.array(out)
