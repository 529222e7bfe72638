"""Every feed-forward rollout kernel `rl_rollout` can pick, against the CPU oracle.

`rl_rollout` picks a kernel from the env, the module's shape and activation, `lanes_per_env`, the actor, the noise mode
and the env count (rollout.cu: K2a thread per env, K2g GL threads per env, K2b / K2c CartPole with L threads per env, K2t
tensor cores, K2q warp-specialised).  Each case below names the kernel its inputs select, runs one or two
collection periods and checks them against the oracle, never against a sibling kernel:

* replaying the kernel's own actions through the oracle reproduces the trajectory: lane lengths, successor codes (RL_PAD
  past each lane's end, the dangling-step Interrupt), rewards, observations (exact for the integer envs, 1e-6 for CartPole)
  and the Interrupt observations;
* the summary over every lane, and the stored step and episode counts, equal the oracle's;
* every action is the oracle's: the inverse-CDF choice of the softmax for the categorical actor, the exploration draw or
  the first argmax for the epsilon-greedy one, with the actor stream regenerated from the replayed words or from Philox.

`test_each_case_runs_the_kernel_it_names` reruns the table under the CUDA profiler so that a change of the selection
rules cannot move a case onto another kernel unnoticed.
"""
from __future__ import annotations

import json
import re
import zlib
from dataclasses import dataclass

import numpy as np
import pytest

import oracle as O
import relearn_b200 as R
from relearn_b200 import _lib as L
from tests import parity as P

pytestmark = pytest.mark.gpu

CAT, EPS = L.RL_ACTOR_CATEGORICAL_POLICY, L.RL_ACTOR_EPS_GREEDY_Q
TC, WS = L.RL_LANES_TENSOR_CORE, L.RL_LANES_WARP_SPECIALIZED
SHORT = R.CartPoleConfig().wrap(R.VisibleStepLimit(23))  # Interrupts, Terminates and resets within a period
WIDE_ANGLE = R.CartPoleConfig(max_angle=0.6).wrap(R.VisibleStepLimit(23))  # K2c serves only max_angle <= 0.5
LATENT = R.CartPoleConfig().wrap(R.LatentStepLimit(23))
BANDIT = R.MetaEnv(R.UniformBernoulliBandits(3), 4)
SAMPLED_LANES = 256  # per-step action checks on large env counts


@dataclass(frozen=True)
class Case:
    id: str
    kernel: str              # demangled name (without namespaces) of the one rollout kernel the inputs select
    cfg: object
    E: int
    hidden: tuple            # MlpConfig::hidden_sizes
    activation: str = "relu"
    actor: int = CAT
    eps: float = 0.0
    philox: bool = True
    lanes: int = 0
    T: int = 30
    slack: int = 10
    periods: int = 1
    scale: float = 2.0       # weight scale: sharper policies than the initialiser's
    ragged_warps: bool = False  # the envs sharing a warp must stop at different steps
    policy_atol: float = 2e-6

    @property
    def cartpole(self):
        return isinstance(self.cfg, R.CartPoleConfig)

    @property
    def params_id(self):
        return pytest.param(self, id=self.id)


def _env_name(cfg):
    return {R.CartPoleConfig: "CartPoleEnv", R.Chain: "ChainEnv", R.MemoryGame: "MemoryEnv", R.MetaEnv: "BanditMetaEnv",
            R.PartitionGame: "PartitionEnv"}[type(cfg)]


def _b(v):
    return "true" if v else "false"


def _actor_tag(actor, eps):
    return "cat" if actor == CAT else f"eps{eps:g}"


def _k2b(L_, cfg, hidden, act, actor, philox, E, eps=0.3):
    tag = f"K2b-L{L_}-{act}-{'lat' if cfg is LATENT else 'wide' if cfg is WIDE_ANGLE else 'vis'}-{_actor_tag(actor, eps)}-" \
          f"{'philox' if philox else 'replay'}-E{E}"
    return Case(tag, f"rollout_cartpole_coop_kernel<{L_}, {_b(not philox)}>", cfg, E, hidden, act, actor,
                eps if actor == EPS else 0.0, philox, L_)


def _build_cases():
    cases = []
    # K2b: a 128-unit module other than the default, L = 8 / 16 / 32 threads per env
    k2b_modules = [(SHORT, (128,), "tanh"), (WIDE_ANGLE, (128,), "relu"), (LATENT, (128,), "sigmoid")]
    for li, L_ in enumerate((8, 16, 32)):
        for mi, (cfg, hidden, act) in enumerate(k2b_modules):
            for ai, actor in enumerate((CAT, EPS)):
                for pi, philox in enumerate((False, True)):  # each (L, module) and each (actor, noise) meets both sizes
                    cases.append(_k2b(L_, cfg, hidden, act, actor, philox, 1000 if (li + mi + ai + pi) % 2 else 97))
    # K2g with eight threads per env (four envs per warp): 2368 <= E below the cost model's crossover, <= 3000 parameters
    k2g8 = [(SHORT, (128,), "tanh", True), (SHORT, (32, 16), "relu", True), (R.MemoryGame(4, 3), (24, 16, 8), "tanh", False)]
    for cfg, hidden, act, ragged in k2g8:
        for actor in (CAT, EPS):
            for philox in (False, True):
                name = f"K2g8-{_env_name(cfg)}-{'-'.join(map(str, hidden))}-{act}-{_actor_tag(actor, 0.3)}-" \
                       f"{'philox' if philox else 'replay'}"
                cases.append(Case(name, f"rollout_warp_kernel<{_env_name(cfg)}, {_b(not philox)}, 8>", cfg, 2999, hidden, act,
                                  actor, 0.3 if actor == EPS else 0.0, philox, 1, slack=25, periods=2 if philox else 1,
                                  ragged_warps=ragged))
    # K2g with a warp per env (few envs): Philox and the epsilon-greedy actor
    for cfg, hidden, act in ((R.PartitionGame(), (64,), "relu"), (BANDIT, (32,), "tanh")):
        for actor, philox in ((CAT, True), (EPS, False), (EPS, True)):
            name = f"K2g32-{_env_name(cfg)}-{_actor_tag(actor, 0.3)}-{'philox' if philox else 'replay'}"
            cases.append(Case(name, f"rollout_warp_kernel<{_env_name(cfg)}, {_b(not philox)}, 32>", cfg, 97, hidden, act, actor,
                              0.3 if actor == EPS else 0.0, philox, periods=2 if philox else 1))
    # K2a with a network: past the crossover, a module too wide for K2g, and an actor that never evaluates its network
    cases += [
        Case("K2a-pack8-CartPoleEnv-128-tanh", "rollout_kernel<CartPoleEnv, false>", SHORT, 30000, (128,), "tanh", CAT,
             philox=True, lanes=1, T=24, slack=6),
        Case("K2a-deep-CartPoleEnv-32-16-relu-eps", "rollout_kernel<CartPoleEnv, false>", SHORT, 30000, (32, 16), "relu", EPS,
             0.3, philox=True, lanes=1, T=24, slack=6),
        Case("K2a-generic-PartitionEnv-64", "rollout_kernel<PartitionEnv, false>", R.PartitionGame(), 40000, (64,), "relu",
             CAT, philox=True, T=24, slack=6),
        Case("K2a-MemoryEnv-16-16-1024", "rollout_kernel<MemoryEnv, true>", R.MemoryGame(16, 16), 197, (1024,), "relu", CAT,
             philox=False, T=40, slack=9, scale=1.0, policy_atol=1e-4),
        Case("K2a-ChainEnv-16-16-eps1", "rollout_kernel<ChainEnv, true>", R.Chain(), 5003, (16, 16), "tanh", EPS, 1.0,
             philox=False),
    ]
    # K2c on the default module with the epsilon-greedy actor (DqnActor on CartPole); lanes_per_env = 0 picks L = 8
    for L_ in (1, 2, 4, 8, 16, 32, 0):
        for eps in (0.0, 0.3):
            for philox in (False, True):
                name = f"K2c-L{L_}-eps{eps:g}-{'philox' if philox else 'replay'}"
                cases.append(Case(name, f"rollout_cartpole_group_kernel<{L_ or 8}, {_b(not philox)}, {EPS}>", SHORT, 97, (128,),
                                  "relu", EPS, eps, philox, L_))
    cases.append(Case("K2c-L8-eps0.3-philox-block128", f"rollout_cartpole_group_kernel<8, false, {EPS}>", SHORT, 10000, (128,),
                      "relu", EPS, 0.3, True, 8, T=24, slack=6))
    # K2c categorical on Philox: the shared actor word of a group
    for L_ in (2, 4, 16, 32):
        cases.append(Case(f"K2c-L{L_}-cat-philox", f"rollout_cartpole_group_kernel<{L_}, false, {CAT}>", SHORT, 97, (128,),
                          "relu", CAT, 0.0, True, L_, periods=2))
    # K2t: the batch variant (grid > 2 x SMs) with a ragged last tile, and the SPEC variant
    cases += [
        Case("K2t-batch-eps0.3-philox", f"rollout_cartpole_tc_kernel<false, {EPS}, false>", SHORT, 40001, (128,), "relu", EPS,
             0.3, True, 0, T=24, slack=6),
        Case("K2t-batch-cat-replay", f"rollout_cartpole_tc_kernel<true, {CAT}, false>", SHORT, 40001, (128,), "relu", CAT,
             0.0, False, 0, T=24, slack=6),
        Case("K2t-spec-eps0.3-philox", f"rollout_cartpole_tc_kernel<false, {EPS}, true>", SHORT, 10000, (128,), "relu", EPS,
             0.3, True, 0, T=24, slack=6),
    ]
    # the `remaining` feature: a table in shared memory up to a step limit of 2047 (its last entry), an f64 division beyond
    for limit in (2047, 2048):
        cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(limit))
        cases += [
            Case(f"limit{limit}-K2c8", f"rollout_cartpole_group_kernel<8, false, {CAT}>", cfg, 1000, (128,), "relu", CAT,
                 philox=True, lanes=8, T=40, slack=5),
            Case(f"limit{limit}-K2t", f"rollout_cartpole_tc_kernel<false, {CAT}, true>", cfg, 1000, (128,), "relu", CAT,
                 philox=True, lanes=TC, T=40, slack=5),
            Case(f"limit{limit}-K2q-E1000", "rollout_cartpole_ws6_kernel", cfg, 1000, (128,), "relu", CAT, philox=True,
                 lanes=WS, T=40, slack=5),
            Case(f"limit{limit}-K2q", "rollout_cartpole_ws6_kernel", cfg, 4096, (128,), "relu", CAT, philox=True, lanes=WS,
                 T=40, slack=5),
        ]
    return cases


CASES = _build_cases()
SEED, LANE_OFFSET, T0 = 0x5EED, 123, 7


def _hidden_arg(hidden):
    return hidden[0] if len(hidden) == 1 else list(hidden)


def _setup(ctx, case):
    """Env, network and replayed words of a case (the words are None under Philox noise)."""
    rng = np.random.default_rng(zlib.crc32(case.id.encode()))
    env = R.build_env(ctx, case.cfg, case.E, seed=SEED, lane_offset=LANE_OFFSET)
    F, A = env.num_features, env.num_actions
    params = R.init_params(rng, F, _hidden_arg(case.hidden), A) * np.float32(case.scale)
    net = R.Mlp(ctx, F, list(case.hidden), A, case.activation)
    net.set_weights(params)
    ewords = awords = None
    if case.philox:
        env.set_noise_philox(SEED, T0)
    else:
        W = 24 * (case.T + case.slack + 1) + 64
        ewords, awords = P.random_words(rng, case.E, W), P.random_words(rng, case.E, W)
        env.set_noise_replay(ewords, awords)
    return env, net, params, F, A, ewords, awords


def _spec(case, net):
    return R.ActorSpec(kind=case.actor, net=net, exploration_rate=case.eps, lanes_per_env=case.lanes)


def _check_lanes(E):
    """Every lane, or on large env counts a sample with the first and last lane and the ragged last 128-lane block."""
    if E <= 4096:
        return np.arange(E)
    tail = np.arange((E - 1) // 128 * 128, E)
    rest = np.random.default_rng(E).choice(E, SAMPLED_LANES, replace=False)
    return np.unique(np.concatenate([[0, E - 1], tail, rest]))


def _philox_actor_words(lanes, t0, n):
    lib = L.lib()
    return np.array([[lib.rl_philox_slot(SEED, LANE_OFFSET + int(e), t0 + i, 2, 0) & 0xFFFFFFFF for i in range(n)] for e in lanes],
                    dtype=np.uint64).astype(np.uint32)


def _check_period(case, host, summ, params, A, ewords, awords, t0):
    what = case.id
    E, T, slack = case.E, case.T, case.slack
    kw = dict(philox_seed=SEED, lane_offset=LANE_OFFSET, t0=t0) if case.philox else dict(env_words=ewords)
    ref = P.oracle_rollout(case.cfg, E, T, slack, actor_kind=O.ACTOR_REPLAY, actions=host["action"][: T + slack].copy(), **kw)
    tol = dict(obs_rtol=1e-6, obs_atol=1e-7) if case.cartpole else {}
    P.compare_traj(host, ref, what=what, **tol)
    P.compare_summary(summ, ref["summary"])
    stored = ref["succ"] != L.RL_PAD
    assert summ.num_stored_steps == int(ref["lane_len"].sum()) == int(stored.sum()), what
    assert summ.num_stored_episodes == int((stored & (ref["succ"] != L.RL_CONTINUE)).sum()), what
    if case.cartpole and case.cfg.max_steps_per_episode < T:  # episodes end and restart inside the period
        ends = stored & (ref["succ"] != L.RL_CONTINUE)
        ends[ref["lane_len"].astype(np.int64) - 1, np.arange(E)] = False
        assert ends.any(), what
    if case.ragged_warps:  # four envs share a warp: some warp holds envs that stopped at different steps
        groups = host["lane_len"][: E // 4 * 4].reshape(-1, 4)
        assert (groups.min(axis=1) != groups.max(axis=1)).any(), what

    lanes = _check_lanes(E)
    sub = {k: host[k][:, lanes] for k in ("obs", "action")}
    sub["lane_len"] = host["lane_len"][lanes]
    hidden = _hidden_arg(case.hidden)
    if case.actor == CAT:
        words = awords[lanes] if not case.philox else _philox_actor_words(lanes, t0, T + slack)
        checked, near = P.check_policy_consistency(sub, params, hidden, A, words, atol=case.policy_atol,
                                                   activation=case.activation)
        assert near <= 3, (what, near)
    else:
        if case.philox:
            # the checker walks lane j of `sub` as lane lane_offset + j: one call per sampled lane keeps the global id
            checked = near = 0
            for j, e in enumerate(lanes):
                one = {k: v[:, j : j + 1] for k, v in sub.items() if k != "lane_len"}
                one["lane_len"] = sub["lane_len"][j : j + 1]
                c, n = P.check_eps_greedy_consistency(one, params, hidden, A, case.eps, philox=(SEED, LANE_OFFSET + int(e), t0),
                                                      activation=case.activation)
                checked, near = checked + c, near + n
        else:
            checked, near = P.check_eps_greedy_consistency(sub, params, hidden, A, case.eps, actor_words=awords[lanes],
                                                           activation=case.activation)
        assert near <= 2, (what, near)
    assert checked == int(sub["lane_len"].sum()), what


def _run(ctx, case, check=True):
    env, net, params, F, A, ewords, awords = _setup(ctx, case)
    traj = R.Trajectory(env, case.T + case.slack)
    t0 = T0
    for _ in range(case.periods):
        summ = R.rollout(env, _spec(case, net), R.HistoryDataBound(case.T, case.slack), traj)
        if check:
            _check_period(case, traj.to_host(), summ, params, A, ewords, awords, t0)
        t0 += case.T + case.slack + 1  # the next period draws from the advanced Philox step counter
    traj.close()
    net.close()
    env.close()


@pytest.mark.parametrize("case", [c.params_id for c in CASES])
def test_rollout_kernel_against_the_oracle(ctx, case):
    _run(ctx, case)


def test_each_case_runs_the_kernel_it_names(ctx, tmp_path):
    """One profiled pass over the case table: the rollout kernels, in launch order, are exactly one per period of every
    case, with the function and template arguments the case names.  No recorded kernel at all fails."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.zeros(1, device="cuda")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for case in CASES:
            _run(ctx, case, check=False)
        ctx.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    kernels = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    assert kernels, "the profiler recorded no CUDA kernels"
    names = [e["name"].replace("(anonymous namespace)::", "") for e in kernels]
    rollout = [n for n in names if re.search(r"\brollout_(kernel|warp_kernel|cartpole_\w+_kernel|meta_kernel)\b", n)]
    expected = [c.kernel for c in CASES for _ in range(c.periods)]
    assert len(rollout) == len(expected), (len(rollout), len(expected))
    for case_kernel, got in zip(expected, rollout):
        assert re.search(r"\b" + re.escape(case_kernel) + r"(\(|$)", got), (case_kernel, got)


def test_module_too_large_for_shared_memory_is_refused(ctx):
    """MemoryGame(31, 1) admits a 32-1024-31 module (65 567 parameters, 262 KB): more than a block's shared memory, so the
    rollout is refused with RL_ERR_UNSUPPORTED.  The refusal leaves no error behind: a rollout on the same context right
    after it, with the widest module that fits (32-1024-16, ~201 KB), runs and matches the oracle."""
    env = R.build_env(ctx, R.MemoryGame(31, 1), 64, seed=1)
    assert (env.num_features, env.num_actions) == (32, 31)
    net = R.Mlp(ctx, 32, [1024], 31)
    net.set_weights(R.init_params(np.random.default_rng(0), 32, 1024, 31))
    traj = R.Trajectory(env, 8)
    with pytest.raises(L.RelearnB200Error) as err:
        R.rollout(env, R.ActorSpec(kind=CAT, net=net), R.HistoryDataBound(8, 0), traj)
    assert err.value.status == L.RL_ERR_UNSUPPORTED and "shared memory" in err.value.message, err.value
    traj.close()
    net.close()
    env.close()
    _run(ctx, next(c for c in CASES if c.id == "K2a-MemoryEnv-16-16-1024"))
