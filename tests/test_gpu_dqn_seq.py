"""GPU parity: DQN with a recurrent action-value module (Chain<Gru, Linear>; DqnAgent over SeqPacked + SeqIterative
modules, dqn.rs:75-83,190-197,341-379) -- the epsilon-greedy actor inside the recurrent rollouts, the sequence minibatch
sampler, the Q-loss pass with back-propagation through time and the whole update -- against the oracle.

Tolerances: the env side and every explored action are bit-exact; greedy actions are the first argmax of the f64
restatement except at near-ties of the Q-values (1e-5 relative, 1e-4 for the hidden-128 tile kernel, whose gates use the
SFU approximations); sampled episodes, codes and reward-to-go targets are bit-exact; losses and gradients are compared
with f64 autograd as in test_gpu_gru_update.py."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from oracle import tensor_oracle as TO
import relearn_b200 as R
from relearn_b200 import _lib as L
from tests import parity as P
from tests.test_gpu_dqn import _fill, _oracle_minibatch

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

CONT, TERM, INTR, PAD = L.RL_CONTINUE, L.RL_TERMINATE, L.RL_INTERRUPT, L.RL_PAD
ACT = {"relu": torch.relu, "tanh": torch.tanh, "identity": lambda t: t, "sigmoid": torch.sigmoid}


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) /
                 max(np.linalg.norm(np.asarray(b, np.float64)), 1e-300))


def _q_params(rng, F, hidden, A, bias_scale=0.3, head_scale=1.0, input_scale=1.0, head_bias=True):
    p = R.init_gru_linear_params(rng, F, hidden, A).astype(np.float32)
    p[:3 * hidden * F] *= input_scale
    o = 3 * hidden * F + 3 * hidden * hidden
    p[o:o + 6 * hidden] = rng.normal(size=6 * hidden) * bias_scale
    p[-A * hidden - A:] *= head_scale
    if not head_bias:
        p[-A:] = 0.0
    return p


# ------------------------------------------------------------------------------------------------
# Rollout: DqnActor::act (dqn.rs:360-379) restated
# ------------------------------------------------------------------------------------------------
def _actor_draws(host, A, eps, actor_words=None, philox=None):
    """Walk each lane's actor stream as DqnActor::act does: gen_bool(eps), then gen_range(A) on an explored step.
    Returns explore flags and explored actions [T, E] (the stream does not depend on the Q-values)."""
    lib = O.lib()
    T, E = host["action"].shape
    explore = np.zeros((T, E), bool)
    drawn = np.zeros((T, E), np.int64)
    for e in range(E):
        rng = O.ScriptRng(actor_words[e]) if philox is None else O.PhiloxRng(philox[0], philox[1] + e, philox[2])
        for i in range(int(host["lane_len"][e])):
            if philox is not None:
                lib.ro_rng_set_step(rng.ref, philox[2] + i)
            if lib.ro_gen_bool(rng.ref, O.STREAM_ACTOR, eps):
                explore[i, e] = True
                drawn[i, e] = int(lib.ro_gen_range(rng.ref, O.STREAM_ACTOR, A))
    return explore, drawn


def _restate_actions(host, params, F, H, A, explore, drawn, *, advance_always=False, tie_rtol=1e-5, activation="relu"):
    """Every stored action against the restatement: explored steps take the drawn action; greedy steps the first argmax of
    Q = Linear(act(gru_cell(x, h))) in f64.  The hidden state starts at zero in every episode and -- the reference's
    order -- is NOT advanced on an explored step (advance_always=True restates the other order).  Returns
    (greedy steps, mismatches beyond a near-tie, near-ties)."""
    T, E = host["action"].shape
    w_ih, w_hh, b_ih, b_hh, lw, lb = [t.to(torch.float64) for t in TO.unflatten_gru_linear(torch.tensor(params), F, H, A)]
    h = torch.zeros(E, H, dtype=torch.float64)
    lens = host["lane_len"].astype(np.int64)
    greedy = mism = near = 0
    for t in range(int(lens.max(initial=0))):
        valid = t < lens
        x = torch.tensor(host["obs"][t], dtype=torch.float64)
        hn = torch.gru_cell(x, h, w_ih, w_hh, b_ih, b_hh)
        z = torch.nn.functional.linear(ACT[activation](hn), lw, lb).numpy()
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
        h = torch.where(keep, h, hn)
        done = torch.tensor(host["succ"][t] != CONT)[:, None]
        h = torch.where(done, torch.zeros_like(h), h)
    return greedy, mism, near


def _rollout_case(ctx, cfg, hidden, eps, E, T, seed, head_scale=1.0):
    """One replayed-noise rollout with the epsilon-greedy GRU actor; the env side is checked against the oracle replaying
    the device's actions.  The module's inputs are scaled up and its head bias is zero so that Q depends on the history."""
    rng = np.random.default_rng(seed)
    env = R.build_env(ctx, cfg, E, seed=seed)
    nwords = 16 * T + 64 * env.num_actions
    ewords, awords = P.random_words(rng, E, nwords), P.random_words(rng, E, nwords)
    env.set_noise_replay(ewords, awords)
    F, A = env.num_features, env.num_actions
    params = _q_params(rng, F, hidden, A, head_scale=head_scale, input_scale=3.0, head_bias=False)
    net = R.GruLinear(ctx, F, hidden, A)
    net.set_weights(params)
    traj = R.Trajectory(env, T)
    actor = R.ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, seq_net=net, exploration_rate=eps)
    summ = R.rollout(env, actor, R.HistoryDataBound(T - 2, 2), traj)
    host = traj.to_host()
    ref = P.oracle_rollout(cfg, E, T - 2, 2, actor_kind=O.ACTOR_REPLAY, actions=host["action"].copy(), env_words=ewords)
    P.compare_traj(host, ref, what=f"eps-greedy GRU {hidden}")
    P.compare_summary(summ, ref["summary"])
    explore, drawn = _actor_draws(host, A, eps, actor_words=awords)
    return host, params, F, A, explore, drawn


ROLLOUT_CASES = [(kind, h, eps) for kind in ("memory", "bandit") for h in (4, 8) for eps in (0.0, 0.3, 1.0)]


def _check_quirk_exercised(run, attempts=6):
    """`run(attempt)` checks one rollout against the restatement and returns the greedy mismatches of the restatement that
    advances the hidden state on every step.  Whether those show depends on how much the module's greedy choice depends on
    its history, so further seeds are tried (each checked in full) until one shows them."""
    for attempt in range(attempts):
        mism_always = run(attempt)
        print(f"  attempt {attempt}: restatement advancing on every step: {mism_always} greedy mismatches")
        if mism_always > 0:
            return
    raise AssertionError("no case exercised the hidden state held on explored steps")


@pytest.mark.parametrize("kind,hidden,eps", ROLLOUT_CASES)
def test_eps_greedy_gru_rollout_small(ctx, kind, hidden, eps):
    """K8a (thread per env; bandit 2 arms at hidden 4 = the specialised 6-4-2 instance) with replayed noise."""
    cfg = R.MemoryGame(4, 3) if kind == "memory" else R.MetaEnv(R.UniformBernoulliBandits(2), 10)
    T = 40

    def run(attempt):
        host, params, F, A, explore, drawn = _rollout_case(ctx, cfg, hidden, eps, 96, T, seed=hidden + int(10 * eps) + 101 * attempt,
                                                           head_scale=3.0)
        greedy, mism, near = _restate_actions(host, params, F, hidden, A, explore, drawn)
        print(f"{kind} h={hidden} eps={eps}: greedy {greedy}, explored {int(explore.sum())}, near-ties {near}")
        assert mism == 0 and near <= 2
        if eps == 1.0:
            assert greedy == 0
        if eps == 0.0:
            assert not explore.any()
        if eps != 0.3:
            return 1
        assert greedy > 0 and explore.any()
        return _restate_actions(host, params, F, hidden, A, explore, drawn, advance_always=True)[1]

    _check_quirk_exercised(run)


@pytest.mark.parametrize("kernel", ["thread", "tile", "tile32", "stepped", None])
@pytest.mark.parametrize("eps", [0.0, 0.3, 1.0])
def test_eps_greedy_gru128_rollout(ctx, monkeypatch, kernel, eps):
    """Hidden 128 on the bandit meta-env (10 arms) through each kernel RL_GRU_KERNEL can pick: K8a (thread), K8h at 64 and
    32 envs per CTA; 'stepped' and the default route the epsilon-greedy actor to K8h.  K8h computes the new state of every
    env before the actor draws and restores it on explored steps."""
    if kernel is None:
        monkeypatch.delenv("RL_GRU_KERNEL", raising=False)
    else:
        monkeypatch.setenv("RL_GRU_KERNEL", kernel)
    cfg = R.MetaEnv(R.UniformBernoulliBandits(10), 3)
    tol = 1e-5 if kernel == "thread" else 1e-4

    def run(attempt):
        host, params, F, A, explore, drawn = _rollout_case(ctx, cfg, 128, eps, 150, 17, seed=5 + int(10 * eps) + 101 * attempt,
                                                           head_scale=4.0)
        greedy, mism, near = _restate_actions(host, params, F, 128, A, explore, drawn, tie_rtol=tol)
        print(f"kernel {kernel} eps={eps}: greedy {greedy}, near-ties {near}")
        assert mism == 0 and near <= 3
        if eps != 0.3:
            return 1
        return _restate_actions(host, params, F, 128, A, explore, drawn, advance_always=True, tie_rtol=tol)[1]

    _check_quirk_exercised(run)


@pytest.mark.parametrize("cfg", [R.MemoryGame(3, 4), R.CartPoleConfig().wrap(R.VisibleStepLimit(30))], ids=["memory", "cartpole"])
def test_eps_greedy_gru_rollout_philox_sharding(ctx, cfg):
    """Production noise: two shards of lanes (lane_offset) reproduce the full env's trajectory, and the actions follow the
    Philox actor stream of the restatement."""
    rng = np.random.default_rng(3)
    env0 = R.build_env(ctx, cfg, 8, seed=1)
    F, A = env0.num_features, env0.num_actions
    params = _q_params(rng, F, 8, A, head_scale=3.0)
    T, eps, seed = 60, 0.3, 11

    def run(n, off):
        env = R.build_env(ctx, cfg, n, seed=seed, lane_offset=off)
        env.set_noise_philox(seed, 0)
        net = R.GruLinear(ctx, F, 8, A)
        net.set_weights(params)
        traj = R.Trajectory(env, T)
        R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, seq_net=net, exploration_rate=eps), R.HistoryDataBound(T, 0), traj)
        return traj.to_host()

    full, a, b = run(64, 0), run(32, 0), run(32, 32)
    for k in ("obs", "action", "reward", "succ"):
        np.testing.assert_array_equal(full[k][:, :32], a[k])
        np.testing.assert_array_equal(full[k][:, 32:], b[k])
    explore, drawn = _actor_draws(full, A, eps, philox=(seed, 0, 0))
    greedy, mism, near = _restate_actions(full, params, F, 8, A, explore, drawn)
    assert greedy > 0 and mism == 0 and near <= 2


# ------------------------------------------------------------------------------------------------
# Sampler: the episodes of the flat minibatch as sequences
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def filled(ctx):
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(15))
    E = 48
    env, rb, _ = _fill(ctx, cfg, 15, E, 120, R.HistoryDataBound(30, 6), periods=6, seed=33)
    lanes = [rb.read_lane(e) for e in range(E)]
    return env, rb, lanes


def _rtg(ep, g):
    n = len(ep["reward"])
    return O.discounted_cumsum_lane(ep["reward"], np.array([CONT] * (n - 1) + [TERM], np.uint8), np.float32(g))


@pytest.mark.parametrize("draw_index,minibatch", [(0, 200), (5, 1), (9, 1500)])
def test_sample_seq_holds_the_flat_minibatch_episodes(ctx, filled, draw_index, minibatch):
    env, rb, lanes = filled
    seed, g = 77, 0.99
    cfg = L.DqnCfg(minibatch, 1, 0, np.float32(g), seed)
    got = rb.sample_seq(cfg, None, draw_index)
    eps = _oracle_minibatch(lanes, seed, draw_index, minibatch)
    B = len(eps)
    lens = np.array([len(e["action"]) for e in eps])
    assert got["num_episodes"] == B and got["num_steps"] == lens.sum() and got["max_len"] == lens.max()
    np.testing.assert_array_equal(got["lane_len"], lens)
    flat = rb.sample(cfg, None, draw_index)
    assert flat["num_steps"] == got["num_steps"] and flat["num_episodes"] == B
    for b, ep in enumerate(eps):
        n = lens[b]
        np.testing.assert_array_equal(got["obs"][:n, b], ep["obs"])
        np.testing.assert_array_equal(got["action"][:n, b], ep["action"])
        np.testing.assert_array_equal(got["reward"][:n, b], ep["reward"])
        np.testing.assert_array_equal(got["succ"][:n, b], [CONT] * (n - 1) + [ep["last_succ"]])
        assert (got["succ"][n:, b] == PAD).all()
        np.testing.assert_array_equal(got["target"][:n, b], _rtg(ep, g))
        if ep["last_succ"] == INTR:
            np.testing.assert_array_equal(got["next_obs"][n - 1, b], ep["next_obs"])
    # the per-step targets are those of the flat minibatch, bit for bit
    seq_t = np.concatenate([got["target"][:lens[b], b] for b in range(B)])
    np.testing.assert_array_equal(seq_t, flat["target"])


def _ext_q(params, F, H, A, eps, activation="relu", dtype=torch.float64):
    """Q on each episode and, for an interrupted one, on its successor observation as one more step of the sequence."""
    prm = [t.to(dtype) for t in TO.unflatten_gru_linear(torch.tensor(params), F, H, A)]
    ext = [np.concatenate([e["obs"], e["next_obs"][None]]) if e["last_succ"] == INTR else e["obs"] for e in eps]
    out = TO.gru_linear_forward(prm, TO.EpisodeBatch(ext, dtype), activation).detach().numpy()
    res, pos = [], 0
    for x in ext:
        res.append(out[pos:pos + len(x)])
        pos += len(x)
    return res


def _td_targets(params, F, H, A, eps, g, dtype=torch.float64):
    qs = _ext_q(params, F, H, A, eps, dtype=dtype)
    out = []
    for ep, q in zip(eps, qs):
        n = len(ep["reward"])
        m = q.max(axis=1)
        nxt = np.zeros(n)
        nxt[:-1] = m[1:n]
        if ep["last_succ"] == INTR:
            nxt[-1] = m[n]
        out.append(ep["reward"].astype(np.float64) + float(np.float32(g)) * nxt)
    return out


@pytest.mark.parametrize("hidden", [8, 32])
def test_sample_seq_one_step_td_targets(ctx, filled, hidden):
    """r + gamma * max_a Q(next) from a SeqPacked forward: the next step's Q on Continue, one more step of the same
    sequence on the successor observation after Interrupt, 0 after Terminate.  Tolerance as the flat OneStepTd test."""
    env, rb, lanes = filled
    F, A = 5, 2
    params = _q_params(np.random.default_rng(hidden), F, hidden, A)
    q = R.GruLinear(ctx, F, hidden, A)
    q.set_weights(params)
    seed, di, minibatch, g = 5, 2, 400, 0.99
    got = rb.sample_seq(L.DqnCfg(minibatch, 1, 1, np.float32(g), seed), q, di)
    eps = _oracle_minibatch(lanes, seed, di, minibatch)
    want = _td_targets(params, F, hidden, A, eps, g)
    assert sum(e["last_succ"] == INTR for e in eps) > 0, "the case must include interrupted episodes"
    for b, (ep, w) in enumerate(zip(eps, want)):
        np.testing.assert_allclose(got["target"][:len(w), b], w, rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# Passes and the whole update
# ------------------------------------------------------------------------------------------------
def _seq_q_loss_grad(params, F, H, A, eps, targets, dtype=torch.float64, activation="relu"):
    prm = TO._seq_params(params, F, H, A, dtype)
    q = TO.gru_linear_forward(prm, TO.EpisodeBatch([e["obs"] for e in eps], dtype), activation)
    act = torch.tensor(np.concatenate([e["action"] for e in eps]), dtype=torch.int64).unsqueeze(-1)
    tgt = torch.tensor(np.concatenate(targets), dtype=dtype)
    loss = torch.nn.functional.mse_loss(q.gather(-1, act).squeeze(-1), tgt, reduction="mean")
    grads = torch.autograd.grad(loss, prm)
    return float(loss.detach()), TO.flatten_tensors(grads).numpy()


def _probe(ctx, rb, cfg, q, di):
    loss = C.c_double()
    grad = np.zeros(q.num_params, np.float32)
    L.check(ctx._lib.rl_dqn_probe_seq(rb.handle, C.byref(cfg), q.handle, di, C.byref(loss), grad.ctypes.data_as(C.POINTER(C.c_float))),
            ctx.handle)
    return loss.value, grad


@pytest.mark.parametrize("hidden,activation", [(4, "relu"), (8, "tanh"), (32, "relu"), (128, "relu")])
@pytest.mark.parametrize("td", [False, True])
def test_qloss_probe_matches_f64(ctx, filled, hidden, activation, td):
    """The Q-loss pass (K9 at hidden <= 8, K10 above; tcgen05 at 128): loss and flat gradient against f64 autograd on the
    oracle's GRU, on the sampled sequences and their targets."""
    env, rb, lanes = filled
    F, A = 5, 2
    params = _q_params(np.random.default_rng(100 + hidden), F, hidden, A, head_scale=2.0)
    q = R.GruLinear(ctx, F, hidden, A, activation)
    q.set_weights(params)
    seed, di, minibatch, g = 9, 4, 700, 0.99
    cfg = L.DqnCfg(minibatch, 1, 1 if td else 0, np.float32(g), seed)
    loss, grad = _probe(ctx, rb, cfg, q, di)
    eps = _oracle_minibatch(lanes, seed, di, minibatch)
    tg = _td_targets(params, F, hidden, A, eps, g) if td else [_rtg(e, g) for e in eps]
    # the targets enter as the device computed them (f32): compare the pass, not the target forward
    got_t = rb.sample_seq(cfg, q, di)["target"]
    tg32 = [got_t[:len(e["action"]), b] for b, e in enumerate(eps)]
    if not td:
        for a, b in zip(tg32, tg):
            np.testing.assert_array_equal(a, b)
    loss64, g64 = _seq_q_loss_grad(params, F, hidden, A, eps, tg32, activation=activation)
    _, g32 = _seq_q_loss_grad(params, F, hidden, A, eps, tg32, dtype=torch.float32, activation=activation)
    print(f"h={hidden} {activation} td={td}: loss {loss:.8f} vs {loss64:.8f}; grad rel err kernel {_rel(grad, g64):.2e}, "
          f"torch-f32 {_rel(g32, g64):.2e}")
    assert abs(loss - loss64) <= 1e-6 * max(1.0, abs(loss64))
    assert _rel(grad, g64) <= 1e-5


def test_qloss_gemm_formulation_serves_the_small_modules_too():
    """K10's Q-loss pass on the modules K9 normally serves: the probe tests in a child process with RL_SEQ_FORCE_BIG=1 (the
    switch is read once per process)."""
    if os.environ.get("RL_SEQ_FORCE_BIG") == "1":
        pytest.skip("already the forced run")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RL_SEQ_FORCE_BIG="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_dqn_seq.py"), "-x", "-q", "-m", "gpu",
                        "-k", "probe and not 32 and not 128"], capture_output=True, text=True, env=env, cwd=root, timeout=1200)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and " passed" in r.stdout


def _oracle_seq_dqn(params, F, H, A, minibatches, g, td, dtype, lr=1e-3):
    prm = TO._seq_params(params, F, H, A, dtype)
    opt = TO.Adam112(prm, lr)
    losses = []
    for eps in minibatches:
        if td:
            with torch.no_grad():
                flat = TO.flatten_tensors([p.detach() for p in prm]).numpy()
            tg = [t.astype(np.float32) for t in _td_targets(flat.astype(np.float32) if dtype == torch.float32 else flat, F, H, A, eps, g,
                                                             dtype=dtype)]
        else:
            tg = [_rtg(e, g) for e in eps]
        q = TO.gru_linear_forward(prm, TO.EpisodeBatch([e["obs"] for e in eps], dtype))
        act = torch.tensor(np.concatenate([e["action"] for e in eps]), dtype=torch.int64).unsqueeze(-1)
        loss = torch.nn.functional.mse_loss(q.gather(-1, act).squeeze(-1), torch.tensor(np.concatenate(tg), dtype=dtype))
        opt.step(torch.autograd.grad(loss, prm))
        losses.append(float(loss.detach()))
    return TO.flatten_tensors([p.detach() for p in prm]).numpy().copy(), losses


_DRAWS = {}


@pytest.mark.parametrize("hidden", [8, 32])
@pytest.mark.parametrize("td", [False, True])
def test_dqn_update_seq_matches_oracle(ctx, filled, hidden, td):
    """opt_steps x {sequence sample, Q-loss with BPTT, Adam} against the torch loop on the same episodes: parameter delta
    within max(2e-4, 4x the torch-f32 run's own distance from the f64 run), as the feed-forward DQN test."""
    env, rb, lanes = filled
    F, A = 5, 2
    params = _q_params(np.random.default_rng(7 + hidden), F, hidden, A)
    steps, minibatch, seed = 5, 500, 321
    agent = R.DqnConfig(action_value_fn_config=R.GruLinearConfig(hidden_dim=hidden), minibatch_steps=minibatch,
                        opt_steps_per_update=steps, target_one_step_td=td, sample_seed=seed, buffer_capacity=120).build_agent(env)
    agent.action_value_fn.set_weights(params)
    assert agent.actor().seq_net is agent.action_value_fn and agent.actor().net is None
    # the buffer's draw counter advances by one per optimizer step, over every update on it (flat and sequence alike)
    base = _DRAWS.get(id(rb), 0)
    _DRAWS[id(rb)] = base + steps
    stats = agent.batch_update(rb, {})
    new = agent.action_value_fn.get_weights()
    mbs = [_oracle_minibatch(lanes, seed, base + s, minibatch) for s in range(steps)]
    g = float(agent.discount_factor)
    new64, losses64 = _oracle_seq_dqn(params, F, hidden, A, mbs, g, td, torch.float64)
    new32, _ = _oracle_seq_dqn(params, F, hidden, A, mbs, g, td, torch.float32)
    d, d64, d32 = new - params, new64 - params.astype(np.float64), new32 - params
    print(f"seq dqn h={hidden} td={td}: delta rel err vs f64 kernel {_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}; "
          f"loss {stats.loss_first:.6f}/{stats.loss_last:.6f} vs {losses64[0]:.6f}/{losses64[-1]:.6f}")
    assert stats.opt_steps == steps and stats.num_steps == sum(len(e["action"]) for e in mbs[-1])
    np.testing.assert_allclose(stats.loss_first, losses64[0], rtol=1e-5)
    np.testing.assert_allclose(stats.loss_last, losses64[-1], rtol=1e-4)
    assert _rel(d, d64) <= max(2e-4, 4 * _rel(d32, d64) + 1e-5)


# ------------------------------------------------------------------------------------------------
# Learning and errors
# ------------------------------------------------------------------------------------------------
def _memory_greedy_reward(ctx, config):
    cfg = R.MemoryGame(2, 4)
    E = 2048
    env = R.build_env(ctx, cfg, E, seed=6)
    agent = R.DqnConfig(action_value_fn_config=config, minibatch_steps=20_000, opt_steps_per_update=40, buffer_capacity=200,
                        optimizer_config=R.AdamConfig(learning_rate=3e-3),
                        exploration_rate=R.ExplorationRateSchedule(1.0, 0.1, 150_000),
                        update_size=R.DataCollectionSchedule(10 * E, 10 * E), sample_seed=2).build_agent(env)
    rng = np.random.default_rng(0)
    if isinstance(config, R.GruLinearConfig):
        agent.action_value_fn.set_weights(R.init_gru_linear_params(rng, env.num_features, config.hidden_dim, 2))
    else:
        agent.action_value_fn.set_weights(R.init_params(rng, env.num_features, config.hidden_sizes, 2))
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
    return means


def test_dqn_gru_learns_memory_game(ctx):
    """MemoryGame(2, 4): the reward depends on the first observation of the episode, which a feed-forward Q-network never
    sees again.  With a recurrent Q-network the greedy mean final reward reaches 0.9; the same schedule with an MLP stays
    near 0 (random play), so the memory is what is learned."""
    gru = _memory_greedy_reward(ctx, R.GruLinearConfig(hidden_dim=8))
    mlp = _memory_greedy_reward(ctx, R.MlpConfig(hidden_sizes=[64]))
    print("greedy mean episode reward, GRU:", [round(x, 3) for x in gru])
    print("greedy mean episode reward, MLP:", [round(x, 3) for x in mlp])
    assert max(gru[-3:]) >= 0.9
    assert max(abs(x) for x in mlp[-3:]) < 0.2


def test_dqn_seq_errors(ctx, filled):
    env, rb, lanes = filled
    F, A = 5, 2
    q = R.GruLinear(ctx, F, 8, A)
    q.set_weights(_q_params(np.random.default_rng(1), F, 8, A))
    other = R.GruLinear(ctx, F, 8, A)
    cfg = L.DqnCfg(100, 2, 0, np.float32(0.99), 1)
    stats = L.OptStats()
    lib = ctx._lib

    def status(*args):
        return lib.rl_dqn_update_seq(*args)

    # an optimizer of another module, an Mlp optimizer, a module of another context, a feature count that does not match
    assert status(rb.handle, q.handle, R.Adam(other, R.AdamConfig()).handle, C.byref(cfg), C.byref(stats)) == L.RL_ERR_INVALID_ARG
    mlp = R.Mlp(ctx, F, [16], A)
    assert status(rb.handle, q.handle, R.Adam(mlp, R.AdamConfig()).handle, C.byref(cfg), C.byref(stats)) == L.RL_ERR_INVALID_ARG
    ctx2 = R.Context(0)
    q2 = R.GruLinear(ctx2, F, 8, A)
    assert status(rb.handle, q2.handle, R.Adam(q2, R.AdamConfig()).handle, C.byref(cfg), C.byref(stats)) == L.RL_ERR_INVALID_ARG
    q6 = R.GruLinear(ctx, F + 1, 8, A)
    assert status(rb.handle, q6.handle, R.Adam(q6, R.AdamConfig()).handle, C.byref(cfg), C.byref(stats)) == L.RL_ERR_UNSUPPORTED
    # an empty ring: Uniform::new(0, 0)
    empty = R.ReplayBuffer(env, 50)
    assert status(empty.handle, q.handle, R.Adam(q, R.AdamConfig()).handle, C.byref(cfg), C.byref(stats)) == L.RL_ERR_INVALID_ARG
    # the rollout: an epsilon-greedy actor needs a network, recurrent or not
    traj = R.Trajectory(env, 8)
    with pytest.raises(L.RelearnB200Error) as ei:
        R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, exploration_rate=0.5), R.HistoryDataBound(8, 0), traj)
    assert ei.value.status == L.RL_ERR_INVALID_ARG
    # an Mlp Q-network with seq_net unset still takes the feed-forward kernels and agrees with their restatement
    mp = R.init_params(np.random.default_rng(2), F, 16, A)
    mlp.set_weights(mp)
    env.set_noise_philox(4, 0)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, net=mlp, exploration_rate=0.5), R.HistoryDataBound(8, 0), traj)
    checked, _ = P.check_eps_greedy_consistency(traj.to_host(), mp, 16, A, 0.5, philox=(4, 0, 0))
    assert checked > 0
    ctx2.close()
