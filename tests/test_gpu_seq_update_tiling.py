"""GPU parity of K10, the GEMM form of the recurrent update passes (gru_big.cu, gru_big_tc.cuh), at the lane counts,
sequence lengths and module sizes where its tiles, splits and drains change, against the f64 oracle.

The other recurrent parity tests run K10 at E <= 96 lanes and T <= 23 steps on 0/1 bandit features, where every GEMM
takes 64-row tiles, no weight-gradient split drains more than once and the observations have no low-order bf16 pieces.
Here the trajectories are synthetic (Trajectory.load): N(0, 1) observations, episodes of length 1, lanes that hold one
episode over all T steps, lanes that end early in a PAD tail, lanes with no steps, and an Interrupt as every lane's last
step.  Each case first recomputes, from the SM count, the selection condition of the path it is there for (citing the line
it mirrors) and fails if the shape no longer reaches it.

Tolerances are those of test_gpu_gru_update.py / test_gpu_lstm.py against the f64 oracle (tests/seq_chunked_oracle.py
over chunks of episodes): loss within 1e-6 relative, entropy within 1e-6, gradient and Fisher-vector product within 1e-5
relative, and within 1e-5 on every parameter block (W_ih, W_hh, b_ih, b_hh, head weights, head bias) measured against
that block's own norm, so that a wrong bias row cannot hide in the norm of the whole vector."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import oracle as O
from oracle import tensor_oracle as TO
import relearn_b200 as R
from relearn_b200 import _lib as L

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from tests import seq_chunked_oracle as SC  # noqa: E402

CONT, TERM, INTR, PAD = L.RL_CONTINUE, L.RL_TERMINATE, L.RL_INTERRUPT, L.RL_PAD
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# gru_big_tc.cuh:327 (weight-gradient operand rows and drain period) and :25 (lanes per big_gemm_tc_kernel CTA)
NT_ROWS_B, NT_DRAIN, BT_LANES = 144, 512, 128

# The tensor-core form (GRU 128) over 10^5 .. 10^6 lane-steps of long sequences misses 1e-5 for a numerical reason, not a
# wrong term.  Measured on a B200 (148 SMs, default power limit), kernel vs f64 with the torch-f32 oracle's own distance:
#   D1 (385 k steps, T 128)  grad 4.2e-5 (torch-f32 3.8e-5), fvp 5.2e-5 (5.2e-7)
#   D2 (773 k steps, T 256)  grad 3.6e-5 (2.7e-6),           fvp 5.0e-5 (1.2e-6)
#   H  (61 k steps, T 600)   grad 7.6e-5 (1.7e-6),           fvp 1.3e-5 (4.1e-6)
#   I  (3.8 M steps, T 199)  tensor-core vs FP32 form: up to 5.4e-5 (grad W_hh), 1.0e-4 (fvp W_hh)
# The error grows with the number of steps and stays in the blocks the tensor cores accumulate (W_ih, W_hh, b_ih, b_hh):
# D1 drains each split once, so no slab is involved; the head blocks (FP32 split-K) stay near 1e-6, and the FP32 form of
# the same module at 74 k steps (case E') is at 1.5e-7.  The bf16 pieces drop only products <= 2^-24 relative; what
# remains is the f32 accumulation inside the tensor core, whose rounding does not average out over many steps.  Those
# cases are held to TC_LONG_TOL, which a lost or misplaced slab, tile or bias row exceeds by orders of magnitude.
TC_LONG_TOL = 2e-4


@pytest.fixture(scope="module")
def ctx():
    """A context of this file's own: the scratch its large cases grow (several GB of planes) goes back to the device when
    the file ends instead of staying with the session's context for every later test."""
    c = R.Context(0)
    yield c
    c.close()


# ------------------------------------------------------------------------------------------------
# K10's selection conditions, restated
# ------------------------------------------------------------------------------------------------
def _sm_count(ctx):
    return ctx.device_info()["sm_count"]


def _tc_form(cell, H, tc_env=True):
    """gru_big.cu:704: the per-step GEMMs of a GRU with hidden 128 on the tensor cores unless RL_SEQ_TC=0."""
    return cell == "gru" and H == 128 and tc_env


def _nt_tc(cell, F, H, tc_env=True):
    """gru_big.cu:709: weight gradients on the tensor cores while [x ; h ; 1] fits the 144-row operand."""
    return _tc_form(cell, H, tc_env) and F + H + 1 <= NT_ROWS_B


def _nt_units_per_split(E, T, sm):
    """gru_big.cu:710-711 and gru_big_tc.cuh:370-372: sm / 2 splits of T * ceil(E / 16) units, split s owning
    [units * s / S, units * (s + 1) / S)."""
    S = max(sm // 2, 1)
    units = T * ((E + 15) // 16)
    return [units * (s + 1) // S - units * s // S for s in range(S)]


def _nt_slabs(n):
    """gru_big_tc.cuh:474-495: a split of n units drains after every NT_DRAIN units and after its last unit."""
    return (n + NT_DRAIN - 1) // NT_DRAIN


def _gemm_128_rows(M, N, sm):
    """gru_big.cu:664-665: gemm_nn_kernel<8> (128-row tiles) when they give at least two CTAs per SM."""
    return M >= 128 and -(-N // 128) * -(-M // 128) >= 2 * sm


def _splitk_flushes(E, T):
    """gru_big.cu:142-143, 203: gemm_nt_splitk_kernel's 32 splits flush their f32 sums into f64 every 128 units."""
    return T * ((E + 15) // 16) // 32 > 128


def _reached(cond, what):
    assert cond, f"this shape no longer selects {what}: the case has to be re-derived from the selection condition"
    print(f"path reached: {what}")


# ------------------------------------------------------------------------------------------------
# Synthetic trajectories and modules
# ------------------------------------------------------------------------------------------------
def _planes(seed, E, T, F, A, one_episode=0.25):
    """obs / next_obs [T, E, F] ~ N(0.5, 1), action [T, E] uniform < A, reward 0/1, adv ~ N(0.5, 1), succ [T, E]: a
    quarter of the lanes one episode over all T steps, the others of random length with random episode ends (lanes 5k + 2
    start with three episodes of length 1), lanes 1, E / 2 and E - 2 empty, every lane's last step an Interrupt.

    The means keep the batch conditioned like a real one.  With zero-mean advantages and features independent of
    everything else, the mean gradient is a 1/sqrt(N) residue of its terms, and at 10^5 .. 10^6 steps no f32 computation
    meets 1e-5: on a B200 the torch-f32 oracle itself missed f64 by 1.0e-4 at case D1's shape, the loss at case I's shape
    was -1.9e-4, and the two forms of K10 differed by 4.9e-4 there, all from f32 accumulation order rather than a wrong
    term."""
    rng = np.random.default_rng(seed)
    succ = np.full((T, E), PAD, np.uint8)
    single = rng.random(E) < one_episode
    lens = np.where(single, T, rng.integers(1, T + 1, size=E))
    lens[[1, E // 2, E - 2]] = 0
    p_end = min(1.0, 4.0 / T)
    for e in range(E):
        n = int(lens[e])
        if n == 0:
            continue
        col = np.full(n, CONT, np.uint8)
        if not single[e]:
            ends = rng.random(n) < p_end
            if e % 5 == 2:
                ends[:3] = True
            col[ends] = np.where(rng.random(int(ends.sum())) < 0.5, TERM, INTR)
        col[-1] = INTR
        succ[:n, e] = col
    live = (succ != PAD)
    obs = (0.5 + rng.normal(size=(T, E, F))).astype(np.float32) * live[..., None]
    next_obs = (0.5 + rng.normal(size=(T, E, F))).astype(np.float32) * live[..., None]
    action = (rng.integers(0, A, size=(T, E)) * live).astype(np.uint8)
    reward = ((rng.random(size=(T, E)) < 0.6) * live).astype(np.float32)
    adv = ((0.5 + rng.normal(size=(T, E))) * live).astype(np.float32)
    return dict(obs=obs, next_obs=next_obs, action=action, reward=reward, succ=succ, adv=adv)


def _params(cell, seed, F, H, A):
    """The rl2 initialisation with N(0, 0.2) biases (zero biases would leave the bias rows of every GEMM untested)."""
    rng = np.random.default_rng(seed)
    G = 3 if cell == "gru" else 4
    p = (R.init_gru_linear_params if cell == "gru" else R.init_lstm_linear_params)(rng, F, H, A).astype(np.float32)
    o = G * H * F + G * H * H
    p[o:o + 2 * G * H] = rng.normal(size=2 * G * H) * 0.2
    p[-A:] = rng.normal(size=A) * 0.2
    return p


def _blocks(cell, F, H, A):
    G = 3 if cell == "gru" else 4
    sizes = [("W_ih", G * H * F), ("W_hh", G * H * H), ("b_ih", G * H), ("b_hh", G * H), ("head W", A * H), ("head b", A)]
    out, o = [], 0
    for name, n in sizes:
        out.append((name, slice(o, o + n)))
        o += n
    return out


def _load(ctx, pl, E, T, F):
    """A trajectory of the bandit meta-env with F - 4 arms (F features) filled with the planes."""
    env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(F - 4), 4), E, seed=1)
    assert env.num_features == F
    traj = R.Trajectory(env, T)
    traj.load(pl["obs"], pl["action"], pl["reward"], pl["succ"], pl["next_obs"])
    return env, traj


def _net(ctx, cell, F, H, A, params, activation="relu"):
    net = (R.GruLinear if cell == "gru" else R.LstmLinear)(ctx, F, H, A, activation)
    net.set_weights(params)
    return net


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) /
                 max(np.linalg.norm(np.asarray(b, np.float64)), 1e-300))


def _device_probe(ctx, cell, pl, E, T, F, H, A, params, vec, reg=1e-5):
    env, traj = _load(ctx, pl, E, T, F)
    net = _net(ctx, cell, F, H, A, params)
    policy = R.Trpo(net, R.TrpoConfig(optimizer_config=R.ConjugateGradientOptimizerConfig(hpv_reg_coeff=reg)))
    return policy.probe(traj, ctx.to_device(pl["adv"]), vec)


def _check_probe(got, cell, pl, F, H, A, params, vec, reg=1e-5, what="", tol=1e-5):
    """The device probe against the chunked f64 oracle, whole vectors and every parameter block; prints the torch-f32
    oracle's own distance from f64 beside the kernel's."""
    args = (cell, params, F, H, A, pl["obs"], pl["action"], pl["adv"], pl["succ"], vec, reg)
    loss64, kl64, ent64, g64, hv64 = SC.policy_loss_kl_grad_fvp(*args, dtype=torch.float64)
    _, _, _, g32, hv32 = SC.policy_loss_kl_grad_fvp(*args, dtype=torch.float32)
    print(f"{what}: steps={int((pl['succ'] != PAD).sum())} grad rel err: kernel {_rel(got['grad'], g64):.2e} torch-f32 "
          f"{_rel(g32, g64):.2e}; fvp rel err: kernel {_rel(got['fvp'], hv64):.2e} torch-f32 {_rel(hv32, hv64):.2e}")
    worst = []
    for name, sl in _blocks(cell, F, H, A):
        eg, ef = _rel(got["grad"][sl], g64[sl]), _rel(got["fvp"][sl], hv64[sl])
        print(f"    {name:7s} grad kernel {eg:.2e} torch-f32 {_rel(g32[sl], g64[sl]):.2e}; "
              f"fvp kernel {ef:.2e} torch-f32 {_rel(hv32[sl], hv64[sl]):.2e}")
        worst += [(eg, "grad " + name), (ef, "fvp " + name)]
    assert abs(got["loss"] - loss64) <= 1e-6 * max(1.0, abs(loss64))
    assert abs(got["kl"]) <= 1e-7 and abs(kl64) <= 1e-12
    assert abs(got["entropy"] - ent64) <= 1e-6
    assert _rel(got["grad"], g64) <= tol
    assert _rel(got["fvp"], hv64) <= tol
    bad = [(e, n) for e, n in worst if not e <= tol]
    assert not bad, f"parameter blocks beyond {tol} of f64: {bad}"


def _check_forward(ctx, cell, pl, E, T, F, H, A, params):
    """SeqPacked forward (rl_grunet_seq_forward) on every stored step against the f64 outputs."""
    env, traj = _load(ctx, pl, E, T, F)
    got = _net(ctx, cell, F, H, A, params).seq_packed(traj)
    want = SC.outputs(cell, params, F, H, A, pl["obs"], pl["succ"])
    valid = pl["succ"] != PAD
    print(f"seq_forward max abs err {np.abs(got[valid] - want[valid]).max():.2e}")
    np.testing.assert_allclose(got[valid], want[valid], rtol=1e-5, atol=2e-6)
    assert (got[~valid] == 0).all()


def _check_gae(ctx, cell, pl, E, T, F, H, steps=0):
    """rl_gae_seq with a recurrent critic (an interrupted episode bootstraps from one more step of the same sequence)
    against O.gae_lane on the f64 values; with steps > 0 also that many Adam steps of the critic against the oracle."""
    env, traj = _load(ctx, pl, E, T, F)
    vparams = _params(cell, 5, F, H, 1)
    mcfg = (R.GruLinearConfig if cell == "gru" else R.LstmLinearConfig)(hidden_dim=H)
    critic = R.ValuesOpt(ctx, R.ValuesOptConfig(state_value_fn_config=mcfg, opt_steps_per_update=max(steps, 1)), F,
                         env.discount_factor)
    critic.state_value_fn.set_weights(vparams)
    gamma, lam = critic.discount_factor, np.float32(critic.cfg.gae_lambda)
    adv = critic.advantages(traj).download((T, E), np.float32)
    v, vn = SC.outputs(cell, vparams, F, H, 1, pl["obs"], pl["succ"], pl["next_obs"])
    v, vn = v[..., 0].astype(np.float32), vn[..., 0].astype(np.float32)
    succ, reward = pl["succ"], pl["reward"]
    lens = (succ != PAD).sum(0)
    err = 0.0
    for e in range(E):
        n = int(lens[e])
        ref = O.gae_lane(reward[:n, e], v[:n, e], vn[:n, e], succ[:n, e], gamma, lam)
        np.testing.assert_allclose(adv[:n, e], ref, rtol=2e-5, atol=2e-6)
        err = max(err, float(np.abs(adv[:n, e] - ref).max(initial=0.0)))
    print(f"GAE max abs err {err:.2e}, {int((succ == INTR).sum())} interrupted episodes")
    if steps == 0:
        return
    stats = critic.update(traj)
    new = critic.state_value_fn.get_weights()
    spans = SC.episode_spans(succ)
    rtg = np.zeros((T, E), np.float32)
    for e in range(E):
        n = int(lens[e])
        rtg[:n, e] = O.discounted_cumsum_lane(reward[:n, e], succ[:n, e], gamma)
    eps, tg = [pl["obs"][a:b, e] for e, a, b in spans], [rtg[a:b, e] for e, a, b in spans]
    new64, losses64 = TO.seq_value_update(vparams, F, H, eps, tg, n_steps=steps, dtype=torch.float64)
    new32, _ = TO.seq_value_update(vparams, F, H, eps, tg, n_steps=steps, dtype=torch.float32)
    d, d64, d32 = new - vparams, new64 - vparams.astype(np.float64), new32 - vparams
    print(f"critic delta rel err vs f64: kernel {_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}")
    assert stats.opt_steps == steps and stats.num_steps == sum(b - a for _, a, b in spans)
    np.testing.assert_allclose(stats.loss_first, losses64[0], rtol=1e-5)
    np.testing.assert_allclose(stats.loss_last, losses64[-1], rtol=1e-4)
    assert _rel(d, d64) <= max(2e-4, 4 * _rel(d32, d64) + 1e-5)


def _vec(seed, n):
    return np.random.default_rng(seed).normal(size=n).astype(np.float32)


def _probe_case(ctx, cell, E, T, F, H, A, seed, what, reg=1e-5, tol=1e-5):
    pl = _planes(seed, E, T, F, A)
    params = _params(cell, seed + 1, F, H, A)
    vec = _vec(seed + 2, params.size)
    got = _device_probe(ctx, cell, pl, E, T, F, H, A, params, vec, reg)
    _check_probe(got, cell, pl, F, H, A, params, vec, reg, what, tol)
    return pl, params


# ------------------------------------------------------------------------------------------------
# A, B, C: several big_gemm_tc_kernel CTAs, a ragged last one, scalar loads, the 144-row operand's boundary
# ------------------------------------------------------------------------------------------------
def test_case_a_several_ctas_ragged(ctx):
    """GRU 128, F 14, A 10 at E = 300 (three 128-lane CTAs, E % 16 = 12), T = 40: probe, SeqPacked forward, GAE with the
    Interrupt bootstrap, six critic steps and a whole TRPO step at hpv_reg_coeff 0.1."""
    E, T, F, H, A = 300, 40, 14, 128, 10
    _reached(_tc_form("gru", H) and -(-E // BT_LANES) == 3 and E % BT_LANES and E % 16,
             f"{-(-E // BT_LANES)} big_gemm_tc_kernel CTAs, the last one {E % BT_LANES} lanes (gru_big.cu:644, 704)")
    pl, params = _probe_case(ctx, "gru", E, T, F, H, A, 10, "A")
    _check_forward(ctx, "gru", pl, E, T, F, H, A, params)
    _check_gae(ctx, "gru", pl, E, T, F, H, steps=6)
    # a whole trust-region step
    reg = 0.1
    env, traj = _load(ctx, pl, E, T, F)
    net = _net(ctx, "gru", F, H, A, params)
    policy = R.Trpo(net, R.TrpoConfig(optimizer_config=R.ConjugateGradientOptimizerConfig(hpv_reg_coeff=reg)))
    log = {}
    status = policy.update(traj, ctx.to_device(pl["adv"]), log)
    new = net.get_weights()
    spans = SC.episode_spans(pl["succ"])
    take = lambda x: [x[a:b, e] for e, a, b in spans]  # noqa: E731
    eps, acts, advs = take(pl["obs"]), take(pl["action"]), take(pl["adv"])
    ocfg = TO.CgConfig(hpv_reg_coeff=reg)
    new64, log64 = TO.seq_trpo_update(params, F, H, A, eps, acts, advs, cfg=ocfg, dtype=torch.float64)
    new32, log32 = TO.seq_trpo_update(params, F, H, A, eps, acts, advs, cfg=ocfg, dtype=torch.float32)
    d, d64, d32 = new - params, new64 - params.astype(np.float64), new32 - params
    print(f"TRPO step: status={status} backtracks kernel/f64/f32 = {log['num_backtracks']}/{log64['num_backtracks']}/"
          f"{log32['num_backtracks']}; delta rel err vs f64: kernel {_rel(d, d64):.2e}, torch-f32 {_rel(d32, d64):.2e}")
    assert status == L.RL_OK and log64["error"] is None
    assert log["num_steps"] == sum(b - a for _, a, b in spans)
    assert log["num_backtracks"] == log64["num_backtracks"]
    np.testing.assert_allclose(log["entropy"], log64["entropy"], rtol=1e-5)
    np.testing.assert_allclose(log["step_size"], log64["step_size"], rtol=2e-5)
    np.testing.assert_allclose(log["loss_initial"], log64["loss_initial"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(log["loss_final"], log64["loss_final"], rtol=1e-5, atol=1e-7)
    assert _rel(d, d64) <= max(2e-5, 1.25 * _rel(d32, d64)) and _rel(d, d64) <= 1e-4


def test_case_b_scalar_loads(ctx):
    """GRU 128, F 14 at E = 301: E % 4 != 0 sends the weight-gradient producers to their scalar loads."""
    E, T, F, H, A = 301, 40, 14, 128, 10
    _reached(_nt_tc("gru", F, H) and E % 4 != 0, f"big_nt_tc_kernel scalar loads, E % 4 = {E % 4} (gru_big_tc.cuh:411)")
    _probe_case(ctx, "gru", E, T, F, H, A, 20, "B")


@pytest.mark.parametrize("F", [15, 16])
def test_case_c_operand_boundary(ctx, F):
    """GRU 128 at F = 15 ([x ; h ; 1] fills all 144 rows, the ones row last: tensor-core weight gradients) and F = 16
    (145 rows: the FP32 split-K fallback)."""
    E, T, H = 300, 40, 128
    A = F - 4
    if F + H + 1 == NT_ROWS_B:
        _reached(_nt_tc("gru", F, H), "big_nt_tc_kernel with the ones row in the last of the 144 rows (gru_big.cu:709)")
    else:
        _reached(_tc_form("gru", H) and not _nt_tc("gru", F, H),
                 f"gemm_nt_splitk_kernel weight gradients, F + H + 1 = {F + H + 1} > 144 (gru_big.cu:709, 837-839)")
    _probe_case(ctx, "gru", E, T, F, H, A, 30 + F, f"C F={F}")


# ------------------------------------------------------------------------------------------------
# D: the weight-gradient drains
# ------------------------------------------------------------------------------------------------
def test_case_d1_drain_at_last_step(ctx):
    """Every split gets exactly NT_DRAIN units: its one drain falls on its last step."""
    sm = _sm_count(ctx)
    S = max(sm // 2, 1)
    T, F, H, A = 128, 15, 128, 11
    E = 16 * (NT_DRAIN * S // T) - 4  # T * ceil(E / 16) = 512 * S, E % 16 = 12
    per = _nt_units_per_split(E, T, sm)
    _reached(_nt_tc("gru", F, H) and set(per) == {NT_DRAIN},
             f"E = {E}, T = {T}: all {S} splits own exactly {NT_DRAIN} units (gru_big_tc.cuh:371, 405, 474)")
    _probe_case(ctx, "gru", E, T, F, H, A, 40, "D1", tol=TC_LONG_TOL)


def test_case_d2_three_slabs(ctx):
    """1024 .. 1100 units per split: two full slabs and a short third one, added in f64 by splitk_reduce_f32_kernel."""
    sm = _sm_count(ctx)
    S = max(sm // 2, 1)
    T, F, H, A = 256, 15, 128, 11
    E = 16 * -(-1040 * S // T) - 10
    per = _nt_units_per_split(E, T, sm)
    _reached(_nt_tc("gru", F, H) and min(per) > 2 * NT_DRAIN and max(per) <= 1100 and {_nt_slabs(n) for n in per} == {3},
             f"E = {E}, T = {T}: {min(per)} .. {max(per)} units per split, three slabs (gru_big_tc.cuh:474-495)")
    _probe_case(ctx, "gru", E, T, F, H, A, 50, "D2", tol=TC_LONG_TOL)


# ------------------------------------------------------------------------------------------------
# E, E': 128-row FP32 tiles and the split-K f64 flush
# ------------------------------------------------------------------------------------------------
def _e_shape(sm):
    """E, T of cases E and E': ceil(E / 128) * ceil(4H / 128) >= 2 * sm for 4H in (384, 512], E % 128 = 28."""
    return 128 * -(-sm // 2) + 28, 12


@pytest.mark.parametrize("cell,H", [("lstm", 128), ("gru", 100)])
def test_case_e_128_row_tiles(ctx, cell, H):
    """LSTM 128 and GRU 100 (4H = 400: a ragged 128-row tile; F + H not a multiple of 8) on the FP32 pipe at a lane
    count that selects gemm_nn_kernel<8>; the split-K weight gradients flush to f64.  For the LSTM also the SeqPacked
    forward and GAE."""
    sm = _sm_count(ctx)
    E, T = _e_shape(sm)
    F, A = 14, 10
    _reached(not _tc_form(cell, H) and _gemm_128_rows(4 * H, E, sm) and _splitk_flushes(E, T),
             f"{cell} {H}, E = {E}: gemm_nn_kernel<8> for the {4 * H}-row gate GEMMs (gru_big.cu:664-667), split-K f64 "
             f"flushes (gru_big.cu:203)")
    pl, params = _probe_case(ctx, cell, E, T, F, H, A, 60 + H, f"E {cell} {H}")
    if cell == "lstm":
        _check_forward(ctx, cell, pl, E, T, F, H, A, params)
        _check_gae(ctx, cell, pl, E, T, F, H)


def _child(fn, tc, out, *args):
    """Run `fn(ctx, *args)` of this module in a child process with RL_SEQ_TC=tc (read once per process) and load the
    arrays it saves to `out`."""
    code = (f"import sys; sys.path.insert(0, {ROOT!r}); import numpy as np; import relearn_b200 as R; "
            f"from tests import test_gpu_seq_update_tiling as M; ctx = R.Context(0); "
            f"np.savez({out!r}, **M.{fn}(ctx, *{args!r})); ctx.close()")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=1200,
                       env=dict(os.environ, RL_SEQ_TC=str(tc)))
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0
    return dict(np.load(out))


def _probe_arrays(ctx, cell, E, T, F, H, A, seed):
    pl = _planes(seed, E, T, F, A)
    params = _params(cell, seed + 1, F, H, A)
    got = _device_probe(ctx, cell, pl, E, T, F, H, A, params, _vec(seed + 2, params.size))
    return {k: np.asarray(v) for k, v in got.items()}


def test_case_e_prime_gru128_fp32_form(ctx):
    """GRU 128 with RL_SEQ_TC=0 (a child process: the switch is read once per process) at case E's shape: the FP32 form
    of the rl2-sized module, 128-row tiles included, against f64."""
    sm = _sm_count(ctx)
    E, T = _e_shape(sm)
    F, H, A, seed = 14, 128, 10, 70
    _reached(not _tc_form("gru", H, tc_env=False) and _gemm_128_rows(4 * H, E, sm) and _splitk_flushes(E, T),
             f"gru 128 under RL_SEQ_TC=0, E = {E}: gemm_nn_kernel<8> (gru_big.cu:664-667, 704), split-K f64 flushes")
    with tempfile.TemporaryDirectory() as tmp:
        got = _child("_probe_arrays", 0, os.path.join(tmp, "p.npz"), "gru", E, T, F, H, A, seed)
    got = {k: (float(v) if v.ndim == 0 else v) for k, v in got.items()}
    pl = _planes(seed, E, T, F, A)
    params = _params("gru", seed + 1, F, H, A)
    _check_probe(got, "gru", pl, F, H, A, params, _vec(seed + 2, params.size), what="E' gru 128 FP32 form")


# ------------------------------------------------------------------------------------------------
# G: the wide head; H: long BPTT
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H", [24, 128])
@pytest.mark.parametrize("A", [20, 32])
def test_case_g_wide_head(ctx, H, A):
    """More than 16 outputs: big_head_kernel<MODE, 32> (gru_big.cu:656-657)."""
    E, T, F = 300, 30, 14
    _reached(16 < A <= 32, f"big_head_kernel<MODE, 32> at A = {A} (gru_big.cu:656-657)")
    pl, params = _probe_case(ctx, "gru", E, T, F, H, A, 80 + H + A, f"G H={H} A={A}")
    _check_forward(ctx, "gru", pl, E, T, F, H, A, params)


def test_case_h_long_bptt(ctx):
    """T = 600 with half the lanes holding one episode over all of it: backpropagation through 600 steps."""
    E, T, F, H, A, seed = 130, 600, 15, 128, 11, 90
    pl = _planes(seed, E, T, F, A, one_episode=0.5)
    longest = max(b - a for _, a, b in SC.episode_spans(pl["succ"]))
    _reached(longest == T and (pl["succ"][-1] != PAD).sum() >= E // 4, f"episodes of {longest} steps")
    params = _params("gru", seed + 1, F, H, A)
    vec = _vec(seed + 2, params.size)
    got = _device_probe(ctx, "gru", pl, E, T, F, H, A, params, vec)
    _check_probe(got, "gru", pl, F, H, A, params, vec, what="H", tol=TC_LONG_TOL)


# ------------------------------------------------------------------------------------------------
# I: the production shape, tensor-core form against the FP32 form
# ------------------------------------------------------------------------------------------------
def test_case_i_production_shape_tc_vs_fp32(ctx):
    """GRU 128, F 14, A 10 at E = 18 944, T = 199 (the rl2 rollout): grad and FVP of the tensor-core form (RL_SEQ_TC=1)
    and the FP32 form (RL_SEQ_TC=0) agree per parameter block.  No f64 oracle at 3.8 M lane-steps; cases D and E' pin
    each form against f64 at smaller sizes.  The bound is TC_LONG_TOL, not 3e-6: see the measurements above it."""
    sm = _sm_count(ctx)
    E, T, F, H, A, seed = 18944, 199, 14, 128, 10, 100
    per = _nt_units_per_split(E, T, sm)
    _reached(_nt_tc("gru", F, H) and min(_nt_slabs(n) for n in per) > 2 and _gemm_128_rows(4 * H, E, sm),
             f"{min(per)} .. {max(per)} units per split ({_nt_slabs(max(per))} slabs); the FP32 form on 128-row tiles")
    with tempfile.TemporaryDirectory() as tmp:
        tc = _child("_probe_arrays", 1, os.path.join(tmp, "tc.npz"), "gru", E, T, F, H, A, seed)
        fp = _child("_probe_arrays", 0, os.path.join(tmp, "fp.npz"), "gru", E, T, F, H, A, seed)
    print(f"I: loss {float(tc['loss']):.9f} / {float(fp['loss']):.9f}")
    bad = []
    for key in ("grad", "fvp"):
        for name, sl in _blocks("gru", F, H, A):
            err = _rel(tc[key][sl], fp[key][sl])
            print(f"    {key} {name:7s} tensor-core vs FP32 {err:.2e}")
            if not err <= TC_LONG_TOL:
                bad.append((key, name, err))
    assert abs(float(tc["loss"]) - float(fp["loss"])) <= 1e-6 * max(1.0, abs(float(fp["loss"])))
    assert abs(float(tc["entropy"]) - float(fp["entropy"])) <= 1e-6
    assert not bad, bad
