"""CPU checks of tests/seq_chunked_oracle.py: on small random trajectory planes (episodes of length 1, lanes that run one
episode to the end, PAD tails, lanes with no steps, open and interrupted last episodes) the chunked oracle equals one call
of the wrapped oracle on all episodes, for the GRU and the LSTM chain: loss, KL, entropy, gradient, Fisher-vector product,
and the outputs with the Interrupt bootstrap that GAE's value targets are built from."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import relearn_b200 as R  # noqa: E402
from relearn_b200 import _lib as L  # noqa: E402
from oracle import tensor_oracle as TO  # noqa: E402
from tests import lstm_oracle as LO  # noqa: E402
from tests import seq_chunked_oracle as SC  # noqa: E402

CONT, TERM, INTR, PAD = L.RL_CONTINUE, L.RL_TERMINATE, L.RL_INTERRUPT, L.RL_PAD
F, H, A, T, E = 5, 6, 3, 13, 9


def _planes(seed):
    rng = np.random.default_rng(seed)
    succ = np.full((T, E), PAD, np.uint8)
    lens = [T, 0, 1, 7, T, 4, 0, 11, T]
    for e, n in enumerate(lens):
        col = rng.choice([CONT, CONT, TERM, INTR], size=n).astype(np.uint8)
        if e == 0:
            col[:] = CONT  # one episode spanning the lane, left open at the end
        elif e == 4:
            col[:] = TERM  # every episode of length 1
        elif n:
            col[-1] = INTR
        succ[:n, e] = col
    obs = rng.normal(size=(T, E, F))
    next_obs = rng.normal(size=(T, E, F))
    action = rng.integers(0, A, size=(T, E))
    adv = rng.normal(size=(T, E))
    return obs, next_obs, action, adv, succ


def _params(cell, seed):
    rng = np.random.default_rng(seed)
    G = 3 if cell == "gru" else 4
    p = (R.init_gru_linear_params if cell == "gru" else R.init_lstm_linear_params)(rng, F, H, A).astype(np.float64)
    o = G * H * F + G * H * H
    p[o:o + 2 * G * H] = rng.normal(size=2 * G * H) * 0.3
    return p


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(np.asarray(b)), 1e-300))


def test_episode_spans():
    _, _, _, _, succ = _planes(0)
    spans = SC.episode_spans(succ)
    # every stored step in exactly one episode, episodes end at a non-CONTINUE step or the lane's last step
    assert sum(b - a for _, a, b in spans) == int((succ != PAD).sum())
    assert {e for e, _, _ in spans} == {0, 2, 3, 4, 5, 7, 8}
    assert [(a, b) for e, a, b in spans if e == 0] == [(0, T)]
    assert [(a, b) for e, a, b in spans if e == 4] == [(t, t + 1) for t in range(T)]
    for e, a, b in spans:
        assert (succ[a:b - 1, e] == CONT).all() and b <= T and (b == T or succ[b - 1, e] != CONT or succ[b, e] == PAD)


@pytest.mark.parametrize("cell", ["gru", "lstm"])
@pytest.mark.parametrize("max_cells", [1, 20, 60])
def test_chunked_probe_equals_one_batch(cell, max_cells):
    obs, _, action, adv, succ = _planes(1)
    params = _params(cell, 2)
    vec = np.random.default_rng(3).normal(size=params.size)
    spans = SC.episode_spans(succ)
    assert len(SC.chunks(spans, max_cells)) > 1
    take = lambda x: [x[a:b, e] for e, a, b in spans]  # noqa: E731
    fn = TO.seq_policy_loss_kl_grad_fvp if cell == "gru" else LO.seq_policy_loss_kl_grad_fvp
    want = fn(params, F, H, A, take(obs), take(action), take(adv), vec, 0.1, torch.float64, "tanh")
    got = SC.policy_loss_kl_grad_fvp(cell, params, F, H, A, obs, action, adv, succ, vec, 0.1, torch.float64, "tanh",
                                     max_cells=max_cells)
    assert abs(got[0] - want[0]) <= 1e-12 * max(1.0, abs(want[0]))
    assert abs(got[1] - want[1]) <= 1e-12
    assert abs(got[2] - want[2]) <= 1e-12 * abs(want[2])
    assert _rel(got[3], want[3]) <= 1e-12 and _rel(got[4], want[4]) <= 1e-12
    # the compared quantities are not trivially small
    assert abs(want[0]) > 1e-3 and np.linalg.norm(want[3]) > 1e-3


@pytest.mark.parametrize("cell", ["gru", "lstm"])
def test_chunked_outputs_and_interrupt_bootstrap(cell):
    obs, next_obs, _, _, succ = _planes(4)
    params = _params(cell, 5)
    episode = TO.gru_linear_episode if cell == "gru" else LO.lstm_linear_episode
    out, out_next = SC.outputs(cell, params, F, H, A, obs, succ, next_obs, max_cells=15)
    one, one_next = SC.outputs(cell, params, F, H, A, obs, succ, next_obs, max_cells=10 ** 9)
    np.testing.assert_allclose(out, one, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(out_next, one_next, rtol=1e-12, atol=1e-12)
    want, want_next = np.zeros_like(out), np.zeros_like(out)
    n_intr = 0
    for e, a, b in SC.episode_spans(succ):
        x = obs[a:b, e]
        if succ[b - 1, e] == INTR:
            y = episode(params, F, H, A, np.concatenate([x, next_obs[b - 1:b, e]]), "relu", torch.float64)
            want[a:b, e], want_next[b - 1, e] = y[:-1], y[-1]
            n_intr += 1
        else:
            want[a:b, e] = episode(params, F, H, A, x, "relu", torch.float64)
    assert n_intr >= 5
    np.testing.assert_allclose(out, want, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(out_next, want_next, rtol=1e-12, atol=1e-12)
    assert (out[succ == PAD] == 0).all()
