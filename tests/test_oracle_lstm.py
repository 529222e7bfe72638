"""CPU checks of the Chain<Lstm, Linear> restatement (tests/lstm_oracle.py) and of the Python module helpers: the packed
forward agrees with the iterated lstm_cell (the reference's seq_packed_matches_iter_steps), the flat parameter order is
torch.nn.LSTM's weight_ih_l0 .. bias_hh_l0 followed by the Linear, and the initializer follows RnnBaseConfig::default()."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import relearn_b200 as R  # noqa: E402
from oracle import tensor_oracle as TO  # noqa: E402
from tests import lstm_oracle as LO  # noqa: E402


@pytest.mark.parametrize("activation", ["relu", "tanh"])
def test_packed_matches_iterated_steps(activation):
    rng = np.random.default_rng(0)
    F, H, A = 5, 7, 3
    params = R.init_lstm_linear_params(rng, F, H, A)
    params[4 * H * F + 4 * H * H:4 * H * F + 4 * H * H + 8 * H] = rng.normal(size=8 * H) * 0.3
    episodes = [rng.normal(size=(n, F)) for n in (4, 1, 6, 6, 2)]
    packed = LO.lstm_packed_episodes(params, F, H, A, episodes, activation, torch.float64)
    for ep, got in zip(episodes, packed):
        want = LO.lstm_linear_episode(params, F, H, A, ep, activation, torch.float64)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    # the composed cell the autograd restatements differentiate is the same function
    prm = [t.to(torch.float64) for t in LO.unflatten_lstm_linear(params, F, H, A)]
    comp = LO.lstm_linear_forward(prm, TO.EpisodeBatch(episodes, torch.float64), activation).numpy()
    np.testing.assert_allclose(comp, np.concatenate(packed), rtol=1e-12, atol=1e-12)


def test_parameter_count_and_order_match_torch_lstm():
    F, H, A = 6, 4, 2
    torch.manual_seed(0)
    lstm, lin = torch.nn.LSTM(F, H, num_layers=1, bias=True), torch.nn.Linear(H, A)
    names = [n for n, _ in lstm.named_parameters()]
    assert names == ["weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"]
    flat = torch.cat([p.detach().reshape(-1) for p in list(lstm.parameters()) + [lin.weight, lin.bias]]).double().numpy()
    assert flat.size == R.lstm_linear_num_params(F, H, A) == 4 * H * (F + H) + 8 * H + A * H + A
    x = np.random.default_rng(1).normal(size=(5, F))
    with torch.no_grad():
        out, _ = lstm.double()(torch.tensor(x)[:, None, :])
        want = lin.double()(torch.relu(out[:, 0])).numpy()
    np.testing.assert_allclose(LO.lstm_linear_episode(flat, F, H, A, x, "relu", torch.float64), want, rtol=1e-12, atol=1e-12)


def test_init_follows_rnn_base_config_default():
    F, H, A = 6, 8, 3
    p = R.init_lstm_linear_params(np.random.default_rng(3), F, H, A)
    assert p.dtype == np.float32 and p.size == R.lstm_linear_num_params(F, H, A)
    w_ih, w_hh, b_ih, b_hh, lw, lb = [t.numpy().astype(np.float64) for t in LO.unflatten_lstm_linear(p, F, H, A)]
    assert np.abs(w_ih).max() <= np.sqrt(6.0 / (F + 4 * H))
    np.testing.assert_allclose(w_hh.T @ w_hh, np.eye(H), atol=1e-5)  # orthonormal columns of the [4H, H] matrix
    assert (b_ih == 0).all() and (b_hh == 0).all()
    lim = np.sqrt(6.0 / (H + 1 + A))
    assert np.abs(lw).max() <= lim and np.abs(lb).max() <= lim


def test_config_builds_the_lstm_module_type():
    cfg = R.LstmLinearConfig()
    assert cfg.hidden_dim == 128 and cfg.activation == "relu"
    assert issubclass(R.LstmLinear, R.modules.SeqLinear) and issubclass(R.GruLinear, R.modules.SeqLinear)
    assert not hasattr(R, "LstmMlpConfig")
