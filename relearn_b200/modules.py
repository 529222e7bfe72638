"""Mlp module (src/torch/modules/ff/mlp.rs) and the recurrent modules (GRU or LSTM, then a Linear) over the C ABI."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L
from .runtime import Context

ACTIVATIONS = {"identity": L.RL_ACT_IDENTITY, "relu": L.RL_ACT_RELU, "sigmoid": L.RL_ACT_SIGMOID, "tanh": L.RL_ACT_TANH}


@dataclass
class MlpConfig:
    """mlp.rs:25-34 defaults: hidden_sizes [128], Relu, output Identity."""

    hidden_sizes: list = field(default_factory=lambda: [128])
    activation: str = "relu"

    def build_module(self, ctx: Context, in_dim: int, out_dim: int) -> "Mlp":
        return Mlp(ctx, in_dim, self.hidden_sizes, out_dim, self.activation)


def _layer_dims(in_dim, hidden, out_dim):
    sizes = [hidden] if isinstance(hidden, (int, np.integer)) else list(hidden)
    dims = [in_dim] + [int(h) for h in sizes] + [out_dim]
    return list(zip(dims[:-1], dims[1:]))


def num_params(in_dim, hidden, out_dim):
    """`hidden`: MlpConfig::hidden_sizes (an int for one hidden layer)."""
    return sum(o * i + o for i, o in _layer_dims(in_dim, hidden, out_dim))


def init_params(rng: np.random.Generator, in_dim: int, hidden, out_dim: int) -> np.ndarray:
    """Initializer::Uniform(FanAvg) with Linear's fan_in = in_dim + 1 (initializers.rs:31-38,159-163;
    linear.rs:56): every tensor of a Linear ~ U(+-sqrt(6 / (in+1+out))).  libtorch's generator is not
    reproducible from relearn, so values come from numpy and are injected.  `hidden`: an int or hidden_sizes."""
    parts = []
    for (i, o) in _layer_dims(in_dim, hidden, out_dim):
        lim = np.sqrt(6.0 / (i + 1 + o))
        parts.append(rng.uniform(-lim, lim, size=(o, i)).astype(np.float32).ravel())
        parts.append(rng.uniform(-lim, lim, size=(o,)).astype(np.float32))
    return np.concatenate(parts)


class Mlp:
    def __init__(self, ctx: Context, in_dim: int, hidden_sizes, out_dim: int, activation: str = "relu"):
        self.ctx, self._lib = ctx, ctx._lib
        self.in_dim, self.hidden_sizes, self.out_dim = in_dim, list(hidden_sizes), out_dim
        hs = (C.c_int32 * len(self.hidden_sizes))(*self.hidden_sizes)
        h = C.c_void_p()
        L.check(self._lib.rl_mlp_create(ctx.handle, in_dim, hs, len(self.hidden_sizes), out_dim,
                                        ACTIVATIONS[activation], C.byref(h)), ctx.handle)
        self.handle = h
        n = C.c_uint64()
        L.check(self._lib.rl_mlp_num_params(h, C.byref(n)), ctx.handle)
        self.num_params = n.value

    def close(self):
        if self.handle and self.ctx.handle:
            self._lib.rl_mlp_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_weights(self, flat: np.ndarray):
        """Flat f32 in Module::variables() order (kernel[out,in] row-major, bias) per Linear."""
        a = np.ascontiguousarray(flat, dtype=np.float32)
        L.check(self._lib.rl_mlp_set_weights(self.handle, a.ctypes.data_as(C.c_void_p), a.size), self.ctx.handle)

    def set_weights_async(self, pinned: np.ndarray):
        """The same copy enqueued without a host round trip; `pinned` must be a page-locked f32 array
        (`Context.pinned_array`) that stays unchanged until the next synchronising call."""
        assert pinned.dtype == np.float32 and pinned.flags["C_CONTIGUOUS"]
        L.check(self._lib.rl_mlp_set_weights_async(self.handle, pinned.ctypes.data, pinned.size), self.ctx.handle)

    def get_weights(self) -> np.ndarray:
        a = np.empty(self.num_params, np.float32)
        L.check(self._lib.rl_mlp_get_weights(self.handle, a.ctypes.data_as(C.c_void_p), a.size), self.ctx.handle)
        return a

    def forward(self, x: np.ndarray) -> np.ndarray:
        """x [n, in_dim] -> [n, out_dim] (host convenience; uploads planes, downloads planes)."""
        x = np.ascontiguousarray(x, np.float32).reshape(-1, self.in_dim)
        n = x.shape[0]
        xin = self.ctx.to_device(np.ascontiguousarray(x.T))
        out = self.ctx.alloc(max(n, 1) * self.out_dim * 4)
        L.check(self._lib.rl_mlp_forward(self.handle, xin.c, n, out.c), self.ctx.handle)
        res = out.download((self.out_dim, n), np.float32).T.copy()
        xin.free()
        out.free()
        return res


# ------------------------------------------------------------------------------------------------
# Chain<Gru, Linear> (src/torch/modules/chain.rs, seq/rnn/gru.rs, ff/linear.rs)
# ------------------------------------------------------------------------------------------------
@dataclass
class GruLinearConfig:
    """ChainConfig<GruConfig, LinearConfig> (chain.rs:12-52): hidden_dim 128, activation between the two."""

    hidden_dim: int = 128
    activation: str = "relu"

    def build_module(self, ctx: Context, in_dim: int, out_dim: int) -> "GruLinear":
        return GruLinear(ctx, in_dim, self.hidden_dim, out_dim, self.activation)


def gru_linear_num_params(in_dim, hidden, out_dim):
    return 3 * hidden * in_dim + 3 * hidden * hidden + 6 * hidden + out_dim * hidden + out_dim


def init_gru_linear_params(rng: np.random.Generator, in_dim: int, hidden: int, out_dim: int) -> np.ndarray:
    """Weights shaped like the rl2 configuration (rl2-bandits.rs:379-393): input weights U(FanAvg), hidden weights
    orthogonal, zero biases; Linear as in `init_params`.  Values come from numpy and are injected."""
    lim = np.sqrt(6.0 / (in_dim + 3 * hidden))
    w_ih = rng.uniform(-lim, lim, size=(3 * hidden, in_dim))
    q, _ = np.linalg.qr(rng.normal(size=(3 * hidden, hidden)))
    lim2 = np.sqrt(6.0 / (hidden + 1 + out_dim))
    parts = [w_ih, q, np.zeros(3 * hidden), np.zeros(3 * hidden), rng.uniform(-lim2, lim2, size=(out_dim, hidden)),
             rng.uniform(-lim2, lim2, size=(out_dim,))]
    return np.concatenate([np.asarray(p, np.float32).ravel() for p in parts])


class SeqLinear:
    """The handle methods of a recurrent module -> activation -> Linear (one rl_grunet handle, GRU or LSTM cell).
    Subclasses name the create call."""

    _create = ""

    def __init__(self, ctx: Context, in_dim: int, hidden: int, out_dim: int, activation: str = "relu"):
        self.ctx, self._lib = ctx, ctx._lib
        self.in_dim, self.hidden, self.out_dim = in_dim, hidden, out_dim
        h = C.c_void_p()
        L.check(getattr(self._lib, self._create)(ctx.handle, in_dim, hidden, out_dim, ACTIVATIONS[activation], C.byref(h)),
                ctx.handle)
        self.handle = h
        n = C.c_uint64()
        L.check(self._lib.rl_grunet_num_params(h, C.byref(n)), ctx.handle)
        self.num_params = n.value

    def close(self):
        if self.handle and self.ctx.handle:
            self._lib.rl_grunet_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_weights(self, flat: np.ndarray):
        a = np.ascontiguousarray(flat, dtype=np.float32)
        L.check(self._lib.rl_grunet_set_weights(self.handle, a.ctypes.data_as(C.c_void_p), a.size), self.ctx.handle)

    def get_weights(self) -> np.ndarray:
        a = np.empty(self.num_params, np.float32)
        L.check(self._lib.rl_grunet_get_weights(self.handle, a.ctypes.data_as(C.c_void_p), a.size), self.ctx.handle)
        return a

    def seq_packed(self, traj) -> np.ndarray:
        """SeqPacked::seq_packed over the stored episodes of `traj`: returns [T, E, out_dim] (zeros in unused slots)."""
        v = traj.view()
        T, E = int(v.step_capacity), int(v.num_lanes)
        out = self.ctx.alloc(T * E * self.out_dim * 4)
        L.check(self._lib.rl_grunet_seq_forward(self.handle, traj.handle, out.c), self.ctx.handle)
        res = out.download((T, self.out_dim, E), np.float32).transpose(0, 2, 1).copy()
        out.free()
        return res


class GruLinear(SeqLinear):
    """One GRU layer -> activation -> Linear.  Flat parameters in Module::variables() order:
    w_ih[3H,in], w_hh[3H,H], b_ih[3H], b_hh[3H] (rnn/mod.rs:223-258), kernel[out,H], bias[out] (linear.rs:108-110)."""

    _create = "rl_grunet_create"


# ------------------------------------------------------------------------------------------------
# Chain<Lstm, Linear> (src/torch/modules/chain.rs, seq/rnn/lstm.rs, ff/linear.rs)
# ------------------------------------------------------------------------------------------------
@dataclass
class LstmLinearConfig:
    """ChainConfig<LstmConfig, LinearConfig>: one LSTM layer (hidden_dim 128), the activation, then a Linear."""

    hidden_dim: int = 128
    activation: str = "relu"

    def build_module(self, ctx: Context, in_dim: int, out_dim: int) -> "LstmLinear":
        return LstmLinear(ctx, in_dim, self.hidden_dim, out_dim, self.activation)


def lstm_linear_num_params(in_dim, hidden, out_dim):
    return 4 * hidden * in_dim + 4 * hidden * hidden + 8 * hidden + out_dim * hidden + out_dim


def init_lstm_linear_params(rng: np.random.Generator, in_dim: int, hidden: int, out_dim: int) -> np.ndarray:
    """RnnBaseConfig::default(): input weights U(+-sqrt(6 / (in + 4H))), hidden weights orthogonal [4H, H], zero biases;
    the Linear as in `init_params`.  Values come from numpy and are injected."""
    lim = np.sqrt(6.0 / (in_dim + 4 * hidden))
    w_ih = rng.uniform(-lim, lim, size=(4 * hidden, in_dim))
    q, _ = np.linalg.qr(rng.normal(size=(4 * hidden, hidden)))
    lim2 = np.sqrt(6.0 / (hidden + 1 + out_dim))
    parts = [w_ih, q, np.zeros(4 * hidden), np.zeros(4 * hidden), rng.uniform(-lim2, lim2, size=(out_dim, hidden)),
             rng.uniform(-lim2, lim2, size=(out_dim,))]
    return np.concatenate([np.asarray(p, np.float32).ravel() for p in parts])


class LstmLinear(SeqLinear):
    """One LSTM layer -> activation -> Linear.  Flat parameters in Module::variables() order:
    w_ih[4H,in], w_hh[4H,H], b_ih[4H], b_hh[4H] (gate order i, f, g, o), kernel[out,H], bias[out]."""

    _create = "rl_lstmnet_create"
