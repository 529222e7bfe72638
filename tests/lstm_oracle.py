"""Torch-CPU restatement of Chain<Lstm, Linear> (src/torch/modules/seq/rnn/lstm.rs, chain.rs, ff/linear.rs) and of the
updates that run through it: the LSTM counterparts of oracle/tensor_oracle.py's GRU functions, built on the same pieces
(Categorical, HessianVectorProduct, the trust-region step, Adam112, EpisodeBatch).  TEST INFRASTRUCTURE ONLY.

libtorch's lstm_cell, what the reference's Lstm evaluates per step (gate order i, f, g, o):
    gates = (W_ih x + b_ih) + (W_hh h + b_hh);  c' = sigmoid(f) c + sigmoid(i) tanh(g);  h' = sigmoid(o) tanh(c')
(h, c) are zero at the start of every episode.  Flat parameters in Module::variables() order:
w_ih[4H,in], w_hh[4H,H], b_ih[4H], b_hh[4H], kernel[out,H], bias[out]."""
from __future__ import annotations

import numpy as np
import torch

from oracle import tensor_oracle as TO

ACT = {"relu": torch.relu, "identity": lambda t: t, "tanh": torch.tanh, "sigmoid": torch.sigmoid}


def unflatten_lstm_linear(flat, n_in, hidden, n_out):
    flat = torch.as_tensor(np.asarray(flat))
    sizes = [(4 * hidden, n_in), (4 * hidden, hidden), (4 * hidden,), (4 * hidden,), (n_out, hidden), (n_out,)]
    out, off = [], 0
    for sh in sizes:
        n = int(np.prod(sh))
        out.append(flat[off:off + n].reshape(sh))
        off += n
    assert off == flat.numel()
    return out


def lstm_linear_episode(flat, n_in, hidden, n_out, obs, activation="relu", dtype=torch.float32):
    """SeqIterative::step over one episode: (h, c) = 0, per step (h, c) = lstm_cell(x, (h, c)), out = Linear(act(h)).
    obs [L, F] -> [L, out]."""
    w_ih, w_hh, b_ih, b_hh, lw, lb = [t.to(dtype) for t in unflatten_lstm_linear(flat, n_in, hidden, n_out)]
    x = torch.tensor(np.asarray(obs), dtype=dtype)
    h = torch.zeros(1, hidden, dtype=dtype)
    c = torch.zeros(1, hidden, dtype=dtype)
    outs = []
    for t in range(x.shape[0]):
        h, c = torch.lstm_cell(x[t:t + 1], (h, c), w_ih, w_hh, b_ih, b_hh)
        outs.append(torch.nn.functional.linear(ACT[activation](h), lw, lb)[0])
    return torch.stack(outs).numpy() if outs else np.zeros((0, n_out), np.float32)


def lstm_packed_episodes(flat, n_in, hidden, n_out, episodes, activation="relu", dtype=torch.float32):
    """SeqPacked::seq_packed: the functional packed `lstm` over pack_sequence(episodes) with the given weights; returns the
    per-episode outputs, unpacked again, so that packed == iterated can be checked (modules/testing.rs:124-157)."""
    w_ih, w_hh, b_ih, b_hh, lw, lb = [t.to(dtype) for t in unflatten_lstm_linear(flat, n_in, hidden, n_out)]
    order = sorted(range(len(episodes)), key=lambda i: -len(episodes[i]))
    seqs = [torch.tensor(np.asarray(episodes[i]), dtype=dtype) for i in order]
    packed = torch.nn.utils.rnn.pack_sequence(seqs, enforce_sorted=True)
    z = torch.zeros(1, len(seqs), hidden, dtype=dtype)
    out, _, _ = torch._VF.lstm(packed.data, packed.batch_sizes, (z, z), [w_ih, w_hh, b_ih, b_hh], True, 1, 0.0, True, False)
    logits = torch.nn.functional.linear(ACT[activation](out), lw, lb)
    unpacked, lens = torch.nn.utils.rnn.pad_packed_sequence(
        torch.nn.utils.rnn.PackedSequence(logits, packed.batch_sizes), batch_first=True)
    res = [None] * len(episodes)
    for k, i in enumerate(order):
        res[i] = unpacked[k, :int(lens[k])].numpy()
    return res


def lstm_linear_forward(params, batch: TO.EpisodeBatch, activation="relu"):
    """The composed lstm_cell over padded episodes (autograd differentiates it twice for the Fisher-vector product)."""
    w_ih, w_hh, b_ih, b_hh, lw, lb = params
    B, Lmax, _ = batch.obs.shape
    h = torch.zeros(B, w_hh.shape[1], dtype=batch.obs.dtype)
    c = torch.zeros_like(h)
    outs = []
    for t in range(Lmax):
        gates = torch.nn.functional.linear(batch.obs[:, t], w_ih, b_ih) + torch.nn.functional.linear(h, w_hh, b_hh)
        i, f, g, o = gates.chunk(4, 1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
        h = torch.sigmoid(o) * torch.tanh(c)
        outs.append(torch.nn.functional.linear(ACT[activation](h), lw, lb))
    return batch.select(torch.stack(outs, dim=1))


def seq_params(flat_params, n_in, hidden, n_out, dtype):
    flat = torch.tensor(np.asarray(flat_params), dtype=dtype)
    return [p.clone().requires_grad_(True) for p in unflatten_lstm_linear(flat, n_in, hidden, n_out)]


def _cat(xs, dtype):
    return torch.tensor(np.concatenate([np.asarray(x) for x in xs]), dtype=dtype)


def seq_policy_loss_kl_grad_fvp(flat_params, n_in, hidden, n_out, episodes, actions, advantages, vector, reg=0.0,
                                dtype=torch.float64, activation="relu"):
    """TO.seq_policy_loss_kl_grad_fvp for the LSTM chain: loss, kl, entropy, grad, (H + reg I) v."""
    params = seq_params(flat_params, n_in, hidden, n_out, dtype)
    batch = TO.EpisodeBatch(episodes, dtype)
    act_t, adv_t = _cat(actions, torch.int64), _cat(advantages, dtype)
    with torch.no_grad():
        dist0 = TO.Categorical(lstm_linear_forward(params, batch, activation))
        logp0 = dist0.log_prob(act_t)
        entropy = float(dist0.entropy().mean())
    dist = TO.Categorical(lstm_linear_forward(params, batch, activation))
    loss = -((dist.log_prob(act_t) - logp0).exp() * adv_t).mean()
    kl = dist0.kl_divergence_from(dist).mean()
    g = TO.flatten_tensors(torch.autograd.grad(loss, params, retain_graph=True))
    hv = TO.HessianVectorProduct(kl, params, reg).mat_vec_mul(torch.tensor(np.asarray(vector), dtype=dtype))
    return float(loss.detach()), float(kl.detach()), entropy, g.detach().numpy(), hv.detach().numpy()


def seq_trpo_update(flat_params, n_in, hidden, n_out, episodes, actions, advantages, max_kl=0.01,
                    cfg: TO.CgConfig | None = None, dtype=torch.float32, activation="relu"):
    cfg = cfg or TO.CgConfig()
    params = seq_params(flat_params, n_in, hidden, n_out, dtype)
    batch = TO.EpisodeBatch(episodes, dtype)
    act_t, adv_t = _cat(actions, torch.int64), _cat(advantages, dtype)
    log = {}
    with torch.no_grad():
        dist0 = TO.Categorical(lstm_linear_forward(params, batch, activation))
        logp0 = dist0.log_prob(act_t)
        log["entropy"] = float(dist0.entropy().mean())

    def loss_distance_fn():
        dist = TO.Categorical(lstm_linear_forward(params, batch, activation))
        loss = -((dist.log_prob(act_t) - logp0).exp() * adv_t).mean()
        return loss, dist0.kl_divergence_from(dist).mean()

    log["error"] = None
    try:
        TO.trust_region_backward_step(params, loss_distance_fn, max_kl, cfg, log)
    except TO.OptimizerStepError as e:
        log["error"] = e.kind
    return TO.flatten_tensors([p.detach() for p in params]).numpy().copy(), log


def seq_value_update(flat_params, n_in, hidden, episodes, targets, n_steps=80, lr=1e-3, dtype=torch.float32,
                     activation="relu"):
    params = seq_params(flat_params, n_in, hidden, 1, dtype)
    opt = TO.Adam112(params, lr)
    batch = TO.EpisodeBatch(episodes, dtype)
    tgt_t = _cat(targets, dtype)
    losses = []
    for _ in range(n_steps):
        v = lstm_linear_forward(params, batch, activation).squeeze(-1)
        loss = torch.nn.functional.mse_loss(v, tgt_t, reduction="mean")
        opt.step(torch.autograd.grad(loss, params))
        losses.append(float(loss.detach()))
    return TO.flatten_tensors([p.detach() for p in params]).numpy().copy(), losses


def seq_q_loss_grad(flat_params, n_in, hidden, n_out, episodes, actions, targets, dtype=torch.float64, activation="relu"):
    """mse(Q(obs).gather(action), targets) over the episodes (dqn.rs:316-326): loss and flat gradient."""
    params = seq_params(flat_params, n_in, hidden, n_out, dtype)
    q = lstm_linear_forward(params, TO.EpisodeBatch(episodes, dtype), activation)
    act = _cat(actions, torch.int64).unsqueeze(-1)
    loss = torch.nn.functional.mse_loss(q.gather(-1, act).squeeze(-1), _cat(targets, dtype), reduction="mean")
    return float(loss.detach()), TO.flatten_tensors(torch.autograd.grad(loss, params)).numpy()


def seq_q_values(flat_params, n_in, hidden, n_out, episodes, dtype=torch.float64, activation="relu"):
    """Q on each episode [L_i, F] -> list of [L_i, out]."""
    prm = [t.to(dtype) for t in unflatten_lstm_linear(torch.tensor(np.asarray(flat_params)), n_in, hidden, n_out)]
    out = lstm_linear_forward(prm, TO.EpisodeBatch(episodes, dtype), activation).detach().numpy()
    res, pos = [], 0
    for x in episodes:
        res.append(out[pos:pos + len(x)])
        pos += len(x)
    return res
