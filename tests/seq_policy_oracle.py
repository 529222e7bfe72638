"""Torch-CPU restatement of Ppo::update (src/torch/agents/policies/ppo.rs:97-147) and Reinforce::update (reinforce.rs:64-89)
with a recurrent policy, over packed episodes: oracle/tensor_oracle.py's ppo_update / reinforce_update with an EpisodeBatch
in place of the flat Mlp batch.  TEST INFRASTRUCTURE ONLY.

Both take the module's unflatten and forward functions, so that one restatement serves every cell:
  GRU:  tensor_oracle.unflatten_gru_linear, tensor_oracle.gru_linear_forward   (CELLS["gru"])
  LSTM: lstm_oracle.unflatten_lstm_linear, lstm_oracle.lstm_linear_forward     (CELLS["lstm"])
episodes / actions / advantages are per-episode arrays ([L_i, F], [L_i], [L_i])."""
from __future__ import annotations

import numpy as np
import torch

from oracle import tensor_oracle as TO
from tests import lstm_oracle as LO

CELLS = {"gru": (TO.unflatten_gru_linear, TO.gru_linear_forward), "lstm": (LO.unflatten_lstm_linear, LO.lstm_linear_forward)}


def _inputs(unflatten, flat_params, n_in, hidden, n_out, episodes, actions, advantages, dtype):
    flat = torch.tensor(np.asarray(flat_params), dtype=dtype)
    params = [p.clone().requires_grad_(True) for p in unflatten(flat, n_in, hidden, n_out)]
    act = torch.tensor(np.concatenate([np.asarray(a) for a in actions]), dtype=torch.int64)
    adv = torch.tensor(np.concatenate([np.asarray(a) for a in advantages]), dtype=dtype)
    return params, TO.EpisodeBatch(episodes, dtype), act, adv


def seq_ppo_update(unflatten, forward, flat_params, n_in, hidden, n_out, episodes, actions, advantages, opt_steps=10,
                   clip_distance=0.2, lr=1e-3, dtype=torch.float32, activation="relu"):
    """no_grad initial log-probs and entropy, then opt_steps x Adam on -mean(min(ratio adv, clip(ratio) adv)).
    Returns (new flat params, per-step losses, entropy, per-step share of samples on the clipped branch, where the
    surrogate's gradient is zero)."""
    params, batch, act, adv = _inputs(unflatten, flat_params, n_in, hidden, n_out, episodes, actions, advantages, dtype)
    opt = TO.Adam112(params, lr)
    with torch.no_grad():
        d0 = TO.Categorical(forward(params, batch, activation))
        lp0 = d0.log_prob(act)
        entropy = float(d0.entropy().mean())
    losses, clipped_share = [], []
    lo, hi = 1.0 - clip_distance, 1.0 + clip_distance
    for _ in range(opt_steps):
        lp = TO.Categorical(forward(params, batch, activation)).log_prob(act)
        ratio = (lp - lp0).exp()
        clipped = ratio.clip(lo, hi)
        loss = -torch.minimum(ratio * adv, clipped * adv).mean()
        with torch.no_grad():
            flat = ~(((ratio >= lo) & (ratio <= hi)) | (ratio * adv < clipped * adv))
            clipped_share.append(float(flat.to(dtype).mean()))
        opt.step(torch.autograd.grad(loss, params))
        losses.append(float(loss.detach()))
    return TO.flatten_tensors([p.detach() for p in params]).numpy().copy(), losses, entropy, clipped_share


def seq_reinforce_update(unflatten, forward, flat_params, n_in, hidden, n_out, episodes, actions, advantages, lr=1e-3,
                         dtype=torch.float32, activation="relu"):
    """One Adam step on -(log_probs * advantages).mean(); returns (new flat params, loss, entropy of that evaluation)."""
    params, batch, act, adv = _inputs(unflatten, flat_params, n_in, hidden, n_out, episodes, actions, advantages, dtype)
    opt = TO.Adam112(params, lr)
    dist = TO.Categorical(forward(params, batch, activation))
    loss = -(dist.log_prob(act) * adv).mean()
    entropy = float(dist.entropy().mean().detach())
    opt.step(torch.autograd.grad(loss, params))
    return TO.flatten_tensors([p.detach() for p in params]).numpy().copy(), float(loss.detach()), entropy
