"""The f64 recurrent-update oracles of oracle/tensor_oracle.py (Chain<Gru, Linear>) and tests/lstm_oracle.py
(Chain<Lstm, Linear>) over trajectories too large for one padded batch.  TEST INFRASTRUCTURE ONLY.

Those oracles pad every episode of a batch to the longest one and differentiate the whole batch at once, which does not
fit in memory at 10^5 .. 10^6 lane-steps.  The quantities the recurrent passes compute are means over all stored steps,
so they split over any partition of the episodes: with N steps in all and n_c in chunk c,
    loss = sum_c (n_c / N) loss_c,   entropy, KL and the gradient of the mean loss likewise,
    (H + reg I) v = sum_c (n_c / N) (H_c + reg I) v   (the chunk weights add up to 1, so reg is counted once).
This module cuts a trajectory's planes [T, E] into episodes, calls the existing oracle on chunks of them and combines the
results that way.  It restates no cell: every forward and backward pass is the wrapped oracle's own."""
from __future__ import annotations

import numpy as np
import torch

from oracle import tensor_oracle as TO
from relearn_b200 import _lib as L
from tests import lstm_oracle as LO

CONT, INTR, PAD = L.RL_CONTINUE, L.RL_INTERRUPT, L.RL_PAD

_PROBE = {"gru": TO.seq_policy_loss_kl_grad_fvp, "lstm": LO.seq_policy_loss_kl_grad_fvp}
_FORWARD = {"gru": TO.gru_linear_forward, "lstm": LO.lstm_linear_forward}
_UNFLATTEN = {"gru": TO.unflatten_gru_linear, "lstm": LO.unflatten_lstm_linear}


def episode_spans(succ):
    """Episodes of a trajectory's succ plane [T, E] as (lane, first step, end step) in lane order: a step whose succ is not
    CONTINUE ends an episode, the first PAD ends the lane (a lane may have no steps at all), and steps left open when the
    lane ends form one more episode."""
    succ = np.asarray(succ)
    T, E = succ.shape
    spans = []
    for e in range(E):
        col = succ[:, e]
        pads = np.flatnonzero(col == PAD)
        n = int(pads[0]) if len(pads) else T
        ends = np.flatnonzero(col[:n] != CONT) + 1
        if n > 0 and (len(ends) == 0 or ends[-1] != n):
            ends = np.append(ends, n)
        a = 0
        for b in ends:
            spans.append((e, a, int(b)))
            a = int(b)
    return spans


def chunks(spans, max_cells):
    """Groups of spans, longest episodes first, each group's padded batch (episodes x longest episode) at most max_cells
    cells (a longer episode goes alone)."""
    order = sorted(spans, key=lambda s: -(s[2] - s[1]))
    out, cur = [], []
    for s in order:
        if cur and (len(cur) + 1) * (cur[0][2] - cur[0][1]) > max_cells:
            out.append(cur)
            cur = []
        cur.append(s)
    if cur:
        out.append(cur)
    return out


def _take(x, group):
    return [x[a:b, e] for e, a, b in group]


def policy_loss_kl_grad_fvp(cell, flat_params, n_in, hidden, n_out, obs, action, adv, succ, vector, reg=0.0,
                            dtype=torch.float64, activation="relu", max_cells=65536):
    """TO / LO.seq_policy_loss_kl_grad_fvp over the episodes of the planes obs [T, E, F], action / adv / succ [T, E]:
    loss, kl, entropy, grad, (H + reg I) v of the means over all stored steps."""
    spans = episode_spans(succ)
    N = sum(b - a for _, a, b in spans)
    loss = kl = ent = 0.0
    g = hv = 0.0
    for group in chunks(spans, max_cells):
        w = sum(b - a for _, a, b in group) / N
        r = _PROBE[cell](flat_params, n_in, hidden, n_out, _take(obs, group), _take(action, group), _take(adv, group),
                         vector, reg, dtype, activation)
        loss, kl, ent = loss + w * r[0], kl + w * r[1], ent + w * r[2]
        g, hv = g + w * r[3].astype(np.float64), hv + w * r[4].astype(np.float64)
    return loss, kl, ent, g, hv


def outputs(cell, flat_params, n_in, hidden, n_out, obs, succ, next_obs=None, dtype=torch.float64, activation="relu",
            max_cells=65536):
    """The module's outputs on every stored step, out [T, E, n_out] (zeros elsewhere), each episode from a zero state.
    With next_obs, also out_next [T, E, n_out]: at the last step of an episode that ends in Interrupt, the output on its
    successor observation as one more step of the same sequence (what GAE bootstraps from), zeros elsewhere."""
    succ = np.asarray(succ)
    T, E = succ.shape
    out = np.zeros((T, E, n_out))
    out_next = np.zeros((T, E, n_out)) if next_obs is not None else None
    prm = [t.to(dtype) for t in _UNFLATTEN[cell](torch.tensor(np.asarray(flat_params)), n_in, hidden, n_out)]
    for group in chunks(episode_spans(succ), max_cells):
        eps = []
        for e, a, b in group:
            x = obs[a:b, e]
            if next_obs is not None and succ[b - 1, e] == INTR:
                x = np.concatenate([x, next_obs[b - 1:b, e]])
            eps.append(x)
        with torch.no_grad():
            y = _FORWARD[cell](prm, TO.EpisodeBatch(eps, dtype), activation).numpy()
        pos = 0
        for (e, a, b), x in zip(group, eps):
            out[a:b, e] = y[pos:pos + b - a]
            if len(x) > b - a:
                out_next[b - 1, e] = y[pos + b - a]
            pos += len(x)
    return (out, out_next) if next_obs is not None else out
