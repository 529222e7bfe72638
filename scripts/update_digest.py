"""Fingerprint of every update entry point, run from fixed seeds on one GPU.

For each run it prints a SHA-256 of what the run leaves behind (the module's parameters, the Adam moments and step count,
every statistics field but the timings; for a probe, everything it returns) and then the kernels the run launched, in
launch order, with their grids (torch.profiler; a block of launches repeated N times is written once under "xN").  Two builds that compute the same thing and
launch the same kernels print the same text, so a change to the host code around the updates can be shown to move
neither a bit nor a launch: run the script on both builds and diff the outputs.

Covered: TRPO update and probe, critic update, critic probe on both pass kernels, PPO, REINFORCE, DQN with reward-to-go
and one-step TD targets, on the default 5-128 modules (once on the tensor-core pass kernel and once on its FP32-pipe twin,
rl_pass_kernel_select(RL_PASS_KERNEL_FFMA)) and on a two-hidden-layer tanh Mlp; TRPO update and probe, critic update,
DQN update and probe on GRU and LSTM modules of hidden 8 and 128.

usage: python scripts/update_digest.py > digest.txt
"""
import ctypes as C
import hashlib
import json
import os
import re
import struct
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

import relearn_b200 as R
from relearn_b200 import _lib as L

E, T = 512, 48
ADAM = R.AdamConfig(learning_rate=3e-3, beta1=0.85, beta2=0.995, weight_decay=1e-4, eps=1e-7)


def sha(*parts) -> str:
    h = hashlib.sha256()
    for p in parts:
        h.update(np.ascontiguousarray(p).tobytes() if isinstance(p, np.ndarray) else repr(p).encode())
    return h.hexdigest()


def fields(stats) -> list:
    """Every field of a stats struct except the device timings."""
    return [(n, getattr(stats, n)) for n, _ in stats._fields_ if not n.endswith("_ms")]


def adam_state(ctx, opt, P):
    """Moments and step count of an optimizer.  rl_adam is opaque in the C ABI: its moment pointers and step count follow
    the stored rl_adam_cfg, which is found by its values (distinct from any pointer)."""
    base = opt.handle.value
    word = lambda k: C.c_uint64.from_address(base + 8 * k).value
    dbl = lambda k: struct.unpack("<d", struct.pack("<Q", word(k)))[0]
    cfg = [ADAM.learning_rate, ADAM.beta1, ADAM.beta2, ADAM.weight_decay, ADAM.eps]
    k = next(k for k in range(8) if all(dbl(k + i) == c for i, c in enumerate(cfg)))
    return ctx.read(word(k + 5), (P,), np.float32), ctx.read(word(k + 6), (P,), np.float32), word(k + 7)


class Digest:
    def __init__(self, ctx):
        self.ctx, self.lines = ctx, []

    def run(self, name, fn):
        """fn() runs the entry point and returns what to hash."""
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            torch.zeros(1, device="cuda")  # the profiler can miss a window's first kernel
            torch.cuda.synchronize()
            out = fn()
            self.ctx.synchronize()
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(path)
            events = json.load(open(path))["traceEvents"]
        kernels = sorted((e for e in events if e.get("cat") == "kernel" and "at::native" not in e["name"]), key=lambda e: e["ts"])
        launches = [f"{kernel_name(e['name'])} grid={list(e['args'].get('grid', ()))}" for e in kernels]
        self.lines.append(f"{name}: {sha(*out)} ({len(launches)} kernels)")
        print(self.lines[-1], file=sys.stderr)
        for block, n in fold(launches):
            if len(block) == 1:
                self.lines.append(f"    {block[0]}" + (f" x{n}" if n > 1 else ""))
            else:
                self.lines.append(f"    x{n}:")
                self.lines += [f"        {k}" for k in block]


def kernel_name(demangled: str) -> str:
    """The function and its template arguments."""
    name = demangled.replace("(anonymous namespace)::", "")
    name = re.sub(r"^void ", "", name)
    return name[:name.index("(")] if "(" in name else name


def fold(seq, max_block=4):
    """Consecutive repeats of a block of up to max_block launches, as (block, repeats): the launch order, written short."""
    out, i = [], 0
    while i < len(seq):
        best_len, best_n = 1, 1
        for L in range(1, max_block + 1):
            n = 1
            while seq[i + n * L:i + (n + 1) * L] == seq[i:i + L]:
                n += 1
            if n > 1 and n * L > best_len * best_n:
                best_len, best_n = L, n
        out.append((seq[i:i + best_len], best_n))
        i += best_len * best_n
    return out


def mlp_runs(d, ctx, lib, env, traj, hidden, act, tag):
    rng = np.random.default_rng(11)
    F, A = 5, 2
    adv = ctx.to_device(rng.normal(size=(T, E)).astype(np.float32))
    tgt = ctx.to_device((rng.normal(size=(T, E)) * 3.0).astype(np.float32))

    def module(out_dim, seed):
        m = R.Mlp(ctx, F, hidden, out_dim, act)
        m.set_weights(R.init_params(np.random.default_rng(seed), F, hidden, out_dim))
        return m

    def trpo_update():
        p, s = module(A, 1), L.TrpoStats()
        cfg = L.TrpoCfg()
        lib.rl_trpo_cfg_default(C.byref(cfg))
        st = L.check(lib.rl_trpo_update(traj.handle, adv.c, p.handle, C.byref(cfg), C.byref(s)), ctx.handle)
        return p.get_weights(), st, fields(s)

    def trpo_probe():
        p = module(A, 2)
        P = p.num_params
        vec = np.random.default_rng(12).normal(size=P).astype(np.float32)
        loss, kl, ent = C.c_double(), C.c_double(), C.c_double()
        grad, fvp = np.zeros(P, np.float32), np.zeros(P, np.float32)
        L.check(lib.rl_trpo_probe(traj.handle, adv.c, p.handle, vec.ctypes.data_as(C.c_void_p), 1e-5, C.byref(loss),
                                  C.byref(kl), C.byref(ent), grad.ctypes.data_as(C.c_void_p), fvp.ctypes.data_as(C.c_void_p)),
                ctx.handle)
        return loss.value, kl.value, ent.value, grad, fvp

    def value_update():
        v, s = module(1, 3), L.OptStats()
        opt = R.Adam(v, ADAM)
        L.check(lib.rl_value_update(traj.handle, tgt.c, v.handle, opt.handle, 6, C.byref(s)), ctx.handle)
        return (v.get_weights(), *adam_state(ctx, opt, v.num_params), fields(s))

    def value_probe(kernel):
        def run():
            v = module(1, 4)
            loss, grad = C.c_double(), np.zeros(v.num_params, np.float32)
            L.check(lib.rl_value_probe(traj.handle, tgt.c, v.handle, kernel, C.byref(loss), grad.ctypes.data_as(C.c_void_p)),
                    ctx.handle)
            return loss.value, grad
        return run

    def policy_adam(ppo):
        def run():
            p, s = module(A, 5), L.PolicyOptStats()
            opt = R.Adam(p, ADAM)
            if ppo:
                cfg = L.PpoCfg(4, 0.2)
                L.check(lib.rl_ppo_update(traj.handle, adv.c, p.handle, opt.handle, C.byref(cfg), C.byref(s)), ctx.handle)
            else:
                L.check(lib.rl_reinforce_update(traj.handle, adv.c, p.handle, opt.handle, C.byref(s)), ctx.handle)
            return (p.get_weights(), *adam_state(ctx, opt, p.num_params), fields(s))
        return run

    def dqn(td):
        def run():
            q, s = module(A, 6), L.OptStats()
            opt = R.Adam(q, ADAM)
            cfg = L.DqnCfg(700, 4, int(td), np.float32(0.97), 21)
            L.check(lib.rl_dqn_update(rb.handle, q.handle, opt.handle, C.byref(cfg), C.byref(s)), ctx.handle)
            return (q.get_weights(), *adam_state(ctx, opt, q.num_params), fields(s))
        return run

    rb = R.ReplayBuffer(env, 200)
    rb.write_experience(traj)
    d.run(f"{tag} rl_trpo_update", trpo_update)
    d.run(f"{tag} rl_trpo_probe", trpo_probe)
    d.run(f"{tag} rl_value_update", value_update)
    d.run(f"{tag} rl_value_probe tcgen05", value_probe(L.RL_PASS_KERNEL_TCGEN05))
    d.run(f"{tag} rl_value_probe ffma", value_probe(L.RL_PASS_KERNEL_FFMA))
    d.run(f"{tag} rl_ppo_update", policy_adam(True))
    d.run(f"{tag} rl_reinforce_update", policy_adam(False))
    d.run(f"{tag} rl_dqn_update reward-to-go", dqn(False))
    d.run(f"{tag} rl_dqn_update one-step-td", dqn(True))


def seq_runs(d, ctx, lib, env, traj, hidden, cls, init, tag):
    rng = np.random.default_rng(23)
    F, A = 5, 2
    adv = ctx.to_device(rng.normal(size=(T, E)).astype(np.float32))
    tgt = ctx.to_device((rng.normal(size=(T, E)) * 3.0).astype(np.float32))
    tag = f"{tag}-{hidden}"

    def module(out_dim, seed):
        g = cls(ctx, F, hidden, out_dim)
        g.set_weights(init(np.random.default_rng(seed), F, hidden, out_dim).astype(np.float32))
        return g

    def trpo_update():
        p, s = module(A, 1), L.TrpoStats()
        cfg = L.TrpoCfg()
        lib.rl_trpo_cfg_default(C.byref(cfg))
        st = L.check(lib.rl_trpo_update_seq(traj.handle, adv.c, p.handle, C.byref(cfg), C.byref(s)), ctx.handle)
        return p.get_weights(), st, fields(s)

    def trpo_probe():
        p = module(A, 2)
        P = p.num_params
        vec = np.random.default_rng(12).normal(size=P).astype(np.float32)
        loss, kl, ent = C.c_double(), C.c_double(), C.c_double()
        grad, fvp = np.zeros(P, np.float32), np.zeros(P, np.float32)
        L.check(lib.rl_trpo_probe_seq(traj.handle, adv.c, p.handle, vec.ctypes.data_as(C.c_void_p), 1e-5, C.byref(loss),
                                      C.byref(kl), C.byref(ent), grad.ctypes.data_as(C.c_void_p),
                                      fvp.ctypes.data_as(C.c_void_p)), ctx.handle)
        return loss.value, kl.value, ent.value, grad, fvp

    def value_update():
        v, s = module(1, 3), L.OptStats()
        opt = R.Adam(v, ADAM)
        L.check(lib.rl_value_update_seq(traj.handle, tgt.c, v.handle, opt.handle, 4, C.byref(s)), ctx.handle)
        return (v.get_weights(), *adam_state(ctx, opt, v.num_params), fields(s))

    def dqn(td):
        def run():
            q, s = module(A, 6), L.OptStats()
            opt = R.Adam(q, ADAM)
            cfg = L.DqnCfg(700, 3, int(td), np.float32(0.97), 21)
            L.check(lib.rl_dqn_update_seq(rb.handle, q.handle, opt.handle, C.byref(cfg), C.byref(s)), ctx.handle)
            return (q.get_weights(), *adam_state(ctx, opt, q.num_params), fields(s))
        return run

    def dqn_probe(td):
        def run():
            q = module(A, 7)
            cfg = L.DqnCfg(700, 1, int(td), np.float32(0.97), 21)
            loss, grad = C.c_double(), np.zeros(q.num_params, np.float32)
            L.check(lib.rl_dqn_probe_seq(rb.handle, C.byref(cfg), q.handle, 5, C.byref(loss), grad.ctypes.data_as(C.POINTER(C.c_float))),
                    ctx.handle)
            return loss.value, grad
        return run

    rb = R.ReplayBuffer(env, 200)
    rb.write_experience(traj)
    d.run(f"{tag} rl_trpo_update_seq", trpo_update)
    d.run(f"{tag} rl_trpo_probe_seq", trpo_probe)
    d.run(f"{tag} rl_value_update_seq", value_update)
    d.run(f"{tag} rl_dqn_update_seq reward-to-go", dqn(False))
    d.run(f"{tag} rl_dqn_update_seq one-step-td", dqn(True))
    d.run(f"{tag} rl_dqn_probe_seq reward-to-go", dqn_probe(False))
    d.run(f"{tag} rl_dqn_probe_seq one-step-td", dqn_probe(True))


def main():
    torch.zeros(1, device="cuda")
    ctx = R.Context(0)
    lib = ctx._lib
    L.check(lib.rl_pass_kernel_select(L.RL_PASS_KERNEL_TCGEN05))
    env = R.build_env(ctx, R.CartPoleConfig().wrap(R.VisibleStepLimit(40)), E, seed=7)
    env.set_noise_philox(7, 0)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_RANDOM), R.HistoryDataBound(T, 0), traj)
    d = Digest(ctx)
    mlp_runs(d, ctx, lib, env, traj, [128], "relu", "mlp-5-128")
    L.check(lib.rl_pass_kernel_select(L.RL_PASS_KERNEL_FFMA))
    mlp_runs(d, ctx, lib, env, traj, [128], "relu", "mlp-5-128-ffma")
    L.check(lib.rl_pass_kernel_select(L.RL_PASS_KERNEL_TCGEN05))
    mlp_runs(d, ctx, lib, env, traj, [32, 32], "tanh", "mlp-5-32x32-tanh")
    for hidden in (8, 128):
        seq_runs(d, ctx, lib, env, traj, hidden, R.GruLinear, R.init_gru_linear_params, "gru")
    for hidden in (8, 128):
        seq_runs(d, ctx, lib, env, traj, hidden, R.LstmLinear, R.init_lstm_linear_params, "lstm")
    print("\n".join(d.lines))


if __name__ == "__main__":
    main()
