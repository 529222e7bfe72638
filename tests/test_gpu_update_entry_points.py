"""GPU: what every update entry point refuses, for Mlp and recurrent (Chain<Gru, Linear>) modules alike, and the kernel
choice of rl_value_probe staying with that one call.

Each refusal is checked by its status alone (the messages are free to change): NULL arguments, an optimizer built for
another module (an Mlp optimizer given to a recurrent entry point and the reverse included), optimizer step counts out of
range, a state-value module with two outputs, a module of another context, a module whose feature count does not match
the batch, and an unknown pass kernel."""
import ctypes as C
import re
from types import SimpleNamespace

import numpy as np
import pytest

import relearn_b200 as R
from relearn_b200 import _lib as L

pytestmark = pytest.mark.gpu

INVALID, UNSUPPORTED = L.RL_ERR_INVALID_ARG, L.RL_ERR_UNSUPPORTED
E, T = 64, 16


@pytest.fixture(scope="module")
def w(ctx):
    env = R.build_env(ctx, R.CartPoleConfig().wrap(R.VisibleStepLimit(20)), E, seed=3)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_RANDOM), R.HistoryDataBound(T, 0), traj)
    rng = np.random.default_rng(0)
    n = SimpleNamespace(ctx=ctx, env=env, traj=traj.handle, keep=[traj], lib=ctx._lib)
    n.adv = ctx.to_device(rng.normal(size=(T, E)).astype(np.float32))
    n.tgt = ctx.to_device(rng.normal(size=(T, E)).astype(np.float32))
    n.rb = R.ReplayBuffer(env, 50)

    def mlp(F, hidden, A):
        m = R.Mlp(ctx, F, [hidden], A)
        m.set_weights(R.init_params(rng, F, hidden, A))
        n.keep.append(m)
        return m

    def gru(F, hidden, A, c=ctx):
        g = R.GruLinear(c, F, hidden, A)
        g.set_weights(R.init_gru_linear_params(rng, F, hidden, A).astype(np.float32))
        n.keep.append(g)
        return g

    n.mlp, n.gru = mlp, gru
    n.policy, n.value, n.gpolicy, n.gvalue = mlp(5, 128, 2), mlp(5, 128, 1), gru(5, 8, 2), gru(5, 8, 1)
    n.ctx2 = R.Context(0)
    n.keep.append(n.ctx2)
    return n


def adam(w, module):
    a = R.Adam(module, R.AdamConfig())
    w.keep.append(a)
    return a.handle


def each_null(fn, args, pointers):
    """Every pointer argument in `pointers` replaced by NULL in turn: the status of each call."""
    return [fn(*[None if i == k else a for i, a in enumerate(args)]) for k in pointers]


def test_null_arguments(w):
    lib, b = w.lib, C.byref
    trpo_cfg, stats, opt, pstats = L.TrpoCfg(), L.TrpoStats(), L.OptStats(), L.PolicyOptStats()
    lib.rl_trpo_cfg_default(b(trpo_cfg))
    ppo_cfg, dqn_cfg = L.PpoCfg(2, 0.2), L.DqnCfg(20, 2, 0, np.float32(0.99), 1)
    out, loss, kl, ent = C.c_void_p(), C.c_double(), C.c_double(), C.c_double()
    grad = np.zeros(4096, np.float32).ctypes.data_as(C.c_void_p)
    mq, gq = w.mlp(5, 16, 2), w.gru(5, 8, 2)
    cases = {
        "rl_trpo_update": ((w.traj, w.adv.c, w.policy.handle, b(trpo_cfg), b(stats)), range(4)),
        "rl_trpo_update_seq": ((w.traj, w.adv.c, w.gpolicy.handle, b(trpo_cfg), b(stats)), range(4)),
        "rl_trpo_probe": ((w.traj, w.adv.c, w.policy.handle, None, 1e-5, b(loss), b(kl), b(ent), grad, None), range(3)),
        "rl_trpo_probe_seq": ((w.traj, w.adv.c, w.gpolicy.handle, None, 1e-5, b(loss), b(kl), b(ent), grad, None), range(3)),
        "rl_value_update": ((w.traj, w.tgt.c, w.value.handle, adam(w, w.value), 2, b(opt)), range(4)),
        "rl_value_update_seq": ((w.traj, w.tgt.c, w.gvalue.handle, adam(w, w.gvalue), 2, b(opt)), range(4)),
        "rl_value_probe": ((w.traj, w.tgt.c, w.value.handle, L.RL_PASS_KERNEL_TCGEN05, b(loss), grad), range(3)),
        "rl_ppo_update": ((w.traj, w.adv.c, w.policy.handle, adam(w, w.policy), b(ppo_cfg), b(pstats)), range(5)),
        "rl_reinforce_update": ((w.traj, w.adv.c, w.policy.handle, adam(w, w.policy), b(pstats)), range(4)),
        "rl_dqn_update": ((w.rb.handle, mq.handle, adam(w, mq), b(dqn_cfg), b(opt)), range(4)),
        "rl_dqn_update_seq": ((w.rb.handle, gq.handle, adam(w, gq), b(dqn_cfg), b(opt)), range(4)),
        "rl_dqn_probe_seq": ((w.rb.handle, b(dqn_cfg), gq.handle, 0, b(loss), None), range(3)),
        "rl_adam_create": ((mq.handle, b(L.AdamCfg()), b(out)), range(3)),
        "rl_adam_create_seq": ((gq.handle, b(L.AdamCfg()), b(out)), range(3)),
    }
    for name, (args, pointers) in cases.items():
        assert each_null(getattr(lib, name), args, pointers) == [INVALID] * len(pointers), name


def test_optimizer_of_another_module(w):
    lib, opt, pstats = w.lib, C.byref(L.OptStats()), C.byref(L.PolicyOptStats())
    ppo, dqn = C.byref(L.PpoCfg(2, 0.2)), C.byref(L.DqnCfg(20, 2, 0, np.float32(0.99), 1))
    mq, gq = w.mlp(5, 16, 2), w.gru(5, 8, 2)
    for other in (adam(w, w.mlp(5, 128, 1)), adam(w, w.gvalue)):  # another Mlp, a recurrent module
        assert lib.rl_value_update(w.traj, w.tgt.c, w.value.handle, other, 2, opt) == INVALID
    for other in (adam(w, w.gru(5, 8, 1)), adam(w, w.value)):  # another recurrent module, an Mlp
        assert lib.rl_value_update_seq(w.traj, w.tgt.c, w.gvalue.handle, other, 2, opt) == INVALID
    for other in (adam(w, w.value), adam(w, w.gpolicy)):
        assert lib.rl_ppo_update(w.traj, w.adv.c, w.policy.handle, other, ppo, pstats) == INVALID
        assert lib.rl_reinforce_update(w.traj, w.adv.c, w.policy.handle, other, pstats) == INVALID
    for other in (adam(w, w.policy), adam(w, gq)):
        assert lib.rl_dqn_update(w.rb.handle, mq.handle, other, dqn, opt) == INVALID
    for other in (adam(w, w.gpolicy), adam(w, mq)):
        assert lib.rl_dqn_update_seq(w.rb.handle, gq.handle, other, dqn, opt) == INVALID


@pytest.mark.parametrize("n_steps", [-1, 100001])
def test_optimizer_steps_out_of_range(w, n_steps):
    lib, opt, pstats = w.lib, C.byref(L.OptStats()), C.byref(L.PolicyOptStats())
    assert lib.rl_value_update(w.traj, w.tgt.c, w.value.handle, adam(w, w.value), n_steps, opt) == INVALID
    assert lib.rl_value_update_seq(w.traj, w.tgt.c, w.gvalue.handle, adam(w, w.gvalue), n_steps, opt) == INVALID
    ppo = L.PpoCfg(n_steps % (1 << 64), 0.2)  # opt_steps_per_update is unsigned: -1 is all ones
    assert lib.rl_ppo_update(w.traj, w.adv.c, w.policy.handle, adam(w, w.policy), C.byref(ppo), pstats) == INVALID
    dqn = C.byref(L.DqnCfg(20, n_steps, 0, np.float32(0.99), 1))
    mq, gq = w.mlp(5, 16, 2), w.gru(5, 8, 2)
    assert lib.rl_dqn_update(w.rb.handle, mq.handle, adam(w, mq), dqn, opt) == INVALID
    assert lib.rl_dqn_update_seq(w.rb.handle, gq.handle, adam(w, gq), dqn, opt) == INVALID


def test_value_module_with_two_outputs(w):
    lib, opt, loss = w.lib, C.byref(L.OptStats()), C.c_double()
    m, g = w.mlp(5, 16, 2), w.gru(5, 8, 2)
    assert lib.rl_value_update(w.traj, w.tgt.c, m.handle, adam(w, m), 2, opt) == INVALID
    assert lib.rl_value_probe(w.traj, w.tgt.c, m.handle, L.RL_PASS_KERNEL_TCGEN05, C.byref(loss), None) == INVALID
    assert lib.rl_value_update_seq(w.traj, w.tgt.c, g.handle, adam(w, g), 2, opt) == UNSUPPORTED


def test_module_of_another_context(w):
    lib, b, loss = w.lib, C.byref, C.c_double()
    trpo_cfg = L.TrpoCfg()
    lib.rl_trpo_cfg_default(b(trpo_cfg))
    gp, gv = w.gru(5, 8, 2, w.ctx2), w.gru(5, 8, 1, w.ctx2)
    assert lib.rl_trpo_update_seq(w.traj, w.adv.c, gp.handle, b(trpo_cfg), None) == INVALID
    assert lib.rl_trpo_probe_seq(w.traj, w.adv.c, gp.handle, None, 1e-5, b(loss), None, None, None, None) == INVALID
    assert lib.rl_value_update_seq(w.traj, w.tgt.c, gv.handle, adam(w, gv), 2, None) == INVALID
    dqn = b(L.DqnCfg(20, 2, 0, np.float32(0.99), 1))
    assert lib.rl_dqn_update_seq(w.rb.handle, gp.handle, adam(w, gp), dqn, None) == INVALID
    assert lib.rl_dqn_probe_seq(w.rb.handle, dqn, gp.handle, 0, b(loss), None) == INVALID


def test_feature_count_mismatch(w):
    """Batches of 5 features: an Mlp of 6 inputs is an invalid argument, a recurrent module of 6 inputs an unsupported one."""
    lib, b, opt, pstats, loss = w.lib, C.byref, C.byref(L.OptStats()), C.byref(L.PolicyOptStats()), C.c_double()
    trpo_cfg = L.TrpoCfg()
    lib.rl_trpo_cfg_default(b(trpo_cfg))
    dqn = b(L.DqnCfg(20, 2, 0, np.float32(0.99), 1))
    mp, mv, gp, gv = w.mlp(6, 16, 2), w.mlp(6, 16, 1), w.gru(6, 8, 2), w.gru(6, 8, 1)
    assert lib.rl_trpo_update(w.traj, w.adv.c, mp.handle, b(trpo_cfg), None) == INVALID
    assert lib.rl_trpo_probe(w.traj, w.adv.c, mp.handle, None, 1e-5, b(loss), None, None, None, None) == INVALID
    assert lib.rl_value_update(w.traj, w.tgt.c, mv.handle, adam(w, mv), 2, opt) == INVALID
    assert lib.rl_value_probe(w.traj, w.tgt.c, mv.handle, L.RL_PASS_KERNEL_FFMA, b(loss), None) == INVALID
    assert lib.rl_ppo_update(w.traj, w.adv.c, mp.handle, adam(w, mp), b(L.PpoCfg(2, 0.2)), pstats) == INVALID
    assert lib.rl_reinforce_update(w.traj, w.adv.c, mp.handle, adam(w, mp), pstats) == INVALID
    assert lib.rl_dqn_update(w.rb.handle, mp.handle, adam(w, mp), dqn, opt) == INVALID
    assert lib.rl_trpo_update_seq(w.traj, w.adv.c, gp.handle, b(trpo_cfg), None) == UNSUPPORTED
    assert lib.rl_trpo_probe_seq(w.traj, w.adv.c, gp.handle, None, 1e-5, b(loss), None, None, None, None) == UNSUPPORTED
    assert lib.rl_value_update_seq(w.traj, w.tgt.c, gv.handle, adam(w, gv), 2, opt) == UNSUPPORTED
    assert lib.rl_dqn_update_seq(w.rb.handle, gp.handle, adam(w, gp), dqn, opt) == UNSUPPORTED
    assert lib.rl_dqn_probe_seq(w.rb.handle, dqn, gp.handle, 0, b(loss), None) == UNSUPPORTED


def test_value_probe_unknown_kernel(w):
    loss = C.c_double()
    assert w.lib.rl_value_probe(w.traj, w.tgt.c, w.value.handle, 2, C.byref(loss), None) == INVALID
    assert w.lib.rl_value_probe(w.traj, w.tgt.c, w.value.handle, -1, C.byref(loss), None) == INVALID


@pytest.mark.parametrize("selected,probed", [(L.RL_PASS_KERNEL_TCGEN05, L.RL_PASS_KERNEL_FFMA),
                                             (L.RL_PASS_KERNEL_FFMA, L.RL_PASS_KERNEL_TCGEN05)],
                         ids=["tcgen05-selected", "ffma-selected"])
def test_value_probe_kernel_leaves_the_selection(request, tmp_path, selected, probed):
    """rl_value_probe runs the kernel it is given; the next rl_value_update runs the process-wide selection.

    The kernels are read from a torch.profiler trace taken in a child process.  Late in a long session the profiler of
    the session's process loses kernel records: after the whole GPU suite, a trace of this window held the launch calls
    of every kernel but the kernel records of only the last two, not even the torch fill kernel that opens the window."""
    import os
    import subprocess
    import sys

    if os.environ.get("RL_PROFILE_CHILD") != "1":
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        r = subprocess.run([sys.executable, "-m", "pytest", f"{__file__}::{request.node.name}", "-q", "-m", "gpu",
                            "-p", "no:cacheprovider"], capture_output=True, text=True, cwd=root, timeout=600,
                           env=dict(os.environ, RL_PROFILE_CHILD="1"))
        print(r.stdout[-3000:], r.stderr[-2000:])
        assert r.returncode == 0 and "1 passed" in r.stdout
        return
    _value_probe_kernel_leaves_the_selection(request.getfixturevalue("w"), tmp_path, selected, probed)


def _value_probe_kernel_leaves_the_selection(w, tmp_path, selected, probed):
    import json

    import torch
    from torch.profiler import ProfilerActivity, profile

    name = {L.RL_PASS_KERNEL_TCGEN05: "mlp_pass_tc_kernel", L.RL_PASS_KERNEL_FFMA: "mlp_pass_kernel"}
    lib, loss = w.lib, C.c_double()
    a = adam(w, w.value)
    torch.zeros(1, device="cuda")
    L.check(lib.rl_pass_kernel_select(selected))
    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            torch.zeros(1, device="cuda")  # late in a long session the profiler can miss a window's first kernel
            torch.cuda.synchronize()
            L.check(lib.rl_value_probe(w.traj, w.tgt.c, w.value.handle, probed, C.byref(loss), None), w.ctx.handle)
            L.check(lib.rl_value_update(w.traj, w.tgt.c, w.value.handle, a, 2, None), w.ctx.handle)
            w.ctx.synchronize()
    finally:
        L.check(lib.rl_pass_kernel_select(L.RL_PASS_KERNEL_TCGEN05))
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    kernels = sorted((e for e in json.loads(path.read_text())["traceEvents"] if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    passes = [m.group(1) for e in kernels for m in [re.search(r"\b(mlp_pass_kernel|mlp_pass_tc_kernel)<", e["name"])] if m]
    assert passes == [name[probed], name[selected], name[selected]], [e["name"] for e in kernels]
