"""Time DQN with a recurrent Q-network on one GPU: the epsilon-greedy GRU rollout next to the categorical GRU rollout on the
same module, and rl_dqn_update_seq per 50-step update at a minibatch of 100 000 steps with the padding fraction of its
sequence minibatches (B episodes x L longest / M steps).

Rollouts: MemoryGame(4, 16) with hidden 8 at 65 536 envs (K8a), bandit meta-env (10 arms, 100 episodes) with hidden 128 at
131 072 envs (categorical: K8s by default and K8h forced; epsilon-greedy: K8h).  Each row is the median of REPS timed
rollouts after one warm-up."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import relearn_b200 as R
from relearn_b200 import _lib as L

REPS = int(os.environ.get("REPS", 5))


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still printed; the row says where the device name is missing
        return f"unknown ({e})"


def time_rollout(ctx, cfg, E, T, hidden, kind, eps=0.1, kernel=None):
    if kernel:
        os.environ["RL_GRU_KERNEL"] = kernel
    else:
        os.environ.pop("RL_GRU_KERNEL", None)
    env = R.build_env(ctx, cfg, E, seed=1)
    env.set_noise_philox(3, 0)
    net = R.GruLinear(ctx, env.num_features, hidden, env.num_actions)
    net.set_weights(R.init_gru_linear_params(np.random.default_rng(0), env.num_features, hidden, env.num_actions))
    actor = (R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net) if kind == "categorical" else
             R.ActorSpec(kind=L.RL_ACTOR_EPS_GREEDY_Q, seq_net=net, exploration_rate=eps))
    traj = R.Trajectory(env, T)
    bound = R.HistoryDataBound(T, 0)
    R.rollout(env, actor, bound, traj)
    ms = []
    for _ in range(REPS):
        e0 = ctx.event().record()
        R.rollout(env, actor, bound, traj, want_summary=False)
        e1 = ctx.event().record()
        ms.append(e0.elapsed_ms(e1))
    traj.close()
    os.environ.pop("RL_GRU_KERNEL", None)
    med = float(np.median(ms))
    return {"what": "rollout", "env": type(cfg).__name__, "E": E, "T": T, "hidden": hidden, "actor": kind,
            "eps": eps if kind != "categorical" else None, "kernel": kernel or "default", "ms": round(med, 3),
            "env_steps_per_s": round(E * T / (med * 1e-3)), "ms_all": [round(x, 3) for x in ms]}


def time_update(ctx, name, cfg, E, T, hidden, periods, minibatch=100_000, steps=50, td=False):
    env = R.build_env(ctx, cfg, E, seed=2)
    env.set_noise_philox(5, 0)
    agent = R.DqnConfig(action_value_fn_config=R.GruLinearConfig(hidden_dim=hidden), minibatch_steps=minibatch,
                        opt_steps_per_update=steps, target_one_step_td=td, buffer_capacity=4 * T, sample_seed=1).build_agent(env)
    agent.action_value_fn.set_weights(R.init_gru_linear_params(np.random.default_rng(1), env.num_features, hidden, env.num_actions))
    rb = agent.buffer()
    traj = R.Trajectory(env, T)
    for _ in range(periods):
        R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_RANDOM), R.HistoryDataBound(T, 0), traj)
        rb.write_experience(traj)
    cfg_c = agent.c_cfg()
    pads = []
    for di in range(3):
        s = rb.sample_seq(cfg_c, agent.action_value_fn, 10_000 + di)
        pads.append(s["num_episodes"] * s["max_len"] / s["num_steps"])
    agent.batch_update(rb, {})  # warm-up
    rows = []
    for _ in range(3):
        t0 = time.perf_counter()
        st = agent.batch_update(rb, {})
        wall = (time.perf_counter() - t0) * 1e3
        rows.append((st.update_ms, wall))
    dev = float(np.median([r[0] for r in rows])); wall = float(np.median([r[1] for r in rows]))
    return {"what": "dqn_update_seq", "case": name, "hidden": hidden, "one_step_td": td, "minibatch_steps": minibatch, "opt_steps": steps,
            "update_ms_device": round(dev, 2), "update_ms_wall": round(wall, 2), "ms_per_opt_step": round(dev / steps, 3),
            "padding_B_L_over_M": [round(p, 3) for p in pads], "stored_steps": int(rb.stats().num_steps)}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    ctx = R.Context(0)
    rows = [{"gpu": gpu_info()}]
    mem = R.MemoryGame(4, 16)
    for kind in ("categorical", "eps_greedy"):
        rows.append(time_rollout(ctx, mem, 65_536, 200, 8, kind))
    bandit = R.MetaEnv(R.UniformBernoulliBandits(10), 100)
    rows.append(time_rollout(ctx, bandit, 131_072, 199, 128, "categorical"))
    rows.append(time_rollout(ctx, bandit, 131_072, 199, 128, "categorical", kernel="tile"))
    rows.append(time_rollout(ctx, bandit, 131_072, 199, 128, "eps_greedy"))
    rows.append(time_rollout(ctx, bandit, 131_072, 199, 128, "eps_greedy", eps=1.0))
    rows.append(time_update(ctx, "MemoryGame(4,16)", mem, 4096, 68, 8, periods=3))
    rows.append(time_update(ctx, "MemoryGame(4,16) OneStepTd", mem, 4096, 68, 8, periods=3, td=True))
    rows.append(time_update(ctx, "CartPole(limit 500)", R.CartPoleConfig().wrap(R.VisibleStepLimit(500)), 4096, 64, 8, periods=3))
    rows.append(time_update(ctx, "bandit meta (10 arms, 100 episodes)", bandit, 1024, 199, 128, periods=2))
    text = "\n".join(json.dumps(r) for r in rows)
    print(text)
    if out:
        os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
        with open(out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
