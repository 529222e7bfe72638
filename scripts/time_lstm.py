"""Time Chain<Lstm, Linear> next to Chain<Gru, Linear> of the same size on one GPU, in one process.

Rows (each LSTM row beside the GRU row of the same shape):
  - rollout at config 4's shape: bandit meta-env (2 arms, 10 episodes), hidden 4, E = 131 072, T = 190 (K8a for both cells);
  - rollout at the rl2 shape: bandit meta-env (10 arms, 100 episodes), hidden 128, E = 18 944, T = 199 (GRU: the default
    pick, K8s; LSTM: K8a);
  - one TRPO step and one 50-step critic update at the rl2 size (E = 18 944, T = 199; K10 for both cells, the GRU's per-step
    GEMMs on the tensor cores, the LSTM's on the FP32 pipe).
Rollouts: median of REPS timed calls after one warm-up, CUDA events.  Updates: device time reported by the update itself,
median of REPS after one warm-up.  The first row names the card, its power limit and its maximum SM clock.

usage: python scripts/time_lstm.py [out.jsonl]
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import relearn_b200 as R
from relearn_b200 import _lib as L

REPS = int(os.environ.get("REPS", 3))
CELLS = {"gru": (R.GruLinear, R.GruLinearConfig, R.init_gru_linear_params),
         "lstm": (R.LstmLinear, R.LstmLinearConfig, R.init_lstm_linear_params)}


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still printed; the row says where the device name is missing
        return f"unknown ({e})"


def time_rollout(ctx, cell, label, cfg, E, T, hidden):
    Net, _, init = CELLS[cell]
    env = R.build_env(ctx, cfg, E, seed=1)
    env.set_noise_philox(3, 0)
    net = Net(ctx, env.num_features, hidden, env.num_actions)
    net.set_weights(init(np.random.default_rng(0), env.num_features, hidden, env.num_actions))
    spec = R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net)
    traj = R.Trajectory(env, T)
    bound = R.HistoryDataBound(T, 0)
    R.rollout(env, spec, bound, traj, want_summary=False)
    ms = []
    for _ in range(REPS):
        e0 = ctx.event().record()
        R.rollout(env, spec, bound, traj, want_summary=False)
        e1 = ctx.event().record()
        ms.append(e0.elapsed_ms(e1))
    traj.close(); env.close()
    med = float(np.median(ms))
    return {"what": "rollout", "cell": cell, "shape": label, "E": E, "T": T, "hidden": hidden, "ms": round(med, 3), "env_steps_per_s": round(E * T / (med * 1e-3)),
            "ms_all": [round(x, 3) for x in ms]}


def time_updates(ctx, cell, E, T, hidden=128):
    Net, Cfg, init = CELLS[cell]
    env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(10), 100), E, seed=2)
    env.set_noise_philox(5, 0)
    F, A = env.num_features, env.num_actions
    agent = R.ActorCriticConfig(policy_config=R.TrpoConfig(policy_fn_config=Cfg(hidden_dim=hidden)),
                                critic_config=R.ValuesOptConfig(state_value_fn_config=Cfg(hidden_dim=hidden), opt_steps_per_update=50)
                                ).build_agent(env)
    rng = np.random.default_rng(1)
    p0, v0 = init(rng, F, hidden, A), init(rng, F, hidden, 1)
    traj = R.Trajectory(env, T)
    agent.policy.policy_fn.set_weights(p0)
    R.rollout(env, agent.actor(), R.HistoryDataBound(T, 0), traj, want_summary=False)
    adv = agent.critic.advantages(traj)
    trpo, critic = [], []
    for rep in range(REPS + 1):
        agent.policy.policy_fn.set_weights(p0)
        agent.critic.state_value_fn.set_weights(v0)
        log = {}
        agent.policy.update(traj, adv, log)
        cs = agent.critic.update(traj, log)
        if rep > 0:
            trpo.append(log["policy/update_time"] * 1e3)
            critic.append(cs.update_ms)
    traj.close(); env.close()
    return {"what": "update", "cell": cell, "E": E, "T": T, "hidden": hidden, "lane_steps": E * T,
            "trpo_step_ms": round(float(np.median(trpo)), 2), "critic_50_adam_ms": round(float(np.median(critic)), 2),
            "trpo_ms_all": [round(x, 2) for x in trpo], "critic_ms_all": [round(x, 2) for x in critic]}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    ctx = R.Context(0)
    rows = [{"gpu": gpu_info(), "reps": REPS}]
    config4 = R.MetaEnv(R.UniformBernoulliBandits(2), 10)
    rl2 = R.MetaEnv(R.UniformBernoulliBandits(10), 100)
    for cell in ("gru", "lstm"):
        rows.append(time_rollout(ctx, cell, "config 4: bandit meta-env (2 arms, 10 episodes)", config4, 131_072, 190, 4))
    for cell in ("gru", "lstm"):
        rows.append(time_rollout(ctx, cell, "rl2: bandit meta-env (10 arms, 100 episodes)", rl2, 18_944, 199, 128))
    for cell in ("gru", "lstm"):
        rows.append(time_updates(ctx, cell, 18_944, 199))
    text = "\n".join(json.dumps(r) for r in rows)
    print(text)
    if out:
        os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
        with open(out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
