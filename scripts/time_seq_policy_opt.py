"""Time the PPO and REINFORCE updates through a recurrent policy next to one TRPO step on the same batch, on one GPU.

Rows, for Chain<Gru, Linear> and Chain<Lstm, Linear>:
  - config 4's shape: bandit meta-env (2 arms, 10 episodes), hidden 4, E = 131 072, T = 19 (K9; the GRU on its
    compile-time <6, 4, 2> instances, the LSTM on the run-time-sized ones);
  - the rl2 shape: bandit meta-env (10 arms, 100 episodes), hidden 128, E = 18 944, T = 199 (K10; the GRU's per-step GEMMs
    on the tensor cores, the LSTM's on the FP32 pipe).
Each row: one PPO update (10 Adam steps, clip 0.2), one REINFORCE update (one Adam step) and one TRPO step on the same
rolled-out batch and advantages ~ N(0, 1), each from the same initial parameters and a fresh optimizer.  Times are the
device time the update reports itself (CUDA events around it), median of REPS after one warm-up.  The first row names the
card, its power limit and its maximum SM clock.

usage: python scripts/time_seq_policy_opt.py [out.jsonl]
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
CELLS = {"gru": (R.GruLinear, R.init_gru_linear_params), "lstm": (R.LstmLinear, R.init_lstm_linear_params)}
SHAPES = [("config 4: bandit meta-env (2 arms, 10 episodes)", 2, 10, 131_072, 19, 4),
          ("rl2: bandit meta-env (10 arms, 100 episodes)", 10, 100, 18_944, 199, 128)]


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still printed; the row says where the device name is missing
        return f"unknown ({e})"


def time_updates(ctx, cell, label, arms, episodes, E, T, hidden):
    Net, init = CELLS[cell]
    env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(arms), episodes), E, seed=2)
    env.set_noise_philox(5, 0)
    F, A = env.num_features, env.num_actions
    net = Net(ctx, F, hidden, A)
    p0 = init(np.random.default_rng(1), F, hidden, A)
    net.set_weights(p0)
    traj = R.Trajectory(env, T)
    R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net), R.HistoryDataBound(T, 0), traj, want_summary=False)
    adv = ctx.to_device(np.random.default_rng(3).normal(size=(T, E)).astype(np.float32))
    makers = {"ppo_10_adam": lambda: R.Ppo(net, R.PpoConfig()), "reinforce": lambda: R.Reinforce(net, R.ReinforceConfig()),
              "trpo_step": lambda: R.Trpo(net, R.TrpoConfig())}
    times = {k: [] for k in makers}
    num_steps = None
    for rep in range(REPS + 1):
        for name, make in makers.items():
            net.set_weights(p0)
            policy = make()
            log = {}
            policy.update(traj, adv, log)
            num_steps = log["num_steps"]
            if rep > 0:
                times[name].append(log["policy/update_time"] * 1e3)
            if hasattr(policy, "optimizer"):
                policy.optimizer.close()
    traj.close(); env.close(); net.close()
    row = {"cell": cell, "shape": label, "E": E, "T": T, "hidden": hidden, "arms": arms, "valid_steps": num_steps,
           "kernel": "K9" if hidden <= 8 else "K10"}
    for name, ms in times.items():
        row[f"{name}_ms"] = round(float(np.median(ms)), 3)
    for name, ms in times.items():
        row[f"{name}_ms_all"] = [round(x, 3) for x in ms]
    return row


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    ctx = R.Context(0)
    rows = [{"gpu": gpu_info(), "reps": REPS}]
    for shape in SHAPES:
        for cell in ("gru", "lstm"):
            rows.append(time_updates(ctx, cell, *shape))
            print(json.dumps(rows[-1]), file=sys.stderr)
    text = "\n".join(json.dumps(r) for r in rows)
    print(text)
    if out:
        os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
        with open(out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
