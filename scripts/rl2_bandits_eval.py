#!/usr/bin/env python
"""rl2_bandits_eval.py -- the `eval` half of relearn's rl2-bandits experiment (relearn_experiments/src/bin/rl2-bandits.rs:
166-245, 459-492) on the device: classical bandit agents lifted onto MetaEnv<UniformBernoulliBandits(k)> with
TrialEpisodeLimit(n) by ResettingMetaAgent, the baselines an RL^2 policy is compared against.

Each lane runs whole trials: a trial is always 2n - 1 meta steps (n pulls, n - 1 inner resets), so the bound
(m (2n - 1), 0) gives exactly m trials per lane and `--num-trials` trials spread over the lanes.  The result is
EvalResults: the mean trial reward and its population standard deviation (OnlineMeanVariance::stddev, utils/stats.rs).

Agents as at rl2-bandits.rs:197-220: random, eps-greedy (tabular Q, epsilon 0.2), greedy (epsilon 0), TS (Beta Thompson
sampling, one sample), OTS (the same with the mean of 10 samples, as the reference defines it) and UCB1 (exploration rate
0.2).  The tabular configs there set initial_action_count 2 / initial_action_value 0.5, which build_agent ignores
(tabular.rs:61-77): every table starts from zeros, here as in the reference.  The Thompson agents draw from the device's
own Beta sampler (DESIGN section 5): the same distribution as the reference's, not its bit stream.

Noise: the device draws env and agent noise from one Philox key; --env-seed and --agent-seed are combined into it.

`--time` also times one rollout of every inner agent, and of the plain random actor on the same env as a floor, at a user
size (config 4's 131 072 lanes, k = 10, n = 100, one trial per lane) with CUDA events after warm-up runs, and reads the
card's name and power limit in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import relearn_b200 as R  # noqa: E402
from relearn_b200 import _lib as L  # noqa: E402

AGENTS = {
    "random": R.RandomAgentConfig(),
    "eps-greedy": R.TabularQLearningAgentConfig(exploration_rate=0.2, initial_action_count=2, initial_action_value=0.5),
    "greedy": R.TabularQLearningAgentConfig(exploration_rate=0.0, initial_action_count=2, initial_action_value=0.5),
    "ts": R.BetaThompsonSamplingAgentConfig(num_samples=1),
    "ots": R.BetaThompsonSamplingAgentConfig(num_samples=10),
    "ucb1": R.UCB1AgentConfig(exploration_rate=0.2),
}


def philox_seed(env_seed: int, agent_seed: int) -> int:
    return ((agent_seed & 0xFFFFFFFF) << 32) ^ (env_seed & 0xFFFFFFFFFFFFFFFF)


def evaluate(ctx, agent: str, num_arms: int, num_episodes: int, num_trials: int, num_envs: int, seed: int) -> dict:
    lanes = max(1, min(num_envs, num_trials))
    m = -(-num_trials // lanes)  # trials per lane
    cfg = R.MetaEnv(R.UniformBernoulliBandits(num_arms), num_episodes)
    env = R.build_env(ctx, cfg, lanes, seed=seed)
    env.set_noise_philox(seed, 0)
    steps = m * (2 * num_episodes - 1)
    traj = R.Trajectory(env, steps)
    actor = R.ResettingMetaAgentConfig(AGENTS[agent]).build_agent(env).actor()
    summ = R.rollout(env, actor, R.HistoryDataBound(steps, 0), traj)
    er = summ.episode_reward
    traj.close()
    return {"agent": agent, "num_arms": num_arms, "num_episodes": num_episodes, "num_trials": int(er.count),
            "trial_reward_mean": er.mean if er.count else math.nan,
            "trial_reward_stddev": math.sqrt(er.variance()) if er.count else math.nan}


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as exc:  # the timing is still reported, marked as unlabelled
        return {"gpu": f"unknown ({exc})", "power_limit": "unknown"}


def time_rollouts(ctx, lanes: int, num_arms: int, num_episodes: int, warmup: int, reps: int) -> list[dict]:
    cfg = R.MetaEnv(R.UniformBernoulliBandits(num_arms), num_episodes)
    env = R.build_env(ctx, cfg, lanes, seed=1)
    steps = 2 * num_episodes - 1
    traj = R.Trajectory(env, steps)
    bound = R.HistoryDataBound(steps, 0)
    actors = [("random actor (K2a floor)", R.ActorSpec(kind=L.RL_ACTOR_RANDOM))]
    for name in ("random", "eps-greedy", "ucb1", "ts", "ots"):
        actors.append((f"meta {name} (K2m)", R.ResettingMetaAgentConfig(AGENTS[name]).build_agent(env).actor()))
    rows = []
    for name, actor in actors:
        env.set_noise_philox(1, 0)
        for _ in range(warmup):
            R.rollout(env, actor, bound, traj, want_summary=False)
        start, stop = ctx.event(), ctx.event()
        start.record()
        for _ in range(reps):
            R.rollout(env, actor, bound, traj, want_summary=False)
        stop.record()
        ms = start.elapsed_ms(stop) / reps
        rows.append({"actor": name, "lanes": lanes, "steps_per_lane": steps, "ms_per_rollout": ms,
                     "env_steps_per_sec": lanes * steps / (ms * 1e-3)})
    traj.close()
    return rows


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("-k", "--num-arms", type=int, default=10)
    ap.add_argument("-n", "--num-episodes", type=int, default=100, help="inner episodes (pulls) per trial")
    ap.add_argument("--num-trials", type=int, default=1000)
    ap.add_argument("--agent", choices=list(AGENTS) + ["all"], default="ucb1")
    ap.add_argument("--env-seed", type=int, default=0)
    ap.add_argument("--agent-seed", type=int, default=1)
    ap.add_argument("--num-envs", type=int, default=131072, help="lanes the trials are spread over (at most num_trials)")
    ap.add_argument("--json", metavar="PATH", help="also write the results as JSON")
    ap.add_argument("--time", action="store_true", help="also time one rollout per agent at 131 072 lanes, k = 10, n = 100")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()

    ctx = R.Context(0)
    seed = philox_seed(args.env_seed, args.agent_seed)
    agents = list(AGENTS) if args.agent == "all" else [args.agent]
    results = [evaluate(ctx, a, args.num_arms, args.num_episodes, args.num_trials, args.num_envs, seed) for a in agents]
    out = {"eval": results}
    for r in results:
        print(f"{r['agent']:>10}  k={r['num_arms']} n={r['num_episodes']} trials={r['num_trials']}  "
              f"trial reward {r['trial_reward_mean']:.3f} +- {r['trial_reward_stddev']:.3f}")
    if args.time:
        info = gpu_info()
        rows = time_rollouts(ctx, 131072, 10, 100, args.warmup, args.reps)
        out["timing"] = {**info, "rows": rows}
        print(f"timing on {info['gpu']} at power limit {info['power_limit']}:")
        for r in rows:
            print(f"  {r['actor']:>26}: {r['ms_per_rollout']:.3f} ms per rollout of {r['lanes']} x {r['steps_per_lane']} steps, "
                  f"{r['env_steps_per_sec'] / 1e9:.3f} G env-steps/s")
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
