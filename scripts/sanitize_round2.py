"""Small runs of the kernels added in round 2 for compute-sanitizer
(`compute-sanitizer --tool memcheck|racecheck|synccheck python scripts/sanitize_round2.py`): the warp-specialised
rollout K2q (ragged last CTA, slack, step-limit Interrupts), a rollout and the update passes through a module with
two hidden layers, the UCB1 actor / fold, rl_pack_history."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import relearn_b200 as R
from relearn_b200 import _lib as L

ctx = R.Context(0)
rng = np.random.default_rng(0)
cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(9))
# K2q with one policy warp (4-env CTAs), five (20-env CTAs) and eight (32-env CTAs); every last CTA ragged
for E in (37, 2401, 4700):
    env = R.build_env(ctx, cfg, E, seed=2, lane_offset=3)
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(R.init_params(rng, 5, 128, 2))
    traj = R.Trajectory(env, 24)
    for _ in range(2):
        summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=L.RL_LANES_WARP_SPECIALIZED),
                         R.HistoryDataBound(20, 4), traj)
    print("E", E, "steps", summ.step_reward.count, "packed", R.pack_history(traj)["num_episodes"])
# deep module: rollout + TRPO + critic + PPO
env = R.build_env(ctx, R.MemoryGame(4, 3), 40, seed=5)
mc = R.MlpConfig(hidden_sizes=[24, 17], activation="tanh")
for pc in (R.TrpoConfig(policy_fn_config=mc), R.PpoConfig(policy_fn_config=mc, opt_steps_per_update=2)):
    agent = R.ActorCriticConfig(policy_config=pc, critic_config=R.ValuesOptConfig(state_value_fn_config=mc, opt_steps_per_update=2)).build_agent(env)
    agent.policy.policy_fn.set_weights(R.init_params(rng, env.num_features, [24, 17], env.num_actions))
    agent.critic.state_value_fn.set_weights(R.init_params(rng, env.num_features, [24, 17], 1))
    traj = R.Trajectory(env, 30)
    R.rollout(env, agent.actor(), R.HistoryDataBound(30, 0), traj, want_summary=False)
    print(type(agent.policy).__name__, "status", agent.batch_update(traj, {}))
# UCB1
env = R.build_env(ctx, R.Chain(), 33, seed=1)
agent = R.UCB1AgentConfig().build_agent(env)
traj = R.Trajectory(env, 20)
for training in (True, False):
    R.rollout(env, agent.actor(training=training), R.HistoryDataBound(20, 0), traj)
    agent.update(traj)
print("ucb1 visits", int(agent.get_tables()[2].sum()))
ctx.synchronize()
print("done")
