"""K2q (the warp-specialised CartPole rollout) against K2c with 8 threads per env where episodes
end all the time: a reset after the very first step, episodes ending on consecutive steps, step-limit Interrupts on
every step or every other step, terminations of the bare env under a saturated policy.  K2q steps the state on a
dynamics warp from a reset state the aux warp drew ahead into a ring and hands it to the policy warps through named
barriers; every stored byte, the lane lengths and the summary must match K2c, which does it all in one thread group."""
import numpy as np
import pytest

import relearn_b200 as R
from relearn_b200 import _lib as L

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("E,T,slack,limit,visible,gain", [
    (2400, 24, 0, 1, True, 2.0),     # every step ends its episode: a reset after step 0 and after every step
    (37, 24, 0, 1, True, 2.0),       # the same with one policy warp per CTA (4-env CTAs, ragged last one)
    (1501, 30, 4, 2, True, 2.0),     # three policy warps, each on a sub-partition of its own; ragged last CTA, slack
    (2405, 30, 4, 2, True, 2.0),     # ragged last CTA, slack, episodes of two steps
    (4096, 48, 3, 0, False, 6.0),    # the bench size, bare env: episodes end by Terminate only (a saturated policy)
    (4096, 40, 0, 3, False, 6.0),    # latent limit (F = 4), Interrupts and Terminates mixed
    (4736, 30, 2, 1, True, 2.0),     # 32-env CTAs (eight policy warps)
    (4736, 36, 5, 0, True, 6.0),
    (9472, 20, 0, 2, False, 6.0),    # two waves
    (9472, 24, 3, 0, True, 6.0),
])
def test_k2q_reset_heavy_rollouts_are_bit_identical_to_k2c(ctx, E, T, slack, limit, visible, gain):
    wrap = R.VisibleStepLimit(limit) if visible else R.LatentStepLimit(limit)
    cfg = R.CartPoleConfig().wrap(wrap) if limit else R.CartPoleConfig()
    F = 5 if visible and limit else 4
    net = R.Mlp(ctx, F, [128], 2)
    net.set_weights(R.init_params(np.random.default_rng(E + T), F, 128, 2) * gain)

    def run(lanes, periods=2):
        env = R.build_env(ctx, cfg, E, seed=7, lane_offset=3)
        traj = R.Trajectory(env, T + slack)
        out = []
        for _ in range(periods):  # the second period starts from mid-episode states and the advanced noise counter
            summ = R.rollout(env, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=lanes),
                             R.HistoryDataBound(T, slack), traj)
            out.append((traj.to_host(), summ))
        traj.close()
        env.close()
        return out

    for (ws, sw), (gk, sg) in zip(run(L.RL_LANES_WARP_SPECIALIZED), run(8)):
        for k in ("lane_len", "succ"):
            np.testing.assert_array_equal(ws[k], gk[k], err_msg=k)
        valid = gk["succ"] != L.RL_PAD
        for k in ("action", "reward", "obs"):
            np.testing.assert_array_equal(ws[k][valid], gk[k][valid], err_msg=k)
        intr = gk["succ"] == L.RL_INTERRUPT
        np.testing.assert_array_equal(ws["next_obs"][intr], gk["next_obs"][intr])
        assert ws["num_steps"] == gk["num_steps"]
        for name in ("step_reward", "episode_reward", "episode_length"):
            a, b = getattr(sw, name), getattr(sg, name)
            assert (a.mean, a.squared_residual_sum, a.count) == (b.mean, b.squared_residual_sum, b.count), name
        assert (sw.num_stored_steps, sw.num_stored_episodes) == (sg.num_stored_steps, sg.num_stored_episodes)
        # the reset path is taken, and often
        ends = (gk["succ"] == L.RL_TERMINATE) | intr
        if limit == 1:
            assert ends[valid].all()  # every stored step ends its episode (the kernel's dangling step excepted)
        else:
            assert ends.sum() >= E // 4, ends.sum()
