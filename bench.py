#!/usr/bin/env python
"""bench.py -- env-steps/sec of the fused rollout (+ policy act) hot path, TRPO update ms, roofline.

Usage: `python bench.py --gpus N --steps K --warmup W`; for N > 1 run it under torchrun (one rank per GPU,
RANK/LOCAL_RANK/WORLD_SIZE/MASTER_* in the env).  One JSON line on stdout from rank 0.  `--dump-outputs DIR`
also writes the trajectory of the last timed step to DIR (see dump_outputs): the inputs are seeded, so two builds
run with the same arguments can be compared output for output.

Workload = BASELINE.json configs[1] "cartpole-trpo": CartPole + VisibleStepLimit(500), MLP policy 5->128->2,
E = 4096 lanes per GPU, T = 256 steps per lane per period (N = 1 048 576 env-steps per GPU per step of this
bench).  A "step" is one collection period: fresh episodes on every lane, policy forward + categorical
sample + dynamics + trajectory write for E*T env-steps.  Weak scaling: every rank owns its own E lanes
(global lane ids rank*E ..), no data-path collective.

`--impl reference` times the reference's CPU implementation of the same path: the C oracle port of
Steps::step + PolicyActor::act on all host cores (the Rust reference cannot be built in this image).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
B_PER_STEP_ROLLOUT = 26      # obs 5 x f32 + action u8 + reward f32 + succ u8 (DESIGN.md, SURVEY 8d K2)
B_PER_STEP_UNFUSED = 98      # K1 (f64 state)
B_PER_STEP_SCAN = 17         # K3
FLOP_PER_STEP_POLICY = 1792  # 2 * (5*128 + 128*2)
# K6 critic pass (SURVEY 8d): forward 1536 + backward 3072 FLOP per sample per Adam iteration (the network's own
# arithmetic).  What the tcgen05 kernel issues per 128-sample tile is larger (bf16-piece operands, padded N):
# MMA1 128x128x48, MMA3 128x32x128, MMA2 128x32x128  =>  2 * (786432 + 524288 + 524288) / 128 = 28672 FLOP per sample.
FLOP_PER_SAMPLE_CRITIC = 4608
FLOP_ISSUED_PER_SAMPLE_CRITIC_TC = 28672
# dram__bytes_read.sum + dram__bytes_write.sum of one K2q launch (the kernel `lanes_per_env = 0` picks) at E = 4096,
# T = 256 from the round-2 `ncu --set full` capture of the final kernel (profiles/r2A_k2q_e4096.md): 58.6 KB + 3.6 KB
# (the write figure is whatever part of the trajectory L2 happened to write back during the launch: 2.8 .. 22 KB over captures).  The 27 MB trajectory of a
# period stays in the 126 MB L2 while the kernel runs and drains afterwards, so the in-kernel DRAM traffic
# is far BELOW the algorithmic 26 B/env-step, not above it.
K2C_NCU_DRAM_BYTES_PER_LAUNCH = 62208
DUMP_MAX_BYTES = 64_000_000  # --dump-outputs: beyond this, a fixed sample of lanes is written


WORKLOAD = "cartpole-trpo rollout (CartPole+VisibleStepLimit(500), MLP 5-128-2 policy: env step + policy act + sample + trajectory write)"


def workload_config(args, world: int) -> dict:
    """The `config` of the JSON line: the same keys and values in both arms (the reference arm runs a bounded sample of
    this workload per step; cpu_baseline.sample says how much)."""
    return {"workload": WORKLOAD, "envs_per_gpu": args.envs, "horizon": args.horizon,
            "env_steps_per_step": world * args.envs * args.horizon, "lanes_per_env": args.lanes,
            "l2": "GPU arm: flushed between timed iterations (256 MiB memset)", "noise": "philox4x32-10",
            "parallelism": f"dp{world} (lanes sharded, no collective)"}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s: the sustained figure (the critic pass runs 80 times back to back inside a long step)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        if "bf16_tflops_sustained" in d:
            return float(d["bf16_tflops_sustained"]), "measured sustained (MEASURED_PEAKS.json)"
    return 1500.0, "fallback (B200_PROFILING.md)"


def cpu_update_baseline(n_steps: int, seed: int = 0):
    """The reference's update on the host: torch-CPU restatement of Trpo::update + ValuesOpt::update (oracle/
    tensor_oracle.py, all host threads) on a bounded sample of the same batch distribution."""
    import torch

    from oracle import tensor_oracle as TO
    from relearn_b200.modules import init_params

    torch.set_num_threads(os.cpu_count() or 1)  # intra-op threads = all cores for updates (SURVEY 8d)
    rng = np.random.default_rng(seed)
    obs = rng.uniform(-1, 1, size=(n_steps, 5)).astype(np.float32)
    act = rng.integers(0, 2, n_steps)
    adv = rng.normal(size=n_steps).astype(np.float32)
    tgt = rng.uniform(0, 50, size=n_steps).astype(np.float32)
    pp, vp = init_params(rng, 5, 128, 2), init_params(rng, 5, 128, 1)
    t0 = time.perf_counter()
    TO.trpo_update(pp, 5, 128, 2, obs, act, adv)
    t1 = time.perf_counter()
    TO.value_update(vp, 5, 128, obs, tgt, n_steps=80)
    t2 = time.perf_counter()
    return {"batch_steps": n_steps, "trpo_policy_ms": (t1 - t0) * 1e3, "critic_80_adam_ms": (t2 - t1) * 1e3,
            "threads": torch.get_num_threads(), "kind": "port (torch-CPU autograd restatement, f32)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_begin(self):
        """Wall-clock start of the region whose samples count (the sampler itself starts earlier: with 8 GPUs nvidia-smi
        needs more than a second before its first line)."""
        self.t_begin = time.time()

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        t_end = time.time()
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        import datetime

        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 10:
                    continue
                try:
                    ts = datetime.datetime.strptime(p[9], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(p[1]), float(p[2]), [n for n, v in zip(names, p[5:9]) if v.lower().startswith("active")]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        t0 = getattr(self, "t_begin", 0.0)
        inside = [r for r in rows if t0 - 0.05 <= r[0] <= t_end + 0.05]
        use, where = (inside, "timed + e2e region") if inside else (rows[-5:], "last samples before the region ended (none fell inside)")
        if use:
            out.update(sm_mhz=float(np.median([r[1] for r in use])), sm_max_mhz=float(max(r[2] for r in use)),
                       reasons=sorted({n for r in use for n in r[3]}), samples=len(use), window=where)
        return out


def dist_setup():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist  # noqa: F811

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def max_over_ranks(dist, local, value: float) -> float:
    if dist is None:
        return value
    import torch

    t = torch.tensor([value], dtype=torch.float64, device=torch.device("cuda", local))
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(dist, ctx):
    ctx.synchronize()
    if dist is not None:
        import torch

        dist.barrier()
        torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------
# CPU arm (the reference's own CPU path, as the C oracle port)
# ------------------------------------------------------------------------------------------------
def cpu_rollout_rate(params: np.ndarray, lanes: int, horizon: int, threads: int, seed: int = 1, t0: int = 0, aten: bool = False):
    """One period of `lanes` lanes x `horizon` steps on `threads` host threads.  aten = False: the C oracle port (scalar C
    MLP); aten = True: the same env loop with PolicyActor::act as batch-1 ATen calls against libtorch_cpu.so
    (oracle/aten_actor.cpp), the calls `tch` forwards the reference's actor to (BASELINE.md section 2)."""
    import ctypes as C

    import oracle as O

    cfg = O.cartpole_cfg(500)
    summ = O.Summary()
    if aten:
        p32 = np.ascontiguousarray(params, np.float32)
        fn = O.aten_lib().ro_rollout_lanes_aten
        t = time.perf_counter()
        fn(C.byref(cfg), p32.ctypes.data_as(C.POINTER(C.c_float)), 5, 128, 2, lanes, 0, horizon, 0, seed, t0, threads, C.byref(summ))
        dt = time.perf_counter() - t
        return lanes * horizon / dt, dt, summ
    mlp = O.mlp_struct(params, 5, 128, 2) if params is not None else None  # None: RandomAgent (env only)
    t = time.perf_counter()
    O.lib().ro_rollout_lanes_philox(C.byref(cfg), C.byref(mlp) if mlp is not None else None, lanes, 0, horizon, 0, seed, t0,
                                    threads, C.byref(summ))
    dt = time.perf_counter() - t
    return lanes * horizon / dt, dt, summ


def cpu_aten_sample(params: np.ndarray, horizon: int, cores: int, budget_s: float):
    """~budget_s seconds of the ATen-actor CPU rollout on all cores (a bounded sample: it runs ~20x slower than the port)."""
    try:
        rate, _, _ = cpu_rollout_rate(params, max(cores, 8), horizon, cores, aten=True)
        lanes = int(max(cores, rate * budget_s / horizon))
        v, dt, _ = cpu_rollout_rate(params, lanes, horizon, cores, t0=horizon + 1, aten=True)
        return {"value": v, "unit": UNIT, "cores": cores, "kind": "port-aten",
                "sample": f"{lanes} lanes x {horizon} steps ({dt:.1f} s wall), oracle env loop + batch-1 ATen linear/relu/linear/"
                          f"log_softmax/exp/multinomial per env-step (libtorch_cpu.so), {cores} threads"}
    except Exception as exc:  # no torch / no g++ on the box
        return {"unavailable": repr(exc)[:200]}


def run_reference(args):
    rank, world, local, _ = dist_setup() if int(os.environ.get("WORLD_SIZE", "1")) > 1 else (0, 1, 0, None)
    if rank != 0:
        return
    import oracle as O  # noqa: F401
    from relearn_b200.modules import init_params

    cores = os.cpu_count() or 1
    params = init_params(np.random.default_rng(0), 5, 128, 2)
    horizon = args.horizon
    # bounded sample: calibrate so that one step is ~1 s of wall time on all cores
    rate, _, _ = cpu_rollout_rate(params, max(cores, 8), horizon, cores)
    lanes = int(max(cores, min(args.envs, rate * 1.0 / horizon)))
    for _ in range(args.warmup):
        cpu_rollout_rate(params, lanes, horizon, cores)
    t = time.perf_counter()
    for i in range(args.steps):
        cpu_rollout_rate(params, lanes, horizon, cores, t0=i * (horizon + 1))
    dt = time.perf_counter() - t
    value = lanes * horizon * args.steps / dt
    sample = f"{lanes} lanes x {horizon} steps per step on {cores} threads (C oracle port of Steps::step + PolicyActor::act)"
    # Two restatements of the reference's CPU path are timed: the scalar C port (above) and the batch-1 ATen actor the
    # reference really calls through tch.  The line's value is the FASTER of the two, so the speed-up the driver computes
    # from it is the conservative one.
    kind = "port"
    extra = {"aten": cpu_aten_sample(params, horizon, cores, 5.0)}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 dynamics / f32 policy", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, **extra},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import relearn_b200 as R
    from relearn_b200 import _lib as L

    rank, world, local, dist = dist_setup()
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    # clocks / throttle reasons: nvidia-smi every 20 ms, started first (its start-up takes over a second on an 8-GPU box);
    # only the samples stamped inside the timed + e2e region are used
    clocks = ClockSampler(local)
    clocks.start()
    ctx = R.Context(local)
    info = ctx.device_info()
    E, T = args.envs, args.horizon
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
    env = R.build_env(ctx, cfg, E, seed=1234, lane_offset=rank * E)
    rng = np.random.default_rng(0)
    params = R.init_params(rng, 5, 128, 2)
    vparams = R.init_params(rng, 5, 128, 1)
    agent = R.ActorCriticConfig().build_agent(env)
    agent.policy.policy_fn.set_weights(params)
    agent.critic.state_value_fn.set_weights(vparams)
    traj = R.Trajectory(env, T)
    bound = R.HistoryDataBound(T, 0)
    actor = agent.actor(args.lanes)
    flush = ctx.alloc(256 << 20)  # > 126 MB L2

    if world > 1:  # data-parallel group for the update's all-reduces
        ids = [R.Context.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx.comm_init(ids[0], rank, world)

    def one_period(timed_events=None):
        flush.zero()
        if timed_events is not None:
            timed_events[0].record()
        R.rollout(env, actor, bound, traj, want_summary=False)
        if timed_events is not None:
            timed_events[1].record()

    for _ in range(max(args.warmup, 3)):
        one_period()
    barrier(dist, ctx)
    clocks.mark_begin()
    evs = [(ctx.event(), ctx.event()) for _ in range(args.steps)]
    launches0 = ctx.launch_count
    barrier(dist, ctx)
    wall0 = time.perf_counter()
    for k in range(args.steps):
        one_period(evs[k])
    barrier(dist, ctx)
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count - launches0
    kernel_ms = sum(a.elapsed_ms(b) for a, b in evs)
    total_ms = max_over_ranks(dist, local, kernel_ms)
    steps_per_period = E * T
    value = world * steps_per_period * args.steps / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, traj.to_host())

    # ---- e2e through the C ABI with host buffers: weights H2D (pinned) -> rollout -> summary D2H ----
    w_pinned = ctx.pinned_array((params.size,), np.float32)
    w_pinned[:] = params
    e2e_s = 0.0
    for k in range(max(3, min(args.warmup, 5)) + args.steps):
        flush.zero()
        ctx.synchronize()
        t0 = time.perf_counter()
        agent.policy.policy_fn.set_weights_async(w_pinned)
        summ = R.rollout(env, actor, bound, traj, want_summary=True)
        dt = time.perf_counter() - t0
        if k >= max(3, min(args.warmup, 5)):
            e2e_s += dt
    e2e_s = max_over_ranks(dist, local, e2e_s)
    clock_info = clocks.stop()
    e2e_value = world * steps_per_period * args.steps / e2e_s
    h2d = int(params.nbytes)
    d2h = 10 * 8

    # ---- roofline of the dominant kernel.  SURVEY 8(d) row K2: the fused rollout is bound by the FP32 FMA pipe / the
    #      latency of its dependent step chain, NOT by HBM (26 B of trajectory per env-step); the roof it is reported
    #      against is the measured FP32 FMA peak, and the HBM figure is given for the write stream only. ----
    hbm_peak, peak_src = measured_peaks()
    write_gbs = B_PER_STEP_ROLLOUT * steps_per_period * args.steps / (kernel_ms * 1e-3) / 1e9
    fp32_peak = ctx.fp32_peak_tflops() if rank == 0 else None
    policy_tflops = FLOP_PER_STEP_POLICY * steps_per_period * args.steps / (kernel_ms * 1e-3) / 1e12
    roofline = {"bound": "fp32-fma / step-chain latency (SURVEY 8d row K2; not hbm)", "achieved": policy_tflops,
                "peak": fp32_peak, "unit": "TFLOP/s", "frac": (policy_tflops / fp32_peak) if fp32_peak else None,
                "peak_source": "FFMA probe kernel timed in this run (rl_ctx_fp32_peak)",
                "flop_per_env_step": FLOP_PER_STEP_POLICY,
                "traffic": K2C_NCU_DRAM_BYTES_PER_LAUNCH if (E == 4096 and T == 256) else None,
                "traffic_note": "ncu dram bytes of one launch (profiles/r2A_k2q_e4096.md).  The 27 MB trajectory of a period stays in "
                                "the 126 MB L2 while the kernel runs; its write-back to HBM happens in the untimed L2 flush "
                                "between iterations, i.e. OUTSIDE the timed region",
                "hbm_write_stream": {"achieved": write_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": write_gbs / hbm_peak,
                                     "bytes_per_env_step": B_PER_STEP_ROLLOUT, "peak_source": peak_src},
                "kernel": "rollout_cartpole_ws6_kernel K2q (fused step+policy+sample; one CTA per SM: one dynamics warp of 28 envs x both "
                          "actions alone on its sub-partition, seven policy warps, an aux Philox warp)",
                "note": "at 4096 envs (28 per SM) the period is 256 x the latency of one step (~980 clk; profiles/r2_summary.md section 5: "
                        "dynamics warp 570 clk for both actions + select / publish, beside it three lock-step policy warps per "
                        "sub-partition at ~750 clk row -> action); ncu: FMA 27 %, FP64 9 %, issue 39 %, barrier 2.9 of 7.5 stall cycles "
                        "per instruction.  The HBM-bound kernels of the path are in kernels[] (77-81 % of the HBM peak)"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 dynamics / f32 policy", "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "what": "rl_mlp_set_weights_async(pinned host) + rl_rollout + StepsSummary read-back per period"},
        "gpu_launches": int(launches), "clocks": clock_info, "roofline": roofline,
        "wall_s_timed_region": wall, "sm_count": info["sm_count"],
    }

    if rank == 0:
        line["fp32"] = {"policy_tflops": policy_tflops, "measured_fma_peak_tflops": fp32_peak}
    # ---- the update that consumes the rollout: GAE + TRPO + critic (ms per iteration) ----
    if not args.no_update:
        upd = {"adv_est_ms": [], "policy_ms": [], "critic_ms": [], "status": []}
        for it in range(1 + args.update_iters):
            R.rollout(env, actor, bound, traj, want_summary=False)
            barrier(dist, ctx)
            e0, e1 = ctx.event().record(), None
            adv = agent.critic.advantages(traj)
            e1 = ctx.event().record()
            log = {}
            status = agent.policy.update(traj, adv, log)
            cstats = agent.critic.update(traj, log)
            if it > 0:
                upd["adv_est_ms"].append(e0.elapsed_ms(e1))
                upd["policy_ms"].append(log["policy/update_time"] * 1e3)
                upd["critic_ms"].append(cstats.update_ms)
                upd["status"].append(int(status))
        adv_ms = float(np.mean(upd["adv_est_ms"]))
        pol_ms = max_over_ranks(dist, local, float(np.mean(upd["policy_ms"])))
        cri_ms = max_over_ranks(dist, local, float(np.mean(upd["critic_ms"])))
        tpeak, tpeak_src = measured_tensor_peak()
        fp32_peak = line.get("fp32", {}).get("measured_fma_peak_tflops")
        alg = FLOP_PER_SAMPLE_CRITIC * steps_per_period * 80 / (cri_ms * 1e-3) / 1e12
        issued = FLOP_ISSUED_PER_SAMPLE_CRITIC_TC * steps_per_period * 80 / (cri_ms * 1e-3) / 1e12
        line["update"] = {
            "batch_steps_per_gpu": steps_per_period, "adv_est_ms": adv_ms, "trpo_policy_ms": pol_ms,
            "critic_80_adam_ms": cri_ms, "total_ms": adv_ms + pol_ms + cri_ms, "status": upd["status"],
            "pass_kernel": os.environ.get("RL_PASS_KERNEL", "tcgen05"),
            "all_reduce": ("none (1 GPU)" if world == 1 else
                           "fused row-reduction + NVLink peer-mailbox exchange (+ Adam), one kernel per pass"
                           if ctx.comm_peer_info()["peer_mailboxes"] else "reduce + ncclAllReduce (f64 sums)"),
            # the critic's 80 passes + Adam steps as one region: the network's own FLOPs per second (compare with the
            # FP32 FMA peak, which bounds any non-tensor implementation) and the bf16 FLOPs the MMAs issue
            "critic_roofline": {"bound": "tensor", "achieved": alg, "peak": tpeak, "unit": "TFLOP/s", "frac": alg / tpeak,
                                "peak_source": tpeak_src, "issued_bf16_tflops": issued, "fp32_fma_peak_tflops": fp32_peak,
                                "note": "achieved = ALGORITHMIC FLOPs (4608 per sample per Adam iteration of the f32 network, SURVEY 8d "
                                        "row K6) / time; issued_bf16_tflops = what the three MMAs issue per tile (bf16 pieces + "
                                        "padding, 28 672 per sample)"},
        }
    # ---- driver-visible correctness of the data-parallel update, and BASELINE configs 3 / 4 at this world size ----
    if not args.no_update and not args.quick:
        if world > 1:
            par = update_parity(ctx, R, L, args, rank, world, dist, local, params, vparams)
            line["update"]["parity_vs_single"] = par
            assert par["params_identical_across_ranks"], "ranks hold different parameters after a data-parallel update"
        line["configs"] = scaled_configs(ctx, R, L, hbm_peak, rank, world, dist, local)
    # ---- per-kernel rooflines for the HBM-bound kernels (rank 0, 1 GPU only) ----
    if rank == 0 and world == 1 and not args.quick:
        line["kernels"] = kernel_rooflines(ctx, R, L, hbm_peak)
        # CPU baseline on this box's host cores (bounded sample)
        cores = os.cpu_count() or 1
        cpu_rollout_rate(params, max(cores, 8), T, cores)
        periods, cpu_s = 0, 0.0
        while cpu_s < 10.0 and periods < 10000:  # ~10 s of wall time on all cores
            _, dt, _ = cpu_rollout_rate(params, E, T, cores, t0=periods * (T + 1))
            cpu_s += dt
            periods += 1
        line["cpu_baseline"] = {"value": periods * E * T / cpu_s, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{periods} periods of {E} lanes x {T} steps ({cpu_s:.1f} s wall) of the same "
                                          f"workload, C oracle port of Steps::step + PolicyActor::act, {cores} threads"}
        # env-only (RandomAgent: no policy network), SURVEY 8d's second CPU number: ~3 s of the same lanes on all cores
        env_s, env_periods = 0.0, 0
        while env_s < 3.0:
            _, dt, _ = cpu_rollout_rate(None, E, T, cores, t0=env_periods * (T + 1))
            env_s += dt
            env_periods += 1
        line["cpu_baseline"]["aten"] = cpu_aten_sample(params, T, cores, 5.0)
        line["cpu_baseline"]["env_only"] = {"value": env_periods * E * T / env_s, "unit": UNIT,
                                            "sample": f"{env_periods} periods of {E} lanes x {T} steps, RandomAgent, {cores} threads"}
        if not args.no_update:
            try:
                line["update"]["cpu_baseline"] = cpu_update_baseline(steps_per_period if args.cpu_update_full else 1 << 16)
            except Exception as exc:  # torch missing on the box: report, do not fail the bench
                line["update"]["cpu_baseline"] = {"unavailable": repr(exc)[:200]}
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir: str, host: dict) -> None:
    """Write a Trajectory.to_host() as DIR/<name>.npy: obs, next_obs [T, E, F], action, reward, succ [T, E] and
    lane_len [E] in float32, and lane [E] in float64, the trajectory lane of each column.  Slots the rollout leaves
    undefined are written as 0 (every field but succ at padding steps, succ == RL_PAD; next_obs except at interrupted
    steps), so two builds that agree compare equal.  When all lanes would exceed DUMP_MAX_BYTES, a fixed seeded
    sample of lanes is written."""
    from relearn_b200 import _lib as L

    T, E, F = host["obs"].shape
    lane_bytes = 4 * T * (2 * F + 3) + 4 + 8
    keep = min(E, DUMP_MAX_BYTES // lane_bytes)
    lanes = np.arange(E) if keep == E else np.sort(np.random.default_rng(0).choice(E, keep, replace=False))
    succ = host["succ"][:, lanes]
    pad, intr = succ == L.RL_PAD, succ == L.RL_INTERRUPT
    out = {"obs": np.where(pad[..., None], 0, host["obs"][:, lanes]),
           "next_obs": np.where(intr[..., None], host["next_obs"][:, lanes], 0),
           "action": np.where(pad, 0, host["action"][:, lanes]),
           "reward": np.where(pad, 0, host["reward"][:, lanes]),
           "succ": succ, "lane_len": host["lane_len"][lanes]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))
    np.save(os.path.join(out_dir, "lane.npy"), lanes.astype(np.float64))


def kernel_rooflines(ctx, R, L, hbm_peak):
    """Unfused step kernel (K1) and GAE scan (K3) at sizes larger than L2, timed alone with CUDA events."""
    import ctypes as C

    out = []
    E = 1 << 22
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
    env = R.build_env(ctx, cfg, E, seed=7)
    env.reset_all()
    actions = ctx.to_device(np.random.default_rng(0).integers(0, 2, E).astype(np.uint8))
    for _ in range(5):
        env.step_device(actions)
    reps = 20
    e0 = ctx.event().record()
    for _ in range(reps):
        env.step_device(actions)
    e1 = ctx.event().record()
    ms = e0.elapsed_ms(e1) / reps
    gbs = B_PER_STEP_UNFUSED * E / (ms * 1e-3) / 1e9
    out.append({"kernel": "env_step_kernel<CartPole> (unfused, f64 SoA state)", "envs": E, "bytes_per_step": B_PER_STEP_UNFUSED,
                "ms": ms, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm_peak, "env_steps_per_s": E / (ms * 1e-3),
                "working_set_mb": E * (B_PER_STEP_UNFUSED + 20) / 1e6})
    env.close()
    # GAE / reward-to-go scan over [T, E] = [256, 131072] (33.5 M steps, 570 MB)
    T, E2 = 256, 1 << 17
    env2 = R.build_env(ctx, cfg, E2, seed=8)
    traj = R.Trajectory(env2, T)
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(R.init_params(np.random.default_rng(1), 5, 128, 2))
    R.rollout(env2, R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net), R.HistoryDataBound(T, 0), traj, want_summary=False)
    adv, rtg = ctx.alloc(T * E2 * 4), ctx.alloc(T * E2 * 4)
    x = ctx.alloc(T * E2 * 4)
    x.zero()
    v = traj.view()
    lib = ctx._lib
    for _ in range(3):
        L.check(lib.rl_gae(traj.handle, None, 0.99, 0.95, adv.c, rtg.c), ctx.handle)
    reps = 10
    e0 = ctx.event().record()
    for _ in range(reps):
        L.check(lib.rl_gae(traj.handle, None, 0.99, 0.95, adv.c, rtg.c), ctx.handle)
    e1 = ctx.event().record()
    ms = e0.elapsed_ms(e1) / reps
    # without a critic the pass reads reward 4 + succ 1 and writes adv 4 + rtg 4 = 13 B/step
    gbs = 13 * T * E2 / (ms * 1e-3) / 1e9
    out.append({"kernel": "gae_scan_kernel<no critic> (reward-to-go + advantages)", "steps": T * E2, "bytes_per_step": 13,
                "ms": ms, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm_peak})
    for _ in range(3):
        L.check(lib.rl_discounted_cumsum(ctx.handle, x.c, C.c_void_p(v.succ), T, E2, 0.99, adv.c), ctx.handle)
    e0 = ctx.event().record()
    for _ in range(reps):
        L.check(lib.rl_discounted_cumsum(ctx.handle, x.c, C.c_void_p(v.succ), T, E2, 0.99, adv.c), ctx.handle)
    e1 = ctx.event().record()
    ms = e0.elapsed_ms(e1) / reps
    gbs = 9 * T * E2 / (ms * 1e-3) / 1e9
    out.append({"kernel": "cumsum_kernel (discounted_cumsum_from_end)", "steps": T * E2, "bytes_per_step": 9, "ms": ms,
                "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm_peak})
    # LazyHistoryFeatures' packed tensors from the same 33.5 M-step trajectory (rl_pack_history: episode scan, stable radix
    # sort by length, gather).  Algorithmic bytes per stored step: read obs 20 + action 1 + reward 4 + succ 1, write
    # obs 20 + extended obs 20 + is_invalid 1 + action (i64) 8 + reward 4 = 79 (the per-episode extra rows and the sort's
    # own traffic -- 24 B per EPISODE -- come on top and are not counted).
    cap = T * E2
    p_obs, p_ext, p_inv = ctx.alloc(cap * 5 * 4), ctx.alloc(2 * cap * 5 * 4), ctx.alloc(2 * cap)
    p_act, p_rew, p_bs, p_ebs = ctx.alloc(cap * 8), ctx.alloc(cap * 4), ctx.alloc((T + 1) * 8), ctx.alloc((T + 2) * 8)
    info = L.PackedInfo()
    pack = lambda: L.check(lib.rl_pack_history(traj.handle, p_obs.c, p_ext.c, p_inv.c, p_act.c, p_rew.c, p_bs.c, p_ebs.c,
                                               C.byref(info)), ctx.handle)
    for _ in range(2):
        pack()
    reps = 5
    e0 = ctx.event().record()
    for _ in range(reps):
        pack()
    e1 = ctx.event().record()
    ms = e0.elapsed_ms(e1) / reps
    gbs = 79 * info.num_steps / (ms * 1e-3) / 1e9
    out.append({"kernel": "rl_pack_history (LazyHistoryFeatures: packed observations, extended observations, actions, rewards)",
                "steps": int(info.num_steps), "episodes": int(info.num_episodes), "bytes_per_step": 79, "ms": ms,
                "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm_peak})
    for b in (p_obs, p_ext, p_inv, p_act, p_rew, p_bs, p_ebs):
        b.free()
    # large-E fused rollout (config 5's throughput end): K2c with one thread per env on the FP32 pipe, and K2t with the
    # policy's hidden layer on tcgen05 (what `lanes_per_env = 0` picks at this size)
    E3, T3 = 1 << 20, 64
    env3 = R.build_env(ctx, cfg, E3, seed=9)
    traj3 = R.Trajectory(env3, T3)
    for lanes, name in ((1, "rollout_cartpole_group_kernel<1> K2c (fused, thread per env, FP32 pipe)"),
                        (L.RL_LANES_TENSOR_CORE, "rollout_cartpole_tc_kernel K2t (fused, 128-env tiles, hidden layer on tcgen05)")):
        spec = R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=lanes)
        for _ in range(2):
            R.rollout(env3, spec, R.HistoryDataBound(T3, 0), traj3, want_summary=False)
        reps = 5
        e0 = ctx.event().record()
        for _ in range(reps):
            R.rollout(env3, spec, R.HistoryDataBound(T3, 0), traj3, want_summary=False)
        e1 = ctx.event().record()
        ms = e0.elapsed_ms(e1) / reps
        rec = {"kernel": name, "envs": E3, "horizon": T3, "ms": ms, "env_steps_per_s": E3 * T3 / (ms * 1e-3),
               "trajectory_write_gbs": B_PER_STEP_ROLLOUT * E3 * T3 / (ms * 1e-3) / 1e9,
               "policy_tflops": FLOP_PER_STEP_POLICY * E3 * T3 / (ms * 1e-3) / 1e12}
        if lanes == L.RL_LANES_TENSOR_CORE:
            # bf16 FLOPs the MMAs issue: [128 x 48] . [48 x 128] per 128 env-steps
            rec["mma_bf16_tflops"] = 2 * 48 * 128 * E3 * T3 / (ms * 1e-3) / 1e12
        out.append(rec)
    out += rl2_sized_rollout(ctx, R, L)
    return out


def scaled_configs(ctx, R, L, hbm_peak, rank, world, dist, local):
    """BASELINE configs 3 and 4, run by EVERY rank (any world size; timed alone with CUDA events, max over ranks):
    config 3 cartpole-dqn: 65 536 envs in total, sharded over the ranks, each rank with the replay rings of its own lanes
    (one ReplayBuffer per worker, dqn.rs:228-230), minibatch_steps / world sampled locally and the Q-loss gradient
    reduced over the group in every Adam step; config 4: the bandit meta-env with the rnn.rs-sized GRU policy at
    131 072 envs per GPU (1 048 576 on 8) and the GAE + TRPO + critic update through the GRU with reduced sums."""
    out = []
    rng = np.random.default_rng(3)
    mx = lambda v: max_over_ranks(dist, local, float(v))
    # ---- config 3: cartpole-dqn, 65 536 envs over the group ----
    E_total = 65536
    E, cfg = E_total // world, R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
    env = R.build_env(ctx, cfg, E, seed=5, lane_offset=rank * E)
    agent = R.DqnConfig(buffer_capacity=762).build_agent(env)  # 50 M steps of replay over the group (examples/cartpole-dqn.rs:34-42)
    agent.action_value_fn.set_weights(R.init_params(rng, 5, 128, 2))
    rb = agent.buffer()
    bound = R.HistoryDataBound(16, 5)  # first update: 1 M steps over 65 536 lanes
    traj = R.Trajectory(env, bound.min_steps + bound.slack_steps)
    times = {"rollout_ms": [], "append_ms": [], "update_ms": []}
    for it in range(4):
        barrier(dist, ctx)
        e0 = ctx.event().record()
        R.rollout(env, agent.actor(), bound, traj, want_summary=False)
        e1 = ctx.event().record()
        rb.write_experience(traj)
        e2 = ctx.event().record()
        stats = agent.batch_update(rb)
        if it > 0:
            times["rollout_ms"].append(e0.elapsed_ms(e1))
            times["append_ms"].append(e1.elapsed_ms(e2))
            times["update_ms"].append(stats.update_ms)
    st = rb.stats()
    steps = traj.view().num_steps
    app_ms = mx(np.mean(times["append_ms"]))
    qhash = params_identical(dist, agent.action_value_fn.get_weights())
    out.append({"config": "3 cartpole-dqn: eps-greedy rollout + replay append + 50 x (sample 100k over the group, Q loss, Adam)",
                "envs_total": E_total, "envs_per_gpu": E, "steps_per_period_per_gpu": int(steps),
                "rollout_ms": mx(np.mean(times["rollout_ms"])), "append_ms": app_ms,
                "append_gbs_per_gpu": 2 * 26 * steps / (app_ms * 1e-3) / 1e9,
                "dqn_update_50_steps_ms": mx(np.mean(times["update_ms"])), "replay_steps_per_gpu": int(st.num_steps),
                "replay_episodes_per_gpu": int(st.num_episodes), "q_params_identical_across_ranks": qhash})
    traj.close(); rb.close(); env.close()
    # ---- config 4: bandit meta-env (k = 2 arms, n = 10 episodes per trial) + GRU(6 -> 4) -> Linear(4 -> 2) ----
    E4, trials = 131072, 10
    mcfg = R.MetaEnv(R.UniformBernoulliBandits(2), 10)
    env4 = R.build_env(ctx, mcfg, E4, seed=6, lane_offset=rank * E4)
    net = R.GruLinear(ctx, env4.num_features, 4, env4.num_actions)
    net.set_weights(R.init_gru_linear_params(rng, env4.num_features, 4, env4.num_actions))
    T4 = trials * 19
    traj4 = R.Trajectory(env4, T4)
    spec = R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net)
    for _ in range(2):
        R.rollout(env4, spec, R.HistoryDataBound(T4, 0), traj4, want_summary=False)
    reps = 5
    barrier(dist, ctx)
    e0 = ctx.event().record()
    for _ in range(reps):
        R.rollout(env4, spec, R.HistoryDataBound(T4, 0), traj4, want_summary=False)
    e1 = ctx.event().record()
    ms = mx(e0.elapsed_ms(e1) / reps)
    bytes_per_step = 4 * env4.num_features + 6  # obs planes + action + reward + succ
    out.append({"config": "4 bandit meta-env + GRU(6->4)->Linear policy, fused rollout (thread per env)", "envs_total": E4 * world,
                "envs_per_gpu": E4, "horizon": T4, "ms": ms, "env_steps_per_s": world * E4 * T4 / (ms * 1e-3),
                "bytes_per_step": bytes_per_step, "trajectory_write_gbs_per_gpu": bytes_per_step * E4 * T4 / (ms * 1e-3) / 1e9,
                "frac_of_hbm_peak": bytes_per_step * E4 * T4 / (ms * 1e-3) / 1e9 / hbm_peak})
    traj4.close()
    # the update that consumes it: GAE + TRPO + 80-step critic through Chain<Gru, Linear> on one trial per lane (T = 19)
    g = R.GruLinearConfig(hidden_dim=4)
    agent4 = R.ActorCriticConfig(policy_config=R.TrpoConfig(policy_fn_config=g),
                                 critic_config=R.ValuesOptConfig(state_value_fn_config=g)).build_agent(env4)
    agent4.policy.policy_fn.set_weights(R.init_gru_linear_params(rng, env4.num_features, 4, env4.num_actions))
    agent4.critic.state_value_fn.set_weights(R.init_gru_linear_params(rng, env4.num_features, 4, 1))
    traj5 = R.Trajectory(env4, 19)
    upd = []
    for it in range(3):
        R.rollout(env4, agent4.actor(), R.HistoryDataBound(19, 0), traj5, want_summary=False)
        barrier(dist, ctx)
        e0 = ctx.event().record()
        adv = agent4.critic.advantages(traj5)
        e1 = ctx.event().record()
        log = {}
        agent4.policy.update(traj5, adv, log)
        cs = agent4.critic.update(traj5, log)
        if it > 0:
            upd.append((e0.elapsed_ms(e1), log["policy/update_time"] * 1e3, cs.update_ms))
    ghash = params_identical(dist, np.concatenate([agent4.policy.policy_fn.get_weights(), agent4.critic.state_value_fn.get_weights()]))
    out.append({"config": "4 update: GAE + TRPO + 80-step critic through GRU(6->4)->Linear (BPTT pass kernel), sums reduced over the group",
                "envs_per_gpu": E4, "batch_steps_per_gpu": E4 * 19, "adv_est_ms": mx(np.mean([u[0] for u in upd])),
                "trpo_policy_ms": mx(np.mean([u[1] for u in upd])), "critic_80_adam_ms": mx(np.mean([u[2] for u in upd])),
                "params_identical_across_ranks": ghash})
    traj5.close(); env4.close()
    return out


def params_identical(dist, params: np.ndarray):
    """Every rank must hold bit-identical parameters after a data-parallel update (the reduced sums are identical on
    every rank by construction; no broadcast happens).  True / False from an all-gather of a digest; None on one GPU."""
    if dist is None:
        return None
    import hashlib

    digest = hashlib.sha1(np.ascontiguousarray(params).tobytes()).hexdigest()
    digests = [None] * dist.get_world_size()
    dist.all_gather_object(digests, digest)
    return all(d == digests[0] for d in digests)


def update_parity(ctx, R, L, args, rank, world, dist, local, params, vparams):
    """Driver-visible correctness of the data-parallel update (world > 1): one GAE + TRPO + critic update on this bench's
    own per-GPU batch (E x T env-steps per rank, lanes rank*E ..) with the sums reduced over the group, against rank 0
    re-running the same update on the CONCATENATED batch (world x E lanes, no communicator) on its own GPU.  The
    rollouts agree bit for bit (Philox is keyed by the global lane; both sides run the warp-specialised kernel)."""
    E, T, seed = args.envs, args.horizon, 4321
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))

    def run(context, n_lanes, offset):
        env = R.build_env(context, cfg, n_lanes, seed=seed, lane_offset=offset)
        # hpv_reg_coeff 0.1: ten f32 CG iterations stay well conditioned, so the comparison measures the reduction and not
        # the amplification of rounding by the reference's own 1e-5 (tests/test_gpu_update.py quantifies that)
        pcfg = R.TrpoConfig(optimizer_config=R.ConjugateGradientOptimizerConfig(hpv_reg_coeff=0.1))
        agent = R.ActorCriticConfig(policy_config=pcfg).build_agent(env)
        agent.policy.policy_fn.set_weights(params)
        agent.critic.state_value_fn.set_weights(vparams)
        traj = R.Trajectory(env, T)
        R.rollout(env, agent.actor(L.RL_LANES_WARP_SPECIALIZED), R.HistoryDataBound(T, 0), traj, want_summary=False)
        log = {}
        status = agent.batch_update(traj, log)
        p, v = agent.policy.policy_fn.get_weights(), agent.critic.state_value_fn.get_weights()
        traj.close(); env.close()
        return p, v, int(status), log

    p_s, v_s, st_s, log_s = run(ctx, E, rank * E)
    same = params_identical(dist, np.concatenate([p_s, v_s]))
    res = {"params_identical_across_ranks": same, "num_steps_group": int(log_s["num_steps"])}
    if rank == 0:
        solo = R.Context(local)  # no communicator: the whole batch on one GPU
        p_f, v_f, st_f, log_f = run(solo, E * world, 0)
        rel = lambda a, b, base: float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b.astype(np.float64) - base), 1e-30))
        res.update({"max_rel": max(rel(p_s, p_f, params), rel(v_s, v_f, vparams)), "policy_delta_rel": rel(p_s, p_f, params),
                    "critic_delta_rel": rel(v_s, v_f, vparams), "num_steps_single": int(log_f["num_steps"]),
                    "status": [st_s, st_f], "num_backtracks": [int(log_s["num_backtracks"]), int(log_f["num_backtracks"])],
                    "hpv_reg_coeff": 0.1,
                    "what": f"one GAE+TRPO+critic update on {world} x {E * T} env-steps with reduced sums vs the same update on the "
                            f"concatenated {world * E * T}-step batch on one GPU; rel = |delta_group - delta_single| / |delta_single|"})
        solo.close() if hasattr(solo, "close") else None
    return res


def rl2_sized_rollout(ctx, R, L):
    """config 4, rl2-sized: k = 10 arms, n = 100 episodes per trial, GRU(14 -> 128) -> Linear(128 -> 10) (K8h); one GPU."""
    rng = np.random.default_rng(4)
    E6, T6 = 148 * 64 * 2, 199
    env6 = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(10), 100), E6, seed=7)
    net6 = R.GruLinear(ctx, env6.num_features, 128, env6.num_actions)
    net6.set_weights(R.init_gru_linear_params(rng, env6.num_features, 128, env6.num_actions))
    traj6 = R.Trajectory(env6, T6)
    spec6 = R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, seq_net=net6)
    R.rollout(env6, spec6, R.HistoryDataBound(T6, 0), traj6, want_summary=False)
    e0 = ctx.event().record()
    for _ in range(3):
        R.rollout(env6, spec6, R.HistoryDataBound(T6, 0), traj6, want_summary=False)
    e1 = ctx.event().record()
    ms = e0.elapsed_ms(e1) / 3
    flop = 2 * 3 * 128 * (env6.num_features + 128) + 2 * 128 * env6.num_actions
    fp32_peak = ctx.fp32_peak_tflops()
    rec = {"kernel": "config 4 rl2-sized: bandit meta-env (10 arms x 100 episodes) + GRU(14->128)->Linear(128->10), rollout K8s (two "
                     "launches per step: the GRU cell of all envs as bf16-piece tcgen05 MMAs with the gates in the TMEM epilogue, then "
                     "sample + env step + record, four threads per env); K8h (persistent 64-env tiles, FP32 FFMA2 GEMM) runs 338 M",
           "envs": E6, "horizon": T6, "ms": ms, "env_steps_per_s": E6 * T6 / (ms * 1e-3), "flop_per_env_step": flop,
           "fp32_tflops": flop * E6 * T6 / (ms * 1e-3) / 1e12, "measured_fma_peak_tflops": fp32_peak,
           "frac_of_fp32_peak": flop * E6 * T6 / (ms * 1e-3) / 1e12 / fp32_peak}
    out = [rec]
    # the update that consumes it (K10, gru_big.cu: tiled FP32 GEMMs over the lanes of a step): one gradient pass and one
    # Fisher-vector product through GRU(14->128)->Linear(128->10) on a quarter of those lanes (942 464 steps)
    E7 = E6 // 4
    env7 = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(10), 100), E7, seed=8)
    traj7 = R.Trajectory(env7, T6)
    R.rollout(env7, spec6, R.HistoryDataBound(T6, 0), traj7, want_summary=False)
    pol = R.Trpo(net6, R.TrpoConfig())
    adv = ctx.to_device(np.random.default_rng(5).normal(size=(T6, E7)).astype(np.float32))
    vec = np.random.default_rng(6).normal(size=net6.num_params).astype(np.float32)
    pol.probe(traj7, adv, vec)
    e0 = ctx.event().record()
    pol.probe(traj7, adv, vec)  # stats + loss/KL + gradient + one Fisher-vector product
    e1 = ctx.event().record()
    ms7 = e0.elapsed_ms(e1)
    Fh, Hh, Ah = env7.num_features, 128, env7.num_actions
    cell = 2 * 3 * Hh * (Fh + Hh)                       # gru_cell forward FLOP per step
    # stats fwd + eval fwd + grad (fwd + dh GEMM + weight grads) + FVP (fwd + tangent 2 GEMMs + dh + weight grads)
    flop7 = (2 * cell + (cell + 2 * Hh * 3 * Hh + cell) + (cell + cell + 2 * 3 * Hh * Hh + 2 * Hh * 3 * Hh + cell)) * E7 * T6
    out.append({"kernel": "config 4 rl2-sized update K10: stats + loss/KL + gradient + Fisher-vector product through GRU(14->128)->Linear "
                          "(tiled FP32 GEMMs per step, split-K weight gradients)", "envs": E7, "horizon": T6, "batch_steps": E7 * T6,
                "probe_ms": ms7, "algorithmic_tflops": flop7 / (ms7 * 1e-3) / 1e12, "measured_fma_peak_tflops": fp32_peak,
                "frac_of_fp32_peak": flop7 / (ms7 * 1e-3) / 1e12 / fp32_peak})
    traj7.close(); env7.close()
    traj6.close(); env6.close()
    return out


def run_sweep(args):
    """BASELINE config 5: rollout throughput of the config-2 env + policy over E_total = 2^10 .. 2^24 envs sharded over the
    ranks, T = 512 steps per lane where the trajectory fits (else the largest power of two whose trajectory stays under
    ~60 GB per GPU; the line says which), fused kernel picked by lanes_per_env = 0, plus the unfused step kernel (K1).
    One JSON line per E on stdout (rank 0)."""
    import relearn_b200 as R
    from relearn_b200 import _lib as L

    rank, world, local, dist = dist_setup()
    ctx = R.Context(local)
    cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
    net = R.Mlp(ctx, 5, [128], 2)
    net.set_weights(R.init_params(np.random.default_rng(0), 5, 128, 2))
    for lg in range(10, 25, 2):
        E_total = 1 << lg
        if E_total < world:
            continue
        E = E_total // world
        T = 512
        while E * T * 52 > 60e9 and T > 8:  # obs + next_obs planes, action, reward, succ
            T //= 2
        env = R.build_env(ctx, cfg, E, seed=1, lane_offset=rank * E)
        traj = R.Trajectory(env, T)
        spec = R.ActorSpec(kind=L.RL_ACTOR_CATEGORICAL_POLICY, net=net, lanes_per_env=0)
        bound = R.HistoryDataBound(T, 0)
        for _ in range(2):
            R.rollout(env, spec, bound, traj, want_summary=False)
        reps = 5 if E * T <= (1 << 28) else 2
        barrier(dist, ctx)
        e0 = ctx.event().record()
        for _ in range(reps):
            R.rollout(env, spec, bound, traj, want_summary=False)
        e1 = ctx.event().record()
        ms = max_over_ranks(dist, local, e0.elapsed_ms(e1) / reps)
        # unfused step kernel (K1) on the same lanes: one launch per step, actions resident
        env.reset_all()
        actions = ctx.to_device(np.random.default_rng(0).integers(0, 2, E).astype(np.uint8))
        for _ in range(3):
            env.step_device(actions)
        ksteps = 20
        barrier(dist, ctx)
        e0 = ctx.event().record()
        for _ in range(ksteps):
            env.step_device(actions)
        e1 = ctx.event().record()
        ms1 = max_over_ranks(dist, local, e0.elapsed_ms(e1) / ksteps)
        if rank == 0:
            emit({"sweep": "config 5", "n_gpus": world, "envs_total": E_total, "envs_per_gpu": E, "horizon": T,
                  "fused_ms_per_period": ms, "fused_env_steps_per_s": E_total * T / (ms * 1e-3),
                  "unfused_ms_per_step": ms1, "unfused_env_steps_per_s": E_total / (ms1 * 1e-3),
                  "unfused_gbs_per_gpu": B_PER_STEP_UNFUSED * E / (ms1 * 1e-3) / 1e9})
        traj.close(); env.close()
    if dist is not None:
        dist.destroy_process_group()


_REAL_STDOUT = None


def claim_stdout():
    """Route everything libraries write to fd 1 (e.g. NCCL's version banner) to stderr; the one JSON line
    of the contract goes to the original stdout through emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--envs", type=int, default=4096, help="lanes per GPU")
    ap.add_argument("--horizon", type=int, default=256, help="steps per lane per period")
    ap.add_argument("--lanes", type=int, default=0, help="threads per env in the fused kernel (0 = auto)")
    ap.add_argument("--update-iters", type=int, default=3)
    ap.add_argument("--no-update", action="store_true")
    ap.add_argument("--quick", action="store_true", help="skip the per-kernel rooflines and the CPU baseline")
    ap.add_argument("--cpu-update-sample", dest="cpu_update_full", action="store_false",
                    help="time the CPU update baseline on a 65 536-step sample instead of the full batch")
    ap.add_argument("--sweep", action="store_true", help="BASELINE config 5: rollout throughput over E = 2^10 .. 2^24 (see run_sweep)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the trajectory of the last timed step (rank 0's lanes) to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and (args.sweep or args.impl == "reference"):
        ap.error("--dump-outputs writes the GPU rollout's trajectory: it needs --impl ours and no --sweep")
    if args.sweep:
        run_sweep(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
