#!/usr/bin/env python
"""bench.py -- env-steps/sec (rollout + PPO update), point env, N x B200.

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA hot path)
  python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle port of the
                                                             # reference stack on the host cores
  python bench.py --env car --envs-per-gpu 16384            # BASELINE configs[3]
  python bench.py --gpus 8 --envs-per-gpu 8192 [--env car]  # BASELINE configs[4] (under torchrun)
  python bench.py ... --dump-outputs DIR                     # also write the last timed step's outputs
                                                             # as DIR/<name>.npy (see dump_outputs)

A "step" is one PPO iteration of the workload (default: data/configs/point-ppo-b200.yaml) on every
rank: rollout of n_steps x envs-per-gpu env-steps (point: ONE fused kernel), GAE, then 10 epochs of
minibatches of 18 944 samples (forward, clipped loss, backward, grad-norm clip, Adam) in one persistent
kernel per epoch.  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definitions.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ENVS = 4096          # per GPU (weak scaling), default workload
N_STEPS = 296
BATCH = 18944          # = 148 SMs x 128-sample tiles
N_EPOCHS = 10
DEFAULTS = {"point": (4096, 296), "car": (16384, 74)}   # (envs per GPU, n_steps): 64 minibatches per epoch each
OBS_DIM = {"point": 14, "car": 26}

# algorithmic work of the dominant kernel (ppo_epoch_tc_kernel), DESIGN.md "Kernels":
# per sample and epoch: forward + backward-data + backward-weight of both O-64-64 towers (SURVEY.md section 8d)
FLOP_PER_SAMPLE_EPOCH = 61056
FLOPS = {"point": 61056, "car": 70272}
ENV_STEP_BYTES = 145           # SURVEY.md section 8d, stand-alone point env-step


def metric_name(env):
    return f"env-steps/sec (rollout+PPO update), {env} env"


def workload_name(env, n_envs):
    which = {("point", 4096): "configs[2]", ("car", 16384): "configs[3]", ("point", 8192): "configs[4] (8192/GPU)",
             ("car", 8192): "configs[4] (8192/GPU, car)"}.get((env, n_envs), "custom size")
    return f"{env} env {n_envs} parallel envs/GPU full rollout + GAE + PPO update (BASELINE.json {which})"


METRIC = metric_name("point")
WORKLOAD = workload_name("point", N_ENVS)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--env", default="point", choices=["point", "car"])
    ap.add_argument("--envs-per-gpu", type=int, default=None, help="default 4096 (point) / 16384 (car)")
    ap.add_argument("--n-steps", type=int, default=None, help="rollout length; default 296 (point) / 74 (car)")
    ap.add_argument("--batch", type=int, default=BATCH, help="minibatch size per GPU (multiple of 128; default 18944)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the stand-alone env-step roofline and the "
                    "SB3-host-permutation e2e variant (they do not change value / e2e)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed as DIR/<name>.npy (rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's outputs: it needs --impl ours")
    d_envs, d_steps = DEFAULTS[a.env]
    a.envs_per_gpu = a.envs_per_gpu or d_envs
    a.n_steps = a.n_steps or d_steps
    return a


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.proc, self.lines, self.index = None, [], index
        self.active = True   # only samples taken while a timed region runs are kept

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            if self.active:
                self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback"


# ------------------------------------------------------------------------------------------
def cpu_port_step(n_envs, n_steps, batch, n_epochs, state):
    """One iteration of the reference algorithm on the host: oracle env + torch-CPU PPO."""
    import torch

    from oracle import sb3_oracle

    ro, pol, opt = state["ro"], state["pol"], state["opt"]
    eps = torch.randn((n_steps, n_envs, 2), generator=state["gen"]).numpy()
    buf = ro.collect(eps)
    sb3_oracle.train_epochs(pol, opt, buf, n_epochs, batch, rng=state["rng"], clip_range=0.2, ent_coef=0.05,
                            vf_coef=0.5)
    return n_envs * n_steps


def cpu_port_setup(n_envs, n_steps, seed=0, env="point"):
    import numpy as np
    import torch

    from oracle import sb3_oracle
    from oracle.vec_oracle import GoalVecOracle

    if env == "point":
        from oracle import point_oracle as po

        body = po.PointBody(n_envs)
    else:
        from oracle import car_oracle as co

        body = co.CarBody(n_envs)
    torch.manual_seed(seed)
    pol = sb3_oracle.MlpPolicyOracle(OBS_DIM[env])
    venv = GoalVecOracle(body, seed=seed, time_limit=1000, terminate_on_goal=True)
    ro = sb3_oracle.RolloutOracle(venv, pol, n_steps, gamma=0.99, gae_lambda=0.5)
    return dict(ro=ro, pol=pol, opt=sb3_oracle.make_adam(pol), gen=torch.Generator().manual_seed(seed),
                rng=np.random.RandomState(seed))


def cpu_sample_shape(args):
    """Workload of one CPU-arm step.  Point: the bench workload itself (same envs, rollout length,
    minibatch size and epochs).  Car: the numpy car oracle (per-substep contact solves) runs at ~1.6e3
    env-steps/s, so a step is a bounded sample of 1024 envs x 16 steps with proportionally small
    minibatches (64 per epoch, as in the full workload)."""
    if args.env == "point":
        n_envs, T = args.envs_per_gpu, args.n_steps
        return n_envs, T, min(args.batch, n_envs * T), True
    n_envs, T = 1024, 16
    return n_envs, T, n_envs * T // 64, False


def run_reference(args):
    """CPU arm: the oracle port of the reference stack (numpy fp64 env + torch-CPU PPO = SB3's
    arithmetic) with every host thread torch / numpy will use, on our arm's config."""
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_envs, T, batch, same = cpu_sample_shape(args)
    state = cpu_port_setup(n_envs, T, env=args.env)
    for _ in range(args.warmup):
        cpu_port_step(n_envs, T, batch, N_EPOCHS, state)
    t0 = time.perf_counter()
    done = 0
    for _ in range(args.steps):
        done += cpu_port_step(n_envs, T, batch, N_EPOCHS, state)
    dt = time.perf_counter() - t0
    value = done / dt
    sample = (f"{n_envs} envs x {T} steps per step ({n_envs * T} env-steps), {N_EPOCHS} epochs of "
              f"minibatch {batch}; numpy fp64 oracle env + torch-CPU PPO (SB3 arithmetic)"
              + ("; the full per-GPU workload of our arm" if same else "; bounded sample of our arm's workload"))
    line = {"impl": "reference", "metric": metric_name(args.env), "value": value, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 physics / f32 PPO",
            "data": "synthetic",
            "config": {"workload": workload_name(args.env, args.envs_per_gpu), "n_envs_per_gpu": args.envs_per_gpu,
                       "n_steps": args.n_steps, "batch_size": args.batch, "n_epochs": N_EPOCHS, "sample": sample,
                       "same_workload_as_ours": same,
                       "note": "one host runs ONE rank's share whatever --gpus says (the CPU arm does not shard)"},
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from mobrob_b200 import _lib
    from mobrob_b200.rl_control.ppo import PPOCtrl

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: mobrob_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    env_name, n_envs, n_steps = args.env, args.envs_per_gpu, args.n_steps
    steps_per_iter = n_envs * n_steps  # per rank
    batch = args.batch
    if steps_per_iter % batch:
        raise SystemExit(f"envs-per-gpu x n-steps = {steps_per_iter} is not a multiple of the minibatch {batch}")
    # PPO's default index stream: mr_device_permutation (keyed Feistel bijection on the device);
    # permutation="sb3" would reproduce numpy's stream bit for bit from the host (parity runs)
    cfg = dict(env_name=env_name, time_limit=1000, n_envs=n_envs, vec_env_type="dummy", enable_gui=False, seed=0,
               ppo_kwargs=dict(policy="MlpPolicy", n_steps=n_steps, n_epochs=N_EPOCHS, ent_coef=0.05,
                               gae_lambda=0.5, batch_size=batch, verbose=0))
    ctrl = PPOCtrl.from_config(cfg)
    ctrl.ppo.tensorboard_log = None
    model = ctrl.ppo
    assert model.permutation == "device"
    up = model.updater
    built = [t.clone() for t in (up.params, up.exp_avg, up.exp_avg_sq, up.step)]

    def iteration():
        model.collect_rollouts()
        model.train()

    def restart():
        """Put the model back into the state it was built in: seeded parameters, zero Adam state and counters,
        the environments' seeded first reset.  The update adds the CTAs' partial gradients in L2 in no fixed
        order, so a minibatch is reproducible to rounding only, and over several iterations the rollouts of two
        runs drift apart.  Every timed step therefore starts here: it then reads the same inputs in every run."""
        for t, s in zip((up.params, up.exp_avg, up.exp_avg_sq, up.step), built):
            t.copy_(s)
        model._rollout_count = model._train_count = 0
        model.env.seed(cfg["seed"])
        model._last_obs = model.env.reset_tensor().clone()   # what collect_rollouts does on a new model
        model._last_episode_starts = torch.ones(n_envs, dtype=torch.float32, device=dev)

    for _ in range(max(args.warmup, 3)):
        iteration()
    barrier()

    # ---- value: device-resident, CUDA events around each step, max over ranks ------------------------
    # restart() lies between the steps, outside the events; env.seed synchronises the stream, so a spin kernel
    # keeps the device busy while the host enqueues the step (its launches then run back to back as before)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, launches = 0.0, 0
    for _ in range(args.steps):
        restart()
        barrier()
        torch.cuda._sleep(10_000_000)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = _lib.launch_count()
        e0.record()
        iteration()
        e1.record()
        launches += _lib.launch_count() - launches0
        e1.synchronize()
        ms += e0.elapsed_time(e1)
    barrier()
    ms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    value = steps_per_iter * world * args.steps / (ms / 1e3)
    sampler.active = False
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model)   # before anything below steps the model further

    # ---- phase split and roofline of the dominant kernel (live CUDA events, same stream) -----------
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    barrier()
    ev[0].record()
    model.collect_rollouts()
    ev[1].record()
    model.train()
    ev[2].record()
    barrier()
    rollout_ms, train_ms = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
    launch_ms, launch_epochs = time_update_kernel(model, dev, batch)
    peaks, peaks_src = measured_peaks()
    fp32_peak = 148 * 128 * 2 * peaks.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
    tensor_peak = peaks.get("bf16_tflops", 1590.0)   # burst figure: the kernel is timed alone
    flops = FLOPS[env_name]
    achieved = flops * steps_per_iter * launch_epochs / (launch_ms * 1e-3) / 1e12
    default_cfg = (env_name, n_envs, n_steps, batch) == ("point", N_ENVS, N_STEPS, BATCH)
    kp = 16 if OBS_DIM[env_name] + 1 <= 16 else 32
    roofline = {"kernel": f"ppo_epoch_tc_kernel<{kp}> (one launch = {launch_epochs} epoch(s) = "
                          f"{launch_epochs * (steps_per_iter // batch)} minibatch updates: "
                          "tcgen05 forward/backward GEMMs, bulk-reduced gradient, clip, Adam)",
                "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                "frac": achieved / tensor_peak, "traffic": UPDATE_KERNEL_DRAM_BYTES.get(launch_epochs) if default_cfg else None,
                "ms_per_launch": launch_ms, "epochs_per_launch": launch_epochs,
                "algorithmic": f"{flops} FLOP/sample/epoch (SURVEY 8d) x {steps_per_iter} samples x {launch_epochs} epoch(s) per launch",
                "peak_source": f"bf16_tflops of MEASURED_PEAKS.json ({peaks_src})",
                "tensor_flops_issued_per_algorithmic_flop": 3,
                "frac_issued": 3 * achieved / tensor_peak,
                "frac_of_fp32_fma_peak": achieved / fp32_peak,
                "note": "fp32 products are formed from two fp16 parts per operand (3 MMAs per product, gradients within "
                        "1e-6 of torch fp32), so 3x the algorithmic FLOPs go through the tensor pipe; the kernel is bound by the "
                        "per-minibatch dependency chain (element-wise passes between the GEMMs, one grid barrier), see profiles/",
                "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full, profiles/ (per launch)",
                "step_share": {"rollout_ms": rollout_ms, "update_ms": train_ms,
                               "update_kernel_ms": launch_ms * (N_EPOCHS // launch_epochs)}}
    env_roof = None
    if default_cfg and not args.no_extras and world == 1:
        env_roof = time_env_step_kernel(dev, peaks)

    # ---- e2e: the public API, PPOCtrl.learn(), as a user calls it: host loop, logger and episode-buffer
    #      reads (D2H from the device into pinned memory) every iteration --------------------------------
    def timed_learn():
        barrier()
        model.learn(total_timesteps=steps_per_iter * world * 3, reset_num_timesteps=True)  # warm (logger paths too)
        barrier()
        t0 = time.perf_counter()
        model.learn(total_timesteps=steps_per_iter * world * args.steps, reset_num_timesteps=True)
        barrier()
        wall = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        return steps_per_iter * world * args.steps / float(wall.item())

    model.verbose = 0
    sampler.active = True
    e2e_value = timed_learn()
    sampler.active = False
    d2h = EP_D2H_BYTES + 12 * 4
    e2e_host = None
    if not args.no_extras and env_name == "point" and world == 1:
        # SB3's own semantics for RolloutBuffer.get: permutations drawn on the HOST (thread pool, one iteration
        # ahead) and copied from pinned memory every epoch
        model.permutation = "pool"
        e2e_host = {"value": timed_learn(), "unit": "env-steps/s",
                    "h2d_bytes_per_step": N_EPOCHS * steps_per_iter * 8 * world, "d2h_bytes_per_step": d2h * world,
                    "what": "PPOCtrl.learn() with permutation='pool': int64 minibatch permutations drawn on the host "
                            "and copied H2D every epoch (SB3 draws them on the host too)"}
        model.permutation = "device"
    clocks = sampler.stop() if rank == 0 else None   # sampled every 20 ms inside the value and e2e timed regions

    # ---- with several ranks: are they still the same model, and is the sharded update the single-GPU update? --
    mg = None
    if world > 1:
        from mobrob_b200.selfcheck import sharded_update_check

        torch.cuda.synchronize(dev)
        digest = torch.stack([model.updater.params.double().sum(), model.updater.params.double().abs().sum(),
                              model.updater.exp_avg_sq.double().sum()])
        gathered = [torch.empty_like(model.updater.params) for _ in range(world)]
        dist.all_gather(gathered, model.updater.params)
        identical = all(torch.equal(gathered[0], g) for g in gathered)
        chk = sharded_update_check(dev, modes=("fused",), obs_dim=OBS_DIM[env_name])
        timed_out = bool(model._xchg.timed_out()) if model._xchg is not None else False
        mg = {"identical": bool(identical and chk["fused"]["identical_across_ranks"]),
              "params_identical_after_timed_region": bool(identical),
              "param_digest_rank0": [float(x) for x in digest.tolist()],
              "max_rel_vs_single": chk["fused"]["max_rel_vs_single"], "moved": chk["moved"],
              "exchange_timed_out": bool(timed_out or chk["fused"]["exchange_timed_out"]),
              "what": "all-gather of the parameters after the timed region (bit-identical on every rank); then the "
                      "fused epoch kernel on a small sharded synthetic rollout against a single-GPU update of the whole "
                      "rollout on rank 0 (mobrob_b200/selfcheck.py), difference relative to the update's size",
              "ok": bool(identical and chk["ok"] and not timed_out)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        sys.exit(0 if mg is None or mg["ok"] else 3)

    line = {"metric": metric_name(env_name), "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 physics / f32 policy+PPO", "data": "synthetic",
            "config": {"workload": workload_name(env_name, n_envs), "n_envs_per_gpu": n_envs, "n_steps": n_steps,
                       "batch_size": batch, "n_epochs": N_EPOCHS, "minibatches_per_epoch": steps_per_iter // batch,
                       "permutation": "device (mr_device_permutation, the PPO default)",
                       "parallelism": f"dp{world} (envs sharded, gradient all-reduce)",
                       "l2": f"no flush: every step rewrites its {steps_per_iter * 84 / 1e6:.0f} MB rollout working set and "
                             f"gathers it in {N_EPOCHS} fresh random orders (126 MB L2)"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": d2h * world,
                    "what": "PPOCtrl.learn() wall clock (the call examples/train.py makes): host loop, callbacks, logger; "
                            "every iteration reads the newest episodes and the update's statistics D2H into pinned memory. "
                            "The workload has no per-step host inputs -- envs, action noise and minibatch indices live on "
                            "the device (0 B H2D); e2e_sb3_host_stream is the variant whose indices come from the host"},
            "roofline": roofline}
    if e2e_host is not None:
        line["e2e_sb3_host_stream"] = e2e_host
    if env_roof is not None:
        line["roofline_env_step"] = env_roof
    if mg is not None:
        line["multi_gpu_check"] = mg
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(args)
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    if mg is not None and not mg["ok"]:
        sys.exit(3)


EP_D2H_BYTES = 100 * 12 + 8


# dram bytes of one ppo_epoch_tc_kernel launch of the default workload by epochs per launch (ncu --set full,
# profiles/r02_ncu_full.txt): 10 epochs 1145.2 MB read + 7.6 MB written (the 116 MB of records partly stay in the
# 126 MB L2 from one epoch to the next); a single-epoch launch 154.2 MB + 3.9 MB
UPDATE_KERNEL_DRAM_BYTES = {10: 1152.8e6, 1: 158.05e6}
ENV_STEP_DRAM_BYTES = 808.1e6      # 318.8 MB read + 489.3 MB written at 2^22 envs (profiles/r01_env_step_ncu_final.txt)


DUMP_ROLLOUT_BYTES = 32 << 20


def dump_outputs(out_dir, model):
    """What one timed step hands its caller, as of the last timed step, written as float32 / float64 .npy:
    the rollout buffer collect_rollouts() fills (observations, actions, rewards, episode starts, values, log
    probabilities, GAE advantages and returns), the policy parameters train() leaves and the update's logger
    statistics.  The buffer is n_steps x n_envs deep (107 MB for the default point workload), so it is written
    for a fixed, seeded sample of environments, every time step of each, at most DUMP_ROLLOUT_BYTES;
    sample_env_index holds which.  Every timed step starts from the seeded state the model was built in (see
    restart in run_ours), so two runs with the same arguments feed the path identical inputs and two builds can
    be compared array by array: the rollout bit for bit, the parameters to the rounding of the update's sums."""
    import numpy as np
    import torch

    buf, n_steps, n_envs = model.buf, model.n_steps, model.env.num_envs
    bytes_per_env = n_steps * sum(v[0, 0].numel() * v.element_size() for v in buf.values())
    k = min(n_envs, max(1, DUMP_ROLLOUT_BYTES // bytes_per_env))
    envs = np.sort(np.random.default_rng(0).choice(n_envs, k, replace=False))
    idx = torch.as_tensor(envs, device=model.device)
    arrays = {f"rollout_{name}": v.index_select(1, idx) for name, v in buf.items()}
    arrays["policy_params"] = model.updater.params
    arrays["train_stats"] = model._train_stats
    arrays["sample_env_index"] = torch.as_tensor(envs, dtype=torch.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def time_update_kernel(model, dev, batch=BATCH):
    """Average duration of the update's cooperative launch alone, shaped as PPO.train launches it (every epoch of
    the update in ONE launch when the rollout divides into whole minibatches, else one epoch), CUDA events on the
    launching stream.  Returns (ms per launch, epochs per launch).  Parameters and Adam state are restored
    afterwards (the launches are real updates)."""
    import torch

    up, b = model.updater, model.buf
    T, N = model.n_steps, model.env.num_envs
    saved = [t.clone() for t in (up.params, up.exp_avg, up.exp_avg_sq, up.step)]
    epochs = model.n_epochs if (T * N) % batch == 0 and model.n_epochs <= 32 else 1
    stats, rows = up.prepare_epochs_device(b["advantages"], 12345, list(range(epochs)), batch, N, T)
    stats, rows = stats.view(-1, 3), rows[:epochs].reshape(-1)
    up.pack(b)
    for _ in range(2):
        up.train_epoch_fused(None, None, stats, batch, N, T, rows=rows)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        up.train_epoch_fused(None, None, stats, batch, N, T, rows=rows)
    e1.record()
    torch.cuda.synchronize(dev)
    for t, sv in zip((up.params, up.exp_avg, up.exp_avg_sq, up.step), saved):
        t.copy_(sv)
    return e0.elapsed_time(e1) / reps, epochs


def time_env_step_kernel(dev, peaks):
    """Stand-alone env-step kernel at N = 2^22 envs (state >> L2): HBM roofline of K1."""
    import numpy as np
    import torch

    from mobrob_b200 import GpuVecEnv, _lib as L, seeding

    n = 1 << 22
    env = GpuVecEnv("point", n, seed=None, time_limit=1000, terminate_on_goal=True, device=dev.index)
    # cheap synthetic seeding for 4M envs: replicate a block of real PCG64 streams
    blk = 4096
    init, goal, eng = seeding.vec_env_streams(0, blk)
    reps = n // blk
    init = np.tile(init, (reps, 1)); goal = np.tile(goal, (reps, 1))
    init[:, 1] += np.repeat(np.arange(reps, dtype=np.uint64), blk) * np.uint64(2654435761)
    goal[:, 1] += np.repeat(np.arange(reps, dtype=np.uint64), blk) * np.uint64(40503)
    eng = np.arange(n, dtype=np.int64)
    L.check(env.lib.mr_env_seed(env._h, L.ptr(init), L.ptr(goal), L.ptr(eng), env._stream()))
    env.reset_tensor()
    act = (torch.rand((n, 2), device=dev) * 2 - 1).sign().contiguous()
    for _ in range(3):
        env.step_tensor(act)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 20
    e0.record()
    for _ in range(iters):
        env.step_tensor(act)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    achieved = ENV_STEP_BYTES * n / (ms * 1e-3) / 1e9
    env.close()
    return {"kernel": "point_step_kernel", "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"],
            "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": ENV_STEP_DRAM_BYTES, "ms_per_launch": ms,
            "n_envs": n, "env_steps_per_s": n / (ms * 1e-3),
            "note": "algorithmic 145 B/env-step (SURVEY 8d); the state is fp64, physical traffic is 198 B/env-step (76 read, 122 written)"}


def cpu_baseline(args):
    """One step of the CPU arm's workload (see cpu_sample_shape)."""
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_envs, T, batch, same = cpu_sample_shape(args)
    state = cpu_port_setup(n_envs, T, env=args.env)
    t0 = time.perf_counter()
    done = cpu_port_step(n_envs, T, batch, N_EPOCHS, state)
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": f"one iteration of {n_envs} envs x {T} steps ({done} env-steps), {N_EPOCHS} epochs of "
                      f"minibatch {batch}; numpy fp64 oracle env + torch-CPU PPO; {dt:.1f} s"
                      + ("; the full per-GPU workload" if same else "; bounded sample"),
            "reference_stack_historical": "1026 env-steps/s (SB3 + mujoco-py, 2 subproc envs; BASELINE.md)"}


def _claim_stdout():
    """The contract is ONE JSON line on stdout: keep a private handle to the real stdout and point
    fd 1 at stderr, so that anything a library prints (NCCL's version banner, torch warnings)
    cannot land in front of it."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


if __name__ == "__main__":
    _claim_stdout()
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
