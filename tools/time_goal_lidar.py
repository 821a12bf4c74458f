"""Time observe_goal_lidar: the optional-key env step and a point PPO iteration, with and without the lidar block.

  1. mr_env_step at 2^22 point envs (the optional-key step kernel, one launch per step, CUDA events over --steps
     launches, the configurations alternated --rounds times): observe_goal_dist alone (15 floats) against
     observe_goal_lidar with 10 bins (24 floats) and with 16 bins (30 floats).  The working set (~0.9 GB of state,
     rows and terminal rows) is far beyond the 126 MB L2.
  2. One PPO iteration (collect_rollouts + train) at the flagship shape of data/configs/point-ppo-b200.yaml (4096
     envs x 296 steps, 10 epochs of 64 minibatches), on the observe_goal_dist row against the lidar row (10 bins):
     host clock around iterations that end in a device synchronise, after one warm-up iteration.

Prints one JSON object with the card's name and power limit beside the numbers.

  python tools/time_goal_lidar.py [--steps 200] [--rounds 3] [--iters 3] [--out profiles/goal_lidar.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

STEP_CONFIGS = {
    "goal_dist": {"observe_goal_dist": True},
    "lidar10": {"observe_goal_lidar": True},
    "lidar16": {"observe_goal_lidar": True, "lidar_num_bins": 16},
}
PPO_CONFIGS = {"goal_dist": {"observe_goal_dist": True}, "lidar10": {"observe_goal_lidar": True}}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the number is still worth printing without it
        q = f"unavailable ({e})"
    return {"device": name, "power_limit, max_sm_clock": q}


def time_steps(envs, acts, steps, rounds):
    """ms per mr_env_step launch of every env, the configurations alternated round by round."""
    out = {k: [] for k in envs}
    for k, env in envs.items():   # warm-up: module load, first-touch of every buffer
        for _ in range(10):
            env.step_tensor(acts)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, env in envs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                env.step_tensor(acts)
            b.record()
            b.synchronize()
            out[k].append(a.elapsed_time(b) / steps)
    return out


def time_ppo(cfg, iters):
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    n, T = 4096, 296
    env = GpuVecEnv("point", n, seed=0, time_limit=1000, terminate_on_goal=True, robot_config=cfg)
    model = PPO("MlpPolicy", env, n_steps=T, batch_size=18944, n_epochs=10, ent_coef=0.05, gae_lambda=0.5, seed=0,
                verbose=0)
    model.learn(total_timesteps=n * T)   # warm-up iteration
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    model.learn(total_timesteps=iters * n * T)   # starts with the env's reset, as every learn() does
    torch.cuda.synchronize()
    assert model.num_timesteps == iters * n * T
    dt = (time.perf_counter() - t0) / iters
    assert torch.isfinite(model.updater.params).all()
    return {"obs_dim": env.obs_dim, "s_per_iteration": dt, "env_steps_per_s": n * T / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-envs", type=int, default=1 << 22)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_goal_lidar.py measures on a CUDA device; there is none here")
    from mobrob_b200 import GpuVecEnv

    res = {"card": card(), "n_envs": args.n_envs, "steps_per_window": args.steps}
    envs = {k: GpuVecEnv("point", args.n_envs, seed=0, time_limit=1000, terminate_on_goal=True, robot_config=c)
            for k, c in STEP_CONFIGS.items()}
    for env in envs.values():
        env.reset_tensor()
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.rand((args.n_envs, 2), device="cuda", generator=g) * 3 - 1.5
    ms = time_steps(envs, acts, args.steps, args.rounds)
    res["env_step"] = {k: {"obs_dim": envs[k].obs_dim, "ms_per_step": v, "median_ms": float(np.median(v)),
                           "env_steps_per_s": args.n_envs / (float(np.median(v)) * 1e-3),
                           "row_bytes_written": 4 * envs[k].obs_dim}
                       for k, v in ms.items()}
    del envs, acts
    torch.cuda.empty_cache()
    res["ppo_iteration"] = {k: time_ppo(c, args.iters) for k, c in PPO_CONFIGS.items()}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
