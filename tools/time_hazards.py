"""Time the hazards: the optional-key env step with and without 8 hazards, the layout burst of a step in which every
env does a full reset, the car step, and a point PPO iteration on the hazards row.

  1. mr_env_step at 2^22 point envs (CUDA events over --steps launches, configurations alternated --rounds times):
     observe_goal_dist (15 floats) against observe_goal_dist + 8 hazards with observe_hazards and constrain_hazards
     (25 floats).  Time limit 1000: almost no step resets an env.
  2. The same two configurations with time_limit = 1: every env times out every step, so every env does a full reset
     (for the hazard envs, a layout of robot, goal and 8 hazards drawn on the device) -- the burst after simultaneous
     time-outs.
  3. The car step at 16 384 envs: observe_goal_dist against observe_goal_dist + 8 hazards.
  4. One PPO iteration at the flagship shape (4096 envs x 296 steps, 10 epochs of 64 minibatches) on the
     observe_goal_dist row against the hazards row (observe_hazards, 10 bins: 24 floats).

Prints one JSON object with the card's name and power limit, read in the same run, beside the numbers.

  python tools/time_hazards.py [--steps 200] [--rounds 3] [--iters 3] [--out profiles/hazards.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
import torch

from time_goal_lidar import card, time_ppo, time_steps

HAZ = {"hazards_num": 8, "observe_hazards": True, "constrain_hazards": True}
STEP_CONFIGS = {"goal_dist": {"observe_goal_dist": True}, "hazards8": {"observe_goal_dist": True, **HAZ}}
PPO_CONFIGS = {"goal_dist": {"observe_goal_dist": True}, "hazards8": {"hazards_num": 8, "observe_hazards": True}}


def step_block(kind, n, configs, time_limit, steps, rounds):
    from mobrob_b200 import GpuVecEnv

    envs = {k: GpuVecEnv(kind, n, seed=0, time_limit=time_limit, terminate_on_goal=True, robot_config=c)
            for k, c in configs.items()}
    for env in envs.values():
        env.reset_tensor()
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.rand((n, 2), device="cuda", generator=g) * 3 - 1.5
    ms = time_steps(envs, acts, steps, rounds)
    out = {k: {"obs_dim": envs[k].obs_dim, "ms_per_step": v, "median_ms": float(np.median(v)),
               "env_steps_per_s": n / (float(np.median(v)) * 1e-3)} for k, v in ms.items()}
    for k, env in envs.items():
        if env.hazards_num:
            env._check_layouts()   # no failed layout inside the timed windows
    del envs, acts
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-envs", type=int, default=1 << 22)
    ap.add_argument("--car-envs", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_hazards.py measures on a CUDA device; there is none here")
    res = {"card": card(), "n_envs": args.n_envs, "car_envs": args.car_envs, "steps_per_window": args.steps}
    res["env_step"] = step_block("point", args.n_envs, STEP_CONFIGS, 1000, args.steps, args.rounds)
    res["env_step_all_full_resets"] = step_block("point", args.n_envs, STEP_CONFIGS, 1, max(args.steps // 4, 10),
                                                 args.rounds)
    res["car_env_step"] = step_block("car", args.car_envs, STEP_CONFIGS, 1000, max(args.steps // 4, 10), args.rounds)
    res["ppo_iteration"] = {k: time_ppo(c, args.iters) for k, c in PPO_CONFIGS.items()}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
