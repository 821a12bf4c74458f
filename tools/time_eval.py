"""Time evaluate_policy's device path (mr_evaluate) against the torch loop of tools/eval_policy.py.

Workload (BASELINE.json configs[1] scaled to SB3's evaluate_policy): the shipped point policy, 16 384 envs,
time_limit=1000, terminate_on_goal, deterministic, n_eval_episodes = 4 x 16 384.  The torch loop (one mr_policy_forward,
one mr_env_step and a handful of torch ops per step) is timed over the same number of steps the device path takes.
Then the car at 16 384 envs (per-step path: one launch + mr_env_step + a 4-byte read-back per step).

Rates are END-TO-END: env-steps per second of the whole call (host clock around work that ends in a device
synchronise), and the algorithmic FP32 rate of the policy forward at 20 352 FLOP per env-step (SURVEY section 8d) --
not any kernel's share of peak.

  python tools/time_eval.py [--reps 5] [--car-episodes 16384] [--out profiles/eval_time.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
import torch

FLOP_PER_ENV_STEP = 20352


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the number is still worth printing without it
        q = f"unavailable ({e})"
    return {"device": name, "power_limit, max_sm_clock": q}


def time_device(zip_path, env_name, n, n_episodes, time_limit, reps):
    from mobrob_b200 import GpuVecEnv, evaluate_policy
    from mobrob_b200.ppo import PPO

    model = PPO.load(zip_path)
    env = GpuVecEnv(env_name, n, seed=0, time_limit=time_limit, terminate_on_goal=True)
    evaluate_policy(model, env, n_episodes)   # warm-up: module load, shared-memory opt-in, allocator
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        before = env.eval_steps
        t0 = time.perf_counter()
        mean, std = evaluate_policy(model, env, n_episodes)   # returns after a device synchronise (record read-back)
        dt = time.perf_counter() - t0
        steps = env.eval_steps - before
        out.append({"seconds": dt, "steps": steps, "env_steps_per_s": n * steps / dt, "mean_reward": float(mean)})
    return out


def summarize(runs):
    rates = np.array([r["env_steps_per_s"] for r in runs])
    return {"env_steps_per_s_median": float(np.median(rates)), "env_steps_per_s_min": float(rates.min()),
            "env_steps_per_s_max": float(rates.max()),
            "fp32_forward_flop_per_s_median": float(np.median(rates)) * FLOP_PER_ENV_STEP,
            "steps_per_call": [r["steps"] for r in runs], "seconds_per_call": [round(r["seconds"], 5) for r in runs]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--car-episodes", type=int, default=16384)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_eval.py measures the GPU: no CUDA device here")
    import eval_policy

    pol = os.path.join(ROOT, "tests", "golden", "policies")
    res = {"card": card(), "workload": {"n_envs": a.n, "time_limit": 1000, "deterministic": True,
                                        "point_n_eval_episodes": 4 * a.n, "car_n_eval_episodes": a.car_episodes}}
    point = time_device(os.path.join(pol, "point-ppo.zip"), "point", a.n, 4 * a.n, 1000, a.reps)
    res["point_device"] = summarize(point)
    steps = int(np.median([r["steps"] for r in point]))
    eval_policy.evaluate_gpu(os.path.join(pol, "point-ppo.zip"), a.n, horizon=1000, steps=50)   # warm-up
    loop = []
    for _ in range(a.reps):
        g = eval_policy.evaluate_gpu(os.path.join(pol, "point-ppo.zip"), a.n, horizon=1000, steps=steps)
        loop.append({"env_steps_per_s": g["env_steps_per_s"], "steps": steps, "seconds": a.n * steps / g["env_steps_per_s"]})
    res["point_torch_loop"] = summarize(loop)
    res["point_speedup_median"] = res["point_device"]["env_steps_per_s_median"] / res["point_torch_loop"]["env_steps_per_s_median"]
    car = time_device(os.path.join(pol, "car-ppo.zip"), "car", a.n, a.car_episodes, 1000, max(2, a.reps // 2))
    res["car_device"] = summarize(car)
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
