"""Time follow_waypoints end to end, and the host loop it replaces.

  1. The point robot (shipped policy, default row: the fused kernel) at 16 384 envs x K = 8 waypoints, and the car
     (shipped policy: the per-step path) at 16 384 envs x K = 4.  Waypoints are seeded draws inside the goal box.
     Host clock around the call, which ends in a device synchronise (the results are copied to the host); one warm-up
     call first.  Rate = env-steps the call took (sum of steps_taken) / time.
  2. The host loop over the same semantics (forward, step_tensor, get_pos, set_goals per step, as
     tests/test_waypoints_gpu.py runs it) at --host-n envs for --host-steps steps: the per-step cost a planner pays
     today, and its env-steps/s.

Prints one JSON object with the card's name, power limit and max SM clock read in the same call.

  python tools/time_waypoints.py [--n 16384] [--max-steps 1000] [--host-n 16384] [--host-steps 50] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
import torch

from time_goal_lidar import card  # noqa: E402


def waypoints(n, K, seed):
    return np.random.default_rng(seed).uniform(-2.0, 2.0, (n, K, 2)).astype(np.float32)


def time_call(model, name, n, K, max_steps, reps):
    from mobrob_b200 import GpuVecEnv, follow_waypoints

    out = []
    for r in range(reps + 1):   # the first call is the warm-up
        env = GpuVecEnv(name, n, seed=r, time_limit=None, terminate_on_goal=False)
        env.reset_tensor()
        W = waypoints(n, K, r)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = follow_waypoints(model, env, W, max_steps)
        dt = time.perf_counter() - t0
        if r:
            out.append({"s": dt, "env_steps": int(res["steps"].sum()), "max_steps_used": int(res["steps"].max()),
                        "waypoints_reached": float((res["arrivals"] >= 0).mean())})
    best = min(out, key=lambda x: x["s"])
    return {"n": n, "K": K, "max_steps": max_steps, "calls": out,
            "env_steps_per_s_best": best["env_steps"] / best["s"],
            "env_steps_per_s_median": float(np.median([x["env_steps"] / x["s"] for x in out]))}


def time_host_loop(model, name, n, K, steps):
    """The planner's loop driven from the host, all envs stepping, goals switched with set_goals."""
    from mobrob_b200 import GpuVecEnv

    env = GpuVecEnv(name, n, seed=0, time_limit=None, terminate_on_goal=False)
    env.reset_tensor()
    W = waypoints(n, K, 0)
    k = np.zeros(n, np.int64)
    env.set_goals(W[:, 0])
    obs = env.get_obs_tensor()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        act, _, _ = model.policy.forward_tensor(obs, None)
        env.step_tensor(act.clamp(-1.0, 1.0).contiguous())
        p = env.get_pos().cpu().numpy()
        g = W[np.arange(n), np.minimum(k, K - 1)].astype(np.float64)
        hit = (np.hypot(p[:, 0] - g[:, 0], p[:, 1] - g[:, 1]) < 0.3) & (k < K)
        k[hit] += 1
        sw = np.nonzero(hit & (k < K))[0]
        if len(sw):
            env.set_goals(W[sw, k[sw]], indices=sw)
            obs = env.get_obs_tensor()
        else:
            obs = env.obs
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"n": n, "K": K, "steps": steps, "s": dt, "env_steps_per_s": n * steps / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--max-steps", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-n", type=int, default=16384)
    ap.add_argument("--host-steps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_waypoints needs a CUDA device")
    from mobrob_b200.ppo import PPO

    pol = {m: PPO.load(os.path.join(ROOT, "tests", "golden", "policies", f"{m}-ppo.zip")) for m in ("point", "car")}
    res = {"card": card(),
           "point_fused": time_call(pol["point"], "point", a.n, 8, a.max_steps, a.reps),
           "car_per_step": time_call(pol["car"], "car", a.n, 4, a.max_steps, a.reps),
           "point_host_loop": time_host_loop(pol["point"], "point", a.host_n, 8, a.host_steps),
           "car_host_loop": time_host_loop(pol["car"], "car", a.host_n, 4, a.host_steps)}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
