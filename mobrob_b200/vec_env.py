"""GpuVecEnv: thousands of goal environments resident in HBM behind the SB3 ``VecEnv``
protocol (numpy in/out, for unchanged third-party code) plus a zero-copy tensor path.

Replaces ``make_vec_env(get_env, n_envs, env_kwargs={..., terminate_on_goal, time_limit},
vec_env_cls=DummyVecEnv|SubprocVecEnv, seed=seed)`` of src/mobrob/rl_control/ppo.py:37-48,
i.e. N x Monitor(TimeLimit(PointEnv|CarEnv)).
"""
from __future__ import annotations

import ctypes
import time

import numpy as np
import torch

from . import _lib, seeding
from .spaces import Box

ENV_KINDS = {"point": 0, "car": 1}
OBS_DIMS = {"point": 14, "car": 26}
# Engine config keys (engine.py:124-144) the batched env implements -> mr_env_set_obs_flags bits; every other
# observe_* key must keep the value the reference's get_robot_config leaves it at
OBS_FLAG_BITS = {"observe_goal_dist": 1, "observe_qpos": 2, "observe_qvel": 4, "observe_ctrl": 8, "observe_goal_lidar": 16}
_FIXED_OBSERVE = {"observe_sensors": True, "observe_goal_comp": True, "observe_com": False,
                  "observe_box_comp": False, "observe_box_lidar": False, "observe_circle": False,
                  "observe_remaining": False, "observe_walls": False, "observe_hazards": False, "observe_vases": False,
                  "observe_pillars": False, "observe_buttons": False, "observe_gremlins": False,
                  "observe_vision": False, "observe_freejoint": False}


def obs_flags_of(robot_config: dict | None) -> int:
    """Engine(config) observation switches -> flag bits.  Keys that do not concern the observation (robot_base,
    sensors_obs, box_*) are the reference's constants for the robot and are ignored."""
    flags = 0
    for key, value in (robot_config or {}).items():
        if key in OBS_FLAG_BITS:
            flags |= OBS_FLAG_BITS[key] if value else 0
        elif key in _FIXED_OBSERVE and bool(value) != _FIXED_OBSERVE[key]:
            raise NotImplementedError(f"{key}={value!r}: only {sorted(OBS_FLAG_BITS)} can be switched on the B200 path")
    return flags


# Safety Gym's Engine.DEFAULT pseudo-lidar settings (parity unpinned: restated, the reference's source is not at hand)
LIDAR_DEFAULTS = {"lidar_num_bins": 10, "lidar_max_dist": None, "lidar_exp_gain": 1.0, "lidar_alias": True,
                  "lidar_type": "pseudo"}


def lidar_of(robot_config: dict | None) -> tuple[int, float | None, float, bool]:
    """Engine(config) lidar keys -> (num_bins, max_dist, exp_gain, alias) for observe_goal_lidar, defaults filled in.
    Only the pseudo-lidar exists here: lidar_type 'natural' ray-casts against the model's geoms."""
    cfg = {**LIDAR_DEFAULTS, **{k: v for k, v in (robot_config or {}).items() if k in LIDAR_DEFAULTS}}
    if cfg["lidar_type"] == "natural":
        raise NotImplementedError("lidar_type='natural' (ray-cast lidar) is not available on the B200 path; use 'pseudo'")
    if cfg["lidar_type"] != "pseudo":
        raise ValueError(f"lidar_type={cfg['lidar_type']!r}: must be 'pseudo' or 'natural'")
    bins = cfg["lidar_num_bins"]
    if isinstance(bins, bool) or not isinstance(bins, (int, np.integer)) or bins < 1:
        raise ValueError(f"lidar_num_bins={bins!r}: must be an integer >= 1")
    max_dist = cfg["lidar_max_dist"]
    if max_dist is not None and not float(max_dist) > 0:
        raise ValueError(f"lidar_max_dist={max_dist!r}: must be None or positive")
    return (int(bins), None if max_dist is None else float(max_dist), float(cfg["lidar_exp_gain"]),
            bool(cfg["lidar_alias"]))


class GpuVecEnv:
    def __init__(self, env_name: str = "point", n_envs: int = 1, seed: int | None = 0,
                 time_limit: int | None = 1000, terminate_on_goal: bool = True,
                 device: int | torch.device | None = None, first_rank: int = 0,
                 robot_config: dict | None = None):
        if env_name not in ENV_KINDS:
            raise ValueError(f"Env {env_name} not found")  # wrapper.py:566
        if not torch.cuda.is_available():
            raise RuntimeError("mobrob_b200 needs a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.env_name = env_name
        self.num_envs = int(n_envs)
        self.time_limit = time_limit
        self.terminate_on_goal = bool(terminate_on_goal)
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        self.first_rank = first_rank
        h = ctypes.c_void_p()
        _lib.check(self.lib.mr_env_create(ENV_KINDS[env_name], self.num_envs, self.device.index or 0,
                                          int(time_limit or 0), int(self.terminate_on_goal),
                                          ctypes.byref(h)))
        self._h = h
        self.obs_flags = obs_flags_of(robot_config)
        if self.obs_flags:
            _lib.check(self.lib.mr_env_set_obs_flags(h, self.obs_flags))
        # the lidar keys are read only with observe_goal_lidar on (the Engine ignores them otherwise)
        self.lidar = lidar_of(robot_config) if self.obs_flags & OBS_FLAG_BITS["observe_goal_lidar"] else None
        if self.lidar:
            bins, max_dist, gain, alias = self.lidar
            _lib.check(self.lib.mr_env_set_lidar(h, bins, max_dist or 0.0, gain, int(alias)))
        self.obs_dim = int(self.lib.mr_env_obs_dim(h))
        self.state_dim = int(self.lib.mr_env_state_dim(h))
        self.observation_space = Box(-np.inf, np.inf, (self.obs_dim,), np.float32)
        self.action_space = Box(-1.0, 1.0, (2,), np.float32)
        # MujocoGoalEnv.get_init_space / get_goal_space (wrapper.py:250-264)
        self.init_space = Box(np.array([-1.0, -1.0], np.float32), np.array([1.0, 1.0], np.float32), dtype=np.float32)
        self.goal_space = Box(np.array([-2.0, -2.0], np.float32), np.array([2.0, 2.0], np.float32), dtype=np.float32)
        N, O, dev = self.num_envs, self.obs_dim, self.device
        self.obs = torch.zeros((N, O), dtype=torch.float32, device=dev)
        self.rew = torch.zeros(N, dtype=torch.float32, device=dev)
        self.done = torch.zeros(N, dtype=torch.uint8, device=dev)
        self.trunc = torch.zeros(N, dtype=torch.uint8, device=dev)
        self.term_obs = torch.zeros((N, O), dtype=torch.float32, device=dev)
        self.ep_ret = torch.zeros(N, dtype=torch.float64, device=dev)
        self.ep_len = torch.zeros(N, dtype=torch.int32, device=dev)
        self._actions = None
        self._needs_first_reset = True
        self._seed = None
        # VecEnv steps taken so far by evaluate_policy's device path: the Philox counter at which the next stochastic
        # evaluation on this env starts, so that consecutive evaluations never reuse a draw
        self.eval_steps = 0
        self.t_start = time.time()
        if seed is not None:
            self.seed(seed)

    # -- plumbing ---------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def close(self):
        if getattr(self, "_h", None) is not None:
            self.lib.mr_env_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- seeding / reset -----------------------------------------------------------------
    def seed(self, seed: int | None = None):
        """VecEnv.seed: env rank i gets ``seed + i`` at its next (first) reset."""
        if seed is None:
            seed = int(np.random.randint(0, 2**31 - 1))
        self._seed = int(seed)
        init, goal, eng = seeding.vec_env_streams(self._seed, self.num_envs, self.first_rank)
        _lib.check(self.lib.mr_env_seed(self._h, _lib.ptr(init), _lib.ptr(goal), _lib.ptr(eng),
                                        self._stream()))
        self._needs_first_reset = True
        return [self._seed + self.first_rank + i for i in range(self.num_envs)]

    def reset_tensor(self) -> torch.Tensor:
        first = 1 if self._needs_first_reset else 0
        _lib.check(self.lib.mr_env_reset(self._h, None, first, self.obs.data_ptr(), self._stream()))
        self._needs_first_reset = False
        return self.obs

    def reset(self) -> np.ndarray:
        return self.reset_tensor().cpu().numpy()

    # -- stepping ---------------------------------------------------------------------------
    def step_tensor(self, actions: torch.Tensor):
        """actions: float32 cuda [N, 2] (clipped on device like Engine.step).  Returns views of
        the env-owned output tensors (obs, rew, done u8, trunc u8), valid until the next step."""
        assert actions.is_cuda and actions.dtype == torch.float32 and actions.is_contiguous()
        assert actions.shape == (self.num_envs, 2)
        _lib.check(self.lib.mr_env_step(self._h, actions.data_ptr(), self.obs.data_ptr(),
                                        self.rew.data_ptr(), self.done.data_ptr(),
                                        self.trunc.data_ptr(), self.term_obs.data_ptr(),
                                        self.ep_ret.data_ptr(), self.ep_len.data_ptr(),
                                        self._stream()))
        return self.obs, self.rew, self.done, self.trunc

    def step_async(self, actions):
        a = torch.as_tensor(np.ascontiguousarray(actions, dtype=np.float32))
        self._actions = a.to(self.device, non_blocking=True)

    def step_wait(self):
        obs, rew, done, trunc = self.step_tensor(self._actions)
        obs_h = obs.cpu().numpy()
        rew_h = rew.cpu().numpy()
        done_h = done.cpu().numpy().astype(bool)
        infos = [{} for _ in range(self.num_envs)]
        if done_h.any():
            idx = np.nonzero(done_h)[0]
            trunc_h = trunc.cpu().numpy().astype(bool)
            tobs = self.term_obs.cpu().numpy()
            er = self.ep_ret.cpu().numpy()
            el = self.ep_len.cpu().numpy()
            now = time.time()
            for i in idx:
                infos[i] = {
                    "terminal_observation": tobs[i],
                    "TimeLimit.truncated": bool(trunc_h[i]),
                    "episode": {"r": round(float(er[i]), 6), "l": int(el[i]),
                                "t": round(now - self.t_start, 6)},
                }
        else:
            for d in infos:
                d["TimeLimit.truncated"] = False
        return obs_h, rew_h, done_h, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    # -- EnvWrapper.reset_init_space / reset_goal_space (wrapper.py:209-219) for the whole batch ------------------
    def _set_spaces(self):
        init = np.concatenate([self.init_space.low, self.init_space.high]).astype(np.float32)
        goal = np.concatenate([self.goal_space.low, self.goal_space.high]).astype(np.float32)
        _lib.check(self.lib.mr_env_set_spaces(self._h, init.ctypes.data, goal.ctypes.data, self._stream()))

    def reset_init_space(self, init_space):
        """Later full resets place the robot in `init_space` (a 2-d Box).  Every env keeps its own random stream."""
        self.init_space = init_space
        self._set_spaces()

    def reset_goal_space(self, goal_space):
        """Later resets draw the goal from `goal_space` (a 2-d Box)."""
        self.goal_space = goal_space
        self._set_spaces()

    def set_contacts(self, enabled: bool):
        """car only: switch the floor contacts off for contact-free parity trajectories."""
        _lib.check(self.lib.mr_env_set_contacts(self._h, int(bool(enabled))))

    # -- introspection ------------------------------------------------------------------------
    def get_obs_tensor(self):
        out = torch.empty_like(self.obs)
        _lib.check(self.lib.mr_env_get_obs(self._h, out.data_ptr(), self._stream()))
        return out

    def get_state(self) -> torch.Tensor:
        out = torch.empty((self.num_envs, self.state_dim), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.mr_env_get_state(self._h, out.data_ptr(), self._stream()))
        return out

    def set_state(self, state: torch.Tensor):
        s = state.to(self.device, torch.float64).contiguous()
        assert s.shape == (self.num_envs, self.state_dim)
        _lib.check(self.lib.mr_env_set_state(self._h, s.data_ptr(), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def get_pos(self) -> torch.Tensor:
        out = torch.empty((self.num_envs, 2), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.mr_env_get_pos(self._h, out.data_ptr(), self._stream()))
        return out

    def get_reset_counts(self) -> torch.Tensor:
        out = torch.empty((self.num_envs, 2), dtype=torch.int32, device=self.device)
        _lib.check(self.lib.mr_env_get_reset_counts(self._h, out.data_ptr(), self._stream()))
        return out

    # -- VecEnv protocol leftovers ------------------------------------------------------------------
    def get_attr(self, attr_name, indices=None):
        n = self.num_envs if indices is None else len(list(indices))
        return [getattr(self, attr_name)] * n

    def set_attr(self, attr_name, value, indices=None):
        setattr(self, attr_name, value)

    def env_method(self, method_name, *args, indices=None, **kwargs):
        raise NotImplementedError(f"env_method({method_name}) is not available on GpuVecEnv")

    def env_is_wrapped(self, wrapper_class, indices=None):
        n = self.num_envs if indices is None else len(list(indices))
        return [False] * n

    def render(self, mode=None):
        return None
