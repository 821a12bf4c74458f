"""EnvWrapper API (src/mobrob/envs/wrapper.py:15-228) over a batch-of-one GPU environment.

``get_env("point" | "car", enable_gui, terminate_on_goal, time_limit)`` returns an object with
the reference's methods -- seed / set_goal / reset_random_goal / get_goal / reward_fn / step /
reset / reached / get_pos / set_pos / get_obs / space getters -- so examples/control.py
drives it unchanged.  Physics, observation, reward and flags run in the same CUDA kernels as
the vectorised path (one environment = a batch of one); this class only keeps the host-side
protocol (numpy in/out, gymnasium 5-tuple).
"""
from __future__ import annotations

from abc import ABC, abstractmethod

import numpy as np
import torch

from ..spaces import Box
from ..vec_env import GpuVecEnv

REACH_RADIUS = 0.3


class EnvWrapper(ABC):
    metadata = {"render_modes": ["human", "rgb_array"]}

    def __init__(self, enable_gui: bool = False, terminate_on_goal: bool = False):
        self.enable_gui = enable_gui
        self.terminate_on_goal = terminate_on_goal
        self._goal = None
        self._prev_pos = None
        self.env = self.build_env()
        self.observation_space = self.get_observation_space()
        self.action_space = self.get_action_space()
        self.init_space = self.get_init_space()
        self.goal_space = self.get_goal_space()
        self._first_reset = True
        self.render_mode = "human"

    @abstractmethod
    def _set_goal(self, goal): ...
    @abstractmethod
    def build_env(self): ...
    @abstractmethod
    def get_pos(self): ...
    @abstractmethod
    def set_pos(self, pos): ...
    @abstractmethod
    def get_obs(self) -> np.ndarray: ...
    @abstractmethod
    def get_observation_space(self): ...
    @abstractmethod
    def get_action_space(self): ...
    @abstractmethod
    def get_init_space(self): ...
    @abstractmethod
    def get_goal_space(self): ...

    def seed(self, seed=None):
        self._engine_seed = int(np.random.randint(2**32)) if seed is None else int(seed)
        self.init_space.seed(seed)
        self.goal_space.seed(seed + 1 if seed is not None else None)
        self.action_space.seed(seed)
        self.observation_space.seed(seed)

    def toggle_render_mode(self):
        self.render_mode = "human" if self.render_mode == "rgb_array" else "rgb_array"

    def set_goal(self, goal):
        self._set_goal(goal)
        self._goal = np.array(goal)

    def reset_random_goal(self):
        self.set_goal(self.goal_space.sample())

    def get_goal(self) -> np.ndarray:
        return np.array([]) if self._goal is None else self._goal

    def reward_fn(self) -> float:
        current_pos = self.get_pos()
        if self._goal is None or self._prev_pos is None:
            reward = 0.0
        else:
            reward = np.linalg.norm(self._goal - self._prev_pos) - np.linalg.norm(self._goal - current_pos)
        self._prev_pos = current_pos
        if self.reached():
            reward += 5.0
        return reward

    def step(self, action):
        obs = self._physics_step(action)
        reward = self.reward_fn()
        terminated = self.terminate_on_goal and self.reached()
        return obs, reward, terminated, False, {"cost": 0.0}

    def reset(self, init_pos=None, *args, **kwargs):
        if "seed" in kwargs:
            self.seed(kwargs.pop("seed"))
        if self._first_reset or not self.reached():
            self._engine_reset()
            self.set_pos(self.init_space.sample())
        if init_pos is not None:
            self.set_pos(init_pos)
        self.reset_random_goal()
        self._prev_pos = self.get_pos()
        self._first_reset = False
        return self.get_obs(), {}

    def reached(self, reach_radius: float = REACH_RADIUS) -> bool:
        return bool(np.linalg.norm(self.get_pos() - self.get_goal()) < reach_radius)

    def reset_init_space(self, init_space):
        self.init_space = init_space

    def reset_goal_space(self, goal_space):
        self.goal_space = goal_space

    def render(self):
        return None  # rendering is out of scope (SURVEY.md section 2)

    def close(self):
        self.env.close()


class MujocoGoalEnv(EnvWrapper, ABC):
    BASE_SENSORS = ["accelerometer", "velocimeter", "gyro", "magnetometer"]
    ENV_NAME = ""
    placements_extents = (-2, -2, 2, 2)  # engine.py:101

    def get_robot_config(self) -> dict:
        """Engine config of the robot (wrapper.py:235-240, 293-317).  A subclass may switch on observe_goal_dist /
        observe_qpos / observe_qvel / observe_ctrl (engine.py:125, 140-142) and observe_goal_lidar with its
        lidar_num_bins / lidar_max_dist / lidar_exp_gain / lidar_alias settings; other observation keys are fixed."""
        return {"robot_base": f"xmls/{self.ENV_NAME}.xml", "sensors_obs": self.BASE_SENSORS,
                "observe_com": False, "observe_goal_comp": True}

    def build_env(self):
        # time limit / termination are handled by this class (the GPU env runs raw steps)
        self._engine_seed = 0
        return GpuVecEnv(self.ENV_NAME, 1, seed=None, time_limit=None, terminate_on_goal=False,
                         robot_config=self.get_robot_config())

    def get_observation_space(self):
        return self.env.observation_space

    def get_action_space(self):
        return self.env.action_space

    def get_init_space(self):
        x0, y0, x1, y1 = self.placements_extents
        return Box(low=np.array([x0, y0], dtype=np.float32) / 2, high=np.array([x1, y1], dtype=np.float32) / 2,
                   dtype=np.float32)

    def get_goal_space(self):
        x0, y0, x1, y1 = self.placements_extents
        return Box(low=np.array([x0, y0], dtype=np.float32), high=np.array([x1, y1], dtype=np.float32),
                   dtype=np.float32)

    # -- state plumbing: reference-view state vector of the single env ----------------------
    def _state(self):
        return self.env.get_state().cpu().numpy()[0]

    def _write_state(self, s):
        self.env.set_state(torch.as_tensor(s[None]))

    GOAL_SLOT = 11  # index of the goal (x, y) in the reference-view state vector

    def _set_goal(self, goal):
        s = self._state()
        s[self.GOAL_SLOT:self.GOAL_SLOT + 2] = np.asarray(goal, dtype=np.float32)[:2]
        self._write_state(s)

    def get_pos(self) -> np.ndarray:
        return self.env.get_pos().cpu().numpy()[0].copy()

    def get_obs(self) -> np.ndarray:
        return self.env.get_obs_tensor().cpu().numpy()[0]

    def _physics_step(self, action):
        a = np.asarray(action, dtype=np.float32).reshape(1, 2)
        obs, _, _, _ = self.env.step_tensor(torch.as_tensor(a).to(self.env.device))
        return obs.cpu().numpy()[0]

    def add_wp_marker(self, pos, size, color=(0, 1, 1, 0.5), alpha=0.5, label=""):
        pass


def _engine_heading(seed: int) -> float:
    """Engine.reset -> build_layout -> build_world_config heading draw (engine.py:633-667, 728-729)."""
    rs = np.random.RandomState(seed & 0xFFFFFFFF)
    lo, hi = -2 + 0.4, 2 - 0.4
    for _ in range(10000):
        robot = np.array([rs.uniform(lo, hi), rs.uniform(lo, hi)])
        for _ in range(100):
            goal = np.array([rs.uniform(lo, hi), rs.uniform(lo, hi)])
            if not np.sqrt(np.sum(np.square(goal - robot))) < 0.8:
                return float(rs.uniform(0, 2 * np.pi))
    raise RuntimeError("Failed to sample layout of objects")


class PointEnv(MujocoGoalEnv):
    ENV_NAME = "point"
    render_mode = "rgb_array"

    def _engine_reset(self):
        self._engine_seed += 1

    def set_pos(self, pos):
        # PointEnv.set_pos rebuilds the Engine (wrapper.py:301-305): fresh sim, new heading
        self._engine_seed += 1
        s = self._state()
        s[0:6] = 0.0
        s[6:8] = np.asarray(pos, dtype=np.float64)[:2]
        s[8] = _engine_heading(self._engine_seed)
        s[9:11] = 0.0
        self._write_state(s)


def get_env(env_name: str, enable_gui: bool = False, terminate_on_goal: bool = False,
            time_limit: int | None = None):
    if env_name == "point":
        env = PointEnv(enable_gui, terminate_on_goal)
    elif env_name == "car":
        env = CarEnv(enable_gui, terminate_on_goal)
    elif env_name in ("doggo", "drone", "turtlebot3"):
        raise NotImplementedError(f"{env_name}: outside the scope of the B200 path (SURVEY.md section 2)")
    else:
        raise ValueError(f"Env {env_name} not found")
    if time_limit is not None:
        env = TimeLimit(env, max_episode_steps=time_limit)
    return env


class CarEnv(MujocoGoalEnv):
    """CarEnv (wrapper.py:308-326): free-joint root; set_pos only rewrites qpos[0:2]."""
    ENV_NAME = "car"
    render_mode = "rgb_array"
    GOAL_SLOT = 26  # qpos(13) qvel(11) ctrl(2) goal(2) elapsed ep_ret

    def _engine_reset(self):
        # Engine.reset(): new MjSim -- default pose at the origin, body z from car.xml:12, heading
        # drawn from RandomState(_seed), zero velocities and ctrl (engine.py:1000-1021, world.py:52-54)
        self._engine_seed += 1
        heading = _engine_heading(self._engine_seed)
        s = self._state()
        s[0:24] = 0.0
        s[2] = 0.1
        s[3], s[6] = np.cos(0.5 * heading), np.sin(0.5 * heading)
        s[9] = 1.0            # ball joint quaternion
        s[24:26] = 0.0        # data.ctrl
        self._write_state(s)

    def set_pos(self, pos):
        s = self._state()
        s[0:2] = np.asarray(pos, dtype=np.float64)[:2]
        self._write_state(s)


class TimeLimit:
    """gymnasium.wrappers.TimeLimit (wrapper.py:568-569)."""

    def __init__(self, env, max_episode_steps):
        self.env = env
        self._max_episode_steps = max_episode_steps
        self._elapsed_steps = None

    def __getattr__(self, name):
        return getattr(self.env, name)

    def step(self, action):
        obs, reward, terminated, truncated, info = self.env.step(action)
        self._elapsed_steps += 1
        if self._elapsed_steps >= self._max_episode_steps:
            truncated = True
        return obs, reward, terminated, truncated, info

    def reset(self, **kwargs):
        self._elapsed_steps = 0
        return self.env.reset(**kwargs)
