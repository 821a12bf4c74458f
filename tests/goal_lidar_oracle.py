"""Engine's pseudo-lidar of the goal (``observe_goal_lidar``), restated on top of oracle/vec_oracle.py (test
infrastructure only).

Safety Gym's Engine (src/mobrob/envs/mujoco_robots/robots/engine.py) builds ``obs['goal_lidar'] =
obs_lidar([goal_pos], GROUP_GOAL)``; with ``lidar_type == 'pseudo'`` that is ``obs_lidar_pseudo``
(engine.py:1092-1172), restated line by line in :func:`obs_lidar_pseudo`.  The block sits between goal_dist and gyro
in the flat row (sorted key order, engine.py:1253-1259).

Parity unpinned: the reference's source is not at hand and no shipped artefact was produced with the lidar on.  The
settings' defaults (``lidar_num_bins`` 10, ``lidar_max_dist`` None, ``lidar_exp_gain`` 1.0, ``lidar_alias`` True,
``lidar_type`` 'pseudo') are restated from Safety Gym's ``Engine.DEFAULT``.  Safety Gym spells the egocentric vector
``np.complex(*ego)``, which numpy 1.24 no longer has; the arithmetic below is the same.  One deliberate deviation:
``angle / bin_size`` can round up to ``lidar_num_bins`` (atan2 returns a tiny negative angle and ``% 2 pi`` rounds it
to 2 pi), where the reference raises IndexError; the bin is clamped to ``lidar_num_bins - 1``.
"""
from __future__ import annotations

import numpy as np

from oracle import car_oracle as co
from oracle.vec_oracle import GoalVecOracle, extend_obs

DEFAULTS = dict(num_bins=10, max_dist=None, exp_gain=1.0, alias=True)


def obs_lidar_pseudo(ego_positions, num_bins=10, max_dist=None, exp_gain=1.0, alias=True):
    """Engine.obs_lidar_pseudo over objects at egocentric xy ``ego_positions`` (float64, ``num_bins`` floats)."""
    obs = np.zeros(num_bins)
    for ego in ego_positions:
        z = complex(float(ego[0]), float(ego[1]))
        dist = np.abs(z)
        angle = np.angle(z) % (np.pi * 2)
        bin_size = (np.pi * 2) / num_bins
        bin = min(int(angle / bin_size), num_bins - 1)   # the clamp (see the module docstring)
        bin_angle = bin_size * bin
        if max_dist is None:
            sensor = np.exp(-exp_gain * dist)
        else:
            sensor = max(0, max_dist - dist) / max_dist
        obs[bin] = max(obs[bin], sensor)
        if alias:
            alias_ = (angle - bin_angle) / bin_size
            bin_plus = (bin + 1) % num_bins
            bin_minus = (bin - 1) % num_bins
            obs[bin_plus] = max(obs[bin_plus], alias_ * sensor)
            obs[bin_minus] = max(obs[bin_minus], (1 - alias_) * sensor)
    return obs


def ego_xy(goal_xy, robot_pos, robot_mat):
    """Engine.ego_xy: the goal at z = 0 (its height is dropped), ``(goal3 - robot_pos) @ robot_mat``, first two."""
    world_3vec = np.concatenate([np.asarray(goal_xy, np.float64), [0.0]]) - robot_pos
    return np.matmul(world_3vec, robot_mat)[:2]


def _yaw_mat(psi):
    c, s = np.cos(psi), np.sin(psi)
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def robot_frames(body):
    """(robot_pos [n][3], robot_mat [n][3][3]) of an oracle body.  The point's z is 0: its frame is a pure yaw,
    so the height never reaches the first two ego coordinates."""
    if isinstance(body, co.CarBody):
        return body.p.copy(), co.quat_to_mat(body.quat)
    pos = np.concatenate([body.pos(), np.zeros((body.n, 1))], 1)
    return pos, np.stack([_yaw_mat(p) for p in body.psi0 + body.q[:, 2]])


def robot_frames_of_state(kind, state):
    """The same from GpuVecEnv.get_state() rows (point: qpos body_xy psi0 ...; car: p quat ...)."""
    state = np.asarray(state, np.float64)
    if kind == "car":
        return state[:, 0:3].copy(), co.quat_to_mat(state[:, 3:7])
    psi0 = state[:, 8]
    c0, s0 = np.cos(psi0), np.sin(psi0)
    x = state[:, 6] + c0 * state[:, 0] - s0 * state[:, 1]
    y = state[:, 7] + s0 * state[:, 0] + c0 * state[:, 1]
    pos = np.stack([x, y, np.zeros_like(x)], 1)
    return pos, np.stack([_yaw_mat(p) for p in psi0 + state[:, 2]])


def lidar_rows(goal, robot_pos, robot_mat, **settings):
    """The goal_lidar block of every env, float64 [n][num_bins]."""
    cfg = {**DEFAULTS, **settings}
    goal = np.asarray(goal, np.float64)
    return np.stack([obs_lidar_pseudo([ego_xy(goal[i], robot_pos[i], robot_mat[i])], **cfg) for i in range(len(goal))])


def extend_obs_lidar(body, base, goal, observe, lidar=None):
    """extend_obs plus the goal_lidar block (after goal_dist, before gyro) when observe_goal_lidar is on."""
    observe = observe or {}
    row = extend_obs(body, base, goal, {k: v for k, v in observe.items() if k != "observe_goal_lidar"})
    if not observe.get("observe_goal_lidar"):
        return row
    at = body.obs_pre + 2 + (2 if observe.get("observe_ctrl") else 0) + (1 if observe.get("observe_goal_dist") else 0)
    block = lidar_rows(goal, *robot_frames(body), **(lidar or {}))
    return np.concatenate([np.asarray(row[:, :at], np.float64), block, np.asarray(row[:, at:], np.float64)],
                          axis=1).astype(np.float32)


class LidarVecOracle(GoalVecOracle):
    """GoalVecOracle whose rows (reset, step, terminal observations) carry the goal_lidar block."""

    def __init__(self, body, lidar=None, **kw):
        super().__init__(body, **kw)
        self.lidar = lidar or {}

    def _obs(self):
        return extend_obs_lidar(self.body, self.body.obs(self.goal), self.goal, self.observe, self.lidar)
