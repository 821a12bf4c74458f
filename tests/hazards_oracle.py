"""Safety Gym's hazards restated on top of oracle/vec_oracle.py and tests/goal_lidar_oracle.py (test infrastructure
only): the Engine's layout with numpy's own RandomState (the reference's generator), the hazards' pseudo-lidar and the
hazard cost.

- Layout: Engine.reset seeds ``RandomState(_seed)``; build_layout calls sample_layout up to 10 000 times; each object
  of the placements dict (robot, goal, hazard0 ..) takes up to 100 draws ``(uniform(xmin, xmax), uniform(ymin, ymax))``
  from ``constrain_placement(box, keepout)`` until its distance to every placed object is at least
  ``other_keepout + placements_margin + keepout``; build_world_config then draws ``robot_rot = uniform(0, 2 pi)``.
  A fixed location replaces the box by ``(x - k, y - k, x + k, y + k)``, ``k = keepout + 1e-9``.
- Lidar: ``obs_lidar_pseudo(hazards_pos)``, every hazard's height dropped (ego_xy).
- Cost: ``sum over hazards with dist_xy <= size of hazards_cost * (size - dist_xy)``; the indicator makes it
  ``float(x > 0)``.

Parity unpinned, like the goal lidar: the reference's source is not at hand; the defaults are Engine.DEFAULT's.
"""
from __future__ import annotations

import numpy as np

import goal_lidar_oracle as L

ROBOT_KEEPOUT = GOAL_KEEPOUT = 0.4
MARGIN = 0.0
EXTENTS = (-2, -2, 2, 2)


class CountingRandomState(np.random.RandomState):
    """RandomState that counts the 32-bit words its uniform() draws consume (two per float64)."""

    def __init__(self, seed):
        super().__init__(seed)
        self.words = 0

    def uniform(self, low=0.0, high=1.0, size=None):
        self.words += 2
        return super().uniform(low, high, size)


def _constrain(box, keepout):
    xmin, ymin, xmax, ymax = box
    return (xmin + keepout, ymin + keepout, xmax - keepout, ymax - keepout)


def placements(num, keepout, locations=()):
    """Engine.placements for the goal task with ``num`` hazards: name -> (draw box, keepout), in dict order."""
    out = {"robot": (_constrain(EXTENTS, ROBOT_KEEPOUT), ROBOT_KEEPOUT),
           "goal": (_constrain(EXTENTS, GOAL_KEEPOUT), GOAL_KEEPOUT)}
    for i in range(num):
        if i < len(locations):
            x, y = locations[i]
            k = keepout + 1e-9
            box = _constrain((x - k, y - k, x + k, y + k), keepout)
        else:
            box = _constrain(EXTENTS, keepout)
        out[f"hazard{i}"] = (box, keepout)
    return out


def layout(seed, num, keepout=0.4, locations=()):
    """Engine.reset's layout for Engine._seed = seed: (ok, heading, hazards [num][2], words drawn).  ok False: 10 000
    layouts failed (the reference raises ResamplingError)."""
    rs = CountingRandomState(seed & 0xFFFFFFFF)
    place = placements(num, keepout, locations)
    for _ in range(10000):
        lay = {}
        for name, (box, keep) in place.items():
            for _ in range(100):
                xy = np.array([rs.uniform(box[0], box[2]), rs.uniform(box[1], box[3])])
                if all(not np.sqrt(np.sum(np.square(xy - other))) < place[o][1] + MARGIN + keep
                       for o, other in lay.items()):
                    lay[name] = xy
                    break
            else:
                break
        else:
            heading = rs.uniform(0, 2 * np.pi)
            return True, float(heading), np.array([lay[f"hazard{i}"] for i in range(num)]).reshape(num, 2), rs.words
    return False, None, None, rs.words


def hazards_block(hazards, robot_pos, robot_mat, **lidar):
    """The hazards_lidar block of one env, float64 [num_bins]."""
    cfg = {**L.DEFAULTS, **lidar}
    return L.obs_lidar_pseudo([L.ego_xy(h, robot_pos, robot_mat) for h in np.asarray(hazards, np.float64)], **cfg)


def hazards_rows(hazards, robot_pos, robot_mat, **lidar):
    return np.stack([hazards_block(hazards[i], robot_pos[i], robot_mat[i], **lidar) for i in range(len(hazards))])


def cost(hazards, robot_xy, size=0.3, hazards_cost=1.0, indicator=True):
    """Engine.cost with constrain_hazards: info['cost'] (== info['cost_hazards'])."""
    c = 0.0
    for h in np.asarray(hazards, np.float64):
        d = np.sqrt(np.sum(np.square(h - np.asarray(robot_xy, np.float64)[:2])))
        if d <= size:
            c += hazards_cost * (size - d)
    return float(c > 0.0) if indicator else c
