"""INI -> ebc_config.  Key names and fallbacks are the reference's, verbatim:
simulator/env.py:58-87, simulator/utils/reward.py:18-75, simulator/scene/scene_generator.py:26-72,
simulator/agents/agent.py:16-34, rl/policy/cadrl.py:73-82, rl/policy/sarl.py:90-128,
simulator/policy/orca.py:57-69 (SURVEY Appendix D).

One key is this project's own: `[sim] orca_obstacles` (boolean, default false).  With it set, humans (and the ORCA
robot of imitation learning) avoid the scene's obstacle polygons with RVO2's obstacle half-planes.  The reference
does not read it, so an INI that sets it still runs there unchanged, with humans that walk through walls."""
import configparser
from dataclasses import dataclass, field
from typing import List

from . import abi


@dataclass
class SimConfig:
    # [env]
    time_step: float = 0.25
    time_limit: float = 25.0
    # [reward]
    new_reward: bool = False
    time_max: float = 0.0
    time_good: float = 10.0
    max_goal_distance: float = None
    success_reward: float = 1.0
    collision_penalty_adult: float = None
    collision_penalty_bicycle: float = None
    collision_penalty_obstacle: float = None
    collision_penalty_child: float = None
    discomfort_dist: float = 0.2
    discomfort_dist_adult: float = 0.2
    discomfort_dist_bicycle: float = 0.2
    discomfort_dist_child: float = 0.2
    discomfort_penalty_factor_adult: float = 0.5
    discomfort_penalty_factor_bicycle: float = 0.5
    discomfort_penalty_factor_child: float = 0.5
    rotation_penalty_factor: float = 0.0
    # [map]
    map_size_m: float = 9.0
    map_resolution: float = 0.1
    # policy
    robot_kinematics: str = "holonomic"   # policy [action_space] kinematics, verbatim string
    with_agent_type: bool = False
    gamma: float = 0.9
    robot_visible: bool = False
    human_policy: List[str] = field(default_factory=lambda: ["orca", "orca", "orca"])
    # ORCA (simulator/policy/orca.py:63-69)
    orca_neighbor_dist: float = 10.0
    orca_max_neighbors: int = 10
    orca_time_horizon: float = 5.0
    orca_safety_space: float = 0.0
    # ORCA obstacle half-planes (SURVEY 8f-4): off = the reference's live behaviour (humans ignore walls)
    orca_obstacles: bool = False
    orca_time_horizon_obst: float = 5.0

    @classmethod
    def from_ini(cls, env_config, policy_config=None):
        g = env_config
        c = cls()
        c.time_step = g.getfloat("env", "time_step")
        c.time_limit = float(g.getint("env", "time_limit"))
        c.new_reward = g.getboolean("reward", "new_reward", fallback=False)
        tm = g.getfloat("reward", "time_max", fallback=None)
        c.time_max = 0.0 if tm is None else tm
        c.max_goal_distance = g.getfloat("reward", "max_goal_distance", fallback=None)
        c.time_good = g.getfloat("reward", "time_good", fallback=10.0)
        c.success_reward = g.getfloat("reward", "success_reward")
        for t in ("adult", "bicycle", "obstacle", "child"):
            setattr(c, "collision_penalty_" + t, g.getfloat("reward", "collision_penalty_" + t, fallback=None))
        c.discomfort_dist = g.getfloat("reward", "discomfort_dist")
        pf = g.getfloat("reward", "discomfort_penalty_factor")
        for t in ("adult", "bicycle", "child"):
            setattr(c, "discomfort_dist_" + t, g.getfloat("reward", "discomfort_dist_" + t, fallback=c.discomfort_dist))
            setattr(c, "discomfort_penalty_factor_" + t,
                    g.getfloat("reward", "discomfort_penalty_factor_" + t, fallback=pf))
        c.rotation_penalty_factor = g.getfloat("reward", "rotation_penalty_factor")
        c.map_size_m = g.getfloat("map", "map_size_m")
        c.map_resolution = g.getfloat("map", "map_resolution")
        c.robot_visible = g.getboolean("robot", "visible")
        c.human_policy = [g.get(sec, "policy", fallback="orca") if g.has_section(sec) else "orca"
                          for sec in ("adults", "bicycles", "children")]
        # this project's key, not the reference's: walls-aware humans (SURVEY 8f-4).  The reference's RawConfigParser
        # ignores it, so the same INI still runs there, with humans that ignore walls.
        c.orca_obstacles = g.getboolean("sim", "orca_obstacles", fallback=False)
        if policy_config is not None:
            p = policy_config
            c.gamma = p.getfloat("rl", "gamma")
            c.robot_kinematics = p.get("action_space", "kinematics")
            if p.has_option("sarl", "with_agent_type"):
                c.with_agent_type = p.getboolean("sarl", "with_agent_type")
        return c

    @property
    def D(self):
        return 17 if self.with_agent_type else 13

    def to_abi(self, n_episodes, max_humans, max_statics, max_rects, n_actions, max_obst=0):
        a = abi.EbcConfig()
        a.abi_version = abi.ABI_VERSION
        a.n_episodes, a.max_humans, a.max_statics = n_episodes, max_humans, max_statics
        a.max_rects, a.n_actions = max_rects, n_actions
        a.robot_kinematics = abi.KIN_HOLONOMIC if self.robot_kinematics == "holonomic" else abi.KIN_UNICYCLE
        a.rotate_theta = int(self.robot_kinematics == "unicycle")   # cadrl.py:261-265: exact string
        a.with_agent_type = int(self.with_agent_type)
        a.robot_visible = int(self.robot_visible)
        for i, p in enumerate(self.human_policy):
            if p not in ("orca", "linear"):
                raise ValueError("human policy %r is not on the hot path (orca | linear)" % p)
            a.human_policy[i] = abi.POLICY_ORCA if p == "orca" else abi.POLICY_LINEAR
        a.new_reward = int(self.new_reward)
        a.has_max_goal_distance = int(self.max_goal_distance is not None)
        a.orca_max_neighbors = self.orca_max_neighbors
        a.time_step, a.time_limit = self.time_step, self.time_limit
        a.time_max, a.time_good = self.time_max, self.time_good
        a.max_goal_distance = self.max_goal_distance or 0.0
        a.success_reward = self.success_reward
        # a None penalty only crashes the reference if that collision happens (SURVEY Appendix D)
        for t in ("adult", "bicycle", "obstacle", "child"):
            v = getattr(self, "collision_penalty_" + t)
            setattr(a, "collision_penalty_" + t, float("nan") if v is None else v)
        for t in ("adult", "bicycle", "child"):
            setattr(a, "discomfort_dist_" + t, getattr(self, "discomfort_dist_" + t))
            setattr(a, "discomfort_penalty_factor_" + t, getattr(self, "discomfort_penalty_factor_" + t))
        a.rotation_penalty_factor = self.rotation_penalty_factor
        a.map_size_m, a.map_resolution = self.map_size_m, self.map_resolution
        a.gamma = self.gamma
        a.orca_safety_space = self.orca_safety_space
        a.orca_neighbor_dist = self.orca_neighbor_dist
        a.orca_time_horizon = self.orca_time_horizon
        a.orca_obstacles = int(self.orca_obstacles)
        a.max_obst = int(max_obst)
        a.orca_time_horizon_obst = self.orca_time_horizon_obst
        return a


def read_ini(path):
    cp = configparser.RawConfigParser()
    if not cp.read(path):
        raise FileNotFoundError(path)
    return cp
