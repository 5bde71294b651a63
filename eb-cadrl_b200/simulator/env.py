"""EntityBasedCollisionAvoidance — the reference's gym-style environment (simulator/env.py:19-466),
backed by the batched B200 hot path.

This class is the N = 1 view: same constructor-less set-up (`configure`, `set_robot`), same
`reset / step / onestep_lookahead` signatures and return tuples, same attributes read by callers
(`global_time`, `time_step`, `time_limit`, `scene.*`, `robot`).  All arithmetic of the step lives in
libebcadrl.so (`self.native`, an ebc.engine.BatchedSim of one episode); the Agent objects are refreshed from
the device state after every committed step.  N > 1 callers use ebc.batched_env.BatchedEnv, which drives the
same BatchedSim with whole batches.

`local_map` (SURVEY §8f-3): with [map] use_grid_map = false the angular map of env.py:570-628 is computed on the
device (`ebc_local_map_angular`) for reset / step, like the reference does on every call; the lookahead skips it
(the reference computes and drops it there).  With use_grid_map = true it is the binary grid sub-map of env.py:630-708
(`ebc_local_map_grid`: the window of scene.map around the robot, rotated like cv2.warpAffine does, thresholded).
Rendering is out of scope.

With the env INI's `[sim] orca_obstacles = true` (this project's key, off by default like the reference) humans avoid
walls: every reset turns scene.obstacle_vertices -- generated or loaded from `load_scene_path` -- into RVO2 obstacle
records on the device (`ebc_build_obstacles`, the same function BatchedEnv.reset_batch runs), and the lookahead's probe
carries them too.
"""
import dataclasses

import numpy as np
import torch

from ebc import abi
from ebc.config import SimConfig
from ebc.engine import BatchedSim
from ebc.scene import rects_from_zero_cells
from simulator.scene.scene_generator import SceneGenerator
from simulator.utils import info as info_mod
from simulator.utils.action import ActionRot, ActionXY
from simulator.utils.reward import Reward
from simulator.utils.state import ObservableState
from simulator.utils.utils import AgentType


class EntityBasedCollisionAvoidance(object):
    metadata = {"render.modes": ["adult"]}
    PHASES = ["train", "val", "test"]

    def __init__(self):
        self.name = "EntityBasedCollisionAvoidance"
        self.time_step = None
        self.time_limit = None
        self.robot = None
        self.global_time = None
        self.case_capacity = None
        self.config = None
        self.scene = None
        self.reward = None
        self.native = None
        self.sim_config = None
        self.phase = None
        self.states = None
        self.action_values = None
        self.attention_weights = None
        self._policy_bound = None
        self._probe = None
        self._map_probe = None
        self._grid_probe = None
        self._poly = None
        self.local_maps = None
        self.local_maps_angular = None
        self.local_map_enabled = True       # False: reset / step return local_map = None without the extra launch

    # ---- set-up (env.py:58-92) ----------------------------------------------------------------------
    def configure(self, config):
        self.config = config
        self.scene = SceneGenerator(config)
        self.time_step = config.getfloat("env", "time_step")
        self.time_limit = config.getint("env", "time_limit")
        self.reward = Reward(config)
        self.case_capacity = {"train": np.iinfo(np.uint32).max - 2000, "val": 1000, "test": 1000}
        self.use_grid_map = config.getboolean("map", "use_grid_map")
        if self.use_grid_map:
            self.submap_size_m = config.getfloat("map", "submap_size_m")
        else:
            self.angular_map_max_range = config.getfloat("map", "angular_map_max_range")
            self.angular_map_dim = config.getint("map", "angular_map_dim")
            self.angular_map_min_angle = config.getfloat("map", "angle_min") * np.pi
            self.angular_map_max_angle = config.getfloat("map", "angle_max") * np.pi
        self.sim_config = SimConfig.from_ini(config)

    def set_robot(self, robot):
        self.robot = robot
        self.scene.set_robot(robot)
        self.reward.set_robot(robot)

    # ---- helpers -------------------------------------------------------------------------------------
    def _humans(self):
        return self.scene.adults + self.scene.bicycles + self.scene.children

    def _policy_config(self):
        """Fold what the robot's policy contributes to the device configuration."""
        c = self.sim_config
        pol = self.robot.policy
        c.robot_kinematics = getattr(pol, "kinematics", None) or "holonomic"
        c.with_agent_type = bool(getattr(pol, "with_agent_type", False))
        c.gamma = getattr(pol, "gamma", None) or c.gamma
        c.robot_visible = bool(self.robot.visible)
        return c

    def _build_native(self):
        humans, statics = self._humans(), self.scene.static_obstacles_as_pedestrians
        rects = rects_from_zero_cells(self.scene.map == 0)
        H, S, R = max(len(humans), 1), len(statics), len(rects)
        pol = self.robot.policy
        A = len(pol.action_space) if getattr(pol, "action_space", None) else getattr(pol, "n_actions", 81)
        cfg = self._policy_config()
        key = (H, S, R, A, cfg.robot_kinematics, cfg.with_agent_type, cfg.robot_visible, cfg.orca_obstacles)
        if self.native is None or self._native_key != key:
            self.native = BatchedSim(cfg, 1, H, S, R, A, max_obst=64 if cfg.orca_obstacles else 0)
            self._native_key = key
            self._policy_bound = None
            self._probe = None
        pv = np.zeros((1, H, 4), np.float32)
        gr = np.zeros((1, H, 4), np.float32)
        ty = np.zeros((1, H), np.uint8)
        for i, h in enumerate(humans):
            pv[0, i] = (h.px, h.py, h.vx, h.vy)
            gr[0, i] = (h.gx, h.gy, h.v_pref, h.radius)
            ty[0, i] = int(h.agent_type)
        sd = np.zeros((1, max(S, 1), 4), np.float32)
        for i, s in enumerate(statics):
            sd[0, i, :3] = (s.px, s.py, s.radius)
        rc = np.zeros((1, max(R, 1), 4), np.int16)
        rc[0, :R] = rects
        rb = self.robot
        self.native.load_episodes(0, pv, gr, ty, np.array([len(humans)], np.int32), sd, np.array([S], np.int32), rc,
                                  np.array([R], np.int32), np.array([[rb.px, rb.py, rb.vx, rb.vy]], np.float32),
                                  np.array([[rb.gx, rb.gy, rb.v_pref, rb.radius]], np.float32),
                                  np.array([rb.theta], np.float32), np.array([self.global_time], np.float64))
        if cfg.orca_obstacles:      # walls-aware humans: the scene's polygons -> RVO2 obstacle records, on the device
            need = int(self.native.build_obstacles(*self._polygons())[0].item())
            if need < 0:
                raise abi.EbcError("the scene's obstacles need more than %d ORCA obstacle records" % self.native.Omax)

    def bind_policy(self, policy):
        """Register the policy's action table and value-network weights with the device (once per change)."""
        stamp = (id(policy), getattr(policy, "weights_version", 0), id(self.native))
        if self._policy_bound == stamp:
            return
        if getattr(policy, "action_space", None):
            self.native.set_actions(np.array([tuple(a)[:2] for a in policy.action_space], dtype=np.float64))
        model = policy.get_model() if hasattr(policy, "get_model") else None
        if model is not None and hasattr(model, "state_dict"):
            sd = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
            if "mlp1.0.weight" in sd:
                self.native.set_weights(sd, with_global_state=getattr(model, "with_global_state", True),
                                        self_state_dim=getattr(model, "self_state_dim", 6))
                mode = getattr(policy, "value_mode", None)
                if mode:
                    self.native.set_value_mode(mode)
        self._policy_bound = stamp

    def _sync_agents_from_device(self):
        n = self.native
        pv = n.hum_pv[0].cpu().numpy().astype(np.float64)
        for h, row in zip(self._humans(), pv):
            h.px, h.py, h.vx, h.vy = (float(x) for x in row)
        rb = n.rob_pv[0].cpu().numpy().astype(np.float64)
        self.robot.px, self.robot.py, self.robot.vx, self.robot.vy = (float(x) for x in rb)
        self.robot.theta = float(n.rob_theta[0].item())
        self.global_time = float(n.time[0].item())

    # ---- angular local map (env.py:570-628) on the device ---------------------------------------------------
    def _polygons(self):
        """scene.obstacle_vertices as the device arrays of ebc_local_map_angular (rebuilt when the scene changes)."""
        verts = np.asarray(self.scene.obstacle_vertices, dtype=np.float64).reshape(-1, 4, 2)
        key = (verts.tobytes(), str(self.native.device))
        if self._poly is None or self._poly[0] != key:
            dev = self.native.device
            P = len(verts)
            xy = torch.zeros(1, max(P, 1), 4, 2, dtype=torch.float64)
            if P:
                xy[0, :P] = torch.as_tensor(verts)
            self._poly = (key, xy.to(dev), torch.tensor([P], dtype=torch.int32, device=dev))
        return self._poly[1], self._poly[2]

    def get_local_map_angular(self, ob=None, normalize=True, append=True):
        """Distance to the closest obstacle outline per angular sector around `ob` (a FullState; default: the
        robot's current state on the device), simulator/env.py:570-628."""
        n = self.native
        xy, cnt = self._polygons()
        sim = n
        if ob is not None:
            if self._map_probe is None or self._map_probe.device != n.device:
                self._map_probe = BatchedSim(dataclasses.replace(n.cfg, orca_obstacles=False), 1, 1, 0, 0, 1, device=n.device)
            sim = self._map_probe
            sim.rob_pv[0, 0], sim.rob_pv[0, 1] = float(ob.px), float(ob.py)
            sim.rob_gr[0, 3] = float(ob.radius)
            sim.rob_theta[0] = float(ob.theta)
        vec = sim.local_map_angular(xy, cnt, self.angular_map_max_range, self.angular_map_min_angle,
                                    self.angular_map_max_angle, self.angular_map_dim, normalize=normalize)[0].cpu().numpy()
        if append and self.local_maps_angular is not None:
            self.local_maps_angular.append(vec)
        return vec

    def get_local_map(self, ob=None, append=True):
        """Binary sub-map of scene.map around `ob` (a FullState; default: the robot's current state on the device)
        rotated into the robot's heading, simulator/env.py:630-692: float64 [size, size] of zeros and ones."""
        n = self.native
        sim = n
        if ob is not None:
            # a one-episode probe that shares the scene's rectangle list
            if self._grid_probe is None or self._grid_probe.device != n.device or self._grid_probe.Rmax != n.Rmax:
                self._grid_probe = BatchedSim(dataclasses.replace(n.cfg, orca_obstacles=False), 1, 1, 0, n.Rmax, 1,
                                              device=n.device)
            sim = self._grid_probe
            sim.rect.copy_(n.rect[:1])
            sim.rect_count.copy_(n.rect_count[:1])
            sim.rob_pv[0, 0], sim.rob_pv[0, 1] = float(ob.px), float(ob.py)
            sim.rob_theta[0] = float(ob.theta)
        grid = sim.local_map_grid(self.submap_size_m)[0].cpu().numpy().astype(np.float64)
        if append and self.local_maps is not None:
            self.local_maps.append(grid)
        return grid

    def _local_map(self, compute_local_map):
        if not (compute_local_map and self.local_map_enabled):
            return None
        return self.get_local_map() if self.use_grid_map else self.get_local_map_angular()

    def _observation(self):
        ob = [h.get_observable_state() for h in self._humans()]
        if self.robot.policy.name != "SDOADRL":
            ob += self.scene.static_obstacles_as_pedestrians
        return ob

    # ---- reset (env.py:128-205) ------------------------------------------------------------------------
    def reset(self, phase="test", test_case=None, imitation_learning=False, compute_local_map=True,
              save_scene_path=None, load_scene_path=None, scene_number=None):
        if self.robot is None:
            raise AttributeError("robot has to be set!")
        self.phase = phase
        assert phase in self.PHASES, "phase must be one of {}".format(self.PHASES)
        if test_case is not None:
            self.scene.case_counter[phase] = test_case
        self.global_time = 0
        counter_offset = {"train": self.case_capacity["val"] + self.case_capacity["test"], "val": 0,
                          "test": self.case_capacity["val"]}
        self.robot.set(0, -self.scene.circle_radius, 0, self.scene.circle_radius, 0, 0, np.pi / 2)
        if load_scene_path is not None:
            self.scene.load_scene(phase, load_scene_path)
        else:
            self.scene.generate_random_scene(counter_offset, phase, save_scene_path, scene_number=scene_number)
        for agent in [self.robot] + self._humans():
            agent.time_step = self.time_step
            if agent.policy is not None:
                agent.policy.time_step = self.time_step
        self.adult_times = [0] * len(self.scene.adults)
        self.bicycle_times = [0] * len(self.scene.bicycles)
        self.children_times = [0] * len(self.scene.children)
        self.states = list()
        self.local_maps = list()
        self.local_maps_angular = list()
        if hasattr(self.robot.policy, "action_values"):
            self.action_values = list()
        if hasattr(self.robot.policy, "get_attention_weights"):
            self.attention_weights = list()
        self._build_native()
        self._sync_agents_from_device()      # the hot path's state is fp32: objects mirror it exactly
        ob = self._observation()
        local_map = self._local_map(compute_local_map)
        if self.robot.policy.name == "ORCA":
            return ob, self.scene.obstacle_vertices, local_map
        return ob, local_map

    # ---- step (env.py:388-466) and lookahead (env.py:207-209) ----------------------------------------------
    def _action_pair(self, action):
        if isinstance(action, ActionXY):
            return float(action.vx), float(action.vy)
        if isinstance(action, ActionRot):
            return float(action.v), float(action.r)
        raise AssertionError("unsupported action type %r" % (action,))

    def _info(self, event, dist_to_goal, dmin):
        c = self.sim_config
        return info_mod.from_code(event, dist_to_goal, dmin,
                                  (c.discomfort_dist_adult, c.discomfort_dist_bicycle, c.discomfort_dist_child))

    def step(self, action, update=True, compute_local_map=True, border=None):
        if not update:
            ob, reward, done, info = self.onestep_lookahead(action)
            return ob, None, reward, done, info
        n = self.native
        self.robot.check_validity(action)
        self.states.append([self.robot.get_full_state(), [a.get_full_state() for a in self.scene.adults],
                            [b.get_full_state() for b in self.scene.bicycles],
                            [c.get_full_state() for c in self.scene.children]])
        if hasattr(self.robot.policy, "action_values"):
            self.action_values.append(self.robot.policy.action_values)
        if hasattr(self.robot.policy, "get_attention_weights"):            # env.py:355-356
            self.attention_weights.append(self.robot.policy.get_attention_weights())
        act = torch.tensor([self._action_pair(action)], dtype=torch.float64, device=n.device)
        n.step(action=act, fused_orca=True)          # humans' policies + collisions + reward + commit, one launch
        reward, done = float(n.reward[0].item()), bool(n.done[0].item())
        info = self._info(int(n.event[0].item()), n.dist_to_goal[0].item(), n.dmin[0].cpu().numpy())
        self._sync_agents_from_device()
        for group, times in ((self.scene.adults, self.adult_times), (self.scene.bicycles, self.bicycle_times),
                             (self.scene.children, self.children_times)):
            for i, agent in enumerate(group):      # first arrival times (env.py:365-378)
                if times[i] == 0 and agent.reached_destination():
                    times[i] = self.global_time
        return self._observation(), self._local_map(compute_local_map), reward, done, info

    def onestep_lookahead(self, action):
        """Simulate one step without committing it; returns (next entity states, reward, done, info)."""
        n = self.native
        if self._probe is None:
            self._probe = BatchedSim(n.cfg, 1, n.Hmax, n.Smax, n.Rmax, 1, device=n.device, max_obst=n.Omax)
        p = self._probe
        names = ("hum_pv", "hum_gr", "hum_type", "hum_count", "stat", "stat_count", "rect", "rect_count", "rob_pv",
                 "rob_gr", "rob_theta", "time") + (("obst", "obst_count") if n.Omax else ())
        for name in names:
            getattr(p, name).copy_(getattr(n, name))
        p.set_actions(np.array([self._action_pair(action)], dtype=np.float64))
        p.orca()
        p.lookahead(build_inputs=False)
        dt = self.time_step
        nv = p.hum_nv[0].cpu().numpy().astype(np.float64)
        ob = []
        for h, v in zip(self._humans(), nv):        # agent.py:80-93 with the human's new (ORCA) action
            ob.append(ObservableState(h.px + v[0] * dt, h.py + v[1] * dt, float(v[0]), float(v[1]), h.radius, h.agent_type))
        if self.robot.policy.name != "SDOADRL":
            ob += self.scene.static_obstacles_as_pedestrians
        # the committed-step kernel shares evaluate_action with the lookahead: dmin / dist come from a dry step
        q = p.la_event[0, 0].item()
        reward, done = float(p.la_reward[0, 0].item()), bool(p.la_done[0, 0].item())
        p.step(action_idx=torch.zeros(1, dtype=torch.int32, device=p.device))
        info = self._info(int(q), p.dist_to_goal[0].item(), p.dmin[0].cpu().numpy())
        return ob, reward, done, info

    def render(self, mode="adult", output_file=None):
        raise NotImplementedError("rendering is out of scope of the B200 hot path (SURVEY §2 #18)")
