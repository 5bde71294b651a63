"""BatchedEnv — N reference episodes at once: the batched face of simulator/env.py.

    env = BatchedEnv(env_config, policy, n_episodes, device)      # policy: rl.policy.sarl.SARL (configured)
    env.reset_batch("test", seeds)         # env.reset x N   (the reference's seeded scenes, replayed in one launch)
    env.lookahead_batch()                  # onestep_lookahead x 81 x N  -> la_reward / la_event / vin
    env.step_batch(action_idx=...)         # env.step x N
    stats = env.run_episodes("test", seeds)                        # the Explorer's inner loop, on the device

Episode r of rank k uses seed seeds[r]; sharding over ranks is the caller's slice of `seeds` (no collective).

reset_batch builds every episode's scene on the device: ebc_replay_scenes replays numpy's seeded MT19937 stream and the
scene generator's rules (simulator/scene/scene_generator.py, generate_random_scene with scene_number = seed) one thread
per episode, and writes the humans, static discs, grid rectangles and obstacle polygons straight into the bound state.
With the env INI's `[sim] orca_obstacles = true` (this project's key; off by default, like the reference) the humans
avoid walls: ebc_build_obstacles turns the polygons into RVO2 obstacle records on the device right after the replay.
The host uploads the seeds and reads back one array of counts to check the capacity.  The host SceneGenerator
still parses the INI (and serves the N = 1 env, simulator/env.py); its case counter advances as if it had generated
the scenes.
"""
import configparser
import dataclasses

import numpy as np
import torch

from . import abi
from .actions import build_action_space
from .config import SimConfig
from .engine import BatchedSim
from .scene import replay_config, replay_rect_bound


class _RobotStub(object):
    """What the scene generator needs from the robot (position, goal, radius, policy flags)."""

    def __init__(self, config, policy):
        self.radius = config.getfloat("robot", "radius")
        self.v_pref = config.getfloat("robot", "v_pref")
        self.visible = config.getboolean("robot", "visible")
        self.policy = policy
        self.px = self.py = self.gx = self.gy = self.vx = self.vy = self.theta = 0.0

    def set(self, px, py, gx, gy, vx, vy, theta):
        self.px, self.py, self.gx, self.gy, self.vx, self.vy, self.theta = px, py, gx, gy, vx, vy, theta


class TargetValue(object):
    """The TARGET value network of the TD update (rl/utils/explorer.py:174-186) on the K4 kernels: a second library
    handle that only ever runs ebc_value, with its own copy of the weights (the online network keeps changing)."""

    def __init__(self, env):
        sim = env.sim
        cfg = dataclasses.replace(env.cfg, orca_obstacles=False)       # runs K4 only: no obstacle slots needed
        self.sim = BatchedSim(cfg, 1, sim.Hmax, sim.Smax, 0, sim.A, device=sim.device)
        self.value_mode = getattr(env.policy, "value_mode", None)

    def set_model(self, model):
        sd = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
        self.sim.set_weights(sd, with_global_state=model.with_global_state, self_state_dim=model.self_state_dim)
        if self.value_mode:
            self.sim.set_value_mode(self.value_mode)

    def __call__(self, states, rows):
        return self.sim.value(states.contiguous(), rows.to(torch.int32).contiguous())


class EpisodeStats(object):
    """Per-episode outcome arrays (what rl/utils/explorer.py:33-94 accumulates one episode at a time)."""

    def __init__(self, n):
        self.event = np.zeros(n, np.int64)          # terminal event code
        self.time = np.zeros(n, np.float64)         # env.global_time at the end
        self.steps = np.zeros(n, np.int64)
        self.cum_reward = np.zeros(n, np.float64)   # sum_t gamma^(t dt v_pref) r_t
        self.too_close = np.zeros(n, np.int64)      # Danger steps
        self.min_dist_sum = np.zeros(n, np.float64)


class BatchedEnv(object):
    COUNTER_OFFSET = {"train": 2000, "val": 0, "test": 1000}     # env.py:153-158

    def __init__(self, env_config, policy=None, n_episodes=1, device="cuda:0", max_humans=None, max_statics=None,
                 max_rects=None, max_obst=None):
        from simulator.scene.scene_generator import SceneGenerator   # the INI's scene settings (and the case counter)
        if not isinstance(env_config, configparser.RawConfigParser):
            cp = configparser.RawConfigParser()
            cp.read(env_config)
            env_config = cp
        self.config = env_config
        self.policy = policy
        self.cfg = SimConfig.from_ini(env_config)
        if policy is not None:
            self.cfg.robot_kinematics = policy.kinematics or "holonomic"
            self.cfg.with_agent_type = bool(getattr(policy, "with_agent_type", False))
            self.cfg.gamma = policy.gamma or self.cfg.gamma
        self.scene = SceneGenerator(env_config)
        self._replay_configs = {}      # ebc_replay_config per (phase, multiagent_training, list sizes)
        self.robot = _RobotStub(env_config, policy if policy is not None else type("P", (), dict(
            multiagent_training=True, name="none", kinematics="holonomic"))())
        self.cfg.robot_visible = self.robot.visible
        self.scene.set_robot(self.robot)
        self.time_step, self.time_limit = self.cfg.time_step, self.cfg.time_limit
        sg = self.scene
        H = max_humans or max(sg.adult_num + sg.bicycle_num + sg.children_num, 20 if "mixed_20" in (
            sg.test_sim_adult, sg.train_val_sim_adult) else 1)
        walls, circles = sg.num_walls or 0, sg.num_circles or 0
        discs_per_wall = int(np.ceil(sg.max_wall_length / np.sqrt(2.0)))
        S = max_statics if max_statics is not None else walls * discs_per_wall + circles
        # the replay's per-obstacle rectangles: one per obstacle inside the map, a lattice for a striped border patch
        R = max_rects if max_rects is not None else replay_rect_bound(sg)
        # [sim] orca_obstacles: RVO2 obstacle records of the scene's polygons, built on the device at every reset
        O = max_obst if max_obst is not None else (64 if self.cfg.orca_obstacles else 0)
        self.N = n_episodes
        n_actions = policy.n_actions if policy is not None and hasattr(policy, "n_actions") else 81
        self.sim = BatchedSim(self.cfg, n_episodes, H, S, R, n_actions, device=device, max_obst=O)
        self.device = self.sim.device
        if policy is not None:
            if policy.action_space is None:
                policy.build_action_space(self.robot.v_pref)
            self.sim.set_actions(np.array([tuple(a)[:2] for a in policy.action_space], dtype=np.float64))
            self.sync_weights()
        self._weights_version = getattr(policy, "weights_version", 0)
        # epsilon-greedy exploration stream: ONE generator for the life of the env, keyed by (seed, rank), so that
        # neither successive run_episodes calls nor different ranks replay the same explore mask / random actions
        # (the reference draws from numpy's global stream, reseeded per scene: multi_human_rl.py:31)
        self.target_value = TargetValue(self) if (policy is not None and self.device.type == "cuda") else None
        rank = int(__import__("os").environ.get("RANK", "0"))
        self._explore_gen = torch.Generator(device=self.device)
        self.seed_exploration(20261018, rank)

    def seed_exploration(self, seed, rank=0):
        self._explore_gen.manual_seed(int(np.random.SeedSequence([int(seed), int(rank)]).generate_state(1, np.uint64)[0] >> 1))

    @classmethod
    def synthetic(cls, cfg, shape, n_episodes, device, actions, weights, value_mode=None, first_episode_id=0,
                  id_stride=None, with_global_state=True, self_state_dim=6):
        """The N-episode face over a SYNTHETIC workload (ebc.synth.SceneShape, SURVEY 8d) instead of an INI file:
        scenes come from the device generator (ebc_generate, counter-based in the global episode id), finished
        episodes are re-generated with FRESH scenes (`reset_done`), weights / action table are given directly.
        Same batched calls as the INI-driven env: lookahead_batch / decide_batch / step_batch."""
        self = cls.__new__(cls)
        self.config, self.policy, self.scene = None, None, None
        self.cfg, self.shape = cfg, shape
        self.time_step, self.time_limit = cfg.time_step, cfg.time_limit
        self.robot = type("RobotStub", (), dict(radius=shape.robot_radius, v_pref=shape.robot_v_pref, visible=cfg.robot_visible))()
        self.N = n_episodes
        self.sim = BatchedSim(cfg, n_episodes, shape.H, shape.Smax, shape.Rmax, len(actions), device=device)
        self.device = self.sim.device
        self.sim.set_actions(np.asarray(actions, dtype=np.float64))
        self.sim.set_weights(weights, with_global_state=with_global_state, self_state_dim=self_state_dim)
        if value_mode:
            self.sim.set_value_mode(value_mode)
        self.sim.fused_input = self.sim.value_mode().startswith("tc")      # K4 builds its own input: no N*A*n*D buffer
        self._weights_version = 0
        self.target_value = None
        self._explore_gen = torch.Generator(device=self.device)
        self.seed_exploration(20261018, int(__import__("os").environ.get("RANK", "0")))
        # global episode ids: this rank owns [first, first + N); a finished episode e continues with id + stride
        self.episode_ids = torch.arange(first_episode_id, first_episode_id + n_episodes, dtype=torch.int64, device=self.device)
        self.id_stride = int(id_stride if id_stride is not None else n_episodes)
        self.sim.generate(shape, self.episode_ids)
        return self

    def reset_done(self, done=None):
        """env.reset for the episodes that just ended (default: sim.done of the last step): a fresh scene from the
        device generator, keyed by the next global id of that slot.  No host round trip."""
        done = self.sim.done if done is None else done
        self.episode_ids += done.to(torch.int64) * self.id_stride
        self.sim.generate(self.shape, self.episode_ids, mask=done)

    def sync_weights(self):
        model = self.policy.get_model()
        sd = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
        self.sim.set_weights(sd, with_global_state=model.with_global_state, self_state_dim=model.self_state_dim)
        if getattr(self.policy, "value_mode", None):
            self.sim.set_value_mode(self.policy.value_mode)
        self.sim.fused_input = self.sim.value_mode().startswith("tc")      # K4 builds its own input: no N*A*n*D buffer
        self._weights_version = getattr(self.policy, "weights_version", 0)

    # ---- env.reset x N ---------------------------------------------------------------------------------
    def reset_batch(self, phase, seeds):
        """seeds[e] = scene_number of episode e (the reference: counter offset + case counter, or explicit): the scene
        generate_random_scene(phase, scene_number = seeds[e]) makes, regenerated on the device in one launch.

        With [sim] orca_obstacles set, the scene's polygons then become RVO2 obstacle records on the device
        (ebc_build_obstacles), before the one readback of the counts.

        A scene that does not fit the batch's capacity (humans, static discs, grid rectangles, obstacle records) raises
        EbcError naming its seed; polygons are never dropped to make a scene fit.  The check needs the kernel's counts,
        so by then every episode's state in the sim has been overwritten (the oversized scenes truncated): reset again
        before stepping.  self.poly_xy / poly_count and the
        scene generator's counters are left as they were."""
        sim, sg = self.sim, self.scene
        assert len(seeds) == self.N
        seeds = np.asarray([int(x) for x in seeds], dtype=object)
        bad = [int(x) for x in seeds if not 0 <= int(x) <= 0xFFFFFFFF]
        if bad:
            raise ValueError("Seed must be between 0 and 2**32 - 1 (got %d)" % bad[0])      # np.random.seed's bound
        seeds = seeds.astype(np.uint32)
        multi = bool(self.robot.policy.multiagent_training)
        key = (phase, multi, sg.adult_num, sg.bicycle_num, sg.children_num)
        if key not in self._replay_configs:
            self._replay_configs[key] = replay_config(sg, phase, multi, max((sg.num_circles or 0) + (sg.num_walls or 0), 1))
        cfg = self._replay_configs[key]
        rad = sg.circle_radius
        self.robot.set(0, -rad, 0, rad, 0, 0, np.pi / 2)
        dev_seeds = torch.from_numpy(seeds.view(np.int32)).to(self.device)
        poly_xy, poly_count, need = sim.replay_scenes(cfg, dev_seeds)
        if self.cfg.orca_obstacles:
            need = torch.cat([need, sim.build_obstacles(poly_xy, poly_count)[:, None]], 1)
        need = need.cpu().numpy()
        obst_bad = need[:, 5] < 0 if self.cfg.orca_obstacles else np.zeros(self.N, bool)
        for e in np.nonzero((need[:, 0] > sim.Hmax) | (need[:, 1] > sim.Smax) | (need[:, 2] > sim.Rmax) | obst_bad)[0][:1]:
            if need[e, 0] > sim.Hmax or need[e, 1] > sim.Smax:
                raise abi.EbcError("scene %d exceeds the batch capacity (H=%d, S=%d)" % (seeds[e], need[e, 0], need[e, 1]))
            if need[e, 2] > sim.Rmax:
                raise abi.EbcError("scene %d needs %d grid rectangles (capacity %d)" % (seeds[e], need[e, 2], sim.Rmax))
            raise abi.EbcError("scene %d needs more than %d ORCA obstacle records" % (seeds[e], sim.Omax))
        self.poly_xy, self.poly_count = poly_xy, poly_count
        # what the host generator leaves behind: the case counter advanced once per scene, and the adult count the
        # mixed rules draw (the last scene's)
        sg.case_counter[phase] = (sg.case_counter[phase] + self.N) % sg.case_size[phase]
        if self.N and cfg.rule[0] in (abi.REPLAY_RULES["mixed"], abi.REPLAY_RULES["mixed_20"]):
            sg.adult_num = int(need[-1, 4])

    # ---- thin batched calls ------------------------------------------------------------------------------
    def lookahead_batch(self):
        self.sim.orca()
        self.sim.lookahead()
        return self.sim.la_reward, self.sim.la_done, self.sim.la_event

    def decide_batch(self):
        if self.policy is not None and getattr(self.policy, "weights_version", 0) != self._weights_version:
            self.sync_weights()
        return self.sim.decide()

    def step_batch(self, action_idx=None, action=None, active=None):
        self.sim.step(action_idx=action_idx, action=action, active=active, fused_orca=action_idx is None)
        return self.sim.reward, self.sim.done, self.sim.event

    def local_map_batch(self, normalize=True, out=None):
        """`local_map` of env.reset / env.step for every episode, one launch: with [map] use_grid_map = false the
        angular map (simulator/env.py:570-628, ebc_local_map_angular), [N, angular_map_dim] float64 on the device;
        with use_grid_map = true the binary grid sub-map (env.py:630-708, ebc_local_map_grid), [N, size, size] uint8."""
        c = self.config
        if c.getboolean("map", "use_grid_map"):
            return self.sim.local_map_grid(c.getfloat("map", "submap_size_m"), out=out)
        return self.sim.local_map_angular(self.poly_xy, self.poly_count, c.getfloat("map", "angular_map_max_range"),
                                          c.getfloat("map", "angle_min") * np.pi, c.getfloat("map", "angle_max") * np.pi,
                                          c.getint("map", "angular_map_dim"), normalize=normalize, out=out)

    # ---- the explorer's inner loop on the device (rl/utils/explorer.py:33-94) ------------------------------
    @torch.no_grad()
    def run_episodes(self, phase, seeds, epsilon=None, record=False, imitation=False, safety_space=0.0, rng=None,
                     poll_every=8, record_dmin=False):
        """Run every episode to its end.  Returns (EpisodeStats, trajectory or None); trajectory =
        dict(states [T, N, n, D], rewards [T, N], alive [T, N], rows [N]) on the device.

        The running statistics (discounted return, step / danger counts, min-distance sum, final event, alive mask)
        are accumulated by the step kernel itself (ebc_bind_stats): the loop issues launches only and reads ONE int
        (episodes still alive) every `poll_every` steps -- no per-step host synchronisation, no eager torch
        arithmetic.  `rng`: a torch.Generator on this device for the epsilon-greedy draws (default: the env's own,
        persistent across calls and keyed by the rank)."""
        sim = self.sim
        self.reset_batch(phase, seeds)
        N, dev = self.N, self.device
        sx = sim.bind_stats()
        states, rewards, alive = [], [], []
        dmins = []
        nan_seen = torch.zeros(N, dtype=torch.uint8, device=dev)
        gen = rng if rng is not None else self._explore_gen
        max_steps = int(self.time_limit / self.time_step) + 2
        try:
            for t in range(max_steps):
                if t % poll_every == 0 and t > 0:
                    if int(sx["alive_count"].item()) == 0:
                        break
                    if bool(nan_seen.any()):
                        raise ValueError("Value network is not well trained. ")      # multi_human_rl.py:81-82
                if record or record_dmin:
                    alive.append(sx["alive"].bool().clone())
                if record:
                    states.append(sim.transform().clone())
                if imitation:
                    act = sim.robot_orca(safety_space)
                    sim.orca()
                    sim.step(action=act)
                else:
                    idx = self.decide_batch()
                    nan_seen |= sim.nan_flag & sx["alive"]
                    if epsilon:
                        explore = torch.rand(N, device=dev, generator=gen) < epsilon
                        rnd = torch.randint(0, sim.A, (N,), device=dev, generator=gen, dtype=torch.int32)
                        idx = torch.where(explore, rnd, idx).contiguous()
                    sim.step(action_idx=idx)
                if record:
                    rewards.append(torch.where(alive[-1], sim.reward, torch.zeros_like(sim.reward)))
                if record_dmin:
                    dmins.append(sim.dmin.clone())
            if bool(nan_seen.any()):
                raise ValueError("Value network is not well trained. ")
        finally:
            sim.unbind_stats()
        st = EpisodeStats(N)
        st.event = sx["final_event"].cpu().numpy().astype(np.int64)
        st.time = sim.time.cpu().numpy().copy()
        st.steps = sx["steps"].cpu().numpy().astype(np.int64)
        st.cum_reward = sx["cum_reward"].cpu().numpy().copy()
        st.too_close = sx["too_close"].cpu().numpy().astype(np.int64)
        st.min_dist_sum = sx["min_dist_sum"].cpu().numpy().copy()
        st.still_running = sx["alive"].cpu().numpy().astype(bool)
        st.dist_to_goal = sim.dist_to_goal.cpu().numpy().copy()
        if record_dmin and dmins:
            st.dmin_trace = torch.stack(dmins).cpu().numpy()          # [T, N, 3]
            st.alive_trace = torch.stack(alive).cpu().numpy()         # [T, N]
        traj = None
        if record and states:
            traj = {"states": torch.stack(states), "rewards": torch.stack(rewards), "alive": torch.stack(alive),
                    "rows": (sim.hum_count + sim.stat_count).clone()}
        return st, traj
