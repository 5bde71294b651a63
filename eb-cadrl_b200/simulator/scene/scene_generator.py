"""Host-side scene generator: what `env.reset` feeds to the hot path.

A restatement of simulator/scene/scene_generator.py that REPLAYS THE REFERENCE'S numpy RNG STREAM
(np.random.seed(seed) then the same draws in the same order), so that for a given seed the agents, the
occupancy grid and the static discs are identical to the reference's (pinned by tests/golden/scenes.npz).
The N = 1 env generates its scenes here, once per episode; BatchedEnv.reset_batch replays this module on the device
(ebc_replay_scenes, csrc/ebc_replay.cu), held to it bit for bit by tests/test_scene_replay.py; throughput runs use the
counter-based generator in ebc/synth.py instead.

Crossing rules: square_crossing (:672-712), circle_crossing (:593-650), mixed (:523-577), mixed_20
(:466-501,578-582), one_static (:583-589).  Static map: walls/circles (:113-290), grid (:888-922),
static discs (:380-422).  JSON scene format: save_scene / load_scene (:807-886).
"""
import collections
import json

import numpy as np
from numpy.linalg import norm

from simulator.agents.agents import Adult, Bicycle, Child
from simulator.utils.state import ObservableState
from simulator.utils.utils import AgentType

MAX_TRIES = 100000
Obstacle = collections.namedtuple("Obstacle", ["location_x", "location_y", "dim", "patch"])


class SceneGenerator(object):
    def __init__(self, config):
        self.config = config
        self.robot = None
        sim = lambda key, **kw: config.get("sim", key, **kw)  # noqa: E731
        self.adult_num = config.getint("sim", "adult_num")
        self.bicycle_num = config.getint("sim", "bicycle_num", fallback=0)
        self.bicycle_type = sim("bicycle_type", fallback=None)
        self.children_num = config.getint("sim", "children_num", fallback=0)
        self.case_counter = {"train": 0, "test": 0, "val": 0}
        self.case_size = {"train": np.iinfo(np.uint32).max - 2000, "val": config.getint("env", "val_size"),
                          "test": config.getint("env", "test_size")}
        self.train_val_sim_adult, self.test_sim_adult = sim("train_val_sim_adult"), sim("test_sim_adult")
        self.train_val_sim_bicycle = sim("train_val_sim_bicycle", fallback=None)
        self.test_sim_bicycle = sim("test_sim_bicycle", fallback=None)
        self.train_val_sim_children = sim("train_val_sim_children", fallback=None)
        self.test_sim_children = sim("test_sim_children", fallback=None)
        self.square_width = config.getfloat("sim", "square_width")
        self.circle_radius = config.getfloat("sim", "circle_radius")
        self.last_circle_radius = self.circle_radius
        self.randomize_attributes = config.getboolean("env", "randomize_attributes")
        self.map_resolution = config.getfloat("map", "map_resolution")
        self.map_size_m = config.getfloat("map", "map_size_m")
        self.min_wall_length = config.getint("map", "min_wall_length", fallback=2)
        self.max_wall_length = config.getint("map", "max_wall_length", fallback=4)
        self.num_circles = config.getint("map", "num_circles")
        self.num_walls = config.getint("map", "num_walls")
        self.discomfort_dist = config.getfloat("reward", "discomfort_dist")
        self.other_robots_num = config.getint("env", "robot_num") if config.has_option("env", "robot_num") else 0
        self.adults, self.bicycles, self.children = [], [], []
        self.map = None
        self.obstacles, self.obstacle_vertices, self.static_obstacles_as_pedestrians = [], [], []

    def set_robot(self, robot):
        self.robot = robot

    # ---- dynamic agents ----------------------------------------------------------------------------
    def _too_close(self, px, py, agent, others, with_goals):
        for other in [self.robot] + others:
            d = agent.radius + other.radius + self.discomfort_dist
            if norm((px - other.px, py - other.py)) < d:
                return True
            if with_goals and norm((px - other.gx, py - other.gy)) < d:
                return True
        return False

    def _square_crossing(self, agent, others):
        if self.randomize_attributes:
            agent.sample_random_attributes()
        hw = self.square_width / 2
        for index in range(MAX_TRIES):
            side = np.random.choice(["top", "bottom", "left", "right"])
            u = np.random.uniform(-hw, hw)
            px, py = {"top": (u, hw), "bottom": (u, -hw), "left": (-hw, u), "right": (hw, u)}[side]
            if self._too_close(px, py, agent, others, False) and index != MAX_TRIES - 1:
                continue
            g = np.random.uniform(-hw, hw)
            gx, gy = {"top": (g, -hw), "bottom": (g, hw), "left": (hw, g), "right": (-hw, g)}[side]
            break
        agent.set(px, py, gx, gy, 0, 0, 0)

    def _square_crossing_old(self, agent, others):
        """Legacy rule (scene_generator.py:714-761): start on the top or right edge of one half, goal mirrored."""
        if self.randomize_attributes:
            agent.sample_random_attributes()
        sign = np.random.choice([1, -1], p=[0.5, 0.5])
        for index in range(MAX_TRIES):
            px = np.random.random() * self.square_width * 0.5 * sign
            py = self.square_width * 0.5
            if np.random.random() > 0.5:
                px, py = py, px
            if self._too_close(px, py, agent, others, False) and index != MAX_TRIES - 1:
                continue
            mirror = [(-1, 1), (1, -1), (-1, -1)][np.random.randint(3)]
            gx, gy = px * mirror[0], py * mirror[1]
            clear = agent.radius + self.robot.radius + self.discomfort_dist
            if index == MAX_TRIES - 1 or not norm((gx - self.robot.gx, gy - self.robot.gy)) < clear:
                break
        agent.set(px, py, gx, gy, 0, 0, 0)

    def _circle_crossing(self, agent, others):
        if self.randomize_attributes:
            agent.sample_random_attributes()
        for _ in range(MAX_TRIES):
            angle = np.random.random() * np.pi * 2
            px, py = self.circle_radius * np.cos(angle) + 0, self.circle_radius * np.sin(angle) + 0
            if not self._too_close(px, py, agent, others, True):
                break
        agent.set(px, py, -px, -py, 0, 0, 0)
        return agent

    def _static_adults(self, count, width, height):
        for i in range(count):
            adult = Adult(self.config, "adults")
            if i == 0:
                adult.set(-0.5, -2.5, -0.5, -2.5, 0, 0, 0)
            else:
                sign = np.random.choice([1, -1], p=[0.5, 0.5])
                for _ in range(MAX_TRIES):
                    px = np.random.random() * width * 0.5 * sign
                    py = (np.random.random() - 0.5) * height
                    collide = self._too_close(px, py, adult, self.adults, False)
                    last = self.adults[-1] if self.adults else self.robot
                    near_goal = norm((px - self.robot.gx, py - self.robot.gy)) < adult.radius + last.radius + self.discomfort_dist
                    if not collide and not near_goal:
                        break
                adult.set(px, py, px, py, 0, 0, 0)
            self.adults.append(adult)

    def generate_random_adult_position(self, adult_num, rule):
        self.adults = []
        new = lambda: Adult(self.config, "adults")  # noqa: E731
        if rule == "square_crossing":
            for _ in range(adult_num):
                a = new()
                self._square_crossing(a, self.adults)
                self.adults.append(a)
        elif rule == "circle_crossing":
            for _ in range(adult_num):
                self.adults.append(self._circle_crossing(new(), self.adults))
        elif rule == "mixed":
            static_num = {0: 0.05, 1: 0.2, 2: 0.2, 3: 0.3, 4: 0.1, 5: 0.15}
            dynamic_num = {1: 0.3, 2: 0.3, 3: 0.2, 4: 0.1, 5: 0.1}
            static = bool(np.random.random() < 0.2)
            prob = np.random.random()
            for key, value in sorted(static_num.items() if static else dynamic_num.items()):
                if prob - value <= 0:
                    adult_num = key
                    break
                prob -= value
            self.adult_num = adult_num
            if static:
                if adult_num == 0:
                    a = new()
                    a.set(0, -10, 0, -10, 0, 0, 0)
                    self.adults.append(a)
                for _ in range(adult_num):
                    a = new()
                    sign = -1 if np.random.random() > 0.5 else 1
                    for _ in range(MAX_TRIES):
                        px = np.random.random() * 4 * 0.5 * sign
                        py = (np.random.random() - 0.5) * 8
                        if not self._too_close(px, py, a, self.adults, False):
                            break
                    a.set(px, py, px, py, 0, 0, 0)
                    self.adults.append(a)
            else:
                for i in range(adult_num):
                    a = new()
                    if i < 2:
                        self._circle_crossing(a, self.adults)
                    else:
                        self._square_crossing(a, self.adults)
                    self.adults.append(a)
        elif rule == "mixed_20":
            static_num = np.random.randint(20)
            dynamic_num = 20 - static_num
            self.adult_num = 20
            self._static_adults(static_num, width=6, height=8)
            for i in range(dynamic_num):
                a = new()
                if i < dynamic_num // 2:
                    self._circle_crossing(a, self.adults)
                else:
                    self._square_crossing(a, self.adults)
                self.adults.append(a)
        elif rule == "one_static":
            for x in (-2, -3):
                a = new()
                a.set(x, -8, x, -8, 0, 0, 0)
                self.adults.append(a)
        else:
            raise ValueError("Rule doesn't exist")

    def generate_random_bicycle_position(self, bicycle_num, rule):
        self.bicycles = []
        for _ in range(bicycle_num):
            b = Bicycle(self.config, "bicycles")
            if rule == "circle_crossing":
                self._circle_crossing(b, self.bicycles)
            elif rule == "square_crossing":
                self._square_crossing(b, self.bicycles)
            elif rule == "square_crossing_old":
                self._square_crossing_old(b, self.bicycles)
            else:
                raise Exception("Wrong rule for bicycle: %s" % rule)
            self.bicycles.append(b)

    def generate_random_children_position(self, children_num, rule):
        self.children = []
        for _ in range(children_num):
            if rule != "square_crossing":
                raise Exception("Wrong rule for children: %s" % rule)
            c = Child(self.config, "children")
            self._square_crossing(c, self.children)
            self.children.append(c)

    # ---- static map ---------------------------------------------------------------------------------
    def _near_robot(self, xm, ym, half_x, half_y, circle):
        clear = self.robot.radius + self.discomfort_dist
        for rx, ry in ((self.robot.px, self.robot.py), (self.robot.gx, self.robot.gy)):
            if circle:
                if norm((xm - rx, ym - ry)) < half_x + clear:
                    return True
            elif abs(xm - rx) < half_x + clear and abs(ym - ry) < half_y + clear:
                return True
        return False

    def generate_static_map_input(self, max_size, phase, config=None):
        num_circles = self.num_circles or 0
        num_walls = self.num_walls or 0
        self.final_num_circles, self.final_num_walls = num_circles, num_walls
        res = self.map_resolution
        grid = int(round(max_size / res))
        self.map = np.ones((grid, grid))
        max_loc = int(round(grid))
        obstacles, self.obstacle_vertices = [], []

        def add(loc_x, loc_y, xm, ym, half_x, half_y, dim):
            obstacles.append(Obstacle(int(round(loc_x + grid / 2.0)), int(round(loc_y + grid / 2.0)), dim,
                                      np.zeros([dim[0], dim[1]])))
            self.obstacle_vertices.append([(xm + half_x, ym + half_y), (xm - half_x, ym + half_y),
                                           (xm - half_x, ym - half_y), (xm + half_x, ym - half_y)])

        for _ in range(num_circles):
            for _ in range(MAX_TRIES):
                lx = np.random.randint(-max_loc / 2.0, max_loc / 2.0)
                ly = np.random.randint(-max_loc / 2.0, max_loc / 2.0)
                radius = (np.random.random() + 0.5) * 0.7
                if not self._near_robot(lx * res, ly * res, radius, radius, True):
                    break
            d = int(round(2 * radius / res))
            add(lx, ly, lx * res, ly * res, 1 * radius, 1 * radius, (d, d))
        for _ in range(num_walls):
            for _ in range(MAX_TRIES):
                lx = np.random.randint(-max_loc / 2.0, max_loc / 2.0)
                ly = np.random.randint(-max_loc / 2.0, max_loc / 2.0)
                if np.random.random() > 0.5:
                    x_dim, y_dim = np.random.randint(self.min_wall_length, self.max_wall_length + 1), 1
                else:
                    y_dim, x_dim = np.random.randint(self.min_wall_length, self.max_wall_length + 1), 1
                if not self._near_robot(lx * res, ly * res, x_dim / 2.0, y_dim / 2.0, False):
                    break
            add(lx, ly, lx * res, ly * res, 1 * x_dim / 2.0, 1 * y_dim / 2.0,
                (int(round(x_dim / res)), int(round(y_dim / res))))
        self.place_obstacles_on_map(obstacles, grid)
        self.create_observation_from_static_obstacles(obstacles)
        self.obstacles = obstacles

    def place_obstacles_on_map(self, obstacles, grid):
        """scene_generator.py:888-922, including its cell-by-cell edge path (Python's banker's rounding)."""
        for ob in obstacles:
            dx, dy = ob.dim
            inside = (dx / 2.0 < ob.location_x < grid - dx / 2.0) and (dy / 2.0 < ob.location_y < grid - dy / 2.0)
            if inside:
                x0, y0 = int(round(ob.location_x - dx / 2.0)), int(round(ob.location_y - dy / 2.0))
                self.map[x0:x0 + dx, y0:y0 + dy] = np.minimum(self.map[x0:x0 + dx, y0:y0 + dy], ob.patch)
            else:
                for ix in range(dx):
                    for iy in range(dy):
                        sx, sy = int(round(ob.location_x + ix - dx / 2.0)), int(round(ob.location_y + iy - dy / 2.0))
                        if 0 < sx < grid and 0 < sy < grid:
                            self.map[sx, sy] = ob.patch[ix, iy]

    def create_observation_from_static_obstacles(self, obstacles):
        """Walls / boxes as ADULT_STATIC discs for the robot's observation (scene_generator.py:380-422)."""
        self.static_obstacles_as_pedestrians = []
        put = lambda x, y, r: self.static_obstacles_as_pedestrians.append(  # noqa: E731
            ObservableState(x, y, 0, 0, r, AgentType.ADULT_STATIC))
        for ob, v in zip(obstacles, self.obstacle_vertices):
            cx, cy = (v[0][0] + v[2][0]) / 2.0, (v[0][1] + v[2][1]) / 2.0
            if ob.dim[0] == ob.dim[1]:
                put(cx, cy, (v[0][0] - cx) * np.sqrt(2))
            elif ob.dim[0] > ob.dim[1]:
                r = (v[0][1] - cy) * np.sqrt(2)
                x = v[1][0] + r
                while x < v[0][0]:
                    put(x, cy, r)
                    x = x + 2 * r
            else:
                r = (v[0][0] - cx) * np.sqrt(2)
                y = v[2][1] + r
                while y < v[0][1]:
                    put(cx, y, r)
                    y = y + 2 * r

    # ---- episodes -------------------------------------------------------------------------------------
    def generate_random_scene(self, counter_offset, phase, save_scene_path=None, scene_number=None):
        multi = self.robot.policy.multiagent_training
        if phase in ("train", "val"):
            nums = [n if multi else 1 for n in (self.adult_num, self.bicycle_num, self.children_num)]
            rules = (self.train_val_sim_adult, self.train_val_sim_bicycle, self.train_val_sim_children)
        else:
            nums = [self.adult_num, self.bicycle_num, self.children_num]
            rules = (self.test_sim_adult, self.test_sim_bicycle, self.test_sim_children)
        seed = scene_number if scene_number is not None else counter_offset[phase] + self.case_counter[phase]
        np.random.seed(seed)
        self.generate_random_adult_position(adult_num=nums[0], rule=rules[0])
        self.generate_random_bicycle_position(bicycle_num=nums[1], rule=rules[1])
        self.generate_random_children_position(children_num=nums[2], rule=rules[2])
        self.generate_static_map_input(self.map_size_m, phase)
        self.case_counter[phase] = (self.case_counter[phase] + 1) % self.case_size[phase]
        if save_scene_path is not None:
            self.save_scene(save_scene_path)

    def load_scene(self, phase, load_scene_path):
        with open(load_scene_path, "r") as f:
            scene = json.load(f)
        groups = (("adults", Adult, "adults"), ("bicycles", Bicycle, "bicycles"), ("children", Child, "children"))
        for key, cls, section in groups:
            agents = []
            for state in scene.get(key, []):
                a = cls(self.config, section)
                a.set_from_state_dict(state)
                agents.append(a)
            setattr(self, key, agents)
        self.adult_num, self.bicycle_num, self.children_num = len(self.adults), len(self.bicycles), len(self.children)
        self.obstacle_vertices = scene["map"]["obstacle_vertices"]
        assert len(self.obstacle_vertices) == scene["map"]["num_circles"] + scene["map"]["num_walls"], \
            "Error: length of obstacle_vertices != num_circles + num_walls"
        self.final_num_circles, self.final_num_walls = scene["map"]["num_circles"], scene["map"]["num_walls"]
        grid = int(round(self.map_size_m / self.map_resolution))
        self.map = np.ones((grid, grid))
        obstacles = [Obstacle(o["location"][0], o["location"][1], o["dim"], np.zeros([o["dim"][0], o["dim"][1]]))
                     for o in scene["map"]["obstacles"]]
        self.place_obstacles_on_map(obstacles, grid)
        self.create_observation_from_static_obstacles(obstacles)
        self.obstacles = obstacles
        self.case_counter[phase] = (self.case_counter[phase] + 1) % self.case_size[phase]

    def save_scene(self, path):
        result = {key: [a.get_state_dict() for a in getattr(self, key)] for key in ("adults", "bicycles", "children")}
        result["map"] = {"num_circles": self.final_num_circles, "num_walls": self.final_num_walls,
                         "obstacle_vertices": self.obstacle_vertices,
                         "obstacles": [{"location": (o[0], o[1]), "dim": o[2]} for o in self.obstacles]}
        with open(path, "w") as f:
            json.dump(result, f, indent=4, sort_keys=True)
