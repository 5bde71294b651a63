"""Host-side scene helpers: what `env.reset` hands to the hot path.

The occupancy grid (simulator/scene/scene_generator.py:292-328,888-922) is uploaded as a list
of half-open zero-cell rectangles; the robot/wall test of simulator/env.py:227-261 (window
sum over scene.map) is then an integer AABB-overlap test, bit-identical to the grid test.

`replay_config` turns a SceneGenerator's settings for one phase into the ebc_replay_config with which
ebc_replay_scenes regenerates the reference's seeded scenes on the device; `replay_scene_host` runs the
same replay on the host for one seed (the library's diagnostics export).
"""
import ctypes
import math
from fractions import Fraction

import numpy as np


def rects_from_zero_cells(zero):
    """Exact decomposition of a boolean grid (True = obstacle cell, scene.map == 0) into
    disjoint rectangles [x0, x1) x [y0, y1) (x = first index, y = second index).
    Greedy: maximal runs along y per row, merged along x while identical."""
    zero = np.asarray(zero, dtype=bool)
    gx, gy = zero.shape
    open_runs = {}   # (y0, y1) -> x0
    rects = []
    for x in range(gx + 1):
        runs = set()
        if x < gx:
            row = zero[x]
            if row.any():
                d = np.diff(np.concatenate(([0], row.astype(np.int8), [0])))
                starts, ends = np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]
                runs = set(zip(starts.tolist(), ends.tolist()))
        for run in list(open_runs):
            if run not in runs:
                rects.append((open_runs.pop(run), run[0], x, run[1]))
        for run in runs:
            if run not in open_runs:
                open_runs[run] = x
    rects.sort()
    return np.asarray(rects, dtype=np.int16).reshape(-1, 4)


def wall_polygon(cx, cy, x_dim, y_dim, inflation=1.0):
    """The 4 vertices the reference records for a wall (scene_generator.py:269-290): counter-clockwise from the
    (+, +) corner, inflated by `inflation` (its inflation_rate_il)."""
    hx, hy = inflation * x_dim / 2.0, inflation * y_dim / 2.0
    return [(cx + hx, cy + hy), (cx - hx, cy + hy), (cx - hx, cy - hy), (cx + hx, cy - hy)]


def pack_obstacles(polygons, cap=64):
    """RVO2 addObstacle for every polygon + processObstacles (simulator/policy/orca_obstacles.py:102-107) through
    the library's host entry point ebc_pack_obstacles -> structured array of ebc_obst_vertex records.  When the
    kd-tree's edge splitting needs more than `cap` vertices, polygons are dropped from the END of the list until it
    fits (returned as the second value: how many polygons were kept)."""
    import ctypes
    from . import abi
    lib = abi.load()
    polys = [list(p) for p in polygons]
    while True:
        out = np.zeros(max(cap, 1), dtype=abi.OBST_DTYPE)
        n = ctypes.c_int32(0)
        xy = np.asarray([c for p in polys for v in p for c in v[:2]], dtype=np.float32)
        sizes = np.asarray([len(p) for p in polys], dtype=np.int32)
        rc = lib.ebc_pack_obstacles(xy.ctypes.data_as(ctypes.c_void_p), sizes.ctypes.data_as(ctypes.c_void_p), len(polys),
                                    out.ctypes.data_as(ctypes.c_void_p), cap, ctypes.byref(n))
        if rc == 0:
            return out[:n.value].copy(), len(polys)
        if not polys:
            raise abi.EbcError("ebc_pack_obstacles failed on an empty polygon list")
        polys.pop()


_norm_fused = None


def numpy_norm_is_fused():
    """Whether numpy.linalg.norm((x, y)), which the scene generator's distance tests use, computes
    sqrt(fma(y, y, x * x)) -- OpenBLAS's ddot on FMA-capable x86 cores -- or sqrt(x * x + y * y).  The two differ in the
    last bit for about one pair in ten; probed once on pairs where they differ."""
    global _norm_fused
    if _norm_fused is None:
        rng = np.random.default_rng(20261021)
        votes = set()
        for _ in range(256):
            x, y = float(rng.normal()), float(rng.normal())
            plain = math.sqrt(x * x + y * y)
            fused = math.sqrt(float(Fraction(y) ** 2 + Fraction(x * x)))    # one rounding of y*y + round(x*x)
            if plain != fused:
                got = float(np.linalg.norm((x, y)))
                votes.add(1 if got == fused else 0 if got == plain else -1)
        if votes != {1} and votes != {0}:
            from . import abi
            raise abi.EbcError("numpy.linalg.norm of a 2-vector is neither sqrt(x*x + y*y) nor sqrt(fma(y, y, x*x)) here")
        _norm_fused = votes.pop()
    return _norm_fused


def _runs_max(d):
    """Most runs of zero cells the per-cell path of place_obstacles_on_map writes along an axis of d cells: one for an
    even d (consecutive integers), ceil(d / 2) for an odd d (half-integers rounded half to even: every other cell)."""
    return 0 if d <= 0 else 1 if d % 2 == 0 else (d + 1) // 2


def _rects_max(dx, dy):
    return 0 if dx <= 0 or dy <= 0 else max(1, _runs_max(dx) * _runs_max(dy))


def replay_rect_bound(sg):
    """Grid rectangles ebc_replay_scenes may need for a scene of SceneGenerator `sg`: per obstacle, one for the slice of
    an obstacle inside the map, runs(x) * runs(y) for one on the border -- walls over their length range (a wall is
    round(L / res) x round(1 / res) cells), circles over d = round(2 r / res) for the radius range [0.35, 1.05)
    (scene_generator.py: (random() + 0.5) * 0.7)."""
    res = sg.map_resolution
    walls = sg.num_walls or 0
    circles = sg.num_circles or 0
    wall = max([_rects_max(int(round(L / res)), int(round(1 / res)))
                for L in range(sg.min_wall_length, sg.max_wall_length + 1)] + [0]) if walls else 0
    circle = max(_rects_max(d, d) for d in range(int(round(0.7 / res)), int(round(2.1 / res)) + 1)) if circles else 0
    return walls * wall + circles * circle


def replay_config(sg, phase, multiagent_training, max_polys):
    """ebc_replay_config for generate_random_scene(phase) of SceneGenerator `sg` (its robot set): the lists' counts and
    rules as that phase resolves them (one agent per list in train / val without multiagent_training), the agent
    sections' radius / v_pref and their ranges, the map and the robot."""
    from . import abi
    c = abi.EbcReplayConfig()
    if phase in ("train", "val"):
        counts = [n if multiagent_training else 1 for n in (sg.adult_num, sg.bicycle_num, sg.children_num)]
        rules = (sg.train_val_sim_adult, sg.train_val_sim_bicycle, sg.train_val_sim_children)
    else:
        counts = [sg.adult_num, sg.bicycle_num, sg.children_num]
        rules = (sg.test_sim_adult, sg.test_sim_bicycle, sg.test_sim_children)
    allowed = (("square_crossing", "circle_crossing", "mixed", "mixed_20", "one_static"),
               ("square_crossing", "circle_crossing", "square_crossing_old"), ("square_crossing",))
    for t, (section, n, rule) in enumerate(zip(("adults", "bicycles", "children"), counts, rules)):
        if rule not in allowed[t] and (t == 0 or n > 0):
            raise ValueError("Rule %r doesn't exist for %s" % (rule, section))
        c.count[t] = n
        c.rule[t] = abi.REPLAY_RULES.get(rule, 0)
        get = lambda key: sg.config.getfloat(section, key, fallback=None) if sg.config.has_section(section) else None  # noqa: E731
        vals = {k: get(k) for k in ("v_pref", "radius", "v_pref_min", "v_pref_max", "radius_min", "radius_max")}
        standing = t == 0 and rule in ("mixed", "mixed_20", "one_static")     # places agents without drawing them
        if n > 0 or standing:
            need = ["v_pref", "radius"] if standing or not sg.randomize_attributes else []
            need += ["v_pref_min", "v_pref_max", "radius_min", "radius_max"] if sg.randomize_attributes else []
            missing = [k for k in need if vals[k] is None]
            if missing:
                raise ValueError("[%s] lacks %s for the %s phase's scenes" % (section, ", ".join(missing), phase))
        for k, v in vals.items():
            getattr(c, k)[t] = 0.0 if v is None else v
    c.randomize_attributes = int(bool(sg.randomize_attributes))
    c.num_circles, c.num_walls = sg.num_circles or 0, sg.num_walls or 0
    c.min_wall_length, c.max_wall_length = sg.min_wall_length, sg.max_wall_length
    c.max_polys = max_polys
    c.norm_fused = numpy_norm_is_fused()
    c.square_width, c.circle_radius, c.discomfort_dist = sg.square_width, sg.circle_radius, sg.discomfort_dist
    c.robot_radius, c.robot_v_pref = sg.robot.radius, sg.robot.v_pref
    c.map_size_m, c.map_resolution = sg.map_size_m, sg.map_resolution
    return c


def replay_scene_host(cfg, seed, max_humans, max_statics, max_rects):
    """ebc_replay_scenes' replay of one seed, run on the host (diagnostics export of the library): dict of numpy arrays
    in the ebc_state layout of one episode (hum_pv, hum_gr, hum_type, stat, rect, poly_xy) and need = (humans, static
    discs, rectangles, polygons, adult_num)."""
    from . import abi
    lib = abi.load()
    out = {"hum_pv": np.zeros((max_humans, 4), np.float32), "hum_gr": np.zeros((max_humans, 4), np.float32),
           "hum_type": np.zeros(max_humans, np.uint8), "stat": np.zeros((max_statics, 4), np.float32),
           "rect": np.zeros((max_rects, 4), np.int16), "poly_xy": np.zeros((cfg.max_polys, 4, 2), np.float64),
           "need": np.zeros(5, np.int32)}
    p = {k: v.ctypes.data_as(ctypes.c_void_p) for k, v in out.items()}
    rc = lib.ebc_replay_scene_host(ctypes.byref(cfg), int(seed), max_humans, max_statics, max_rects, p["hum_pv"],
                                   p["hum_gr"], p["hum_type"], p["stat"], p["rect"], p["poly_xy"], p["need"])
    if rc != 0:
        raise abi.EbcError("ebc_replay_scene_host: bad argument")
    return out
