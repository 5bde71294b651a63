"""The device scene replay (ebc_replay_scenes) on the host: its numpy primitives against numpy itself, and the whole
per-episode replay -- the same __host__ __device__ function, through the library's diagnostics export
ebc_replay_scene_host -- against simulator/scene/scene_generator.py, bit for bit.  CPU only."""
import configparser
import ctypes
import os

import numpy as np
import pytest

import oracle_backend as ob
from ebc import abi
from ebc import scene as S

CFG = os.path.join(ob.GOLDEN, "configs")
SIM_CONFIGS = sorted(f for f in os.listdir(CFG) if f.endswith(".config") and "[sim]" in open(os.path.join(CFG, f)).read())


@pytest.fixture(scope="module")
def lib():
    return abi.load()


# ---- numpy primitives ---------------------------------------------------------------------------------------------
def _twin(lib, state, op, a=0.0, b=0.0):
    """Run one primitive of the replay on numpy's state tuple; returns (result, new key, new pos)."""
    key = np.array(state[1], dtype=np.uint32)
    pos = ctypes.c_int32(int(state[2]))
    out = ctypes.c_double(0.0)
    assert lib.ebc_replay_rng_host(key.ctypes.data_as(ctypes.c_void_p), ctypes.byref(pos), op, a, b, ctypes.byref(out)) == 0
    return out.value, key, pos.value


def _random_states(n, seed):
    rng = np.random.default_rng(seed)
    for _ in range(n):
        yield ("MT19937", rng.integers(0, 2 ** 32, 624, dtype=np.uint64).astype(np.uint32), int(rng.integers(0, 625)), 0, 0.0)


def _numpy(state, fn):
    np.random.set_state(state)
    value = fn()
    after = np.random.get_state()
    return value, after[1], after[2]


def _same(twin, ref):
    assert twin[0] == ref[0], (twin[0], ref[0])
    assert twin[2] == ref[2], "draw count differs: pos %d vs numpy %d" % (twin[2], ref[2])
    assert np.array_equal(twin[1], ref[1])


def test_seed_is_init_genrand(lib):
    blank = ("MT19937", np.zeros(624, np.uint32), 0, 0, 0.0)
    for seed in (0, 1, 5489, 1000000, 2 ** 31, 2 ** 32 - 1, 123456789):
        np.random.seed(seed)
        ref = np.random.get_state()
        _, key, pos = _twin(lib, blank, abi.REPLAY_RNG_SEED, float(seed))
        assert pos == ref[2] == 624 and np.array_equal(key, ref[1]), seed


def test_random_matches_numpy(lib):
    for st in _random_states(400, 1):
        _same(_twin(lib, st, abi.REPLAY_RNG_RANDOM), _numpy(st, np.random.random))


def test_uniform_matches_numpy(lib):
    rng = np.random.default_rng(2)
    for st in _random_states(400, 3):
        lo, hi = sorted(rng.normal(size=2) * 5)
        if rng.random() < 0.3:
            lo, hi = -abs(lo), abs(lo)              # the generator's symmetric ranges (-hw, hw)
        _same(_twin(lib, st, abi.REPLAY_RNG_UNIFORM, lo, hi), _numpy(st, lambda: np.random.uniform(lo, hi)))


@pytest.mark.parametrize("lo,hi", [(-45.0, 45.0), (-22.5, 22.5), (-45.5, 45.5), (-70.0, 70.0), (0, 20), (0, 3), (0, 4),
                                   (1, 6), (2, 4), (3, 4), (-0.5, 1.5), (0, 1000), (-7.5, -2.5)])
def test_randint_matches_numpy(lib, lo, hi):
    """Masked rejection on 32-bit outputs; float bounds truncated toward zero; a one-value range draws nothing."""
    for st in _random_states(300, int(abs(lo) * 10 + hi)):
        _same(_twin(lib, st, abi.REPLAY_RNG_RANDINT, lo, hi), _numpy(st, lambda: float(np.random.randint(lo, hi))))


def test_choice_matches_numpy(lib):
    for st in _random_states(300, 5):
        _same(_twin(lib, st, abi.REPLAY_RNG_CHOICE_SIGN),
              _numpy(st, lambda: float(np.random.choice([1, -1], p=[0.5, 0.5]))))
    sides = ["top", "bottom", "left", "right"]
    for st in _random_states(300, 6):                # choice(list) without p: one randint(0, len)
        _same(_twin(lib, st, abi.REPLAY_RNG_RANDINT, 0, 4),
              _numpy(st, lambda: float(sides.index(np.random.choice(sides)))))


def test_norm_probe_matches_numpy():
    """The norm the replay is configured with (ebc_replay_config.norm_fused) is numpy's on 2000 random pairs."""
    from fractions import Fraction
    x, y = np.random.default_rng(7).normal(size=(2, 2000)) * 3
    fused = S.numpy_norm_is_fused()
    for a, b in zip(x.tolist(), y.tolist()):
        want = float(np.linalg.norm((a, b)))
        assert want == (float(np.sqrt(float(Fraction(b) ** 2 + Fraction(a * a)))) if fused else float(np.sqrt(a * a + b * b)))


# ---- the whole replay against the host generator ------------------------------------------------------------------
class _Policy(object):
    name, kinematics = "none", "holonomic"

    def __init__(self, multi):
        self.multiagent_training = multi


def _generator(cp, multi=True):
    from ebc.batched_env import _RobotStub
    from simulator.scene.scene_generator import SceneGenerator
    sg = SceneGenerator(cp)
    robot = _RobotStub(cp, _Policy(multi))
    sg.set_robot(robot)
    return sg, robot


def _read(name, over=None):
    cp = configparser.RawConfigParser()
    assert cp.read(os.path.join(CFG, name))
    for (section, key), value in (over or {}).items():
        if not cp.has_section(section):
            cp.add_section(section)
        cp.set(section, key, str(value))
    return cp


def compare_replay(cp, phase, seeds, multi=True):
    """Host twin vs SceneGenerator on every seed: every stored field bit for bit, the rectangles' union equal to
    scene.map == 0 and within the configured bound.  Returns the number of scenes with a striped border patch."""
    sg, robot = _generator(cp, multi)
    P = max((sg.num_circles or 0) + (sg.num_walls or 0), 1)
    bound = S.replay_rect_bound(sg)
    striped = 0
    try:
        robot.set(0, -sg.circle_radius, 0, sg.circle_radius, 0, 0, np.pi / 2)
        sg.generate_random_scene(None, phase, scene_number=0)
    except Exception:               # a list without a rule for this phase: the config cannot generate scenes at all
        with pytest.raises(ValueError):
            S.replay_config(sg, phase, multi, P)
        return None
    for seed in seeds:
        cfg = S.replay_config(sg, phase, multi, P)
        robot.set(0, -sg.circle_radius, 0, sg.circle_radius, 0, 0, np.pi / 2)
        sg.generate_random_scene({"train": 2000, "val": 0, "test": 1000}, phase, scene_number=int(seed))
        hs = sg.adults + sg.bicycles + sg.children
        st = sg.static_obstacles_as_pedestrians
        H, Sn = len(hs), len(st)
        o = S.replay_scene_host(cfg, seed, 64, Sn + 2, bound + 2)
        tag = "seed %d" % seed
        assert list(o["need"][:4]) == [H, Sn, o["need"][2], P if (sg.num_circles or 0) + (sg.num_walls or 0) else 0], tag
        if cfg.rule[0] in (abi.REPLAY_RULES["mixed"], abi.REPLAY_RULES["mixed_20"]):
            assert o["need"][4] == sg.adult_num, tag
        assert np.array_equal(o["hum_pv"][:H], np.array([[h.px, h.py, h.vx, h.vy] for h in hs], np.float32).reshape(-1, 4)), tag
        assert np.array_equal(o["hum_gr"][:H], np.array([[h.gx, h.gy, h.v_pref, h.radius] for h in hs], np.float32).reshape(-1, 4)), tag
        assert np.array_equal(o["hum_type"][:H], np.array([int(h.agent_type) for h in hs], np.uint8)), tag
        assert not o["hum_pv"][H:].any() and not o["hum_gr"][H:].any() and not o["hum_type"][H:].any(), tag
        assert np.array_equal(o["stat"][:Sn], np.array([[s.px, s.py, s.radius, 0] for s in st], np.float32).reshape(-1, 4)), tag
        assert not o["stat"][Sn:].any(), tag
        verts = np.asarray(sg.obstacle_vertices, np.float64).reshape(-1, 4, 2)
        assert np.array_equal(o["poly_xy"][:len(verts)], verts) and not o["poly_xy"][len(verts):].any(), tag
        nr = int(o["need"][2])
        assert nr <= bound and not o["rect"][nr:].any(), (tag, nr, bound)
        zero = np.zeros(sg.map.shape, bool)
        for x0, y0, x1, y1 in o["rect"][:nr].astype(int):
            assert 0 <= x0 < x1 <= zero.shape[0] and 0 <= y0 < y1 <= zero.shape[1], tag
            zero[x0:x1, y0:y1] = True
        assert np.array_equal(zero, sg.map == 0), tag
        striped += nr > len(sg.obstacles)
    return striped


@pytest.mark.parametrize("phase", ["train", "val", "test"])
@pytest.mark.parametrize("config", SIM_CONFIGS)
def test_replay_matches_scene_generator(config, phase):
    start = {"train": 2000, "val": 0, "test": 1000}[phase]
    compare_replay(_read(config), phase, range(start, start + 500))


VARIANTS = {
    # (base config, overrides, multiagent_training)
    "mixed": ("env_adults_5_bikes_5_static_5.config", {("sim", "test_sim_adult"): "mixed", ("sim", "train_val_sim_adult"): "mixed"}, True),
    "mixed_randomized": ("env_ebcadrl.config", {("sim", "test_sim_adult"): "mixed", ("sim", "train_val_sim_adult"): "mixed",
                                                ("adults", "radius"): 0.3, ("adults", "v_pref"): 1.0}, True),
    "mixed_20": ("env_adults_5_bikes_5_static_5.config", {("sim", "test_sim_adult"): "mixed_20", ("sim", "train_val_sim_adult"): "mixed_20"}, True),
    "one_static": ("env_adults_3_bikes_3_static_2.config", {("sim", "test_sim_adult"): "one_static", ("sim", "train_val_sim_adult"): "one_static"}, True),
    "single_agent": ("env_fast_train.config", {}, False),
    "single_agent_ebcadrl": ("env_ebcadrl.config", {}, False),
    "map_14m": ("env_adults_3_bikes_3_static_2.config", {("map", "map_size_m"): 14, ("map", "num_walls"): 3, ("map", "num_circles"): 2}, True),
    "odd_grid": ("env_adults_3_bikes_3_static_2.config", {("map", "map_size_m"): 9.1, ("map", "num_walls"): 3, ("map", "num_circles"): 2}, True),
    # walls of 267 x 67 cells (odd both ways): a border wall is a lattice of up to 134 x 34 rectangles
    "fine_grid": ("env_adults_5_bikes_5_static_5.config", {("map", "map_resolution"): 0.015, ("map", "min_wall_length"): 4,
                                                           ("map", "max_wall_length"): 4}, True),
    "coarse_grid": ("env_adults_5_bikes_5_static_5.config", {("map", "map_resolution"): 0.3, ("map", "num_circles"): 2}, True),
    "bikes_circle": ("env_adults_5_bikes_5_static_5.config", {("sim", "test_sim_bicycle"): "circle_crossing",
                                                              ("sim", "train_val_sim_bicycle"): "circle_crossing"}, True),
}


@pytest.mark.parametrize("phase", ["train", "test"])
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_replay_matches_scene_generator_variants(variant, phase):
    base, over, multi = VARIANTS[variant]
    compare_replay(_read(base, over), phase, range(1000, 1500), multi=multi)


def test_replay_extreme_seeds():
    for config in SIM_CONFIGS:
        compare_replay(_read(config), "test", [0, 1, 2 ** 31, 2 ** 32 - 2, 2 ** 32 - 1])


def test_striped_circles_are_lattices():
    """env_adults_3_bikes_3_static_2's test seeds put its circle on the border with an odd cell count about one time in
    six; the union of the lattice rectangles is still exactly the map, within the configured bound."""
    assert compare_replay(_read("env_adults_3_bikes_3_static_2.config"), "test", range(1000, 2000)) > 100


def test_golden_scenes():
    """tests/golden/scenes.npz (the reference's own scenes) straight from the replay."""
    z = np.load(os.path.join(ob.GOLDEN, "scenes.npz"))
    for tag, config in (("adults5", "env_adults_5.config"), ("ebcadrl", "env_ebcadrl.config")):
        sg, _ = _generator(_read(config))
        cfg = S.replay_config(sg, "test", True, max((sg.num_circles or 0) + (sg.num_walls or 0), 1))
        for seed in (1002, 1003, 1000000):
            o = S.replay_scene_host(cfg, seed, 64, 16, 16)
            H, Sn, nr = int(o["need"][0]), int(o["need"][1]), int(o["need"][2])
            assert np.array_equal(o["hum_pv"][:H], z["%s_%d_hum_pv" % (tag, seed)].astype(np.float32))
            assert np.array_equal(o["hum_gr"][:H], z["%s_%d_hum_gr" % (tag, seed)].astype(np.float32))
            assert np.array_equal(o["hum_type"][:H], z["%s_%d_hum_type" % (tag, seed)])
            assert np.array_equal(o["stat"][:Sn], z["%s_%d_stat" % (tag, seed)].astype(np.float32).reshape(-1, 4))
            grid = int(round(sg.map_size_m / sg.map_resolution))
            zero = np.zeros((grid, grid), bool)
            for x0, y0, x1, y1 in o["rect"][:nr].astype(int):
                zero[x0:x1, y0:y1] = True
            assert np.array_equal(np.packbits(zero.astype(np.uint8), axis=None), z["%s_%d_map_zero" % (tag, seed)])


def test_capacity_is_reported_not_overrun():
    sg, _ = _generator(_read("env_ebcadrl.config"))
    cfg = S.replay_config(sg, "test", True, 1)
    full = S.replay_scene_host(cfg, 1000, 64, 16, 16)
    small = S.replay_scene_host(cfg, 1000, 5, 2, 1)
    assert list(small["need"]) == list(full["need"]) and full["need"][0] == 24 and full["need"][3] == 3
    assert np.array_equal(small["hum_pv"], full["hum_pv"][:5]) and np.array_equal(small["stat"], full["stat"][:2])
    assert np.array_equal(small["poly_xy"], full["poly_xy"][:1])


def test_default_rect_bound_follows_the_config():
    sg, _ = _generator(_read("env_adults_3_bikes_3_static_2.config"))
    assert S.replay_rect_bound(sg) == 1 + 11 ** 2          # one wall + a 21-cell circle striped both ways
    sg, _ = _generator(_read("env_ebcadrl.config"))
    assert S.replay_rect_bound(sg) == 3
    sg, _ = _generator(_read("env_adults_5.config"))
    assert S.replay_rect_bound(sg) == 0
    sg, _ = _generator(_read("env_adults_5_bikes_5_static_5.config", {("map", "map_resolution"): 0.3}))
    assert S.replay_rect_bound(sg) == 5 * 2 * 9            # 3-cell thickness: 2 runs; lengths up to 17 cells: 9 runs
