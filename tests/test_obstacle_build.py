"""Walls-aware humans on the reference's seeded scenes (SURVEY 8f-4), the CPU half: the env INI key that turns them on,
and the obstacle packer -- the __host__ __device__ function that ebc_build_obstacles runs per episode on the device and
ebc_pack_obstacles on the host -- against the oracle's independent restatement of RVO2, byte for byte, on the
polygons the scene replay really produces."""
import configparser
import ctypes
import os

import numpy as np

import oracle_backend as ob
from ebc import abi
from ebc import scene as S
from ebc.config import SimConfig

CFG = os.path.join(ob.GOLDEN, "configs")
ENV_CONFIGS = sorted(f for f in os.listdir(CFG) if f.endswith(".config") and "[env]" in open(os.path.join(CFG, f)).read())


def read_config(name, over=None):
    cp = configparser.RawConfigParser()
    assert cp.read(os.path.join(CFG, name))
    for (section, key), value in (over or {}).items():
        cp.set(section, key, str(value))
    return cp


# the scenes both halves of the suite pack: a circle (as a square) and a wall, the 5-wall config, env_ebcadrl, and
# env_ebcadrl with 10 walls (whose splitting can exceed 64 records)
WALLS10 = {("map", "num_walls"): 10}
SCENES = [("env_adults_3_bikes_3_static_2.config", None), ("env_adults_5_bikes_5_static_5.config", None),
          ("env_ebcadrl.config", None), ("env_ebcadrl.config", WALLS10)]


def pack(fn, poly_xy, count, cap):
    """One episode's quadrilaterals (float64 [P, 4, 2], the first `count` real) through a packer with the C signature of
    ebc_pack_obstacles, narrowed to float32 like the device builder -> (status, records as bytes)."""
    xy = np.ascontiguousarray(poly_xy[:count], dtype=np.float32).ravel()
    sizes = np.full(max(count, 1), 4, np.int32)
    out = np.zeros(64, dtype=abi.OBST_DTYPE)
    n = ctypes.c_int32(-1)
    rc = fn(xy.ctypes.data_as(ctypes.c_void_p), sizes.ctypes.data_as(ctypes.c_void_p), count,
            out.ctypes.data_as(ctypes.c_void_p), cap, ctypes.byref(n))
    return (rc, out[:n.value].tobytes() if rc == 0 else b"")


def scene_polygons(cp, phase, seeds):
    """scene.obstacle_vertices of each seed, from the library's host replay of the reference's scene generator."""
    from ebc.batched_env import _RobotStub
    from simulator.scene.scene_generator import SceneGenerator
    sg = SceneGenerator(cp)
    sg.set_robot(_RobotStub(cp, type("P", (), dict(multiagent_training=True, name="none", kinematics="holonomic"))()))
    P = max((sg.num_circles or 0) + (sg.num_walls or 0), 1)
    cfg = S.replay_config(sg, phase, True, P)
    for seed in seeds:
        o = S.replay_scene_host(cfg, seed, 64, 256, S.replay_rect_bound(sg) + 2)
        yield seed, o["poly_xy"], int(o["need"][3])


def test_orca_obstacles_key():
    for name in ENV_CONFIGS:
        assert SimConfig.from_ini(read_config(name)).orca_obstacles is False, name
    for value, want in (("true", True), ("false", False), ("1", True), ("off", False)):
        cp = read_config("env_ebcadrl.config", {("sim", "orca_obstacles"): value})
        assert SimConfig.from_ini(cp).orca_obstacles is want, value


def test_packer_matches_oracle_on_replayed_scenes(oracle):
    """ebc_pack_obstacles == ebc_ref_pack_obstacles byte for byte on 300 test-phase scenes of every config, at cap 64
    and, where the splitting adds records, at a cap one short of them (which both must refuse)."""
    lib = abi.load()
    splits = overflow64 = forced = 0
    for name, over in SCENES:
        for seed, poly, count in scene_polygons(read_config(name, over), "test", range(1000, 1300)):
            a = pack(lib.ebc_pack_obstacles, poly, count, 64)
            b = pack(oracle.lib.ebc_ref_pack_obstacles, poly, count, 64)
            assert a == b, (name, seed)
            if a[0] != 0:
                assert a[0] == abi.ERR_INVALID
                overflow64 += 1
                continue
            n = len(a[1]) // 48
            if n > 4 * count:
                splits += 1
                c = pack(lib.ebc_pack_obstacles, poly, count, n - 1)
                assert c == pack(oracle.lib.ebc_ref_pack_obstacles, poly, count, n - 1) and c[0] == abi.ERR_INVALID
                forced += 1
                assert pack(lib.ebc_pack_obstacles, poly, count, n) == a       # exactly enough room
    print("splits %d, overflow at 64: %d, forced overflow %d" % (splits, overflow64, forced))
    assert splits > 100 and forced > 100 and overflow64 > 0
