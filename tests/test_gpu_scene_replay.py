"""BatchedEnv.reset_batch on the device (ebc_replay_scenes) against the host scene generator it replaces: the state of
4097 episodes, the obstacle polygons, both local maps, and the simulation kernels on a copy of the batch whose grid
rectangles come from rects_from_zero_cells instead.  Needs a B200."""
import configparser
import os

import numpy as np
import pytest
import torch

import oracle_backend as ob
from ebc import abi
from ebc.actions import build_action_space
from ebc.batched_env import BatchedEnv
from ebc.engine import BatchedSim
from host_scenes import host_batch

pytestmark = pytest.mark.gpu
CFG = os.path.join(ob.GOLDEN, "configs")
DEV = "cuda:0"
N = 4097
OFFSET = BatchedEnv.COUNTER_OFFSET
# the golden configs whose rules exist in every phase (env_adults_5_child_5_static_5 has no children rule)
CONFIGS = ["env_adults_3_bikes_3_static_2.config", "env_adults_5.config", "env_adults_5_bikes_0_static_5.config",
           "env_adults_5_bikes_5_static_5.config", "env_ebcadrl.config", "env_fast_train.config"]


def _read(name, over=None):
    cp = configparser.RawConfigParser()
    assert cp.read(os.path.join(CFG, name))
    for (section, key), value in (over or {}).items():
        cp.set(section, key, str(value))
    return cp


def union(rect, count, shape):
    z = np.zeros(shape, bool)
    for x0, y0, x1, y1 in rect[:count].astype(int):
        z[x0:x1, y0:y1] = True
    return z


def check_positions(name, got, want, circle):
    """Bit-exact, except circle_crossing coordinates (the device's double cos / sin): at most one fp32 ulp there."""
    diff = got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64)
    off = np.abs(diff) > 0
    assert np.abs(diff).max() <= 1, (name, np.abs(diff).max())
    assert not (off & ~circle[..., None]).any(), name
    if off.any():
        print("%s: %d circle_crossing coordinates 1 ulp from the host" % (name, int(off.sum())))
    return int(off.sum())


@pytest.mark.parametrize("phase", ["train", "val", "test"])
@pytest.mark.parametrize("config", CONFIGS)
def test_reset_batch_matches_host_generator(config, phase):
    env = BatchedEnv(_read(config), None, N, DEV)
    seeds = np.arange(N) + OFFSET[phase] + 1000
    ref = host_batch(env, phase, seeds)
    before = env.scene.case_counter[phase]
    env.reset_batch(phase, seeds)
    assert env.scene.case_counter[phase] == (before + N) % env.scene.case_size[phase]
    sim = env.sim
    g = {k: getattr(sim, k).cpu().numpy() for k in ("hum_pv", "hum_gr", "hum_type", "hum_count", "stat", "stat_count",
                                                   "rect", "rect_count", "rob_pv", "rob_gr", "rob_theta", "time", "hum_nv")}
    check_positions("hum_pv", g["hum_pv"], ref["hum_pv"], ref["circle_agents"])
    check_positions("hum_gr", g["hum_gr"], ref["hum_gr"], ref["circle_agents"])
    for k in ("hum_type", "hum_count", "stat_count"):
        assert np.array_equal(g[k], ref[k]), k
    if sim.Smax:
        assert np.array_equal(g["stat"], ref["stat"])
    assert not g["hum_nv"].any() and not g["time"].any()
    rad = env.scene.circle_radius
    assert np.array_equal(g["rob_pv"], np.tile(np.array([0, -rad, 0, 0], np.float32), (N, 1)))
    assert np.array_equal(g["rob_gr"], np.tile(np.array([0, rad, env.robot.v_pref, env.robot.radius], np.float32), (N, 1)))
    assert np.array_equal(g["rob_theta"], np.full(N, np.pi / 2, np.float32))
    assert np.array_equal(env.poly_xy.cpu().numpy(), ref["poly_xy"])
    assert np.array_equal(env.poly_count.cpu().numpy(), ref["poly_count"])
    for e in range(N):
        assert np.array_equal(union(g["rect"][e], g["rect_count"][e], ref["maps"][e].shape), ref["maps"][e]), e
        assert not g["rect"][e, g["rect_count"][e]:].any()


def _loaded_copy(env, ref, rect_lists):
    """A second sim holding the same batch, loaded from the host with the given rectangle lists."""
    sim = env.sim
    R = max([len(r) for r in rect_lists] + [1])
    other = BatchedSim(env.cfg, sim.N, sim.Hmax, sim.Smax, R, sim.A, device=DEV)
    rc = np.zeros((sim.N, R, 4), np.int16)
    for e, r in enumerate(rect_lists):
        rc[e, :len(r)] = r
    other.load_episodes(0, sim.hum_pv.cpu().numpy(), sim.hum_gr.cpu().numpy(), sim.hum_type.cpu().numpy(),
                        sim.hum_count.cpu().numpy(), sim.stat.cpu().numpy(), sim.stat_count.cpu().numpy(), rc,
                        np.array([len(r) for r in rect_lists], np.int32), sim.rob_pv.cpu().numpy(),
                        sim.rob_gr.cpu().numpy(), sim.rob_theta.cpu().numpy(), sim.time.cpu().numpy())
    return other


LAYOUT = [("env_adults_3_bikes_3_static_2.config", "test", 1000), ("env_adults_5_bikes_5_static_5.config", "test", 1000),
          ("env_ebcadrl.config", "train", 2000)]


@pytest.mark.parametrize("config,phase,first", LAYOUT)
def test_rectangle_layout_does_not_change_the_simulation(config, phase, first):
    """The replay's per-obstacle rectangles (lattices for striped border circles) against rects_from_zero_cells of the
    same grid: lookahead outcomes, committed steps and the grid local map bit for bit.  Seeds 1000-1511 of
    env_adults_3_bikes_3_static_2 hold striped circles."""
    n = 512
    cp = _read(config)
    env = BatchedEnv(cp, None, n, DEV)
    seeds = np.arange(first, first + n)
    ref = host_batch(env, phase, seeds)
    env.reset_batch(phase, seeds)
    sim = env.sim
    if config.startswith("env_adults_3"):
        assert (sim.rect_count.cpu().numpy() > 2).sum() > 40       # striped circles are in the batch
    other = _loaded_copy(env, ref, ref["rects"])
    actions = np.array(build_action_space(env.robot.v_pref, "holonomic"), dtype=np.float64)
    for s in (sim, other):
        s.set_actions(actions)
    size = cp.getfloat("map", "submap_size_m")
    assert torch.equal(sim.local_map_grid(size), other.local_map_grid(size))
    gen = torch.Generator(device=DEV)
    gen.manual_seed(5)
    for t in range(40):
        for s in (sim, other):
            s.orca()
            s.lookahead()
        for k in ("la_reward", "la_done", "la_event", "vin", "hum_nv"):
            assert torch.equal(getattr(sim, k), getattr(other, k)), (t, k)
        idx = torch.randint(0, len(actions), (n,), device=DEV, generator=gen, dtype=torch.int32)
        for s in (sim, other):
            s.step(action_idx=idx)
        for k in ("reward", "done", "event", "dmin", "hum_pv", "rob_pv", "time"):
            assert torch.equal(getattr(sim, k), getattr(other, k)), (t, k)
        assert torch.equal(sim.local_map_grid(size), other.local_map_grid(size)), t


@pytest.mark.parametrize("config", ["env_adults_3_bikes_3_static_2.config", "env_ebcadrl.config"])
def test_local_maps_equal_a_host_loaded_batch(config):
    cp = _read(config)
    env = BatchedEnv(cp, None, 1024, DEV)
    seeds = np.arange(1000, 2024)
    ref = host_batch(env, "test", seeds)
    env.reset_batch("test", seeds)
    other = _loaded_copy(env, ref, ref["rects"])
    size = cp.getfloat("map", "submap_size_m")
    assert torch.equal(env.sim.local_map_grid(size), other.local_map_grid(size))
    pxy = torch.as_tensor(ref["poly_xy"]).to(DEV)
    pc = torch.as_tensor(ref["poly_count"]).to(DEV)
    assert torch.equal(env.poly_xy, pxy)
    args = (cp.getfloat("map", "angular_map_max_range"), cp.getfloat("map", "angle_min") * np.pi,
            cp.getfloat("map", "angle_max") * np.pi, cp.getint("map", "angular_map_dim"))
    a = env.sim.local_map_angular(env.poly_xy, env.poly_count, *args)
    b = other.local_map_angular(pxy, pc, *args)
    assert torch.equal(a, b)
    assert torch.equal(env.local_map_batch(), a)


STATE = ("hum_pv", "hum_gr", "hum_type", "hum_count", "hum_nv", "stat", "stat_count", "rect", "rect_count", "rob_pv",
         "rob_gr", "rob_theta", "time")


def test_mask_and_permutation():
    env = BatchedEnv(_read("env_adults_3_bikes_3_static_2.config"), None, 777, DEV)
    sim = env.sim
    a, b = np.arange(1000, 1777), np.arange(5000, 5777)
    env.reset_batch("test", a)
    cfg = next(iter(env._replay_configs.values()))
    before = {k: getattr(sim, k).clone() for k in STATE}
    poly = env.poly_xy.clone(), env.poly_count.clone()
    mask = (torch.arange(777, device=DEV) % 3 == 1).to(torch.uint8)
    need = torch.full((777, 5), -7, dtype=torch.int32, device=DEV)
    dev_b = torch.from_numpy(b.astype(np.uint32).view(np.int32)).to(DEV)
    pxy, pc = poly[0].clone(), poly[1].clone()
    sim.replay_scenes(cfg, dev_b, mask=mask, poly_xy=pxy, poly_count=pc, need=need)
    masked = {k: getattr(sim, k).clone() for k in STATE}
    env.reset_batch("test", b)
    full = {k: getattr(sim, k).clone() for k in STATE}
    on = mask.bool()
    for k in STATE:
        assert torch.equal(masked[k][~on], before[k][~on]), k      # untouched, byte for byte
        if k != "hum_nv":
            assert torch.equal(masked[k][on], full[k][on]), k
    assert torch.equal(pxy[~on], poly[0][~on]) and torch.equal(pxy[on], env.poly_xy[on])
    assert (need[~on] == -7).all() and (need[on] >= 0).all()
    perm = np.random.default_rng(3).permutation(777)
    env.reset_batch("test", b[perm])
    p = torch.as_tensor(perm, device=DEV)
    for k in STATE:
        assert torch.equal(getattr(sim, k), full[k][p]), k


def test_capacity_overflow_names_the_seed():
    """Adults only, mixed rule, room for 4 humans: only a scene whose drawn adult count is 5 overflows, and the error
    names the first such seed.  The polygons of the previous reset stay."""
    over = {("sim", "test_sim_adult"): "mixed", ("map", "num_walls"): 1}
    env = BatchedEnv(_read("env_adults_5.config", over), None, 64, DEV, max_humans=4)
    seeds = np.arange(1000, 1064)
    counts = host_batch(env, "test", seeds)["hum_count"]
    assert counts.min() < 5 and counts.max() == 5
    first = int(seeds[np.argmax(counts > 4)])
    ok = seeds[counts <= 4][:1].repeat(64)
    env.reset_batch("test", ok)
    poly = env.poly_xy.clone()
    counter = dict(env.scene.case_counter)
    with pytest.raises(abi.EbcError, match=r"scene %d exceeds the batch capacity \(H=5, S=" % first):
        env.reset_batch("test", seeds)
    assert torch.equal(env.poly_xy, poly) and env.scene.case_counter == counter
    env = BatchedEnv(_read("env_adults_3_bikes_3_static_2.config"), None, 200, DEV, max_rects=2)
    with pytest.raises(abi.EbcError, match=r"scene \d+ needs \d+ grid rectangles \(capacity 2\)"):
        env.reset_batch("test", np.arange(1000, 1200))
    env = BatchedEnv(_read("env_adults_5.config"), None, 2, DEV)
    for bad in ([0, -1], [0, 2 ** 32]):
        with pytest.raises(ValueError):
            env.reset_batch("test", bad)
    env.reset_batch("test", [0, 2 ** 32 - 1])


def test_mixed_rule_keeps_the_adult_count_side_effect():
    """The mixed rules leave the adult count they drew in SceneGenerator.adult_num, which a later train / val batch of
    a config with another rule there reads; the replay reports it the same way."""
    over = {("sim", "test_sim_adult"): "mixed", ("sim", "train_val_sim_adult"): "circle_crossing"}
    cp = _read("env_adults_5_bikes_5_static_5.config", over)
    env = BatchedEnv(cp, None, 32, DEV)
    host = BatchedEnv(cp, None, 32, DEV)
    seeds = np.arange(1000, 1032)
    host_batch(host, "test", seeds)
    env.reset_batch("test", seeds)
    assert env.scene.adult_num == host.scene.adult_num
    ref = host_batch(env, "train", np.arange(2000, 2032))
    env.reset_batch("train", np.arange(2000, 2032))
    assert np.array_equal(env.sim.hum_count.cpu().numpy(), ref["hum_count"])


def test_striped_test_seeds_reset_at_the_default_capacity():
    """env_adults_3_bikes_3_static_2's test seeds 1000-1999: about one in six puts its circle on the map border with an
    odd cell count; every scene fits the default capacity now."""
    env = BatchedEnv(_read("env_adults_3_bikes_3_static_2.config"), None, 1000, DEV)
    env.reset_batch("test", np.arange(1000, 2000))
    counts = env.sim.rect_count.cpu().numpy()
    assert counts.max() <= env.sim.Rmax and (counts > 2).sum() > 100
