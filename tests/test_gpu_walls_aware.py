"""Walls-aware humans on the reference's seeded scenes (`[sim] orca_obstacles = true`, SURVEY 8f-4) on the device:
ebc_build_obstacles against the host packer, the whole decision loop against the oracle, what the half-planes
guarantee, the key's default, the N = 1 env, and the CLI.  Needs a B200."""
import configparser
import os

import numpy as np
import pytest
import torch

import oracle_backend as ob
from ebc import abi
from ebc import scene as S
from ebc.actions import build_action_space
from ebc.batched_env import BatchedEnv, TargetValue
from ebc.engine import BatchedSim
from test_obstacle_build import SCENES, WALLS10, pack, read_config

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OFFSET = BatchedEnv.COUNTER_OFFSET
ON = {("sim", "orca_obstacles"): "true"}
WALLS5 = "env_adults_5_bikes_5_static_5.config"
STATE = ("hum_pv", "hum_gr", "hum_type", "hum_count", "stat", "stat_count", "rect", "rect_count", "rob_pv", "rob_gr",
         "rob_theta", "time", "obst", "obst_count")


def _env(name, over=None, n=1, **kw):
    return BatchedEnv(read_config(name, {**(over or {}), **ON}), None, n, DEV, **kw)


def _replay(env, phase, seeds, mask=None):
    """The first half of reset_batch, without its capacity check: the replayed polygons and the obstacle build's need."""
    sg = env.scene
    cfg = S.replay_config(sg, phase, True, max((sg.num_circles or 0) + (sg.num_walls or 0), 1))
    dev_seeds = torch.from_numpy(np.asarray(seeds, np.uint32).view(np.int32)).to(DEV)
    pxy, pc, _ = env.sim.replay_scenes(cfg, dev_seeds)
    return pxy, pc, env.sim.build_obstacles(pxy, pc, mask=mask)


def _check_against_host(env, phase, seeds):
    """obst / obst_count / need of every episode == ebc_pack_obstacles on the episode's polygons as float32, at Omax;
    reset_batch then raises for the first seed that overflows, or loads the same records.  -> (splits, overflows)."""
    lib, sim = abi.load(), env.sim
    pxy, pc, need = _replay(env, phase, seeds)
    need, pxy, pc = need.cpu().numpy(), pxy.cpu().numpy(), pc.cpu().numpy()
    obst, cnt = sim.obst.cpu().numpy(), sim.obst_count.cpu().numpy()
    splits = 0
    for e in range(len(seeds)):
        rc, rec = pack(lib.ebc_pack_obstacles, pxy[e], int(pc[e]), sim.Omax)
        if rc != 0:
            assert need[e] == -1 and cnt[e] == 0, e
            continue
        assert need[e] == cnt[e] == len(rec) // 48, e
        assert obst[e, :cnt[e]].tobytes() == rec, e
        splits += cnt[e] > 4 * pc[e]
    bad = np.nonzero(need < 0)[0]
    if len(bad):
        with pytest.raises(abi.EbcError, match=r"scene %d needs more than %d ORCA obstacle records" % (seeds[bad[0]], sim.Omax)):
            env.reset_batch(phase, seeds)
    else:
        env.reset_batch(phase, seeds)
        assert np.array_equal(sim.obst.cpu().numpy(), obst) and np.array_equal(sim.obst_count.cpu().numpy(), cnt)
    return splits, len(bad)


@pytest.mark.parametrize("phase", ["train", "test"])
@pytest.mark.parametrize("name,over", SCENES, ids=["adults3_bikes3_static2", "walls5", "ebcadrl", "ebcadrl_walls10"])
def test_device_builder_matches_host_packer(name, over, phase):
    """4097 episodes (the last block of the kernel partly filled) at Omax = 64, and again at Omax = the polygons' own
    vertex count, where every split overflows."""
    N = 4097
    seeds = np.arange(N) + OFFSET[phase] + 1000
    env = _env(name, over, N)
    assert env.sim.Omax == 64
    splits, overflow = _check_against_host(env, phase, seeds)
    assert splits > 0
    if over is WALLS10:
        assert overflow > 0
    sg = env.scene
    tight = 4 * ((sg.num_circles or 0) + (sg.num_walls or 0))
    splits, overflow = _check_against_host(_env(name, over, N, max_obst=tight), phase, seeds)
    assert splits == 0 and overflow > 0


def test_mask_leaves_other_episodes_alone():
    env = _env("env_ebcadrl.config", n=777)
    sim = env.sim
    a, b = np.arange(1000, 1777), np.arange(5000, 5777)
    env.reset_batch("test", b)
    full = {k: getattr(sim, k).clone() for k in ("obst", "obst_count")}
    env.reset_batch("test", a)
    before = {k: getattr(sim, k).clone() for k in ("obst", "obst_count")}
    mask = (torch.arange(777, device=DEV) % 3 == 1).to(torch.uint8)
    on = mask.bool()
    sg = env.scene
    cfg = S.replay_config(sg, "test", True, (sg.num_circles or 0) + (sg.num_walls or 0))
    pxy, pc, _ = sim.replay_scenes(cfg, torch.from_numpy(b.astype(np.uint32).view(np.int32)).to(DEV), mask=mask,
                                   poly_xy=env.poly_xy.clone(), poly_count=env.poly_count.clone())
    need = sim.build_obstacles(pxy, pc, mask=mask)
    assert (need[~on] == 0).all() and (need[on] == full["obst_count"][on]).all()
    for k in ("obst", "obst_count"):
        assert torch.equal(getattr(sim, k)[~on], before[k][~on]), k       # untouched, byte for byte
    assert torch.equal(sim.obst_count[on], full["obst_count"][on])
    # the masked episodes' records equal the full build's; slots past obst_count are left as they were (never read)
    used = torch.arange(sim.Omax, device=DEV)[None, :] < sim.obst_count[:, None]
    sel = used & on[:, None]
    assert torch.equal(sim.obst[sel], full["obst"][sel])


def test_build_obstacles_needs_the_key():
    env = BatchedEnv(read_config("env_ebcadrl.config"), None, 4, DEV)
    env.reset_batch("test", [1000, 1001, 1002, 1003])
    with pytest.raises(abi.EbcError, match="orca_obstacles"):
        env.sim.build_obstacles(env.poly_xy, env.poly_count)


def _oracle_copy(oracle, env):
    sim = env.sim
    r = BatchedSim(env.cfg, sim.N, sim.Hmax, sim.Smax, sim.Rmax, sim.A, device="cpu", backend=oracle, max_obst=sim.Omax)
    r.set_actions(sim.actions)
    r.load_episodes(0, *[getattr(sim, k).cpu().numpy() for k in STATE])
    return r


@pytest.mark.parametrize("name", ["env_ebcadrl.config", WALLS5])
@pytest.mark.parametrize("imitation", [False, True], ids=["decide", "robot_orca"])
def test_whole_loop_matches_oracle(oracle, name, imitation):
    """40 committed steps of 384 episodes: the GPU's chosen actions (value network argmax, or the IL robot's ORCA
    action) fed to an oracle sim holding the same state and obstacle records; everything bit-identical."""
    N = 384
    env = _env(name, n=N)
    sim = env.sim
    sim.set_actions(build_action_space(env.robot.v_pref))
    sim.set_weights(ob.load_weights("weights_sarl_baseline.npz"))
    env.reset_batch("test", np.arange(1000, 1000 + N))
    assert int(sim.obst_count.min()) > 0
    r = _oracle_copy(oracle, env)
    for t in range(40):
        if imitation:
            act = sim.robot_orca(0.15)
            ract = r.robot_orca(0.15)
            torch.cuda.synchronize()
            assert np.array_equal(act.cpu().numpy(), ract.numpy()), t
            sim.orca()
            r.orca()
        else:
            idx = sim.decide()
            r.orca()
        torch.cuda.synchronize()
        assert np.array_equal(sim.hum_nv.cpu().numpy(), r.hum_nv.numpy()), t
        if imitation:
            sim.step(action=act)
            r.step(action=act.cpu())
        else:
            sim.step(action_idx=idx)
            r.step(action_idx=idx.cpu())
        torch.cuda.synchronize()
        for k in ("hum_pv", "rob_pv", "rob_theta", "time", "reward", "done", "event"):
            assert np.array_equal(getattr(sim, k).cpu().numpy(), getattr(r, k).numpy()), (t, k)


def _wall_boxes(env):
    """Every episode's polygons as axis-aligned boxes (x0, y0, x1, y1) in metres; unused slots far away."""
    p = env.poly_xy.cpu().numpy()
    box = np.concatenate([p.min(2), p.max(2)], axis=2)
    box[np.arange(p.shape[1])[None, :] >= env.poly_count.cpu().numpy()[:, None]] = 1e6
    return box


def _clearance(sim, box):
    p = sim.hum_pv.cpu().numpy()[:, :, :2].astype(np.float64)
    r = sim.hum_gr.cpu().numpy()[:, :, 3]
    dx = np.maximum(np.maximum(box[:, None, :, 0] - p[:, :, None, 0], 0), p[:, :, None, 0] - box[:, None, :, 2])
    dy = np.maximum(np.maximum(box[:, None, :, 1] - p[:, :, None, 1], 0), p[:, :, None, 1] - box[:, None, :, 3])
    return (np.hypot(dx, dy) - r[:, :, None]).min(2)


@pytest.mark.parametrize("name", ["env_ebcadrl.config", WALLS5])
def test_humans_never_enter_walls(name):
    """Humans that start clear of every wall stay at least radius + 0.01 - 1e-4 from it for 100 steps with the key on
    (RVO2 keeps agents at their ORCA radius r + 0.01); with it off the same scenes have humans inside walls."""
    N = 512
    seeds = np.arange(1000, 1000 + N)
    worst = {}
    for key in ("true", "false"):
        env = BatchedEnv(read_config(name, {("sim", "orca_obstacles"): key}), None, N, DEV)
        sim = env.sim
        sim.set_actions(build_action_space(env.robot.v_pref))
        env.reset_batch("test", seeds)
        box = _wall_boxes(env)
        hc = sim.hum_count.cpu().numpy()
        real = np.arange(sim.Hmax)[None, :] < hc[:, None]
        c0 = _clearance(sim, box)
        clear = real & (c0 > 0.05)
        mn = c0.copy()
        zero = torch.zeros(N, dtype=torch.int32, device=DEV)
        for _ in range(100):
            sim.step(action_idx=zero, fused_orca=True)
            mn = np.minimum(mn, _clearance(sim, box))
        assert np.isfinite(sim.hum_pv.cpu().numpy()).all()
        worst[key] = mn[clear].min()
    print(name, worst)
    assert worst["true"] >= 0.01 - 1e-4, worst
    assert worst["false"] < -0.1, worst


def test_key_off_is_the_default_path():
    """No key and `orca_obstacles = false` are the same run, with no obstacle slots; the key on changes the crowd."""
    seeds = np.arange(1000, 1256)
    res = {}
    for label, over in (("absent", {}), ("false", {("sim", "orca_obstacles"): "false"}), ("true", ON)):
        env = BatchedEnv(read_config(WALLS5, over), None, len(seeds), DEV)
        sim = env.sim
        sim.set_actions(build_action_space(env.robot.v_pref))
        sim.set_weights(ob.load_weights("weights_sarl_baseline.npz"))
        assert sim.Omax == (64 if label == "true" else 0)
        st, _ = env.run_episodes("test", seeds, record_dmin=True)
        res[label] = st
    for k in ("event", "time", "steps", "cum_reward", "too_close", "min_dist_sum", "dist_to_goal", "dmin_trace"):
        assert np.array_equal(getattr(res["absent"], k), getattr(res["false"], k)), k
    a, b = res["absent"].dmin_trace, res["true"].dmin_trace
    assert a.shape != b.shape or not np.array_equal(a, b)


def _write_ini(tmp_path, name, over):
    cp = read_config(name, over)
    path = str(tmp_path / name)
    with open(path, "w") as f:
        cp.write(f)
    return path


def test_single_env_matches_batched(tmp_path):
    """env.reset(scene_number = s) with the key on: the N = 1 env's obstacle records are the batched episode's; the same
    actions give the same human states; onestep_lookahead returns what step then commits."""
    from simulator.utils.action import ActionXY
    from simulator.utils.test_utils import configure_env_policy_robot
    # square_crossing scenes: the host generator and the device replay agree bit for bit (circle_crossing's cos / sin
    # need not)
    path = _write_ini(tmp_path, "env_ebcadrl.config", ON)
    env, policy, robot = configure_env_policy_robot(path, os.path.join(ob.GOLDEN, "configs", "policy.config"),
                                                    os.path.join(ob.GOLDEN, "weights_sarl_baseline.npz"))
    seeds = [1000, 1003, 1007, 1011]
    benv = _env("env_ebcadrl.config", n=len(seeds))
    benv.reset_batch("test", seeds)
    actions = build_action_space(benv.robot.v_pref)
    benv.sim.set_actions(actions)
    rng = np.random.default_rng(0)
    picks = rng.integers(0, len(actions), (6, len(seeds))).astype(np.int32)
    traj = []
    for t in range(6):
        benv.sim.step(action_idx=torch.as_tensor(picks[t], device=DEV), fused_orca=True)
        traj.append(benv.sim.hum_pv.cpu().numpy().copy())
    for i, seed in enumerate(seeds):
        env.reset("test", scene_number=seed)
        n = env.native
        assert n.Omax == 64
        c = int(n.obst_count[0])
        assert c == int(benv.sim.obst_count[i]) > 0
        assert torch.equal(n.obst[0, :c], benv.sim.obst[i, :c]), seed
        H = int(n.hum_count[0])
        for t in range(6):
            a = ActionXY(*actions[picks[t, i]])
            _, la_reward, la_done, la_info = env.onestep_lookahead(a)
            _, _, reward, done, info = env.step(a)
            assert (la_reward, la_done, str(la_info)) == (reward, done, str(info)), (seed, t)
            assert np.array_equal(n.hum_pv[0, :H].cpu().numpy(), traj[t][i, :H]), (seed, t)


def test_cli_and_probes(tmp_path, capsys):
    """rl.test runs to the end on a walls INI with the key on and logs its usual summary; the value-only and map
    handles an env builds from the same config still bind."""
    from rl import test as rl_test
    path = _write_ini(tmp_path, WALLS5, ON)
    metrics = rl_test.main(["--env_config", path, "--policy_config", os.path.join(ob.GOLDEN, "configs", "policy.config"),
                            "--policy", "sarl", "--model_path", os.path.join(ob.GOLDEN, "weights_sarl_baseline.npz"),
                            "--start", "1000", "--end", "1016", "--batch", "8"])
    out = capsys.readouterr().out
    assert metrics is not None and "has success rate" in out and "collision rate adult" in out
    env = _env(WALLS5, n=8)
    tv = TargetValue(env)
    assert tv.sim.Omax == 0 and not tv.sim.cfg.orca_obstacles and env.cfg.orca_obstacles
    from simulator.utils.test_utils import configure_env_policy_robot
    for grid in ("false", "true"):
        ini = _write_ini(tmp_path, WALLS5, {**ON, ("map", "use_grid_map"): grid})
        e1, _, robot = configure_env_policy_robot(ini, os.path.join(ob.GOLDEN, "configs", "policy.config"),
                                                  os.path.join(ob.GOLDEN, "weights_sarl_baseline.npz"))
        e1.reset("test", scene_number=1000)
        m = e1.get_local_map(robot.get_full_state()) if grid == "true" else e1.get_local_map_angular(robot.get_full_state())
        assert np.isfinite(m).all()
