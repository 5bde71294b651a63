"""The simulation kernels (K1 ORCA, K3 lookahead, K2 committed step, robot ORCA, transform) at every entity count they
accept, against the oracle, plus a plain fp64 restatement of the collision and reward rule.  The GPU tests need a
B200 and are marked `gpu` one by one; the restatement test runs on the CPU.

These kernels pick their code from the shape of the batch, and each group of tests pins one such choice with the
shape in the test id:

- Entity-count sweep (`test_entity_count_sweep`, ids `H<Hmax>-S<Smax>[-vis]`): every Hmax from 1 to 64, the
  lookahead group boundaries with statics, and a visible robot up to 64 ORCA candidates.  K3 runs 8, 16 or 32 lanes
  per (episode, action) from n = Hmax + Smax; the number of episodes is odd, so with A = 81 the last warp of K3 is
  partly filled at G = 8 / 16 and, at odd Hmax, the last warp of K1 is half empty at 16 lanes per human.  At G = 32
  with Hmax > 32 a lane holds humans l and l + 32 (`n_ch = 2`), and the collision and type masks use their upper
  half; `build_rows` and `robot_orca` put statics on lanes >= 32.  ORCA velocities, lookahead and step outcomes are
  bit-exact against the oracle, the forced whole-warp K1 (`EBC_ORCA_GROUP=32`) equals the default, the fused
  `ebc_orca_step` equals K1 then K2, and every event class, maxNeighbors truncation and collisions or dangers at
  human index >= 32 are asserted to occur.
- ORCA configuration sweep (`test_orca_neighbor_config`, ids `nb<k>-H<Hmax>[-vis]`): K1 runs a half warp per human iff
  `Hmax + robot_visible <= 32 and orca_max_neighbors <= 16`.  maxNeighbors 0 / 1 / 10 / 16 / 17 / 31 / 32 and two
  neighbour ranges, GPU == oracle == forced whole warp.
- Hand-built collisions (`test_upper_mask_half_scenes`, ids `H<Hmax>`): single and double collisions at indices
  0 / 31 / 32 / 33 / 40 / 63, dmin frozen at the first collision across the mask halves, the priority chain between
  a collision and a discomfort of another type on the other half, type boundaries across index 32, and a human
  inside the robot in a padding slot.  GPU == oracle == restatement.
- Garbage past the counts (`test_garbage_past_counts`): NaN, +-inf, +-3e38, random type bytes and map-covering
  rectangles in the slots past hum_count / stat_count / rect_count change no output bit and are never written.
- The restatement (`restate`, CPU test `test_restatement_matches_oracle`): env.py:303-338 and reward.py:103-179 of the
  reference in numpy fp64, in the reference's operation order, held to the oracle on the hand-built scenes and on
  random states.  Above 24 humans there is no reference golden; this gives the kernels a reference that is not one
  of the two twins.
- Action counts other than 81 (`test_action_counts`), the explorer statistics at Hmax 1 / 33 / 64
  (`test_statistics_at_extreme_counts`) and the obstacle path with more than 64 ORCA lines
  (`test_obstacle_path_beyond_64_lines`).

Bars: holonomic robot bit-exact (ORCA velocities, events, done, rewards, dmin, dist_to_goal, states, time, robot
ORCA); rotated rows 2e-5 absolute (positions up to ~12 m, as test_random_batches); unicycle rewards 1e-12 (CUDA's and
glibc's cos / sin of a double may differ in the last bit).
"""
import numpy as np
import pytest
import torch

import oracle_backend as ob
from ebc.actions import build_action_space
from ebc.engine import BatchedSim
from test_gpu_parity import assert_same_bits, np_, pair, random_cfg

VIN_TOL = 2e-5
N_SWEEP = 301                 # odd: N * 81 is odd, and N * Hmax is odd at odd Hmax
STATE_KEYS = ("hum_pv", "hum_gr", "hum_type", "hum_count", "stat", "stat_count", "rect", "rect_count", "rob_pv",
              "rob_gr", "rob_theta", "time")
STEP_KEYS = ("reward", "done", "event", "dmin", "dist_to_goal", "hum_pv", "hum_nv", "rob_pv", "rob_theta", "time")


# ---- the fp64 restatement -------------------------------------------------------------------------------------------
def _seg_dist0(x1, y1, x2, y2):
    """simulator/utils/collisions.py:4-26 with (x3, y3) = (0, 0), element-wise, same operations and order."""
    px, py = x2 - x1, y2 - y1
    zero = (px == 0.0) & (py == 0.0)
    with np.errstate(invalid="ignore", divide="ignore"):
        u = ((0.0 - x1) * px + (0.0 - y1) * py) / (px * px + py * py)
    u = np.where(u > 1.0, 1.0, np.where(u < 0.0, 0.0, u))
    x, y = x1 + u * px, y1 + u * py
    far = np.sqrt((x - 0.0) * (x - 0.0) + (y - 0.0) * (y - 0.0))
    return np.where(zero, np.sqrt((0.0 - x1) * (0.0 - x1) + (0.0 - y1) * (0.0 - y1)), far)


def restate(cfg, st, actions):
    """env.py:303-338 (collisions: per type, list order, dmin frozen at the first collision; the occupancy-grid window
    as an integer AABB overlap with the zero-cell rectangles) and reward.py:103-179 (the priority chain) in fp64, for
    every (episode, action) of a state dict in the ebc_state layout.  Returns reward, done, event [N, A], dmin
    [N, A, 3] and the index of the first collision of each type [N, A, 3] (Hmax when none)."""
    hol = cfg.robot_kinematics == "holonomic"
    dt = cfg.time_step
    N, Hm = st["hum_type"].shape
    a0, a1 = actions[:, 0][None], actions[:, 1][None]                          # [1, A]
    rp = st["rob_pv"].astype(np.float64)
    rg = st["rob_gr"].astype(np.float64)
    rpx, rpy, rrad = rp[:, 0:1], rp[:, 1:2], rg[:, 3:4]                       # [N, 1]
    if hol:
        avx, avy = a0 + 0 * rpx, a1 + 0 * rpx
        end_x, end_y = rpx + a0 * dt, rpy + a1 * dt
    else:
        th = st["rob_theta"].astype(np.float64)[:, None] + a1
        avx, avy = a0 * np.cos(th), a0 * np.sin(th)
        end_x, end_y = rpx + np.cos(th) * a0 * dt, rpy + np.sin(th) * a0 * dt
    pv = st["hum_pv"].astype(np.float64)
    px = (pv[:, :, 0] - rpx)[:, None, :]                                       # [N, 1, H]
    py = (pv[:, :, 1] - rpy)[:, None, :]
    vx = pv[:, None, :, 2] - avx[:, :, None]                                   # [N, A, H]
    vy = pv[:, None, :, 3] - avy[:, :, None]
    ex, ey = px + vx * dt, py + vy * dt
    closest = _seg_dist0(px + 0 * ex, py + 0 * ey, ex, ey) - st["hum_gr"][:, :, 3].astype(np.float64)[:, None, :] \
        - rrad[:, :, None]
    live = np.arange(Hm)[None] < st["hum_count"][:, None]                      # [N, H]
    A = actions.shape[0]
    dmin = np.full((N, A, 3), np.inf)
    first = np.full((N, A, 3), Hm)
    for t in range(3):
        of_t = (live & (st["hum_type"] == t))[:, None, :]
        hit = of_t & (closest < 0.0)
        f = np.where(hit.any(2), hit.argmax(2), Hm)
        first[..., t] = f
        before = of_t & (np.arange(Hm)[None, None] < f[..., None])
        dmin[..., t] = np.where(before, closest, np.inf).min(2)
    coll = first < Hm
    # env.py:227-261: the robot's square window of the grid against the zero-cell rectangles
    ix = np.rint((end_x + cfg.map_size_m / 2.0) / cfg.map_resolution).astype(np.int64)
    iy = np.rint((end_y + cfg.map_size_m / 2.0) / cfg.map_resolution).astype(np.int64)
    sz = np.ceil(rrad / np.sqrt(2.0) / cfg.map_resolution).astype(np.int64)
    G = int(np.rint(cfg.map_size_m / cfg.map_resolution))
    sx, sy = ix - sz, iy - sz
    ex_, ey_ = np.minimum(sx + sz * 2, G), np.minimum(sy + sz * 2, G)
    sx, sy = np.maximum(sx, 0), np.maximum(sy, 0)
    rc = st["rect"].astype(np.int64)
    rlive = np.arange(rc.shape[1])[None] < st["rect_count"][:, None]
    over = ((sx[..., None] < rc[:, None, :, 2]) & (rc[:, None, :, 0] < ex_[..., None]) & (sy[..., None] < rc[:, None, :, 3])
            & (rc[:, None, :, 1] < ey_[..., None]) & rlive[:, None, :])
    coll_obst = (ex_ > sx) & (ey_ > sy) & over.any(2)
    # reward.py:103-179
    gdx, gdy = end_x - rg[:, 0:1], end_y - rg[:, 1:2]
    dist = np.sqrt(gdx * gdx + gdy * gdy)
    gt = st["time"].astype(np.float64)[:, None] + 0 * dist
    base = (1.0 - dist / cfg.max_goal_distance) if (cfg.new_reward and cfg.max_goal_distance is not None) else 0 * dist
    reward, done, event = np.zeros((N, A)), np.zeros((N, A), np.uint8), np.zeros((N, A), np.uint8)
    todo = np.ones((N, A), bool)

    def take(mask, r, d, ev):
        m = todo & mask
        reward[m], done[m], event[m] = r[m] if np.ndim(r) else r, d, ev
        todo[m] = False

    take(gt >= cfg.time_limit, base, 1, 7)
    take(coll[..., 2], base + cfg.collision_penalty_child, 1, 5)
    take(coll[..., 1], base + cfg.collision_penalty_bicycle, 1, 4)
    take(coll[..., 0], base + cfg.collision_penalty_adult, 1, 3)
    take(coll_obst, base + cfg.collision_penalty_obstacle, 1, 6)
    if cfg.new_reward:
        tr = np.where(gt < cfg.time_good, 1.0, np.where(gt <= cfg.time_max, (cfg.time_max - gt) / (cfg.time_max - cfg.time_good), 0.0))
        take(dist < rrad, base + tr, 1, 2)
    else:
        take(dist < rrad, base + cfg.success_reward, 1, 2)
    for t, name in ((2, "child"), (1, "bicycle"), (0, "adult")):
        dd, fac = getattr(cfg, "discomfort_dist_" + name), getattr(cfg, "discomfort_penalty_factor_" + name)
        take(dmin[..., t] < dd, (dmin[..., t] - dd) * fac * dt, 0, 1)
    if not hol and cfg.rotation_penalty_factor != 0.0:
        take(np.abs(a1 + 0 * dist) > 0.0, np.abs(a1 + 0 * dist) * cfg.rotation_penalty_factor, 0, 0)
    take(todo, 0 * dist, 0, 0)
    return reward, done, event, dmin, first


# ---- batches --------------------------------------------------------------------------------------------------------
def sweep_batch(N, H, S, R, seed):
    """A dense ragged batch with zero padding.  The area grows with Hmax so that the density stays about that of
    test_random_batches' dense 24-human case: maxNeighbors truncation and LP3 are live at every size.  Episode 0 has
    one human and no statics, episode 1 is full.  For Hmax > 32, episodes 2..4 have 31, 32 and 33 humans, and every
    third episode from 5 on is full."""
    rng = np.random.default_rng(seed)
    span = 3.0 * max(1.0, np.sqrt(H / 24.0))
    cnt = rng.integers(1, H + 1, N).astype(np.int32)
    cnt[0], cnt[1] = 1, H
    if H > 32:
        cnt[2:5] = (31, 32, 33)
        cnt[5::3] = H           # a third of the batch fills the upper half of the masks
    scnt = rng.integers(0, S + 1, N).astype(np.int32)
    scnt[0], scnt[1] = 0, S
    live = np.arange(H)[None] < cnt[:, None]
    d = {"hum_count": cnt, "stat_count": scnt}
    d["hum_pv"] = np.concatenate([rng.uniform(-span, span, (N, H, 2)), rng.uniform(-1, 1, (N, H, 2))], 2).astype(np.float32)
    d["hum_gr"] = np.concatenate([rng.uniform(-span, span, (N, H, 2)), rng.uniform(0.3, 1.5, (N, H, 1)),
                                  rng.uniform(0.1, 0.5, (N, H, 1))], 2).astype(np.float32)
    d["hum_gr"][::7, 0, :2] = d["hum_pv"][::7, 0, :2] + 0.3
    ty = np.sort(rng.integers(0, 3, (N, H)), axis=1)
    d["hum_type"] = np.where(live, ty, 0).astype(np.uint8)
    d["hum_pv"][~live] = 0
    d["hum_gr"][~live] = 0
    Sx = max(S, 1)
    d["stat"] = np.concatenate([rng.uniform(-span, span, (N, Sx, 2)), rng.uniform(0.3, 0.8, (N, Sx, 1)),
                                np.zeros((N, Sx, 1))], 2).astype(np.float32)
    d["stat"][np.arange(Sx)[None] >= scnt[:, None]] = 0
    d["rect_count"] = rng.integers(0, R + 1, N).astype(np.int32)
    d["rect_count"][1] = R
    x0 = rng.integers(0, 80, (N, max(R, 1), 2))
    wh = rng.integers(1, 31, (N, max(R, 1), 2))
    d["rect"] = np.concatenate([x0, np.minimum(x0 + wh, 90)], 2).astype(np.int16)
    d["rect"][np.arange(max(R, 1))[None] >= d["rect_count"][:, None]] = 0
    rs = min(span, 4.0)
    d["rob_pv"] = np.concatenate([rng.uniform(-rs, rs, (N, 2)), rng.uniform(-1, 1, (N, 2))], 1).astype(np.float32)
    d["rob_gr"] = np.concatenate([rng.uniform(-4, 4, (N, 2)), rng.uniform(0.5, 1.0, (N, 1)),
                                  rng.uniform(0.2, 0.4, (N, 1))], 1).astype(np.float32)
    d["rob_gr"][::11, :2] = d["rob_pv"][::11, :2] + 0.05          # already at the goal
    d["rob_theta"] = rng.uniform(0, 2 * np.pi, N).astype(np.float32)
    d["time"] = (rng.integers(0, 110, N) * 0.25).astype(np.float64)   # some past the time limit
    return d


def truncated(cfg, st):
    """Does some live human have more ORCA candidates in range than maxNeighbors?"""
    pv, cnt = st["hum_pv"][:, :, :2].astype(np.float32), st["hum_count"]
    H = pv.shape[1]
    d = ((pv[:, :, None] - pv[:, None]) ** 2).sum(-1)
    live = np.arange(H)[None] < cnt[:, None]
    ok = live[:, :, None] & live[:, None] & ~np.eye(H, dtype=bool)[None] & (d < np.float32(cfg.orca_neighbor_dist) ** 2)
    n = ok.sum(2)
    if cfg.robot_visible:
        dr = ((pv - st["rob_pv"][:, None, :2]) ** 2).sum(-1)
        n = n + (dr < np.float32(cfg.orca_neighbor_dist) ** 2)
    return bool((live & (n > cfg.orca_max_neighbors)).any())


def _load(sims, batch):
    for s in sims:
        s.load_episodes(0, **batch)


def _orca_both_groups(g, monkeypatch):
    """K1 with the default group choice, then with the whole warp forced: bit-identical."""
    g.orca()
    nv = g.hum_nv.clone()
    monkeypatch.setenv("EBC_ORCA_GROUP", "32")
    g.orca()
    torch.cuda.synchronize()
    monkeypatch.delenv("EBC_ORCA_GROUP")
    assert_same_bits(g.hum_nv, nv, "ORCA velocities, forced whole warp vs default")


def _compare_lookahead(g, r, st, exact=True):
    assert_same_bits(g.la_event, r.la_event, "lookahead events")
    assert_same_bits(g.la_done, r.la_done, "lookahead done")
    if exact:
        assert_same_bits(g.la_reward, r.la_reward, "lookahead rewards")
    else:
        np.testing.assert_allclose(np_(g.la_reward), np_(r.la_reward), rtol=0, atol=1e-12)
    gv = np_(g.vin)
    np.testing.assert_allclose(gv, np_(r.vin), rtol=0, atol=VIN_TOL)
    rows = st["hum_count"] + st["stat_count"]
    pad = np.arange(g.n)[None] >= rows[:, None]                    # [N, n]
    assert not gv[np.broadcast_to(pad[:, None], gv.shape[:3])].any(), "rows past an episode's count must be zero"


def _state(sim):
    return {k: np_(getattr(sim, k)).copy() for k in STATE_KEYS}


# every event class over the whole sweep
SEEN_EVENTS = set()

SWEEP = ([(H, 0, False) for H in range(1, 65)]
         + [(1, 7, False), (1, 8, False), (8, 8, False), (9, 8, False), (1, 15, False), (1, 16, False), (16, 16, False),
            (17, 15, False), (32, 1, False), (1, 63, False), (32, 32, False), (33, 31, False)]
         + [(H, 0, True) for H in (15, 16, 31, 32, 33, 63)])


def _sid(s):
    return "H%d-S%d%s" % (s[0], s[1], "-vis" if s[2] else "")


@pytest.mark.gpu
@pytest.mark.parametrize("H,S,visible", SWEEP, ids=[_sid(s) for s in SWEEP])
def test_entity_count_sweep(oracle, monkeypatch, H, S, visible):
    N, R = N_SWEEP, 3
    cfg = random_cfg("holonomic", typed=True, visible=visible)
    actions = build_action_space(0.8)
    g, r = pair(cfg, N, H, S, R, oracle, actions=actions)
    batch = sweep_batch(N, H, S, R, seed=1000 + 100 * H + S + visible)
    _load((g, r), batch)
    _orca_both_groups(g, monkeypatch)
    r.orca()
    assert_same_bits(g.hum_nv, r.hum_nv, "ORCA velocities")
    if H + visible - 1 > cfg.orca_max_neighbors:
        assert truncated(cfg, batch), "no human has more candidates than maxNeighbors"
    for s in (g, r):
        s.lookahead()
    torch.cuda.synchronize()
    _compare_lookahead(g, r, batch)
    # the independent restatement: events exact, rewards bit-exact (holonomic)
    rw, dn, ev, _, first = restate(cfg, batch, actions)
    assert np.array_equal(np_(g.la_event), ev), "lookahead events vs restatement"
    assert np.array_equal(np_(g.la_reward), rw), "lookahead rewards vs restatement"
    seen = set(np.unique(ev).tolist())
    SEEN_EVENTS.update(seen)
    assert {1, 7} <= seen and seen & {3, 4, 5, 6}, seen
    if H > 32:
        coll_hi = ((first >= 32) & (first < H)).any(2) & np.isin(ev, (3, 4, 5))
        assert coll_hi.any(), "no lookahead collision at a human index >= 32"
    # a committed step with every 5th episode inactive, then a second decision from the stepped state
    rng = np.random.default_rng(H)
    idx = torch.as_tensor(rng.integers(0, 81, N), dtype=torch.int32)
    active = torch.as_tensor((np.arange(N) % 5 != 0).astype(np.uint8))
    before = _state(g)
    g.step(action_idx=idx.cuda(), active=active.cuda())
    r.step(action_idx=idx, active=active)
    torch.cuda.synchronize()
    for k in STEP_KEYS:
        assert_same_bits(getattr(g, k), getattr(r, k), "step " + k)
    after = _state(g)
    for k in ("hum_pv", "rob_pv", "time"):
        assert np.array_equal(after[k][::5], before[k][::5]), "inactive episodes must not move: " + k
    for s in (g, r):
        s.orca()
        s.lookahead()
    torch.cuda.synchronize()
    assert_same_bits(g.hum_nv, r.hum_nv, "ORCA velocities, second decision")
    _compare_lookahead(g, r, batch)
    ga, ra = g.robot_orca(0.15), r.robot_orca(0.15)
    torch.cuda.synchronize()
    assert_same_bits(ga, ra, "robot ORCA action")
    np.testing.assert_allclose(np_(g.transform()), np_(r.transform()), rtol=0, atol=VIN_TOL)
    # ebc_orca_step (K1 for the active episodes, then K2) == K1 then K2; inactive episodes keep hum_pv AND hum_nv
    f = BatchedSim(cfg, N, H, S, R, 81, device="cuda:0")
    f.set_actions(actions)
    f.load_episodes(0, **batch)
    g.load_episodes(0, **batch)
    nv0 = torch.as_tensor(np.random.default_rng(7).uniform(-1, 1, (N, H, 2)).astype(np.float32), device="cuda:0")
    f.hum_nv.copy_(nv0)
    g.orca()
    g.step(action_idx=idx.cuda(), active=active.cuda())
    f.step(action_idx=idx.cuda(), active=active.cuda(), fused_orca=True)
    torch.cuda.synchronize()
    act = np_(active).astype(bool)
    live = act[:, None] & (np.arange(H)[None] < batch["hum_count"][:, None])     # slots past the count: untouched
    for k in ("hum_pv", "hum_nv"):
        assert np.array_equal(np_(getattr(f, k))[live], np_(getattr(g, k))[live]), "fused step " + k
    for k in ("rob_pv", "time"):
        assert np.array_equal(np_(getattr(f, k))[act], np_(getattr(g, k))[act]), "fused step " + k
    for k in ("reward", "event", "done", "dmin", "dist_to_goal"):
        assert np.array_equal(np_(getattr(f, k))[act].view(np.uint8), np_(getattr(g, k))[act].view(np.uint8)), k
    assert np.array_equal(np_(f.hum_pv)[~act], batch["hum_pv"][~act]), "inactive hum_pv"
    assert np.array_equal(np_(f.hum_nv)[~act], np_(nv0)[~act]), "inactive hum_nv"


@pytest.mark.gpu
def test_entity_count_sweep_saw_every_event_class():
    if len(SEEN_EVENTS) == 0:
        pytest.skip("runs after test_entity_count_sweep in the same session")
    assert SEEN_EVENTS == set(range(8)), SEEN_EVENTS


# ---- K1 group switch ------------------------------------------------------------------------------------------------
NEIGHBORS = (0, 1, 10, 16, 17, 31, 32)
ORCA_CFGS = [(nb, H, vis) for nb in NEIGHBORS for vis in (False, True)
             for H in ((16, 17, 32, 33) + ((63,) if vis else (64,)))]     # Hmax + robot_visible <= 64


def half_warp_k1(H, visible, nb):
    """The K1 group rule (orca_group in ebc_sim.cu): 16 lanes per human iff every human has at most 32 candidates
    (Hmax - 1 others, plus the visible robot, on two slots per lane) and at most 16 ORCA lines."""
    return H + int(visible) <= 32 and nb <= 16


def test_orca_config_sweep_runs_both_group_widths():
    rule = [half_warp_k1(H, vis, nb) for nb, H, vis in ORCA_CFGS]
    assert any(rule) and not all(rule)


@pytest.mark.gpu
@pytest.mark.parametrize("nb,H,visible", ORCA_CFGS, ids=["nb%d-H%d%s" % (nb, H, "-vis" if v else "") for nb, H, v in ORCA_CFGS])
def test_orca_neighbor_config(oracle, monkeypatch, nb, H, visible):
    """The 16-lane kernel runs iff half_warp_k1(H, visible, nb): here nb <= 16 at H <= 31 (or 32 without the robot)."""
    N, S, R = 129, 0, 0
    actions = build_action_space(0.8)
    batch = sweep_batch(N, H, S, R, seed=50 * nb + H + visible)
    idx = torch.as_tensor(np.random.default_rng(nb).integers(0, 81, N), dtype=torch.int32)
    for rng_m in (10.0, 1.5):         # a short range: the in-range set, not the slot count, picks the candidates
        cfg = random_cfg("holonomic", typed=True, visible=visible)
        cfg.orca_max_neighbors, cfg.orca_neighbor_dist = nb, rng_m
        g, r = pair(cfg, N, H, S, R, oracle, actions=actions)
        w = BatchedSim(cfg, N, H, S, R, 81, device="cuda:0")
        w.set_actions(actions)
        _load((g, r, w), batch)
        for t in range(3):
            g.step(action_idx=idx.cuda(), fused_orca=True)
            r.step(action_idx=idx, fused_orca=True)
            monkeypatch.setenv("EBC_ORCA_GROUP", "32")
            w.step(action_idx=idx.cuda(), fused_orca=True)
            monkeypatch.delenv("EBC_ORCA_GROUP")
            torch.cuda.synchronize()
            for k in ("hum_nv", "hum_pv", "event", "reward", "dmin"):
                assert_same_bits(getattr(g, k), getattr(r, k), "%s, step %d, range %g" % (k, t, rng_m))
                assert_same_bits(getattr(g, k), getattr(w, k), "%s vs whole warp, step %d, range %g" % (k, t, rng_m))
        if nb == 0:     # no neighbour: every human takes its clamped preferred velocity
            assert np.abs(np_(g.hum_nv)).sum() > 0


# ---- hand-built collisions across the mask halves -------------------------------------------------------------------
def scene_cfg():
    c = random_cfg("holonomic", typed=True)
    c.time_limit = 100.0
    c.discomfort_penalty_factor_adult = 0.5
    return c


# centre distances to the robot.  Radii sum to 0.6 and the robot moves at most 0.2 m: COLLIDE collides whatever the
# action, CLOSE never collides but comes within every discomfort distance for the actions towards it, NEAR neither.
COLLIDE, CLOSE, NEAR = 0.4, 0.85, 1.1


def _far(k, H):
    a = 2 * np.pi * k / 64.0
    rad = 6.0 + 2.0 * (k % 3)
    return rad * np.cos(a), rad * np.sin(a)


def hand_scenes(H):
    """Deterministic episodes at Hmax = H.  Robot at the origin (radius 0.3, still, goal 8 m away), humans of
    radius 0.3 at least 5 m away except the placed ones.  Returns (batch, notes) with notes[e] = what episode e pins."""
    eps, notes = [], []

    def episode(types, placed, count=None, note=""):
        pv = np.zeros((H, 4), np.float32)
        gr = np.zeros((H, 4), np.float32)
        for k in range(H):
            pv[k, :2] = _far(k, H)
            gr[k] = (pv[k, 0], pv[k, 1], 1.0, 0.3)
        for k, dist in placed.items():
            a = 0.37 * k
            pv[k, :2] = (dist * np.cos(a), dist * np.sin(a))
            gr[k, :2] = pv[k, :2]
        c = H if count is None else count
        eps.append((pv, gr, np.asarray(types, np.uint8), c))
        notes.append(note)

    for t in range(3):
        for k in (0, 31, 32, 33, 40, 63):
            if k < H:
                episode([t] * H, {k: COLLIDE}, note="single collision type %d at %d" % (t, k))
    for t in range(3):
        for i in (0, 31):
            for j in (32, H - 1):
                if i < j < H and j > 31:
                    placed = {i: COLLIDE, j: COLLIDE}
                    if j - i > 1:
                        placed[(i + j) // 2 if (i + j) // 2 != i else i + 1] = CLOSE
                    if i > 0:
                        placed[i - 1] = NEAR
                    episode([t] * H, placed, note="two collisions type %d at %d, %d" % (t, i, j))
    lo = min(31, H - 2)
    ty = [0] * (lo + 1) + [2] * (H - lo - 1)
    episode(ty, {5: CLOSE, H - 1: COLLIDE}, note="adult discomfort low, child collision high")
    episode(ty, {5: COLLIDE, H - 1: CLOSE}, note="adult collision low, child discomfort high")
    ty = [1] * (lo + 1) + [2] * (H - lo - 1)
    episode(ty, {3: CLOSE, H - 1: CLOSE}, note="bicycle and child discomfort")
    episode(ty, {3: COLLIDE, H - 1: COLLIDE}, note="bicycle and child collisions")
    # type boundaries across index 32 (adults, bicycles, children; sorted)
    b0, b1 = (36, 50) if H == 64 else ((31, 34) if H == 40 else (30, 32))
    ty = [0] * b0 + [1] * (b1 - b0) + [2] * (H - b1)
    episode(ty, {b0 - 1: CLOSE, b0: COLLIDE, b1: NEAR}, note="bicycle collision at the first bicycle")
    episode(ty, {b0 - 1: COLLIDE, b1 - 1: CLOSE, H - 1: NEAR}, note="adult collision at the last adult")
    episode(ty, {b1 - 1: CLOSE, b1: CLOSE}, note="bicycle / child discomfort at the boundary")
    # a human inside the robot in the first padding slot must not count
    for c in (32, H - 1):
        if c < H:
            episode([0] * H, {c: 0.0, 2: NEAR}, count=c, note="human inside the robot in padding slot %d" % c)
    N = len(eps)
    b = {"hum_pv": np.stack([e[0] for e in eps]), "hum_gr": np.stack([e[1] for e in eps]),
         "hum_type": np.stack([e[2] for e in eps]), "hum_count": np.array([e[3] for e in eps], np.int32),
         "stat": np.zeros((N, 1, 4), np.float32), "stat_count": np.zeros(N, np.int32),
         "rect": np.zeros((N, 1, 4), np.int16), "rect_count": np.zeros(N, np.int32),
         "rob_pv": np.zeros((N, 4), np.float32),
         "rob_gr": np.tile(np.array([0.0, 8.0, 1.0, 0.3], np.float32), (N, 1)),
         "rob_theta": np.full(N, np.pi / 2, np.float32), "time": np.zeros(N)}
    return b, notes


HAND_H = (33, 40, 64)


@pytest.mark.gpu
@pytest.mark.parametrize("H", HAND_H, ids=["H%d" % h for h in HAND_H])
def test_upper_mask_half_scenes(oracle, H):
    cfg = scene_cfg()
    actions = build_action_space(0.8)
    batch, notes = hand_scenes(H)
    N = len(notes)
    g, r = pair(cfg, N, H, 0, 0, oracle, actions=actions)
    _load((g, r), batch)
    for s in (g, r):
        s.orca()
        s.lookahead()
    torch.cuda.synchronize()
    assert_same_bits(g.hum_nv, r.hum_nv, "ORCA velocities")
    _compare_lookahead(g, r, batch)
    rw, dn, ev, dmin, first = restate(cfg, batch, actions)
    assert np.array_equal(np_(g.la_event), ev) and np.array_equal(np_(g.la_done), dn)
    assert np.array_equal(np_(g.la_reward), rw)
    _check_scene_notes(batch, notes, ev, dmin, first)
    idx = np.random.default_rng(H).integers(0, 81, N).astype(np.int32)
    g.step(action_idx=torch.as_tensor(idx, device="cuda:0"))
    r.step(action_idx=torch.as_tensor(idx))
    torch.cuda.synchronize()
    for k in STEP_KEYS:
        assert_same_bits(getattr(g, k), getattr(r, k), "step " + k)
    pick = (np.arange(N), idx)
    assert np.array_equal(np_(g.dmin), dmin[pick]), "step dmin vs restatement"
    assert np.array_equal(np_(g.event), ev[pick]) and np.array_equal(np_(g.reward), rw[pick])


def _check_scene_notes(batch, notes, ev, dmin, first):
    """What each hand-built episode must show, for every action."""
    for e, note in enumerate(notes):
        if note.startswith("single collision"):
            t, k = int(note.split()[3]), int(note.split()[-1])
            assert (first[e, :, t] == k).all() and (ev[e] == 3 + t).all(), note
        elif note.startswith("two collisions"):
            t = int(note.split()[3])
            i = int(note.split()[-2].rstrip(","))
            assert (first[e, :, t] == i).all() and (ev[e] == 3 + t).all(), note
            if i == 0:
                assert np.isinf(dmin[e, :, t]).all(), note         # nobody before the first collision
            else:                                                  # the NEAR human before i, not the CLOSE one after
                assert (dmin[e, :, t] >= NEAR - 0.8).all(), note
        elif note.startswith("human inside the robot"):
            assert (first[e] == batch["hum_type"].shape[1]).all() and not np.isin(ev[e], (3, 4, 5)).any(), note
        elif note == "adult discomfort low, child collision high":
            assert (ev[e] == 5).all(), note
        elif note == "adult collision low, child discomfort high":
            assert (ev[e] == 3).all(), note
        elif note == "bicycle and child collisions":
            assert (ev[e] == 5).all(), note
        elif note == "bicycle and child discomfort":
            assert (ev[e] == 1).any(), note


def test_restatement_matches_oracle(oracle):
    """The numpy restatement against the oracle, on the hand-built scenes and on random states of every size, both
    kinematics.  Events and done exact; rewards and dmin bit-exact for the holonomic robot, 1e-12 for the unicycle."""
    for H in HAND_H:
        cfg = scene_cfg()
        actions = build_action_space(0.8)
        batch, notes = hand_scenes(H)
        N = len(notes)
        r = BatchedSim(cfg, N, H, 0, 0, 81, device="cpu", backend=oracle)
        r.set_actions(actions)
        r.load_episodes(0, **batch)
        r.lookahead(build_inputs=False)
        rw, dn, ev, dmin, first = restate(cfg, batch, actions)
        assert np.array_equal(r.la_event.numpy(), ev) and np.array_equal(r.la_done.numpy(), dn)
        assert np.array_equal(r.la_reward.numpy(), rw)
        _check_scene_notes(batch, notes, ev, dmin, first)
        idx = np.random.default_rng(H).integers(0, 81, N).astype(np.int32)
        r.step(action_idx=torch.as_tensor(idx))
        assert np.array_equal(r.dmin.numpy(), dmin[np.arange(N), idx])
    seen = set()
    for kin in ("holonomic", "unicycle"):
        for H, S, R in ((1, 0, 3), (10, 6, 3), (24, 0, 3), (33, 31, 3), (64, 0, 3)):
            cfg = random_cfg(kin, typed=True)
            actions = build_action_space(0.8, kin)
            batch = sweep_batch(97, H, S, R, seed=5 * H + S + (kin == "unicycle"))
            r = BatchedSim(cfg, 97, H, S, R, 81, device="cpu", backend=oracle)
            r.set_actions(actions)
            r.load_episodes(0, **batch)
            r.orca()
            r.lookahead(build_inputs=False)
            rw, dn, ev, dmin, _ = restate(cfg, batch, actions)
            assert np.array_equal(r.la_event.numpy(), ev), (kin, H)
            assert np.array_equal(r.la_done.numpy(), dn), (kin, H)
            if kin == "holonomic":
                assert np.array_equal(r.la_reward.numpy(), rw), (kin, H)
            else:
                np.testing.assert_allclose(r.la_reward.numpy(), rw, rtol=0, atol=1e-12)
            idx = np.random.default_rng(H).integers(0, 81, 97).astype(np.int32)
            r.step(action_idx=torch.as_tensor(idx))
            got, want = r.dmin.numpy(), dmin[np.arange(97), idx]
            assert np.array_equal(np.isinf(got), np.isinf(want))
            np.testing.assert_allclose(got[np.isfinite(got)], want[np.isfinite(want)], rtol=0,
                                       atol=0 if kin == "holonomic" else 1e-12)
            seen |= set(np.unique(ev).tolist())
    assert seen == set(range(8)), seen


# ---- garbage past the counts ----------------------------------------------------------------------------------------
GARBAGE_SHAPES = [(1, 0, False), (5, 3, False), (9, 8, False), (17, 15, False), (31, 0, True), (33, 31, False),
                  (32, 32, False), (63, 0, True), (64, 0, False)]


def dirty(batch, seed):
    """The same episodes with every slot past the counts filled with values no kernel may read."""
    rng = np.random.default_rng(seed)
    b = {k: v.copy() for k, v in batch.items()}
    N, H = b["hum_type"].shape
    specials = np.array([np.nan, np.inf, -np.inf, 3e38, -3e38], np.float32)

    def junk(shape):
        return specials[rng.integers(0, len(specials), shape)]

    hpad = np.arange(H)[None] >= b["hum_count"][:, None]
    for k in ("hum_pv", "hum_gr"):
        b[k][hpad] = junk(b[k][hpad].shape)
    b["hum_type"][hpad] = rng.integers(0, 256, hpad.sum()).astype(np.uint8)
    first_pad = np.nonzero(hpad.any(1))[0]
    col = b["hum_count"][first_pad]
    b["hum_pv"][first_pad, col] = np.concatenate([b["rob_pv"][first_pad, :2], np.zeros((len(first_pad), 2), np.float32)], 1)
    b["hum_gr"][first_pad, col] = np.array([0, 0, 1, 0.5], np.float32)
    b["hum_type"][first_pad, col] = 0
    S = b["stat"].shape[1]
    spad = np.arange(S)[None] >= b["stat_count"][:, None]
    b["stat"][spad] = junk(b["stat"][spad].shape)
    R = b["rect"].shape[1]
    rpad = np.arange(R)[None] >= b["rect_count"][:, None]
    b["rect"][rpad] = np.array([-32768, -32768, 32767, 32767], np.int16)      # the whole map
    nv = np.zeros((N, H, 2), np.float32)
    nv[hpad] = junk(nv[hpad].shape)
    return b, nv, (hpad, spad, rpad)


@pytest.mark.gpu
@pytest.mark.parametrize("H,S,visible", GARBAGE_SHAPES, ids=[_sid(s) for s in GARBAGE_SHAPES])
def test_garbage_past_counts(H, S, visible):
    N, R = 151, 3
    cfg = random_cfg("holonomic", typed=True, visible=visible)
    actions = build_action_space(0.8)
    w = ob.load_weights("weights_ebcadrl.npz")
    clean = sweep_batch(N, H, S, R, seed=4000 + H + S)
    garbage, nv_junk, (hpad, spad, rpad) = dirty(clean, 5)
    out = []
    for b, nv in ((clean, np.zeros_like(nv_junk)), (garbage, nv_junk)):
        g = BatchedSim(cfg, N, H, S, R, 81, device="cuda:0")
        g.set_actions(actions)
        g.set_weights(w)
        g.enable_attention()
        g.load_episodes(0, **b)
        g.hum_nv.copy_(torch.as_tensor(nv))
        res = {}
        g.orca()
        res["orca"] = g.hum_nv.clone()
        g.lookahead()
        res.update(vin=g.vin.clone(), la_reward=g.la_reward.clone(), la_event=g.la_event.clone(),
                   la_done=g.la_done.clone())
        res["argmax"] = g.decide(fused=True).clone()
        res.update(values=g.values.clone(), attention=g.attention.clone(), action_values=g.action_values.clone(),
                   fused_la_reward=g.la_reward.clone(), nan_flag=g.nan_flag.clone())
        res["robot_orca"] = g.robot_orca(0.15)
        res["transform"] = g.transform()
        res["grid"] = g.local_map_grid(3.0)
        g.step(action_idx=g.argmax)
        for k in STEP_KEYS:
            res["step_" + k] = getattr(g, k).clone()
        res["transform_after"] = g.transform()
        torch.cuda.synchronize()
        res = {k: np_(v) for k, v in res.items()}
        res["state"] = _state(g)
        res["state"]["hum_nv"] = np_(g.hum_nv).copy()
        out.append(res)
    a, b = out
    for k in a:
        if k == "state":
            continue
        if k in ("orca", "step_hum_nv", "step_hum_pv"):    # per-human state: the live slots here, the padding below
            a[k], b[k] = a[k][~hpad], b[k][~hpad]
        assert np.array_equal(np.ascontiguousarray(a[k]).view(np.uint8), np.ascontiguousarray(b[k]).view(np.uint8)), k
    # the bytes past the counts come out as they went in
    st = b["state"]
    for k in ("hum_pv", "hum_gr"):
        assert np.array_equal(st[k][hpad].view(np.uint8), garbage[k][hpad].view(np.uint8)), k
    assert np.array_equal(st["hum_type"][hpad], garbage["hum_type"][hpad])
    assert np.array_equal(st["hum_nv"][hpad].view(np.uint8), nv_junk[hpad].view(np.uint8)), "hum_nv"
    if S:
        assert np.array_equal(st["stat"][spad].view(np.uint8), garbage["stat"][spad].view(np.uint8)), "stat"
    assert np.array_equal(st["rect"][rpad], garbage["rect"][rpad]), "rect"
    assert (a["nan_flag"] == 0).all()


# ---- action counts, statistics, obstacle path -----------------------------------------------------------------------
ACTION_CASES = [(A, H, S) for A in (1, 2, 3, 5, 256) for H, S in ((5, 3), (10, 6), (40, 0))]


@pytest.mark.gpu
@pytest.mark.parametrize("A,H,S", ACTION_CASES, ids=["A%d-H%d-S%d" % c for c in ACTION_CASES])
def test_action_counts(oracle, A, H, S):
    """K3 and K5 at A != 81, with an odd N: the last warp of K3 is partly filled at every A > 1 for G = 8 / 16."""
    N, R = 203, 3
    cfg = random_cfg("holonomic", typed=True)
    rng = np.random.default_rng(A * 7 + H)
    table = np.concatenate([np.zeros((1, 2)), rng.uniform(-0.8, 0.8, (A - 1, 2))], 0)
    g, r = pair(cfg, N, H, S, R, oracle, A=A, actions=table)
    batch = sweep_batch(N, H, S, R, seed=A + H)
    _load((g, r), batch)
    for s in (g, r):
        s.orca()
        s.lookahead()
    torch.cuda.synchronize()
    _compare_lookahead(g, r, batch)
    vals = torch.as_tensor(rng.normal(0, 1, (N, A)).astype(np.float32))
    g.values.copy_(vals)
    r.values.copy_(vals)
    ga, ra = g.select(), r.select()
    torch.cuda.synchronize()
    assert_same_bits(ga, ra, "argmax")
    # gamma^(dt v_pref): CUDA's and glibc's pow may differ in the last bit
    np.testing.assert_allclose(np_(g.action_values), np_(r.action_values), rtol=1e-15, atol=1e-15)
    assert_same_bits(g.nan_flag, r.nan_flag, "nan flag")


@pytest.mark.gpu
@pytest.mark.parametrize("H", (1, 33, 64), ids=["H%d" % h for h in (1, 33, 64)])
def test_statistics_at_extreme_counts(oracle, H):
    """ebc_bind_stats rollouts until every episode ends, by the rules of test_device_statistics_match_oracle."""
    N, S, R = 257, 0, 3
    cfg = random_cfg()
    cfg.time_limit = 8.0
    actions = build_action_space(0.8)
    batch = sweep_batch(N, H, S, R, seed=21 + H)
    batch["time"] = np.zeros(N)
    sims = []
    for dev, be in (("cuda:0", None), ("cpu", oracle)):
        s = BatchedSim(cfg, N, H, S, R, 81, device=dev, backend=be)
        s.set_actions(actions)
        s.load_episodes(0, **batch)
        s.bind_stats()
        sims.append(s)
    g, r = sims
    rng = np.random.default_rng(5)
    for t in range(40):
        idx = torch.as_tensor(rng.integers(0, 81, N), dtype=torch.int32)
        for s, ix in ((g, idx.cuda()), (r, idx)):
            if t % 2:
                s.step(action_idx=ix, fused_orca=True)
            else:
                s.orca()
                s.step(action_idx=ix)
    torch.cuda.synchronize()
    for k in ("alive", "final_event", "steps", "too_close", "alive_count", "min_dist_sum"):
        a, b = np_(g.stats[k]), np_(r.stats[k])
        assert np.array_equal(a, b), (k, a[:8], b[:8])
    for k in ("cum_reward", "discount"):
        np.testing.assert_allclose(np_(g.stats[k]), np_(r.stats[k]), rtol=1e-13, atol=1e-13)
    st = g.stats
    assert int(st["alive_count"]) == int(st["alive"].sum()) == 0
    ev = np_(st["final_event"])
    assert (ev != 0).all() and (ev != 1).all() and 7 in set(ev.tolist())
    assert (np_(st["steps"]) <= 33).all() and np_(st["steps"]).min() >= 1
    if H > 1:
        assert np_(st["too_close"]).sum() > 0


def ring_scene(N, H, seed):
    """Humans inside a clockwise 62-gon of radius 3.5 m (RVO2 treats a clockwise polygon as a wall around the agents):
    every edge faces every human and lies within the obstacle range (time_horizon_obst * v_pref + radius = 5.3 m), and
    on a regular ring no edge's line covers another's, so each human gets about 62 obstacle lines.  With 40 humans
    packed inside, maxNeighbors = 32 adds 32 agent lines: about 94 lines in all, past 64."""
    from ebc.scene import pack_obstacles
    rng = np.random.default_rng(seed)
    ang = np.linspace(0, 2 * np.pi, 62, endpoint=False)[::-1]
    ring = [(3.5 * np.cos(a), 3.5 * np.sin(a)) for a in ang]
    rec, kept = pack_obstacles([ring], cap=64)
    assert kept == 1
    obst = np.zeros((N, 64), dtype=rec.dtype)
    obst[:, :len(rec)] = rec
    b = sweep_batch(N, H, 0, 0, seed)
    b["hum_count"][:] = H
    b["hum_pv"] = np.concatenate([rng.uniform(-2.2, 2.2, (N, H, 2)), rng.uniform(-0.5, 0.5, (N, H, 2))], 2).astype(np.float32)
    b["hum_gr"] = np.concatenate([rng.uniform(-2.2, 2.2, (N, H, 2)), np.ones((N, H, 1)), np.full((N, H, 1), 0.15)],
                                 2).astype(np.float32)
    b["hum_type"][:] = 0
    b["rob_pv"][:] = (0.0, 0.0, 0.0, 0.0)
    b["obst"], b["obst_count"] = obst, np.full(N, len(rec), np.int32)
    return b


@pytest.mark.gpu
@pytest.mark.parametrize("H", (40, 64), ids=["H%d" % h for h in (40, 64)])
def test_obstacle_path_beyond_64_lines(oracle, H):
    """orca_step_kernel (a warp per human, obstacle lines first) with more than 64 ORCA lines per human: see
    ring_scene for why the scene gets there.  RVO2 keeps every line, and so must the kernel.  Fused and unfused steps
    alternate; GPU == oracle bit for bit."""
    N = 97
    cfg = random_cfg()
    cfg.orca_obstacles, cfg.orca_max_neighbors, cfg.map_size_m = True, 32, 14.0
    batch = ring_scene(N, H, seed=H)
    sims = []
    for dev, be in (("cuda:0", None), ("cpu", oracle)):
        s = BatchedSim(cfg, N, H, 0, 0, 81, device=dev, backend=be, max_obst=64)
        s.set_actions(build_action_space(1.0))
        s.load_episodes(0, **batch)
        sims.append(s)
    g, r = sims
    zero = torch.zeros(N, dtype=torch.int32)
    for t in range(6):
        if t % 2:
            g.step(action_idx=zero.cuda(), fused_orca=True)
            r.step(action_idx=zero, fused_orca=True)
        else:
            for s in sims:
                s.orca()
            g.step(action_idx=zero.cuda())
            r.step(action_idx=zero)
        torch.cuda.synchronize()
        for k in ("hum_nv", "hum_pv"):
            assert_same_bits(getattr(g, k), getattr(r, k), "%s, step %d" % (k, t))
    ga, ra = g.robot_orca(0.15), r.robot_orca(0.15)
    torch.cuda.synchronize()
    assert_same_bits(ga, ra, "robot ORCA action")
