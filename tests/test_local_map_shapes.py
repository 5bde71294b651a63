"""The local-map kernels at every shape a user can set in the env INI: the angular map (ebc_local_map_angular,
simulator/env.py:468-628) at every sector count, polygon count and fan, and the binary grid sub-map
(ebc_local_map_grid, env.py:630-708) at every window size and on several map geometries.

References that are not the oracle:
- the grid map's OpenCV leg: the reference's own call chain written out (the clipped window of scene.map, then
  cv2.getRotationMatrix2D + cv2.warpAffine + "> 0.9"), run only where cv2 is importable;
- the angular map's fp64 leg: `angular_ref`, a plain Python restatement of calculate_angular_map_distances +
  get_local_map_angular (sweeps, int() truncation, the wrap rule, interpolation towards earlier points of a sweep,
  minimum per sector from max_range, normalisation), held to the goldens of the unmodified reference.

Bars: the grid map is binary and its arithmetic is integer or exact, so every cell must be equal.  The angular map is
fp64 with libm's cos / sin / atan2 (glibc on the host, CUDA on the device): at most 1e-12 and the same set of touched
sectors, as in test_local_map.py.  The shape of every case is in its test id.
"""
import math
import os

import numpy as np
import pytest
import torch

import oracle_backend as ob
from ebc.config import SimConfig
from ebc.engine import BatchedSim
from test_local_map_grid import _window

TOL = 1e-12
DEV = "cuda:0"


@pytest.fixture(scope="module")
def oracle_be():
    be = ob.OracleBackend()
    be.set_threads(os.cpu_count() or 1)
    return be


def _cv2():
    return pytest.importorskip("cv2")


# ---- grid map ------------------------------------------------------------------------------------------------------
# (map_size_m, map_resolution) -> window sizes S.  20 m / 0.1 m (G = 200) takes every S of the ABI; the others are the
# shipped map (90 cells), whole-map windows (S = G), an odd grid (91 cells) and a coarse grid with half-cell ties.
GEOMS = {
    (9.0, 0.1): [1, 2, 31, 50, 60, 61, 62, 63, 64, 65, 70, 89, 90],
    (9.1, 0.1): [1, 3, 31, 45, 61, 62, 63, 77, 91],
    (14.0, 0.25): [1, 2, 5, 20, 28, 33, 55, 56],
    (7.5, 0.05): [61, 62, 63, 100, 149, 150],
}
GRID_CASES = [(20.0, 0.1, S) for S in range(1, 193)] + [(m, r, S) for (m, r), ss in GEOMS.items() for S in ss]
GRID_IDS = ["map%g-res%g-G%d-S%d" % (m, r, int(round(m / r)), S) for m, r, S in GRID_CASES]
NB = 37          # odd batch: the last block of the grid is not a full warp's worth of anything
RMAX = 8


def _grid_batch(map_size_m, res, S, seed):
    """NB episodes: rectangles [NB, RMAX, 4] int16 (some empty or inverted) with dirty slots past the count, counts
    [NB] int32 (some past RMAX, one negative), poses [NB, 3] fp32-representable float64 (interior, clipped at every border and corner, off the
    map, half-cell ties; headings 0, +-pi/2, pi and random)."""
    rng = np.random.default_rng(seed)
    G = int(round(map_size_m / res))
    half, ext = map_size_m / 2.0, S * res
    rect = np.zeros((NB, RMAX, 4), np.int16)
    cnt = rng.integers(0, RMAX + 1, NB).astype(np.int32)
    for e in range(NB):
        for j in range(RMAX):
            x0, y0 = rng.integers(-5, G + 5, 2)
            w, h = rng.integers(1, max(G // 3, 2), 2)
            rect[e, j] = (max(x0, 0), max(y0, 0), min(x0 + w, G), min(y0 + h, G))
    rect[1, 0] = rect[2, 0] = (0, 0, G, G)                       # rectangles covering the whole map
    cnt[1], cnt[2] = 1, 3
    cnt[3], cnt[4], cnt[5] = RMAX + 5, -3, 0                     # clamped like the oracle; negative; none
    for e in range(NB):                                          # slots past the count: whole-map rectangles
        rect[e, max(cnt[e], 0):] = (0, 0, G, G)
    px = rng.uniform(-half + ext / 2, half - ext / 2, NB) if ext < map_size_m else rng.uniform(-half, half, NB)
    py = rng.uniform(-half + ext / 2, half - ext / 2, NB) if ext < map_size_m else rng.uniform(-half, half, NB)
    r = lambda: rng.uniform(-half, half)  # noqa: E731
    border = [(-half + 0.02, r()), (half - 0.02, r()), (r(), -half + 0.02), (r(), half - 0.02),      # the four borders
              (-half, -half), (-half, half), (half, -half), (half, half),                            # the four corners
              (-half - ext - 1.0, r()), (half + ext + 1.0, half + ext + 1.0),                        # off the map
              (-half - 0.6, r()), (r(), half + 0.6)]                                                 # just past it
    k = rng.integers(0, G, 4)
    ties = [((k[0] // 2 * 2 + 0.5) * res - half, (k[1] // 2 * 2 + 1.5) * res - half),               # even / odd k
            ((k[2] // 2 * 2 + 1.5) * res - half, (k[3] // 2 * 2 + 0.5) * res - half)]
    for i, (x, y) in enumerate(border + ties):
        px[6 + i], py[6 + i] = x, y
    th = rng.uniform(-np.pi, np.pi, NB)
    th[::3] = np.array([0.0, np.pi / 2, -np.pi / 2, np.pi])[np.arange(len(th[::3])) % 4]
    poses = np.stack([px, py, th], 1).astype(np.float32).astype(np.float64)
    return rect, cnt, poses


def _grid_run(map_size_m, res, S, rect, cnt, poses, device, backend=None, out=None):
    cfg = SimConfig()
    cfg.map_size_m, cfg.map_resolution = float(map_size_m), float(res)
    sim = BatchedSim(cfg, len(poses), 1, 0, rect.shape[1], 1, device=device, backend=backend)
    sim.rect.copy_(torch.as_tensor(rect))
    sim.rect_count.copy_(torch.as_tensor(cnt))
    p32 = torch.tensor(poses, dtype=torch.float32)
    sim.rob_pv[:, 0], sim.rob_pv[:, 1], sim.rob_theta[:] = p32[:, 0], p32[:, 1], p32[:, 2]
    return sim.local_map_grid(S * res, out=out).cpu().numpy()


def _grid_cv2(cv2, grid, px, py, theta, S, map_size_m, res):
    """env.py:630-708 as the reference calls it: the clipped window, rotated about (S/2, S/2), thresholded."""
    win = _window(grid, px, py, S, map_size_m, res)
    M = cv2.getRotationMatrix2D((S / 2, S / 2), (-theta + np.pi / 2) * 180 / np.pi, 1)
    rot = cv2.warpAffine(win.astype(np.float64), M, (S, S), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT,
                         borderValue=1)
    return (rot > 0.9).astype(np.uint8)


def _grid_cv2_batch(cv2, map_size_m, res, S, rect, cnt, poses):
    G = int(round(map_size_m / res))
    out = np.empty((len(poses), S, S), np.uint8)
    for e in range(len(poses)):
        grid = np.ones((G, G), np.uint8)
        for x0, y0, x1, y1 in rect[e, :min(max(int(cnt[e]), 0), rect.shape[1])].astype(int):
            if x1 > x0 and y1 > y0:                              # an inverted rectangle is empty (not numpy's x0:-1)
                grid[x0:x1, y0:y1] = 0
        out[e] = _grid_cv2(cv2, grid, poses[e, 0], poses[e, 1], poses[e, 2], S, map_size_m, res)
    return out


def _differ(a, b):
    return "%d of %d cells differ" % (int((a != b).sum()), a.size)


@pytest.mark.parametrize("map_size_m,res,S", GRID_CASES, ids=GRID_IDS)
def test_oracle_grid_map_matches_cv2(map_size_m, res, S, oracle_be):
    cv2 = _cv2()
    rect, cnt, poses = _grid_batch(map_size_m, res, S, S)
    got = _grid_run(map_size_m, res, S, rect, cnt, poses, "cpu", oracle_be)
    want = _grid_cv2_batch(cv2, map_size_m, res, S, rect, cnt, poses)
    assert np.array_equal(got, want), _differ(got, want)
    assert (got[14] == 1).all() and (got[15] == 1).all()         # the windows off the map


def test_grid_batch_reaches_every_branch():
    """The batch holds windows clipped on each side, degenerate windows and maps with free and occupied cells."""
    for map_size_m, res, S in ((20.0, 0.1, 50), (9.0, 0.1, 90), (14.0, 0.25, 5)):
        rect, cnt, poses = _grid_batch(map_size_m, res, S, S)
        G, half = int(round(map_size_m / res)), map_size_m / 2
        cx = np.array([int(round((p + half) / res)) for p in poses[:, 0]])
        six = cx - S // 2
        assert (six < 0).any() and (six + S - 1 > G - 1).any() and (six > G - 1).any()
    rect, cnt, poses = _grid_batch(14.0, 0.25, 5, 5)
    t = (poses[6 + 12:6 + 14, :2] + 7.0) / 0.25 - 0.5                 # exact half-cell ties, even and odd k
    assert np.array_equal(t, np.round(t)) and {int(t[0, 0]) % 2, int(t[0, 1]) % 2} == {0, 1}


@pytest.mark.gpu
@pytest.mark.parametrize("map_size_m,res,S", GRID_CASES, ids=GRID_IDS)
def test_gpu_grid_map_every_size(map_size_m, res, S, oracle_be):
    rect, cnt, poses = _grid_batch(map_size_m, res, S, S)
    run = lambda r=rect, c=cnt, p=poses, **kw: _grid_run(map_size_m, res, S, r, c, p, DEV, **kw)  # noqa: E731
    got = run()
    ref = _grid_run(map_size_m, res, S, rect, cnt, poses, "cpu", oracle_be)
    assert np.array_equal(got, ref), _differ(got, ref)
    clean = rect.copy()
    for e in range(NB):
        clean[e, max(cnt[e], 0):] = 0                              # slots past the count change no bit
    assert np.array_equal(run(r=clean), got)
    perm = np.random.default_rng(S).permutation(NB)
    assert np.array_equal(run(r=rect[perm], c=cnt[perm], p=poses[perm]), got[perm])
    assert np.array_equal(run(r=rect[:19], c=cnt[:19], p=poses[:19]), got[:19])
    if S <= 62:                                                    # the 64-bit-row kernel against the byte kernel
        os.environ["EBC_GRID_MAP_BYTES"] = "1"
        try:
            assert np.array_equal(run(), got)
        finally:
            del os.environ["EBC_GRID_MAP_BYTES"]
    try:
        import cv2
    except ImportError:
        return
    want = _grid_cv2_batch(cv2, map_size_m, res, S, rect, cnt, poses)
    assert np.array_equal(got, want), _differ(got, want)


NOISE_SIZES = [5, 31, 61, 62, 63, 64]


def _noise_batch(S, seed, n=13):
    """n episodes on a 64-cell map (6.4 m at 0.1 m) whose cells are free or occupied at random: the four taps of a
    sample take every pattern, so the thresholded sum lands on exactly 922 / 1024 (the "> 0.9" edge) a few times per
    map.  One rectangle per run of occupied cells (rects_from_zero_cells)."""
    from ebc.scene import rects_from_zero_cells
    rng = np.random.default_rng(seed)
    rects = [np.asarray(rects_from_zero_cells(rng.random((64, 64)) < 0.5), np.int16).reshape(-1, 4) for _ in range(n)]
    R = max(len(r) for r in rects)
    rect = np.zeros((n, R, 4), np.int16)
    cnt = np.array([len(r) for r in rects], np.int32)
    for e, r in enumerate(rects):
        rect[e, :len(r)] = r
    poses = np.stack([rng.uniform(-1.5, 1.5, n), rng.uniform(-1.5, 1.5, n), rng.uniform(-np.pi, np.pi, n)], 1)
    return rect, cnt, poses.astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("S", NOISE_SIZES, ids=lambda S: "map6.4-res0.1-G64-S%d-noise" % S)
def test_oracle_grid_map_noise_matches_cv2(S, oracle_be):
    cv2 = _cv2()
    rect, cnt, poses = _noise_batch(S, S)
    got = _grid_run(6.4, 0.1, S, rect, cnt, poses, "cpu", oracle_be)
    want = _grid_cv2_batch(cv2, 6.4, 0.1, S, rect, cnt, poses)
    assert np.array_equal(got, want), _differ(got, want)
    assert 0.2 < got.mean() < 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("S", NOISE_SIZES, ids=lambda S: "map6.4-res0.1-G64-S%d-noise" % S)
def test_gpu_grid_map_noise(S, oracle_be):
    rect, cnt, poses = _noise_batch(S, S)
    got = _grid_run(6.4, 0.1, S, rect, cnt, poses, DEV)
    ref = _grid_run(6.4, 0.1, S, rect, cnt, poses, "cpu", oracle_be)
    assert np.array_equal(got, ref), _differ(got, ref)
    if S <= 62:
        os.environ["EBC_GRID_MAP_BYTES"] = "1"
        try:
            assert np.array_equal(_grid_run(6.4, 0.1, S, rect, cnt, poses, DEV), got)
        finally:
            del os.environ["EBC_GRID_MAP_BYTES"]


@pytest.mark.gpu
@pytest.mark.parametrize("S", [63, 64, 70, 192])
def test_gpu_grid_map_unaligned_out(S):
    """A contiguous `out` at storage offset 1 (not 4-byte aligned) gets the same maps as an aligned one."""
    rect, cnt, poses = _grid_batch(20.0, 0.1, S, S)
    got = _grid_run(20.0, 0.1, S, rect, cnt, poses, DEV)
    buf = torch.full((NB * S * S + 1,), 7, dtype=torch.uint8, device=DEV)
    out = buf[1:].view(NB, S, S)
    assert out.is_contiguous() and out.data_ptr() % 4 == 1
    assert np.array_equal(_grid_run(20.0, 0.1, S, rect, cnt, poses, DEV, out=out), got)
    assert int(buf[0]) == 7


# ---- angular map ----------------------------------------------------------------------------------------------------
def angular_ref(polys, rx, ry, rad, theta, max_range, min_angle, max_angle, dim, normalize=True):
    """calculate_angular_map_distances + get_local_map_angular in float64, loop by loop.  `polys` [P, 4, 2]."""
    res = (max_angle - min_angle) / dim
    vec = [max_range] * dim
    cs, sn = math.cos(theta), math.sin(theta)
    edges = [(rx - rad, ry - rad), (rx + rad, ry - rad), (rx - rad, ry + rad), (rx + rad, ry + rad)]

    def rotate(x, y):
        return x * cs + y * sn, y * cs - x * sn

    def seen_from(vertex, edge, rad_indeces, locations):
        px, py = rotate(vertex[0] - edge[0], vertex[1] - edge[1])
        rad_idx = int((math.atan2(py, px) - min_angle) / res)
        distance = math.sqrt(px * px + py * py)
        if 0 <= rad_idx < dim:
            vec[rad_idx] = min(vec[rad_idx], distance)
        for old, loc in zip(rad_indeces, locations):
            if abs(rad_idx - old) > math.pi / res:           # the outline crosses the +-pi seam
                wrapped = True
                idx_diff = dim - rad_idx + old if rad_idx > old else dim - old + rad_idx
            else:
                wrapped = False
                idx_diff = abs(rad_idx - old)
            for i in range(idx_diff):
                t = i / idx_diff
                if (rad_idx < old and not wrapped) or (rad_idx > old and wrapped):
                    k = rad_idx + i
                    q = (vertex[0] + t * (loc[0] - vertex[0]) - edge[0], vertex[1] + t * (loc[1] - vertex[1]) - edge[1])
                else:
                    k = old + i
                    q = (loc[0] + t * (vertex[0] - loc[0]) - edge[0], loc[1] + t * (vertex[1] - loc[1]) - edge[1])
                if 0 <= k < dim:
                    px, py = rotate(*q)
                    vec[k] = min(vec[k], math.sqrt(px * px + py * py))
        rad_indeces.append(rad_idx)
        locations.append(vertex)

    for poly in polys:                                       # each robot corner over the polygon's vertices
        for edge in edges:
            idx, loc = [], []
            for vertex in poly:
                seen_from((float(vertex[0]), float(vertex[1])), edge, idx, loc)
    for poly in polys:                                       # each vertex over the robot's corners
        for vertex in poly:
            idx, loc = [], []
            for edge in edges:
                seen_from((float(vertex[0]), float(vertex[1])), edge, idx, loc)
    out = np.array(vec)
    return out / max_range if normalize else out


def _angular_ref_batch(xy, cnt, poses, max_range, amin, amax, dim, normalize):
    P = xy.shape[1]
    return np.stack([angular_ref(xy[e, :min(max(int(cnt[e]), 0), P)], *poses[e], max_range, amin, amax, dim, normalize)
                     for e in range(len(poses))])


def _angular_run(xy, cnt, poses, max_range, amin, amax, dim, normalize, device, backend=None, out=None):
    sim = BatchedSim(SimConfig(), len(poses), 1, 0, 0, 1, device=device, backend=backend)
    p32 = torch.tensor(poses, dtype=torch.float32)
    sim.rob_pv[:, 0], sim.rob_pv[:, 1], sim.rob_gr[:, 3], sim.rob_theta[:] = p32[:, 0], p32[:, 1], p32[:, 2], p32[:, 3]
    return sim.local_map_angular(torch.as_tensor(xy).to(device), torch.as_tensor(cnt).to(device), max_range, amin, amax,
                                 dim, normalize=normalize, out=out).cpu().numpy()


def _check_angular(got, want, full, what):
    assert np.array_equal(got == full, want == full), "%s: a sector is touched in one map and not in the other" % what
    err = np.abs(got - want).max() if got.size else 0.0
    assert err <= TOL, "%s: max |diff| %.3g" % (what, err)


def _quads(rng, n, P, spread=4.0):
    """[n, P, 4, 2] quadrilaterals in the reference's vertex order: rectangles (walls) and rotated boxes (circles)."""
    c = rng.uniform(-spread, spread, (n, P, 1, 2))
    w = rng.uniform(0.05, 1.5, (n, P, 1, 2))
    sgn = np.array([(1, 1), (-1, 1), (-1, -1), (1, -1)], np.float64)[None, None]
    q = sgn * w
    a = rng.uniform(-np.pi, np.pi, (n, P, 1))
    a[:, ::2] = 0.0
    ca, sa = np.cos(a), np.sin(a)
    return c + np.stack([q[..., 0] * ca - q[..., 1] * sa, q[..., 0] * sa + q[..., 1] * ca], -1)


def _poses(rng, n):
    """[n, 4] (px, py, radius, theta), fp32-representable."""
    p = np.stack([rng.uniform(-4.5, 4.5, n), rng.uniform(-4.5, 4.5, n), rng.uniform(0.2, 0.5, n),
                  rng.uniform(-np.pi, np.pi, n)], 1)
    p[::4, 3] = np.array([0.0, np.pi / 2, np.pi, -np.pi / 2])[np.arange(len(p[::4])) % 4]
    return p.astype(np.float32).astype(np.float64)


Z = np.load(os.path.join(ob.GOLDEN, "local_map_angular.npz"))


@pytest.mark.parametrize("normalize", [True, False], ids=["norm", "raw"])
@pytest.mark.parametrize("case", range(int(Z["n_cases"][0])), ids=lambda c: "golden%d" % c)
def test_angular_restatement_matches_reference(case, normalize):
    par, verts, poses = Z["c%d_params" % case], Z["c%d_verts" % case], Z["c%d_poses" % case]
    dim = int(par[3])
    gold = Z["c%d_%s" % (case, "norm" if normalize else "raw")]
    got = np.stack([angular_ref(verts, *[float(v) for v in p], par[0], par[1], par[2], dim, normalize) for p in poses])
    _check_angular(got, gold, 1.0 if normalize else par[0], "dim %d" % dim)


# fans (angle_min, angle_max) in units of pi: full circle, the shipped forward fan, a narrow fan (long interpolation
# runs at dim 256), an asymmetric one and one wider than 2 pi (the INI allows it)
FANS = {"full": (-1.0, 1.0), "forward": (-0.5, 0.5), "narrow": (-0.05, 0.05), "asym": (0.0, 0.7), "wide": (-1.5, 1.5)}


def _fan_case(fan, dim, seed):
    """13 episodes with 0..40 polygons, random poses, plus the special poses: hugging a vertex, inside a
    quadrilateral, a vertex exactly on a robot corner (distance 0)."""
    rng = np.random.default_rng(seed)
    P = 40
    n = 13
    xy = _quads(rng, n, P)
    cnt = np.array([0, 1, 2, 4, 5, 7, 9, 12, 20, 33, 40, 3, 6], np.int32)
    poses = _poses(rng, n)
    poses[11, :2] = xy[11, 0, 1] + 0.01 * np.array([1.0, -1.0])                 # hugging a vertex
    poses[12, :2] = xy[12, 0].mean(0)                                          # inside a quadrilateral
    poses = poses.astype(np.float32).astype(np.float64)
    r = poses[3, 2]
    xy[3, 0, 2] = (poses[3, 0] + r, poses[3, 1] - r)                           # a vertex on robot corner (1, -1)
    return xy, cnt, poses


ANG_FAN_CASES = [(f, d, mr, nz) for f in FANS for d in ([48, 256] if f == "narrow" else [48])
                 for mr in (0.5, 50.0) for nz in (True, False)]


@pytest.mark.parametrize("fan,dim,max_range,normalize", ANG_FAN_CASES,
                         ids=["%s-dim%d-range%g-%s" % (f, d, mr, "norm" if nz else "raw") for f, d, mr, nz in ANG_FAN_CASES])
def test_oracle_angular_map_matches_restatement(fan, dim, max_range, normalize, oracle_be):
    xy, cnt, poses = _fan_case(fan, dim, 7)
    amin, amax = FANS[fan][0] * np.pi, FANS[fan][1] * np.pi
    got = _angular_run(xy, cnt, poses, max_range, amin, amax, dim, normalize, "cpu", oracle_be)
    want = _angular_ref_batch(xy, cnt, poses, max_range, amin, amax, dim, normalize)
    _check_angular(got, want, 1.0 if normalize else max_range, fan)
    assert np.array_equal(got, want)          # same libm, same operation order: bit for bit


@pytest.mark.gpu
@pytest.mark.parametrize("fan,dim,max_range,normalize", ANG_FAN_CASES,
                         ids=["%s-dim%d-range%g-%s" % (f, d, mr, "norm" if nz else "raw") for f, d, mr, nz in ANG_FAN_CASES])
def test_gpu_angular_map_fans(fan, dim, max_range, normalize, oracle_be):
    xy, cnt, poses = _fan_case(fan, dim, 7)
    amin, amax = FANS[fan][0] * np.pi, FANS[fan][1] * np.pi
    full = 1.0 if normalize else max_range
    got = _angular_run(xy, cnt, poses, max_range, amin, amax, dim, normalize, DEV)
    _check_angular(got, _angular_run(xy, cnt, poses, max_range, amin, amax, dim, normalize, "cpu", oracle_be), full, "oracle")
    _check_angular(got, _angular_ref_batch(xy, cnt, poses, max_range, amin, amax, dim, normalize), full, "restatement")
    if fan in ("full", "wide"):          # the vertex on the corner: atan2(+-0, +-0) is +-pi here, inside these fans only
        assert got[3].min() == 0.0
    perm = np.random.default_rng(dim).permutation(len(poses))
    assert np.array_equal(_angular_run(xy[perm], cnt[perm], poses[perm], max_range, amin, amax, dim, normalize, DEV), got[perm])


ANG_PCOUNTS = (0, 1, 4, 5, 40)


def _dim_case(dim):
    """Per polygon count of ANG_PCOUNTS seven episodes, and two more with 40 polygons close by and far away: 37."""
    rng = np.random.default_rng(1000 + dim)
    cnt = np.repeat(np.array(ANG_PCOUNTS, np.int32), 7)
    n = len(cnt) + 2
    cnt = np.concatenate([cnt, np.array([40, 40], np.int32)])
    xy = _quads(rng, n, 40)
    poses = _poses(rng, n)
    xy[-1] = _quads(rng, 1, 40, spread=1.2)[0]                                 # close by: long outlines
    xy[-2] = _quads(rng, 1, 40, spread=12.0)[0]                                # far away: short ones
    return xy, cnt, poses


@pytest.mark.gpu
@pytest.mark.parametrize("dim", range(1, 257), ids=lambda d: "dim%d-P0,1,4,5,40-full" % d)
def test_gpu_angular_map_every_dim(dim, oracle_be):
    xy, cnt, poses = _dim_case(dim)
    out = torch.full((len(poses), dim), float("nan"), dtype=torch.float64, device=DEV)     # every sector is written
    got = _angular_run(xy, cnt, poses, 3.0, -np.pi, np.pi, dim, True, DEV, out=out)
    _check_angular(got, _angular_run(xy, cnt, poses, 3.0, -np.pi, np.pi, dim, True, "cpu", oracle_be), 1.0, "oracle")
    _check_angular(got, _angular_ref_batch(xy, cnt, poses, 3.0, -np.pi, np.pi, dim, True), 1.0, "restatement")
    assert (got[cnt == 0] == 1.0).all()
    perm = np.random.default_rng(dim).permutation(len(poses))
    assert np.array_equal(_angular_run(xy[perm], cnt[perm], poses[perm], 3.0, -np.pi, np.pi, dim, True, DEV), got[perm])


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [48, 256], ids=lambda d: "dim%d-P0..40-full" % d)
def test_gpu_angular_map_every_polygon_count(dim, oracle_be):
    """P = 0..40: 0 to 320 sweeps, up to 10 per lane.  Slots past the count hold NaN, +-inf and 1e300, and counts past
    Pmax (clamped) and negative ones occur: the padding changes no bit."""
    rng = np.random.default_rng(dim)
    P = 40
    cnt = np.concatenate([np.arange(P + 1), [P + 3, 1000, -1, -7]]).astype(np.int32)
    n = len(cnt)
    xy = _quads(rng, n, P, spread=3.0)
    poses = _poses(rng, n)
    xy[41:43], poses[41:43] = xy[40], poses[40]                                # counts past Pmax: episode 40's map
    got = _angular_run(xy, cnt, poses, 3.0, -np.pi, np.pi, dim, True, DEV)
    _check_angular(got, _angular_run(xy, cnt, poses, 3.0, -np.pi, np.pi, dim, True, "cpu", oracle_be), 1.0, "oracle")
    pick = np.array([0, 1, 2, 3, 4, 5, 8, 11, 16, 40, 41, 43, 44])
    _check_angular(got[pick], _angular_ref_batch(xy[pick], cnt[pick], poses[pick], 3.0, -np.pi, np.pi, dim, True), 1.0,
                   "restatement")
    assert (got[[0, 43, 44]] == 1.0).all() and np.array_equal(got[41], got[40]) and np.array_equal(got[42], got[40])
    dirty = xy.copy()
    junk = np.array([np.nan, np.inf, -np.inf, 1e300, -1e300])
    for e in range(n):
        k = min(max(int(cnt[e]), 0), P)
        dirty[e, k:] = junk[rng.integers(0, len(junk), dirty[e, k:].shape)]
    assert np.array_equal(_angular_run(dirty, cnt, poses, 3.0, -np.pi, np.pi, dim, True, DEV), got)
    perm = rng.permutation(n)
    assert np.array_equal(_angular_run(xy[perm], cnt[perm], poses[perm], 3.0, -np.pi, np.pi, dim, True, DEV), got[perm])


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [4, 8], ids=lambda d: "dim%d-axes-full" % d)
def test_gpu_angular_map_points_on_sector_boundaries(dim, oracle_be):
    """Heading 0 (the one axis-aligned heading whose fp32 value has an exact cos and sin) with vertices straight ahead
    of, behind, left and right of the robot's corners: atan2 returns 0, +-pi/2 or pi, the same in glibc and CUDA,
    and at dim 4 and 8 the angles 0 and pi fall exactly on a sector boundary, where int() picks the sector."""
    xy = np.zeros((8, 1, 4, 2))
    poses = np.zeros((8, 4))
    for e in range(8):
        poses[e] = (0.5 * e - 2.0, -0.25 + 0.125 * e, 0.25, 0.0)
        cx, cy = poses[e, 0], poses[e, 1]
        # every vertex straight ahead, behind, left or right of a robot corner of the axis-aligned robot
        xy[e, 0] = [(cx + 0.25 + 1.0, cy - 0.25), (cx - 0.25, cy + 0.25 + 2.0), (cx - 0.25 - 1.5, cy + 0.25),
                    (cx + 0.25, cy - 0.25 - 0.5)]
    poses = poses.astype(np.float32).astype(np.float64)
    cnt = np.ones(8, np.int32)
    for normalize in (True, False):
        full = 1.0 if normalize else 5.0
        got = _angular_run(xy, cnt, poses, 5.0, -np.pi, np.pi, dim, normalize, DEV)
        _check_angular(got, _angular_run(xy, cnt, poses, 5.0, -np.pi, np.pi, dim, normalize, "cpu", oracle_be), full, "oracle")
        _check_angular(got, _angular_ref_batch(xy, cnt, poses, 5.0, -np.pi, np.pi, dim, normalize), full, "restatement")


# ---- end to end: BatchedEnv.local_map_batch after reset_batch ------------------------------------------------------
def _env_config(over):
    import configparser
    cp = configparser.RawConfigParser()
    assert cp.read(os.path.join(ob.GOLDEN, "configs", "env_ebcadrl.config"))
    for (section, key), value in over.items():
        cp.set(section, key, str(value))
    return cp


def _oracle_twin(env, backend):
    s = env.sim
    ref = BatchedSim(env.cfg, env.N, 1, 0, s.Rmax, 1, device="cpu", backend=backend)
    for k in ("rob_pv", "rob_gr", "rob_theta"):
        getattr(ref, k).copy_(getattr(s, k).cpu())
    if s.Rmax:
        ref.rect.copy_(s.rect.cpu())
        ref.rect_count.copy_(s.rect_count.cpu())
    return ref


def _random_robot(env, seed):
    rng = np.random.default_rng(seed)
    half = env.cfg.map_size_m / 2 + 0.5
    p = torch.tensor(np.stack([rng.uniform(-half, half, env.N), rng.uniform(-half, half, env.N)], 1), dtype=torch.float32)
    env.sim.rob_pv[:, :2] = p.to(env.device)
    env.sim.rob_theta[:] = torch.tensor(rng.uniform(-np.pi, np.pi, env.N), dtype=torch.float32).to(env.device)


E2E_N = 4097


@pytest.mark.gpu
def test_gpu_batched_env_angular_map_walls_and_circles(oracle_be):
    from ebc.batched_env import BatchedEnv
    env = BatchedEnv(_env_config({("map", "num_walls"): 10, ("map", "num_circles"): 4}), None, E2E_N, DEV)
    env.reset_batch("test", np.arange(E2E_N) + 1000)
    assert env.poly_xy.shape[1] == 14 and int(env.poly_count.max()) > 10
    for pose in ("reset", "random"):
        if pose == "random":
            _random_robot(env, 3)
        got = env.local_map_batch().cpu().numpy()
        ref = _oracle_twin(env, oracle_be).local_map_angular(env.poly_xy.cpu(), env.poly_count.cpu(), 3.0, -np.pi, np.pi,
                                                             48).numpy()
        _check_angular(got, ref, 1.0, pose)
        assert (got < 1.0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("submap", [5, 7], ids=["S50-bits", "S70-bytes"])
def test_gpu_batched_env_grid_map_striped_borders(submap, oracle_be):
    """9.1 m at 0.1 m (91 cells, odd): circles on the border become the replay's striped lattice rectangles."""
    from ebc.batched_env import BatchedEnv
    from host_scenes import host_batch
    env = BatchedEnv(_env_config({("map", "use_grid_map"): "true", ("map", "submap_size_m"): submap,
                                  ("map", "map_size_m"): 9.1, ("map", "num_circles"): 4}), None, E2E_N, DEV)
    seeds = np.arange(E2E_N) + 1000
    env.reset_batch("test", seeds)
    S = submap * 10
    _random_robot(env, submap)
    got = env.local_map_batch().cpu().numpy()
    twin = _oracle_twin(env, oracle_be)
    ref = twin.local_map_grid(float(submap)).numpy()
    assert got.shape == (E2E_N, S, S) and np.array_equal(got, ref), _differ(got, ref)
    assert 0.01 < (got == 0).mean() < 0.9
    try:
        import cv2
    except ImportError:
        return
    k = 100
    host = host_batch(env, "test", seeds[:k])
    poses = twin.rob_pv[:k, :2].double().numpy()
    theta = twin.rob_theta[:k].double().numpy()
    striped = 0
    for e in range(k):
        grid = (~host["maps"][e]).astype(np.uint8)
        striped += int(len(host["rects"][e]) > 4 + 3)
        want = _grid_cv2(cv2, grid, poses[e, 0], poses[e, 1], theta[e], S, 9.1, 0.1)
        assert np.array_equal(got[e], want), (e, _differ(got[e], want))
    assert striped > 0


# ---- wrapper contract (CPU, oracle backend) --------------------------------------------------------------------------
def _cpu_sim(backend, N=3):
    sim = BatchedSim(SimConfig(), N, 1, 0, 0, 1, device="cpu", backend=backend)
    sim.rob_pv[:, 1] = -1.0
    sim.rob_gr[:, 3] = 0.3
    return sim


def test_local_map_angular_refuses_bad_buffers(oracle_be):
    sim = _cpu_sim(oracle_be)
    xy = torch.as_tensor(_quads(np.random.default_rng(0), 3, 2, spread=2.0))
    cnt = torch.tensor([2, 1, 0], dtype=torch.int32)
    args = (3.0, -np.pi, np.pi, 48)
    want = sim.local_map_angular(xy, cnt, *args).numpy()
    out = torch.full((3, 48), -1.0, dtype=torch.float64)
    assert sim.local_map_angular(xy, cnt, *args, out=out) is out and np.array_equal(out.numpy(), want)
    # a poly_xy that is not contiguous is still made contiguous
    wide = torch.zeros(3, 2, 4, 4, dtype=torch.float64)
    wide[..., ::2] = xy
    assert np.array_equal(sim.local_map_angular(wide[..., ::2], cnt, *args).numpy(), want)
    for bad in (torch.empty(3, 48, dtype=torch.float32), torch.empty(3, 47, dtype=torch.float64),
                torch.empty(3, 48, 1, dtype=torch.float64), torch.empty(3, 64, dtype=torch.float64)[:, :48],
                torch.empty(48, 3, dtype=torch.float64).t()):
        with pytest.raises(AssertionError):
            sim.local_map_angular(xy, cnt, *args, out=bad)
    need = torch.zeros(3, 5, dtype=torch.int32)
    need[:, 3] = cnt
    with pytest.raises(AssertionError):
        sim.local_map_angular(xy, need[:, 3], *args)
    with pytest.raises(AssertionError):
        sim.local_map_angular(xy, cnt[:, None], *args)


def test_build_obstacles_and_replay_scenes_refuse_strided_counts(oracle_be):
    """The checks run before the library is called (the oracle has no twin of either entry point)."""
    sim = BatchedSim(SimConfig(), 3, 1, 0, 0, 1, device="cpu", backend=oracle_be)
    xy = torch.as_tensor(_quads(np.random.default_rng(0), 3, 2, spread=2.0))
    need = torch.zeros(3, 5, dtype=torch.int32)
    need[:, 3] = torch.tensor([2, 1, 0], dtype=torch.int32)
    with pytest.raises(AssertionError):
        sim.build_obstacles(xy, need[:, 3])
    seeds = torch.zeros(3, dtype=torch.int32)
    from ebc import abi
    rc = abi.EbcReplayConfig()
    rc.max_polys = 2
    with pytest.raises(AssertionError):
        sim.replay_scenes(rc, seeds, poly_xy=xy.clone(), poly_count=need[:, 3])
    with pytest.raises(AssertionError):
        sim.replay_scenes(rc, seeds, poly_xy=xy.clone(), need=torch.zeros(5, 3, dtype=torch.int32).t())
