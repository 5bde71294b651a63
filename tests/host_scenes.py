"""The per-episode host path BatchedEnv.reset_batch ran before the device replay (ebc_replay_scenes): SceneGenerator
once per seed, rects_from_zero_cells over its grid, padded numpy arrays.  The GPU tests compare the replay against it,
and tools/scene_replay_rate.py times it."""
import numpy as np

from ebc.scene import rects_from_zero_cells


def host_batch(env, phase, seeds, restore_counter=True):
    """Scenes of `seeds` for BatchedEnv `env`'s capacities: hum_pv / hum_gr / hum_type / hum_count / stat / stat_count /
    rect / rect_count (rects_from_zero_cells, clipped to Rmax) / poly_xy / poly_count as reset_batch used to load them,
    plus every scene's map == 0, its rectangle list and which agents crossed the circle.  The generator's case counter
    is put back afterwards unless `restore_counter` is false."""
    sim, sg = env.sim, env.scene
    n = len(seeds)
    H, S, R = sim.Hmax, max(sim.Smax, 1), max(sim.Rmax, 1)
    out = {"hum_pv": np.zeros((n, H, 4), np.float32), "hum_gr": np.zeros((n, H, 4), np.float32),
           "hum_type": np.zeros((n, H), np.uint8), "hum_count": np.zeros(n, np.int32),
           "stat": np.zeros((n, S, 4), np.float32), "stat_count": np.zeros(n, np.int32),
           "rect": np.zeros((n, R, 4), np.int16), "rect_count": np.zeros(n, np.int32), "maps": [], "rects": [],
           "circle_agents": np.zeros((n, H), bool)}
    rad = sg.circle_radius
    polys = []
    counter = dict(sg.case_counter)
    for e, seed in enumerate(seeds):
        env.robot.set(0, -rad, 0, rad, 0, 0, np.pi / 2)
        sg.generate_random_scene(env.COUNTER_OFFSET, phase, scene_number=int(seed))
        hs = sg.adults + sg.bicycles + sg.children
        for i, h in enumerate(hs[:H]):
            out["hum_pv"][e, i] = (h.px, h.py, h.vx, h.vy)
            out["hum_gr"][e, i] = (h.gx, h.gy, h.v_pref, h.radius)
            out["hum_type"][e, i] = int(h.agent_type)
            out["circle_agents"][e, i] = abs(h.gx + h.px) < 1e-12 and abs(h.gy + h.py) < 1e-12 and h.px != h.gx
        out["hum_count"][e] = len(hs)
        for i, s in enumerate(sg.static_obstacles_as_pedestrians[:S]):
            out["stat"][e, i, :3] = (s.px, s.py, s.radius)
        out["stat_count"][e] = len(sg.static_obstacles_as_pedestrians)
        rects = rects_from_zero_cells(sg.map == 0)
        out["rect"][e, :min(len(rects), R)] = rects[:R]
        out["rect_count"][e] = len(rects)
        out["maps"].append(sg.map == 0)
        out["rects"].append(rects)
        polys.append(np.asarray(sg.obstacle_vertices, dtype=np.float64).reshape(-1, 4, 2))
    if restore_counter:
        sg.case_counter.update(counter)
    P = max([len(v) for v in polys] + [1])
    out["poly_xy"] = np.zeros((n, P, 4, 2), np.float64)
    for e, v in enumerate(polys):
        out["poly_xy"][e, :len(v)] = v
    out["poly_count"] = np.array([len(v) for v in polys], np.int32)
    return out
