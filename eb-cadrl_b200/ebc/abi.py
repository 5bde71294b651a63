"""ctypes view of include/ebcadrl.h — the C ABI of the B200 hot path.

The product library is eb-cadrl_b200/lib/libebcadrl.so (CUDA, sm_100a).  There is no CPU
fallback: `load()` raises if the library is missing.  (The CPU checker used by tests/ lives outside this
package and reuses these struct definitions; nothing in this package loads it.)
"""
import ctypes
import os

ABI_VERSION = 2

EVENT_NAMES = ["Nothing", "Danger", "ReachGoal", "CollisionAdult", "CollisionBicycle",
               "CollisionChild", "CollisionObstacle", "Timeout"]
EV_NOTHING, EV_DANGER, EV_REACH_GOAL, EV_COLLISION_ADULT, EV_COLLISION_BICYCLE, \
    EV_COLLISION_CHILD, EV_COLLISION_OBSTACLE, EV_TIMEOUT = range(8)

KIN_HOLONOMIC, KIN_UNICYCLE = 0, 1
VALUE_FP32, VALUE_TC_FP32, VALUE_TC_BF16, VALUE_TC_FP16X2 = 0, 1, 2, 3
POLICY_ORCA, POLICY_LINEAR = 0, 1
ERR_INVALID, ERR_UNBOUND, ERR_CUDA, ERR_NOMEM = -1, -2, -3, -4
WARN_VALUE_FFMA = 1      # ebc_set_weights: accepted, but K4 runs on the FFMA kernels

c_i32, c_f64, c_f32 = ctypes.c_int32, ctypes.c_double, ctypes.c_float
vp = ctypes.c_void_p


class EbcConfig(ctypes.Structure):
    _fields_ = [
        ("abi_version", c_i32), ("n_episodes", c_i32), ("max_humans", c_i32), ("max_statics", c_i32),
        ("max_rects", c_i32), ("n_actions", c_i32), ("robot_kinematics", c_i32), ("rotate_theta", c_i32),
        ("with_agent_type", c_i32), ("robot_visible", c_i32), ("human_policy", c_i32 * 3),
        ("new_reward", c_i32), ("has_max_goal_distance", c_i32), ("orca_max_neighbors", c_i32),
        ("time_step", c_f64), ("time_limit", c_f64), ("time_max", c_f64), ("time_good", c_f64),
        ("max_goal_distance", c_f64), ("success_reward", c_f64),
        ("collision_penalty_adult", c_f64), ("collision_penalty_bicycle", c_f64),
        ("collision_penalty_obstacle", c_f64), ("collision_penalty_child", c_f64),
        ("discomfort_dist_adult", c_f64), ("discomfort_dist_bicycle", c_f64), ("discomfort_dist_child", c_f64),
        ("discomfort_penalty_factor_adult", c_f64), ("discomfort_penalty_factor_bicycle", c_f64),
        ("discomfort_penalty_factor_child", c_f64), ("rotation_penalty_factor", c_f64),
        ("map_size_m", c_f64), ("map_resolution", c_f64), ("gamma", c_f64), ("orca_safety_space", c_f64),
        ("orca_neighbor_dist", c_f32), ("orca_time_horizon", c_f32),
        ("orca_obstacles", c_i32), ("max_obst", c_i32), ("orca_time_horizon_obst", c_f32), ("reserved0", c_f32),
    ]


class EbcObstVertex(ctypes.Structure):
    _fields_ = [("px", c_f32), ("py", c_f32), ("ux", c_f32), ("uy", c_f32), ("next", ctypes.c_int16),
                ("prev", ctypes.c_int16), ("convex", ctypes.c_int16), ("pad0", ctypes.c_int16),
                ("anc", ctypes.c_uint64), ("anc_left", ctypes.c_uint64), ("pad1", ctypes.c_uint64)]


OBST_DTYPE = [("px", "<f4"), ("py", "<f4"), ("ux", "<f4"), ("uy", "<f4"), ("next", "<i2"), ("prev", "<i2"),
              ("convex", "<i2"), ("pad0", "<i2"), ("anc", "<u8"), ("anc_left", "<u8"), ("pad1", "<u8")]   # numpy view


class EbcState(ctypes.Structure):
    _fields_ = [(n, vp) for n in (
        "hum_pv", "hum_gr", "hum_type", "hum_count", "hum_nv", "stat", "stat_count", "rect", "rect_count",
        "rob_pv", "rob_gr", "rob_theta", "time", "obst", "obst_count")]


class EbcStats(ctypes.Structure):
    _fields_ = [(n, vp) for n in ("alive", "final_event", "steps", "too_close", "cum_reward", "discount",
                                  "min_dist_sum", "alive_count")]


class EbcLinear(ctypes.Structure):
    _fields_ = [("weight", vp), ("bias", vp), ("in_dim", c_i32), ("out_dim", c_i32)]


class EbcWeights(ctypes.Structure):
    _fields_ = [("input_dim", c_i32), ("self_state_dim", c_i32), ("with_global_state", c_i32),
                ("mlp1", EbcLinear * 2), ("mlp2", EbcLinear * 2), ("attention", EbcLinear * 3),
                ("mlp3", EbcLinear * 4)]


# name -> (restype, argtypes) for every entry point include/ebcadrl.h declares for libebcadrl.so
class EbcSceneShape(ctypes.Structure):
    _fields_ = [("n_types", c_i32), ("type_code", c_i32 * 4), ("type_count", c_i32 * 4),
                ("v_pref_lo", c_f64 * 4), ("v_pref_hi", c_f64 * 4), ("radius_lo", c_f64 * 4), ("radius_hi", c_f64 * 4),
                ("rule", c_i32), ("num_walls", c_i32), ("wall_len_lo", c_i32), ("wall_len_hi", c_i32),
                ("discs_per_wall", c_i32), ("max_tries", c_i32),
                ("square_width", c_f64), ("circle_radius", c_f64), ("robot_radius", c_f64), ("robot_v_pref", c_f64),
                ("map_size_m", c_f64), ("map_resolution", c_f64), ("discomfort_dist", c_f64)]


# EBC_REPLAY_* rule codes of ebc_replay_config, by the rule names of the [sim] section
REPLAY_RULES = {"square_crossing": 0, "circle_crossing": 1, "mixed": 2, "mixed_20": 3, "one_static": 4,
                "square_crossing_old": 5}
REPLAY_RNG_SEED, REPLAY_RNG_RANDOM, REPLAY_RNG_UNIFORM, REPLAY_RNG_RANDINT, REPLAY_RNG_CHOICE_SIGN = range(5)


class EbcReplayConfig(ctypes.Structure):     # one phase of simulator/scene/scene_generator.py (ebc_replay_scenes)
    _fields_ = [("count", c_i32 * 3), ("rule", c_i32 * 3), ("randomize_attributes", c_i32),
                ("num_circles", c_i32), ("num_walls", c_i32), ("min_wall_length", c_i32), ("max_wall_length", c_i32),
                ("max_polys", c_i32), ("norm_fused", c_i32), ("reserved", c_i32),
                ("v_pref", c_f64 * 3), ("radius", c_f64 * 3), ("v_pref_min", c_f64 * 3), ("v_pref_max", c_f64 * 3),
                ("radius_min", c_f64 * 3), ("radius_max", c_f64 * 3),
                ("square_width", c_f64), ("circle_radius", c_f64), ("discomfort_dist", c_f64),
                ("robot_radius", c_f64), ("robot_v_pref", c_f64), ("map_size_m", c_f64), ("map_resolution", c_f64)]


class EbcAngularMap(ctypes.Structure):       # [map] section of the env config (simulator/env.py:79-87)
    _fields_ = [("max_range", c_f64), ("min_angle", c_f64), ("max_angle", c_f64), ("dim", c_i32),
                ("normalize", c_i32), ("max_polys", c_i32), ("reserved", c_i32)]


class EbcGridMap(ctypes.Structure):          # [map] submap_size_m (simulator/env.py:81-82, :630-692)
    _fields_ = [("submap_size_m", c_f64), ("size", c_i32), ("reserved", c_i32)]


SIM = vp
PROTOTYPES = {
    "ebc_create": (c_i32, [ctypes.POINTER(EbcConfig), c_i32, ctypes.POINTER(SIM)]),
    "ebc_destroy": (None, [SIM]),
    "ebc_last_error": (ctypes.c_char_p, [SIM]),
    "ebc_abi_version": (c_i32, []),
    "ebc_bind": (c_i32, [SIM, ctypes.POINTER(EbcState)]),
    "ebc_bind_stats": (c_i32, [SIM, ctypes.POINTER(EbcStats)]),
    "ebc_pack_obstacles": (c_i32, [vp, vp, c_i32, vp, c_i32, vp]),
    "ebc_set_actions": (c_i32, [SIM, vp, c_i32]),
    "ebc_set_weights": (c_i32, [SIM, ctypes.POINTER(EbcWeights)]),
    "ebc_reserve": (c_i32, [SIM, ctypes.c_int64]),
    "ebc_set_value_mode": (c_i32, [SIM, c_i32]),
    "ebc_get_value_mode": (c_i32, [SIM]),
    "ebc_orca": (c_i32, [SIM, vp]),
    "ebc_robot_orca": (c_i32, [SIM, c_f64, vp, vp]),
    "ebc_lookahead": (c_i32, [SIM, vp, vp, vp, vp, vp]),
    "ebc_value": (c_i32, [SIM, vp, ctypes.c_int64, vp, vp, vp]),
    "ebc_set_attention_output": (c_i32, [SIM, vp]),
    "ebc_select": (c_i32, [SIM, vp, vp, vp, vp, vp, vp]),
    "ebc_step": (c_i32, [SIM, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "ebc_orca_step": (c_i32, [SIM, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "ebc_transform": (c_i32, [SIM, vp, vp]),
    "ebc_reset": (c_i32, [SIM, ctypes.POINTER(EbcState), c_i32, vp, vp, vp]),
    "ebc_generate": (c_i32, [SIM, ctypes.POINTER(EbcSceneShape), ctypes.c_uint64, vp, vp, vp]),
    "ebc_replay_scenes": (c_i32, [SIM, ctypes.POINTER(EbcReplayConfig), vp, vp, vp, vp, vp, vp]),
    "ebc_build_obstacles": (c_i32, [SIM, vp, vp, c_i32, vp, vp, vp]),
    "ebc_local_map_angular": (c_i32, [SIM, ctypes.POINTER(EbcAngularMap), vp, vp, vp, vp]),
    "ebc_local_map_grid": (c_i32, [SIM, ctypes.POINTER(EbcGridMap), vp, vp]),
    "ebc_debug_trace": (c_i32, [SIM, vp, c_i32]),
    "ebc_launch_count": (ctypes.c_int64, [SIM]),
    "ebc_replay_scene_host": (c_i32, [ctypes.POINTER(EbcReplayConfig), ctypes.c_uint32, c_i32, c_i32, c_i32, vp, vp, vp,
                                      vp, vp, vp, vp]),
    "ebc_replay_rng_host": (c_i32, [vp, vp, c_i32, c_f64, c_f64, vp]),
}

LIB_PATH = os.environ.get("EBCADRL_LIB") or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lib",
                                                        "libebcadrl.so")     # EBCADRL_LIB: another build of the same ABI


class EbcError(RuntimeError):
    pass


_lib = None


def load(path=None):
    """dlopen libebcadrl.so and type every symbol.  Fails loudly when it is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise EbcError("CUDA extension %s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)" % p)
    lib = ctypes.CDLL(p)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)   # AttributeError if the library does not export the header's symbol
        fn.restype = res
        fn.argtypes = args
    if lib.ebc_abi_version() != ABI_VERSION:
        raise EbcError("libebcadrl.so ABI %d != %d" % (lib.ebc_abi_version(), ABI_VERSION))
    if path is None:
        _lib = lib
    return lib
