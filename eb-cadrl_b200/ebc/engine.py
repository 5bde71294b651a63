"""BatchedSim — N independent EB-CADRL episodes advanced at once on one B200.

Host-side owner of the structure-of-arrays episode state (torch tensors on the device,
borrowed by the C ABI through raw pointers).  All compute is in libebcadrl.so
(eb-cadrl_b200/csrc); torch is used for device memory and streams only.

The methods map 1:1 onto the reference's hot path:
    orca()       env.step's per-human policy loop    simulator/env.py:392-405, policy/orca.py:85-157
    lookahead()  env.onestep_lookahead x A actions    simulator/env.py:207-209, rl/policy/multi_human_rl.py:38-61
    value()      SARL value network                   rl/policy/sarl.py:38-82
    select()     reward + gamma^(dt v_pref) V, argmax rl/policy/multi_human_rl.py:72-80
    step()       env.step(action, update=True)        simulator/env.py:388-466
"""
import ctypes

import numpy as np
import torch

from . import abi

_WEIGHT_KEYS = (["mlp1.0", "mlp1.2"], ["mlp2.0", "mlp2.2"], ["attention.0", "attention.2", "attention.4"],
                ["mlp3.0", "mlp3.2", "mlp3.4", "mlp3.6"])


class CudaBackend(object):
    """Thin adapter over libebcadrl.so (the only backend this package ships)."""
    name = "cuda"

    def __init__(self, lib=None):
        self.lib = lib or abi.load()

    def create(self, cfg, device_index):
        h = abi.SIM()
        rc = self.lib.ebc_create(ctypes.byref(cfg), device_index, ctypes.byref(h))
        if rc != 0:
            raise abi.EbcError("ebc_create: %s" % self.lib.ebc_last_error(None).decode())
        return h

    def destroy(self, h):
        self.lib.ebc_destroy(h)

    def last_error(self, h):
        return self.lib.ebc_last_error(h).decode()

    def call(self, name, h, *args, stream=None):
        fn = getattr(self.lib, "ebc_" + name)
        if name in ("bind", "bind_stats", "set_actions", "set_weights", "reserve", "set_attention_output"):
            rc = fn(h, *args)
        else:
            rc = fn(h, *args, stream)
        if rc < 0:
            raise abi.EbcError("ebc_%s failed (%d): %s" % (name, rc, self.last_error(h)))
        if rc > 0:          # accepted with a documented downgrade (EBC_WARN_*): tell the caller, loudly
            import warnings
            warnings.warn("ebc_%s: %s" % (name, self.last_error(h)), RuntimeWarning, stacklevel=3)
        return rc

    def launch_count(self, h):
        return int(self.lib.ebc_launch_count(h))


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class BatchedSim(object):
    def __init__(self, cfg, n_episodes, max_humans, max_statics=0, max_rects=0, n_actions=81,
                 device="cuda:0", backend=None, max_obst=0):
        self.cfg = cfg
        self.N, self.Hmax, self.Smax, self.Rmax, self.A = n_episodes, max_humans, max_statics, max_rects, n_actions
        self.Omax = max_obst
        self.n = max_humans + max_statics
        self.D = cfg.D
        self.device = torch.device(device)
        if backend is None:
            if self.device.type != "cuda":
                raise abi.EbcError("BatchedSim needs a CUDA device: the hot path has no CPU fallback")
            backend = CudaBackend()
        self.be = backend
        self._abi_cfg = cfg.to_abi(n_episodes, max_humans, max_statics, max_rects, n_actions, max_obst)
        dev_index = self.device.index if self.device.type == "cuda" and self.device.index is not None else 0
        if self.device.type == "cuda":
            torch.cuda.set_device(self.device)
        self.h = self.be.create(self._abi_cfg, dev_index)
        N, H, S, R, A = self.N, self.Hmax, max(self.Smax, 1), max(self.Rmax, 1), self.A
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=self.device)  # noqa: E731
        self.hum_pv = z(N, H, 4)
        self.hum_gr = z(N, H, 4)
        self.hum_type = z(N, H, dtype=torch.uint8)
        self.hum_count = z(N, dtype=torch.int32)
        self.hum_nv = z(N, H, 2)
        self.stat = z(N, S, 4)
        self.stat_count = z(N, dtype=torch.int32)
        self.attention = None      # enable_attention()
        self.rect = z(N, R, 4, dtype=torch.int16)
        self.rect_count = z(N, dtype=torch.int32)
        self.rob_pv = z(N, 4)
        self.rob_gr = z(N, 4)
        self.rob_theta = z(N)
        self.time = z(N, dtype=torch.float64)
        # ORCA obstacle vertices (ebc_obst_vertex records of 48 bytes, viewed as bytes; SURVEY 8f-4)
        self.obst = z(N, max(self.Omax, 1), 48, dtype=torch.uint8)
        self.obst_count = z(N, dtype=torch.int32)
        # per-decision buffers
        self.vin = None
        self.fused_input = False      # decide(): K4 builds its own input (set by BatchedEnv when K4 runs on the tensor cores)
        self.la_reward = z(N, A, dtype=torch.float64)
        self.la_done = z(N, A, dtype=torch.uint8)
        self.la_event = z(N, A, dtype=torch.uint8)
        self.values = z(N, A)
        self.action_values = z(N, A, dtype=torch.float64)
        self.argmax = z(N, dtype=torch.int32)
        self.nan_flag = z(N, dtype=torch.uint8)
        # per-step outputs
        self.reward = z(N, dtype=torch.float64)
        self.done = z(N, dtype=torch.uint8)
        self.event = z(N, dtype=torch.uint8)
        self.dmin = z(N, 3, dtype=torch.float64)
        self.dist_to_goal = z(N, dtype=torch.float64)
        self.actions = None
        st = abi.EbcState()
        for name in ("hum_pv", "hum_gr", "hum_type", "hum_count", "hum_nv", "stat", "stat_count", "rect",
                     "rect_count", "rob_pv", "rob_gr", "rob_theta", "time", "obst", "obst_count"):
            setattr(st, name, getattr(self, name).data_ptr())
        self._state = st
        self.be.call("bind", self.h, ctypes.byref(st))
        self.stats = None

    # ---- running episode statistics on the device (ebc_bind_stats) -----------------------------------------
    def bind_stats(self, alive=None):
        """Allocate (first call), re-initialise and bind the per-episode accumulators; every committed step then
        updates them for the episodes it steps, and `step(active=None)` uses stats['alive'] as its mask."""
        N = self.N
        if self.stats is None:
            z = lambda dtype: torch.zeros(N, dtype=dtype, device=self.device)  # noqa: E731
            self.stats = {"alive": z(torch.uint8), "final_event": z(torch.uint8), "steps": z(torch.int32),
                          "too_close": z(torch.int32), "cum_reward": z(torch.float64), "discount": z(torch.float64),
                          "min_dist_sum": z(torch.float64),
                          "alive_count": torch.zeros(1, dtype=torch.int32, device=self.device)}
            sx = abi.EbcStats()
            for k, t in self.stats.items():
                setattr(sx, k, t.data_ptr())
            self._stats_abi = sx
        st = self.stats
        for k in ("final_event", "steps", "too_close", "cum_reward", "min_dist_sum"):
            st[k].zero_()
        st["discount"].fill_(1.0)
        if alive is None:
            st["alive"].fill_(1)
            st["alive_count"].fill_(N)
        else:
            st["alive"].copy_(alive)
            st["alive_count"].copy_(alive.sum().to(torch.int32).reshape(1))
        self.be.call("bind_stats", self.h, ctypes.byref(self._stats_abi))
        return st

    def unbind_stats(self):
        """Stop accumulating (the tensors stay readable); step(active=None) steps every episode again."""
        self.be.call("bind_stats", self.h, None)

    def close(self):
        if getattr(self, "h", None) is not None:
            self.be.destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- configuration ------------------------------------------------------------
    def _stream(self):
        if self.device.type == "cuda":
            return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        return None

    def set_actions(self, table):
        table = np.ascontiguousarray(table, dtype=np.float64)
        assert table.shape == (self.A, 2), table.shape
        self.actions = table
        self.be.call("set_actions", self.h, table.ctypes.data_as(ctypes.c_void_p), self.A)

    def set_weights(self, state_dict, with_global_state=True, self_state_dim=6):
        """state_dict: the reference's ValueNetwork.state_dict() (rl/policy/sarl.py:9-36), tensors or arrays."""
        keep = []

        def lin(key):
            w = np.ascontiguousarray(np.asarray(state_dict[key + ".weight"], dtype=np.float32))
            b = np.ascontiguousarray(np.asarray(state_dict[key + ".bias"], dtype=np.float32))
            keep.extend([w, b])
            l = abi.EbcLinear()
            l.weight, l.bias = w.ctypes.data, b.ctypes.data
            l.out_dim, l.in_dim = w.shape
            return l

        w = abi.EbcWeights()
        w.input_dim, w.self_state_dim, w.with_global_state = self.D, self_state_dim, int(with_global_state)
        for field, keys in zip(("mlp1", "mlp2", "attention", "mlp3"), _WEIGHT_KEYS):
            arr = getattr(w, field)
            for i, k in enumerate(keys):
                arr[i] = lin(k)
        self.be.call("set_weights", self.h, ctypes.byref(w))
        self._have_weights = True
        self._reserved = max(getattr(self, "_reserved", 0), self.N * self.A)

    def reserve(self, n_states):
        """Setup-time: make room for value() batches of up to n_states states (ebc_value never allocates)."""
        if n_states > getattr(self, "_reserved", 0):
            self.be.call("reserve", self.h, ctypes.c_int64(int(n_states)))
            self._reserved = int(n_states)

    def set_value_mode(self, mode):
        """K4 arithmetic: 'fp32' (FFMA), 'tc_fp16x2' (tcgen05, two fp16 parts per operand, 3 MMAs per product,
        fp32-accurate, default when the network fits), 'tc_fp32' (tcgen05, three bf16 parts, 6 MMAs per product,
        fp32-accurate) or 'tc_bf16' (tcgen05, plain bf16 operands, fast, not argmax-exact)."""
        code = {"fp32": abi.VALUE_FP32, "tc_fp32": abi.VALUE_TC_FP32, "tc_bf16": abi.VALUE_TC_BF16,
                "tc_fp16x2": abi.VALUE_TC_FP16X2}[mode]
        rc = self.be.lib.ebc_set_value_mode(self.h, code)
        if rc != 0:
            raise abi.EbcError("ebc_set_value_mode: %s" % self.be.last_error(self.h))

    def value_mode(self):
        return {0: "fp32", 1: "tc_fp32", 2: "tc_bf16", 3: "tc_fp16x2"}[self.be.lib.ebc_get_value_mode(self.h)]

    # ---- scene upload -------------------------------------------------------------
    def load_episodes(self, first, hum_pv, hum_gr, hum_type, hum_count, stat=None, stat_count=None,
                      rect=None, rect_count=None, rob_pv=None, rob_gr=None, rob_theta=None, time=None,
                      obst=None, obst_count=None):
        """Copy host arrays (numpy, already padded to Hmax/Smax/Rmax) into episodes [first, first+k)."""
        k = len(hum_count)
        sl = slice(first, first + k)

        def put(dst, src, dtype):
            if src is None:
                return
            t = torch.as_tensor(np.ascontiguousarray(src), dtype=dtype)
            dst[sl].copy_(t.reshape(dst[sl].shape), non_blocking=False)

        put(self.hum_pv, hum_pv, torch.float32)
        put(self.hum_gr, hum_gr, torch.float32)
        put(self.hum_type, hum_type, torch.uint8)
        put(self.hum_count, hum_count, torch.int32)
        if self.Smax:
            put(self.stat, stat, torch.float32)
        put(self.stat_count, stat_count, torch.int32)
        if self.Rmax:
            put(self.rect, rect, torch.int16)
        put(self.rect_count, rect_count, torch.int32)
        put(self.rob_pv, rob_pv, torch.float32)
        put(self.rob_gr, rob_gr, torch.float32)
        put(self.rob_theta, rob_theta, torch.float32)
        put(self.time, time, torch.float64)
        if self.Omax and obst is not None:
            put(self.obst, np.ascontiguousarray(obst).view(np.uint8).reshape(k, -1, 48), torch.uint8)
            put(self.obst_count, obst_count, torch.int32)

    # ---- hot path -----------------------------------------------------------------
    def orca(self):
        self.be.call("orca", self.h, stream=self._stream())

    def robot_orca(self, safety_space, out=None):
        if out is None:
            out = torch.zeros(self.N, 2, dtype=torch.float64, device=self.device)
        self.be.call("robot_orca", self.h, ctypes.c_double(safety_space), _ptr(out), stream=self._stream())
        return out

    def lookahead(self, build_inputs=True):
        if build_inputs and self.vin is None:
            self.vin = torch.zeros(self.N, self.A, self.n, self.D, dtype=torch.float32, device=self.device)
        self.be.call("lookahead", self.h, _ptr(self.vin if build_inputs else None), _ptr(self.la_reward),
                     _ptr(self.la_done), _ptr(self.la_event), stream=self._stream())

    def value(self, vin=None, row_count=None, out=None, fused=False):
        """K4.  Default: the lookahead batch from `self.vin`.  `fused=True`: no materialised input at all -- the kernel
        builds the rotated rows itself from the bound state and the robot records the preceding
        `lookahead(build_inputs=False)` left (tensor-core modes; SURVEY 7 step 5).  `vin=...`: any batch of states."""
        if fused:
            self.be.call("value", self.h, None, ctypes.c_int64(self.N * self.A), None, _ptr(self.values), stream=self._stream())
            return self.values
        if vin is None:
            vin, out, n_states = self.vin, self.values, self.N * self.A
        else:
            n_states = vin.shape[0]
            if row_count is None:      # an explicit batch never borrows the bound episodes' counts
                row_count = torch.full((n_states,), self.n, dtype=torch.int32, device=self.device)
            if out is None:
                out = torch.zeros(n_states, dtype=torch.float32, device=self.device)
            self.reserve(n_states)
            if self.attention is not None:
                self.enable_attention(n_states)       # grow the borrowed array with the batch
        self.be.call("value", self.h, _ptr(vin), ctypes.c_int64(n_states), _ptr(row_count), _ptr(out),
                     stream=self._stream())
        return out

    def enable_attention(self, n_states=None):
        """Also keep the softmax attention weights of every state K4 evaluates (sarl.py:69-71,
        ValueNetwork.attention_weights): `self.attention` [n_states, n] float32 on the device, row i = state i of the
        last value() call (the lookahead batch: state e * A + a).  Off by default (one more n-float store per state)."""
        rows = int(n_states or self.N * self.A)
        if self.attention is None or self.attention.shape[0] < rows:
            self.attention = torch.zeros(rows, self.n, dtype=torch.float32, device=self.device)
            self.be.call("set_attention_output", self.h, _ptr(self.attention))
        return self.attention

    def select(self):
        self.be.call("select", self.h, _ptr(self.la_reward), _ptr(self.values), _ptr(self.action_values),
                     _ptr(self.argmax), _ptr(self.nan_flag), stream=self._stream())
        return self.argmax

    def decide(self, fused=None):
        """One robot decision for every episode (rl/policy/multi_human_rl.py:12-87, test phase).  With `fused` (default:
        `self.fused_input`) the value-network input is never written to memory: K3 leaves 48 bytes per (episode, action)
        and K4 builds its rows from the state (bit-identical values; `self.vin` is then not updated)."""
        fused = self.fused_input if fused is None else fused
        self.orca()
        if fused:
            self.lookahead(build_inputs=False)
            self.value(fused=True)
        else:
            self.lookahead()
            self.value()
        return self.select()

    def step(self, action_idx=None, action=None, active=None, fused_orca=False):
        """env.step(update=True).  `fused_orca`: run the human policies in the same launch
        (policy-free path); otherwise hum_nv from the preceding orca() is used."""
        name = "orca_step" if fused_orca else "step"
        self.be.call(name, self.h, _ptr(action_idx), _ptr(action), _ptr(active), _ptr(self.reward),
                     _ptr(self.done), _ptr(self.event), _ptr(self.dmin), _ptr(self.dist_to_goal),
                     stream=self._stream())

    def make_pool(self, scenes):
        """Upload pre-generated scenes (dict of numpy arrays in the ebc_state layout, any count P)
        as a device-resident pool for `reset`."""
        return ScenePool(self, scenes)

    def generate(self, shape, episode_ids, mask=None, seed=None):
        """env.reset with a scene generated on the device for the masked episodes (SURVEY 8f-1): `shape` is an
        ebc.synth.SceneShape, `episode_ids` an int64 device tensor of GLOBAL episode ids (the generator's key)."""
        from . import synth
        self.be.call("generate", self.h, ctypes.byref(shape.to_abi()), ctypes.c_uint64(synth.SEED_BASE if seed is None else seed),
                     _ptr(episode_ids), _ptr(mask), stream=self._stream())

    def replay_scenes(self, config, seeds, mask=None, poly_xy=None, poly_count=None, need=None):
        """env.reset with the REFERENCE's seeded scene for the masked episodes: generate_random_scene(scene_number =
        seeds[e]) replayed on the device (ebc_replay_scenes), `config` an abi.EbcReplayConfig (ebc.scene.replay_config),
        `seeds` an int32 device tensor holding the uint32 seeds' bits.  Returns device tensors poly_xy [N, Pmax, 4, 2]
        float64 (scene.obstacle_vertices), poly_count [N] int32 and need [N, 5] int32 (humans, static discs, grid
        rectangles and polygons the scene holds, then the adult count its rule left); a count above the capacity means
        the scene did not fit.  Pass the three outputs to keep the masked-off episodes' entries of earlier calls."""
        assert seeds.dtype == torch.int32 and seeds.shape == (self.N,) and seeds.device == self.device
        P = int(config.max_polys)
        z = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, device=self.device)  # noqa: E731
        poly_xy = z(self.N, max(P, 1), 4, 2, dtype=torch.float64) if poly_xy is None else poly_xy
        poly_count = z(self.N, dtype=torch.int32) if poly_count is None else poly_count
        need = z(self.N, 5, dtype=torch.int32) if need is None else need
        assert tuple(poly_xy.shape) == (self.N, max(P, 1), 4, 2) and poly_xy.dtype == torch.float64 and poly_xy.is_contiguous()
        assert tuple(need.shape) == (self.N, 5) and need.dtype == torch.int32 and need.is_contiguous()
        assert tuple(poly_count.shape) == (self.N,) and poly_count.dtype == torch.int32 and poly_count.is_contiguous()
        self.be.call("replay_scenes", self.h, ctypes.byref(config), _ptr(seeds), _ptr(mask), _ptr(poly_xy), _ptr(poly_count),
                     _ptr(need), stream=self._stream())
        return poly_xy, poly_count, need

    def build_obstacles(self, poly_xy, poly_count, mask=None):
        """RVO2's obstacle records of every masked episode from its polygons (ebc_build_obstacles, SURVEY 8f-4): what
        orca_obstacles.py's addObstacle + processObstacles make of scene.obstacle_vertices, written into obst /
        obst_count on the device.  `poly_xy` [N, Pmax, 4, 2] float64 and `poly_count` [N] int32 as replay_scenes
        returns them.  Returns need [N] int32 on the device: the records each episode needs, -1 where the kd-tree's
        edge splitting overflows Omax (obst_count is then 0); 0 for masked-off episodes."""
        assert poly_xy.dtype == torch.float64 and poly_xy.dim() == 4 and tuple(poly_xy.shape[2:]) == (4, 2)
        assert poly_xy.shape[0] == self.N and poly_xy.is_contiguous()
        assert poly_count.dtype == torch.int32 and tuple(poly_count.shape) == (self.N,) and poly_count.is_contiguous()
        need = torch.zeros(self.N, dtype=torch.int32, device=self.device)
        self.be.call("build_obstacles", self.h, _ptr(poly_xy), _ptr(poly_count), poly_xy.shape[1], _ptr(mask), _ptr(need),
                     stream=self._stream())
        return need

    def reset(self, pool, pool_index=None, mask=None):
        """env.reset for the masked episodes from a device scene pool (simulator/env.py:128-205)."""
        self.be.call("reset", self.h, ctypes.byref(pool.state), pool.size, _ptr(pool_index), _ptr(mask),
                     stream=self._stream())

    def transform(self, out=None):
        if out is None:
            out = torch.zeros(self.N, self.n, self.D, dtype=torch.float32, device=self.device)
        self.be.call("transform", self.h, _ptr(out), stream=self._stream())
        return out

    def local_map_angular(self, poly_xy, poly_count, max_range, min_angle, max_angle, dim, normalize=True, out=None):
        """Angular local map of every episode (simulator/env.py:570-628, SURVEY 8f-3): `poly_xy` [N, Pmax, 4, 2]
        float64 = scene.obstacle_vertices, `poly_count` [N] int32; returns [N, dim] float64 on the device."""
        assert poly_xy.dtype == torch.float64 and poly_xy.dim() == 4 and tuple(poly_xy.shape[2:]) == (4, 2)
        assert poly_xy.shape[0] == self.N and poly_count.dtype == torch.int32 and tuple(poly_count.shape) == (self.N,)
        assert poly_count.is_contiguous()
        if out is None:
            out = torch.empty(self.N, dim, dtype=torch.float64, device=self.device)
        assert out.dtype == torch.float64 and tuple(out.shape) == (self.N, dim) and out.is_contiguous()
        m = abi.EbcAngularMap(max_range, min_angle, max_angle, dim, 1 if normalize else 0, poly_xy.shape[1], 0)
        poly_xy = poly_xy.contiguous()      # held until the call returns: a temporary copy would be freed before it
        self.be.call("local_map_angular", self.h, ctypes.byref(m), _ptr(poly_xy), _ptr(poly_count),
                     _ptr(out), stream=self._stream())
        return out

    def local_map_grid(self, submap_size_m, out=None):
        """Binary grid sub-map of every episode (simulator/env.py:630-708, SURVEY 8f-3, [map] use_grid_map = true):
        the window of scene.map (the bound zero-cell rectangles) around the robot, rotated into its heading like
        cv2.warpAffine does and thresholded; returns [N, size, size] uint8 on the device."""
        size = int(round(submap_size_m / self.cfg.map_resolution))
        if out is None:
            out = torch.empty(self.N, size, size, dtype=torch.uint8, device=self.device)
        assert out.dtype == torch.uint8 and tuple(out.shape) == (self.N, size, size) and out.is_contiguous()
        m = abi.EbcGridMap(submap_size_m, size, 0)
        self.be.call("local_map_grid", self.h, ctypes.byref(m), _ptr(out), stream=self._stream())
        return out

    def launch_count(self):
        return self.be.launch_count(self.h)


class ScenePool(object):
    """P pre-generated scenes resident on the device, in the ebc_state layout of `sim`."""
    _FIELDS = (("hum_pv", torch.float32), ("hum_gr", torch.float32), ("hum_type", torch.uint8),
               ("hum_count", torch.int32), ("stat", torch.float32), ("stat_count", torch.int32),
               ("rect", torch.int16), ("rect_count", torch.int32), ("rob_pv", torch.float32),
               ("rob_gr", torch.float32), ("rob_theta", torch.float32), ("time", torch.float64),
               ("obst", torch.uint8), ("obst_count", torch.int32))

    def __init__(self, sim, scenes):
        self.size = int(len(scenes["hum_count"]))
        self.tensors = {}
        shapes = {"hum_pv": (sim.Hmax, 4), "hum_gr": (sim.Hmax, 4), "hum_type": (sim.Hmax,),
                  "stat": (max(sim.Smax, 1), 4), "rect": (max(sim.Rmax, 1), 4), "obst": (max(sim.Omax, 1), 48)}
        st = abi.EbcState()
        for name, dtype in self._FIELDS:
            src = scenes.get(name)
            if src is None:
                t = torch.zeros((self.size,) + shapes.get(name, ()), dtype=dtype)
            else:
                if name == "obst":
                    src = np.ascontiguousarray(src).view(np.uint8).reshape(self.size, -1, 48)
                t = torch.as_tensor(np.ascontiguousarray(src), dtype=dtype)
                if name in shapes:
                    assert tuple(t.shape[1:]) == shapes[name], (name, tuple(t.shape), shapes[name])
            t = t.to(sim.device).contiguous()
            self.tensors[name] = t
            setattr(st, name, t.data_ptr())
        self.nv = torch.zeros(self.size, sim.Hmax, 2, dtype=torch.float32, device=sim.device)
        st.hum_nv = self.nv.data_ptr()
        self.state = st
