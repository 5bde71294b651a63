// ebc_api.cu — the extern "C" entry points of include/ebcadrl.h (libebcadrl.so).
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <new>

#include "ebc_internal.cuh"

static char g_create_err[256] = "";

int ebc_fail(ebc_sim *s, int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(s ? s->err : g_create_err, 256, fmt, ap);
  va_end(ap);
  return code;
}

static int ebc_tc_index(int mode) { return mode == EBC_VALUE_TC_BF16 ? 0 : (mode == EBC_VALUE_TC_FP16X2 ? 1 : 2); }

int ebc_check_launch(ebc_sim *s, const char *what) {
  const cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return ebc_fail(s, EBC_ERR_CUDA, "%s: %s", what, cudaGetErrorString(err));
  s->launches += 1;
  return EBC_OK;
}

extern "C" {

int ebc_abi_version(void) { return EBC_ABI_VERSION; }

const char *ebc_last_error(const ebc_sim *s) { return s ? s->err : g_create_err; }

int ebc_create(const ebc_config *cfg, int device, ebc_sim **out) {
  if (!cfg || !out) return ebc_fail(nullptr, EBC_ERR_INVALID, "ebc_create: null argument");
  *out = nullptr;
  if (cfg->abi_version != EBC_ABI_VERSION)
    return ebc_fail(nullptr, EBC_ERR_INVALID, "ebc_create: abi_version %d != %d", cfg->abi_version, EBC_ABI_VERSION);
  if (cfg->n_episodes < 1 || cfg->max_humans < 1 || cfg->max_humans > 64 || cfg->max_statics < 0 ||
      cfg->max_humans + cfg->max_statics > 64 || cfg->max_rects < 0 || cfg->n_actions < 1 || cfg->n_actions > 256 ||
      cfg->orca_max_neighbors < 0 || cfg->orca_max_neighbors > 32 || cfg->max_obst < 0 || cfg->max_obst > 64 ||
      (cfg->orca_obstacles && !(cfg->orca_time_horizon_obst > 0.0f)) ||
      cfg->max_humans + (cfg->robot_visible ? 1 : 0) > 64)
    return ebc_fail(nullptr, EBC_ERR_INVALID,
                    "ebc_create: config out of range (1<=Hmax<=64, Hmax+Smax<=64, 1<=A<=256, max_neighbors<=32, Omax<=64)");
  if (!(cfg->time_step > 0.0) || !(cfg->map_resolution > 0.0))
    return ebc_fail(nullptr, EBC_ERR_INVALID, "ebc_create: time_step and map_resolution must be positive");
  int count = 0;
  cudaError_t err = cudaGetDeviceCount(&count);
  if (err != cudaSuccess || count < 1)
    return ebc_fail(nullptr, EBC_ERR_CUDA, "ebc_create: no CUDA device (%s); the hot path has no CPU fallback",
                    cudaGetErrorString(err));
  if (device < 0 || device >= count) return ebc_fail(nullptr, EBC_ERR_INVALID, "ebc_create: device %d of %d", device, count);
  if ((err = cudaSetDevice(device)) != cudaSuccess)
    return ebc_fail(nullptr, EBC_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(err));
  ebc_sim *s = new (std::nothrow) ebc_sim();
  if (!s) return ebc_fail(nullptr, EBC_ERR_NOMEM, "ebc_create: out of host memory");
  memset(s, 0, sizeof(*s));
  s->cfg = *cfg;
  s->device = device;
  cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, device);
  cudaDeviceGetAttribute(&s->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  if ((err = cudaMalloc(&s->d_actions, sizeof(double) * 2 * (size_t)cfg->n_actions)) != cudaSuccess) {
    delete s;
    return ebc_fail(nullptr, EBC_ERR_NOMEM, "cudaMalloc actions: %s", cudaGetErrorString(err));
  }
  *out = s;
  return EBC_OK;
}

void ebc_destroy(ebc_sim *s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->d_actions) cudaFree(s->d_actions);
  if (s->d_la_rec) cudaFree(s->d_la_rec);
  ebc_value_release(s);
  ebc_tc_release(s);
  delete s;
}

int ebc_bind(ebc_sim *s, const ebc_state *st) {
  if (!s || !st) return EBC_ERR_INVALID;
  if (!st->hum_pv || !st->hum_gr || !st->hum_type || !st->hum_count || !st->hum_nv || !st->stat_count ||
      !st->rect_count || !st->rob_pv || !st->rob_gr || !st->rob_theta || !st->time ||
      (s->cfg.max_statics > 0 && !st->stat) || (s->cfg.max_rects > 0 && !st->rect) ||
      (s->cfg.orca_obstacles && (!st->obst || !st->obst_count || s->cfg.max_obst < 1)))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_bind: null state array");
  if ((uintptr_t)st->obst & 15u) return ebc_fail(s, EBC_ERR_INVALID, "ebc_bind: obst must be 16-byte aligned");
  if (((uintptr_t)st->hum_pv | (uintptr_t)st->hum_gr | (uintptr_t)st->stat | (uintptr_t)st->rob_pv |
       (uintptr_t)st->rob_gr) & 15u)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_bind: float4 arrays must be 16-byte aligned");
  if (((uintptr_t)st->hum_nv | (uintptr_t)st->rect | (uintptr_t)st->time) & 7u)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_bind: hum_nv / rect / time must be 8-byte aligned");
  s->st = *st;
  s->bound = true;
  return EBC_OK;
}

int ebc_bind_stats(ebc_sim *s, const ebc_stats *x) {
  if (!s) return EBC_ERR_INVALID;
  if (!x) { memset(&s->stats, 0, sizeof(s->stats)); return EBC_OK; }
  if (!x->alive || !x->final_event || !x->steps || !x->too_close || !x->cum_reward || !x->discount || !x->min_dist_sum ||
      !x->alive_count)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_bind_stats: null statistics array");
  if (((uintptr_t)x->cum_reward | (uintptr_t)x->discount | (uintptr_t)x->min_dist_sum) & 7u)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_bind_stats: double arrays must be 8-byte aligned");
  s->stats = *x;
  return EBC_OK;
}

int ebc_set_actions(ebc_sim *s, const double *actions, int32_t n) {
  if (!s) return EBC_ERR_INVALID;
  if (!actions || n != s->cfg.n_actions) return ebc_fail(s, EBC_ERR_INVALID, "ebc_set_actions: expected %d actions", s->cfg.n_actions);
  cudaSetDevice(s->device);
  const cudaError_t err = cudaMemcpy(s->d_actions, actions, sizeof(double) * 2 * (size_t)n, cudaMemcpyHostToDevice);
  if (err != cudaSuccess) return ebc_fail(s, EBC_ERR_CUDA, "ebc_set_actions: %s", cudaGetErrorString(err));
  s->have_actions = true;
  return EBC_OK;
}

// scratch for the pooled per-state features of K4: [ceil(n/128)*128][ceil(jd/8)*8] floats (the tensor-core kernels keep
// it in 128-state tiles of 8-column chunks: both dimensions rounded up).  Grows monotonically; never called from ebc_value.
static int reserve_states(ebc_sim *s, int64_t n_states) {
  const int jd = s->net.self_dim + s->net.l[3].out;
  const size_t need = (size_t)((n_states + 127) / 128 * 128) * (size_t)((jd + 7) / 8 * 8);
  if (need > s->joint_floats) {
    cudaSetDevice(s->device);
    if (s->d_joint) cudaFree(s->d_joint);     // (synchronises: setup-time only)
    s->d_joint = nullptr;
    s->joint_floats = 0;
    s->joint_cap = 0;
    const cudaError_t err = cudaMalloc(&s->d_joint, need * sizeof(float));
    if (err != cudaSuccess) return ebc_fail(s, EBC_ERR_NOMEM, "cudaMalloc joint scratch: %s", cudaGetErrorString(err));
    s->joint_floats = need;
  }
  if (n_states > s->joint_cap) s->joint_cap = n_states;
  return EBC_OK;
}

int ebc_set_weights(ebc_sim *s, const ebc_weights *w) {
  if (!s || !w) return EBC_ERR_INVALID;
  cudaSetDevice(s->device);
  int rc = ebc_value_prepare(s, w);
  if (rc) return rc;
  // the lookahead batch (N * A states) is reserved here, at setup time: ebc_value itself never allocates
  const int64_t want = (int64_t)s->cfg.n_episodes * s->cfg.n_actions;
  const int64_t keep = s->joint_cap > want ? s->joint_cap : want;   // (the row width may have changed with the network)
  if ((rc = reserve_states(s, keep)) != 0) return rc;
  if (!s->d_la_rec) {      // 48 bytes per (episode, action): the robot part of the rotated rows (fused input path)
    const cudaError_t err = cudaMalloc(&s->d_la_rec, sizeof(float4) * 3 * (size_t)want);
    if (err != cudaSuccess) return ebc_fail(s, EBC_ERR_NOMEM, "cudaMalloc lookahead records: %s", cudaGetErrorString(err));
    s->la_rec_valid = 0;
  }
  // tensor-core programs: [0] bf16, [1] fp16x2 (default), [2] bf16x3
  const int r0 = ebc_tc_prepare(s, w, 0, 1), r1 = ebc_tc_prepare(s, w, 1, 2), r2 = ebc_tc_prepare(s, w, 2, 3);
  if (r0 < 0) return r0;
  if (r1 < 0) return r1;
  if (r2 < 0) return r2;
  if (r0 || r1 || r2) {
    // the shape misses the tensor-core tiling: the weights are accepted, K4 runs on the FFMA kernels, and the caller
    // is TOLD so (a positive status, never a silent downgrade)
    s->tc[0].ready = s->tc[1].ready = s->tc[2].ready = 0;
    s->value_mode = EBC_VALUE_FP32;
    ebc_fail(s, EBC_WARN_VALUE_FFMA, "ebc_set_weights: this network's shape does not fit the tensor-core tiling "
                                     "(layer widths <= 416 / 208, input <= 32, self state <= 8): value mode is EBC_VALUE_FP32");
    return EBC_WARN_VALUE_FFMA;
  }
  if (!s->value_mode_forced) s->value_mode = EBC_VALUE_TC_FP16X2;
  return EBC_OK;
}

int ebc_reserve(ebc_sim *s, int64_t n_states) {
  if (!s) return EBC_ERR_INVALID;
  if (!s->have_weights) return ebc_fail(s, EBC_ERR_UNBOUND, "ebc_reserve: weights not set (the row width is the network's)");
  if (n_states < 0) return ebc_fail(s, EBC_ERR_INVALID, "ebc_reserve: negative size");
  return reserve_states(s, n_states);
}

int ebc_set_value_mode(ebc_sim *s, int32_t mode) {
  if (!s) return EBC_ERR_INVALID;
  if (mode < EBC_VALUE_FP32 || mode > EBC_VALUE_TC_FP16X2) return ebc_fail(s, EBC_ERR_INVALID, "ebc_set_value_mode: unknown mode %d", mode);
  if (mode != EBC_VALUE_FP32 && s->have_weights && !s->tc[ebc_tc_index(mode)].ready)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_set_value_mode: this network's shape does not fit the tensor-core tiling");
  s->value_mode = mode;
  s->value_mode_forced = 1;
  return EBC_OK;
}

int ebc_get_value_mode(const ebc_sim *s) { return s ? s->value_mode : EBC_ERR_INVALID; }

#define REQUIRE_BOUND(name) \
  if (!s) return EBC_ERR_INVALID; \
  if (!s->bound) return ebc_fail(s, EBC_ERR_UNBOUND, name ": state not bound (call ebc_bind)")

int ebc_orca(ebc_sim *s, void *stream) {
  REQUIRE_BOUND("ebc_orca");
  return ebc_launch_orca(s, (cudaStream_t)stream);
}

int ebc_robot_orca(ebc_sim *s, double safety_space, double *out_action, void *stream) {
  REQUIRE_BOUND("ebc_robot_orca");
  if (!out_action) return ebc_fail(s, EBC_ERR_INVALID, "ebc_robot_orca: null output");
  return ebc_launch_robot_orca(s, safety_space, out_action, (cudaStream_t)stream);
}

int ebc_lookahead(ebc_sim *s, float *vin, double *reward, uint8_t *done, uint8_t *event, void *stream) {
  REQUIRE_BOUND("ebc_lookahead");
  if (!s->have_actions) return ebc_fail(s, EBC_ERR_UNBOUND, "ebc_lookahead: action table not set");
  return ebc_launch_lookahead(s, vin, reward, done, event, (cudaStream_t)stream);
}

int ebc_set_attention_output(ebc_sim *s, float *attn) {
  if (!s) return EBC_ERR_INVALID;
  s->attn_out = attn;
  return EBC_OK;
}

int ebc_value(ebc_sim *s, const float *vin, int64_t n_states, const int32_t *row_count, float *values, void *stream) {
  if (!s) return EBC_ERR_INVALID;
  if (!s->have_weights) return ebc_fail(s, EBC_ERR_UNBOUND, "ebc_value: weights not set");
  if (n_states < 0 || (n_states > 0 && !values)) return ebc_fail(s, EBC_ERR_INVALID, "ebc_value: bad argument");
  if (n_states == 0) return EBC_OK;      // an empty batch is valid and launches nothing
  if (!vin) {
    // fused input: K4 builds the rotated rows itself (bound state + the records of the last ebc_lookahead(vin = NULL))
    if (row_count || !s->bound || n_states != (int64_t)s->cfg.n_episodes * s->cfg.n_actions)
      return ebc_fail(s, EBC_ERR_INVALID, "ebc_value: vin == NULL is the lookahead batch (row_count NULL, n_states == n_episodes * n_actions)");
    if (s->value_mode == EBC_VALUE_FP32 || !s->tc[ebc_tc_index(s->value_mode)].ready)
      return ebc_fail(s, EBC_ERR_INVALID, "ebc_value: vin == NULL needs a tensor-core value mode (the FFMA cross-check reads vin)");
    if (!s->d_la_rec || !s->la_rec_valid)
      return ebc_fail(s, EBC_ERR_UNBOUND, "ebc_value: vin == NULL needs a preceding ebc_lookahead with vin == NULL on this state");
  }
  if (n_states > s->joint_cap)
    return ebc_fail(s, EBC_ERR_UNBOUND, "ebc_value: %lld states exceed the reserved %lld (call ebc_reserve at setup time; "
                                        "ebc_value never allocates)", (long long)n_states, (long long)s->joint_cap);
  if (!row_count) {
    // NULL = the lookahead batch: state i belongs to episode i / A and takes that episode's bound entity counts
    if (!s->bound) return ebc_fail(s, EBC_ERR_UNBOUND, "ebc_value: state not bound");
    if (n_states != (int64_t)s->cfg.n_episodes * s->cfg.n_actions)
      return ebc_fail(s, EBC_ERR_INVALID, "ebc_value: row_count == NULL needs n_states == n_episodes * n_actions (%lld), got %lld",
                      (long long)s->cfg.n_episodes * s->cfg.n_actions, (long long)n_states);
  }
  if (s->value_mode != EBC_VALUE_FP32 && s->tc[ebc_tc_index(s->value_mode)].ready)
    return ebc_launch_value_tc(s, s->value_mode, vin, n_states, row_count, values, (cudaStream_t)stream);
  return ebc_launch_value(s, vin, n_states, row_count, values, (cudaStream_t)stream);
}

int ebc_select(ebc_sim *s, const double *reward, const float *values, double *action_values, int32_t *argmax,
               uint8_t *nan_flag, void *stream) {
  REQUIRE_BOUND("ebc_select");
  if (!reward || !values || !argmax) return ebc_fail(s, EBC_ERR_INVALID, "ebc_select: null argument");
  return ebc_launch_select(s, reward, values, action_values, argmax, nan_flag, (cudaStream_t)stream);
}

static int step_common(ebc_sim *s, bool fused, const int32_t *action_idx, const double *action, const uint8_t *active,
                       double *reward, uint8_t *done, uint8_t *event, double *dmin, double *dist_to_goal, void *stream) {
  REQUIRE_BOUND("ebc_step");
  if ((action_idx == nullptr) == (action == nullptr))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_step: give exactly one of action_idx / action");
  if (action_idx && !s->have_actions) return ebc_fail(s, EBC_ERR_UNBOUND, "ebc_step: action table not set");
  return ebc_launch_step(s, fused, action_idx, action, active, reward, done, event, dmin, dist_to_goal,
                         (cudaStream_t)stream);
}

int ebc_step(ebc_sim *s, const int32_t *action_idx, const double *action, const uint8_t *active, double *reward,
             uint8_t *done, uint8_t *event, double *dmin, double *dist_to_goal, void *stream) {
  return step_common(s, false, action_idx, action, active, reward, done, event, dmin, dist_to_goal, stream);
}

int ebc_orca_step(ebc_sim *s, const int32_t *action_idx, const double *action, const uint8_t *active, double *reward,
                  uint8_t *done, uint8_t *event, double *dmin, double *dist_to_goal, void *stream) {
  return step_common(s, true, action_idx, action, active, reward, done, event, dmin, dist_to_goal, stream);
}

int ebc_transform(ebc_sim *s, float *out, void *stream) {
  REQUIRE_BOUND("ebc_transform");
  if (!out) return ebc_fail(s, EBC_ERR_INVALID, "ebc_transform: null output");
  return ebc_launch_transform(s, out, (cudaStream_t)stream);
}

int ebc_reset(ebc_sim *s, const ebc_state *pool, int32_t pool_size, const int32_t *pool_index, const uint8_t *mask,
              void *stream) {
  REQUIRE_BOUND("ebc_reset");
  if (!pool || pool_size < 1 || !pool->hum_pv || !pool->hum_gr || !pool->hum_type || !pool->hum_count ||
      !pool->stat_count || !pool->rect_count || !pool->rob_pv || !pool->rob_gr || !pool->rob_theta || !pool->time ||
      (s->cfg.max_statics > 0 && !pool->stat) || (s->cfg.max_rects > 0 && !pool->rect))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_reset: bad scene pool");
  return ebc_launch_reset(s, pool, pool_size, pool_index, mask, (cudaStream_t)stream);
}

int ebc_generate(ebc_sim *s, const ebc_scene_shape *shape, uint64_t seed, const int64_t *episode_ids, const uint8_t *mask,
                 void *stream) {
  REQUIRE_BOUND("ebc_generate");
  if (!shape || !episode_ids) return ebc_fail(s, EBC_ERR_INVALID, "ebc_generate: null shape or episode ids");
  if (shape->n_types < 1 || shape->n_types > 4 || shape->max_tries < 1 || shape->rule < 0 || shape->rule > 4)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_generate: bad shape");
  int humans = 0;
  for (int t = 0; t < shape->n_types; ++t) {
    if (shape->type_count[t] < 0) return ebc_fail(s, EBC_ERR_INVALID, "ebc_generate: negative group size");
    humans += shape->type_count[t];
  }
  if (shape->rule == 4 && (humans != 2 || shape->n_types != 1))     // scene_generator.py:583-589 ignores adult_num
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_generate: the one_static rule places exactly two agents of one type (got %d in %d groups)",
                    humans, shape->n_types);
  if (humans > s->cfg.max_humans || humans > 64)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_generate: %d humans do not fit (Hmax %d, generator limit 64)", humans, s->cfg.max_humans);
  if (shape->num_walls > s->cfg.max_rects || shape->num_walls * shape->discs_per_wall > s->cfg.max_statics)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_generate: %d walls x %d discs do not fit (Rmax %d, Smax %d)", shape->num_walls,
                    shape->discs_per_wall, s->cfg.max_rects, s->cfg.max_statics);
  return ebc_launch_generate(s, shape, seed, episode_ids, mask, (cudaStream_t)stream);
}

int ebc_replay_scenes(ebc_sim *s, const ebc_replay_config *c, const uint32_t *seeds, const uint8_t *mask, double *poly_xy,
                      int32_t *poly_count, int32_t *need, void *stream) {
  REQUIRE_BOUND("ebc_replay_scenes");
  if (!c || !seeds || !poly_count || !need || (c->max_polys > 0 && !poly_xy))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_replay_scenes: null config, seeds or output");
  for (int t = 0; t < 3; ++t)
    if (c->count[t] < 0 || c->count[t] > 64)
      return ebc_fail(s, EBC_ERR_INVALID, "ebc_replay_scenes: group %d holds %d agents (0..64)", t, c->count[t]);
  const int r0 = c->rule[0], r1 = c->rule[1], r2 = c->rule[2];
  if (r0 < EBC_REPLAY_SQUARE_CROSSING || r0 > EBC_REPLAY_ONE_STATIC ||     // scene_generator.py:589-591
      (c->count[1] > 0 && r1 != EBC_REPLAY_SQUARE_CROSSING && r1 != EBC_REPLAY_CIRCLE_CROSSING &&
       r1 != EBC_REPLAY_SQUARE_CROSSING_OLD) ||
      (c->count[2] > 0 && r2 != EBC_REPLAY_SQUARE_CROSSING))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_replay_scenes: rule (%d, %d, %d) does not exist for its list", r0, r1, r2);
  if (c->num_circles < 0 || c->num_walls < 0 || c->max_polys < 0 || c->min_wall_length > c->max_wall_length ||
      (c->num_walls > 0 && c->min_wall_length < 1))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_replay_scenes: bad obstacle counts or wall lengths");
  if (!(c->map_resolution > 0.0) || !(c->map_size_m > 0.0) || !(c->square_width >= 0.0) || !(c->circle_radius >= 0.0) ||
      !(c->robot_radius >= 0.0) || !(c->discomfort_dist >= 0.0))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_replay_scenes: sizes and distances must be non-negative, map size and resolution positive");
  const double grid = rint(c->map_size_m / c->map_resolution);
  if (c->num_circles + c->num_walls > 0 && !(grid >= 2.0 && grid <= 32767.0))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_replay_scenes: a map of %.0f cells has no room for obstacles (2..32767)", grid);
  if (c->randomize_attributes)          // agent.py:55: the drawn attributes must lie in (0, 20)
    for (int t = 0; t < 3; ++t)
      if (!(c->v_pref_min[t] > 0.0 && c->v_pref_max[t] < 20.0 && c->radius_min[t] > 0.0 && c->radius_max[t] < 20.0) &&
          c->count[t] > 0)
        return ebc_fail(s, EBC_ERR_INVALID, "ebc_replay_scenes: random attributes of group %d outside (0, 20)", t);
  return ebc_launch_replay(s, c, seeds, mask, poly_xy, poly_count, need, (cudaStream_t)stream);
}

int ebc_build_obstacles(ebc_sim *s, const double *poly_xy, const int32_t *poly_count, int32_t max_polys,
                        const uint8_t *mask, int32_t *need, void *stream) {
  REQUIRE_BOUND("ebc_build_obstacles");
  if (!s->cfg.orca_obstacles || s->cfg.max_obst < 1)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_build_obstacles: needs cfg.orca_obstacles and max_obst >= 1");
  if (!poly_count || !need || max_polys < 0 || (max_polys > 0 && !poly_xy))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_build_obstacles: null polygons or output, or max_polys < 0");
  return ebc_launch_build_obstacles(s, poly_xy, poly_count, max_polys, mask, need, (cudaStream_t)stream);
}

int ebc_local_map_angular(ebc_sim *s, const ebc_angular_map *map, const double *poly_xy, const int32_t *poly_count,
                          double *out, void *stream) {
  REQUIRE_BOUND("ebc_local_map_angular");
  if (!map || !poly_count || !out || map->dim < 1 || map->dim > 256 || map->max_polys < 0 ||
      (map->max_polys > 0 && !poly_xy) || !(map->max_angle > map->min_angle) || !(map->max_range > 0.0))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_local_map_angular: bad argument (1 <= dim <= 256, max_angle > min_angle, max_range > 0)");
  return ebc_launch_angular_map(s, map, poly_xy, poly_count, out, (cudaStream_t)stream);
}

int ebc_local_map_grid(ebc_sim *s, const ebc_grid_map *map, uint8_t *out, void *stream) {
  REQUIRE_BOUND("ebc_local_map_grid");
  const int G = (int)rint(s->cfg.map_size_m / s->cfg.map_resolution);           // scene_generator.py:310-311
  if (!map || !out || map->size < 1 || map->size > 192 || map->size > G ||
      map->size != (int)rint(map->submap_size_m / s->cfg.map_resolution))
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_local_map_grid: bad argument (size = round(submap_size_m / map_resolution), 1..192, <= map cells)");
  return ebc_launch_grid_map(s, map, out, (cudaStream_t)stream);
}

int ebc_debug_trace(ebc_sim *s, long long *out, int32_t n) {
  if (!s || !out || n < 1) return EBC_ERR_INVALID;
  if (!s->d_trace) return ebc_fail(s, EBC_ERR_UNBOUND, "ebc_debug_trace: run ebc_value with EBC_TC_TRACE=1 first");
  cudaDeviceSynchronize();
  const cudaError_t err = cudaMemcpy(out, s->d_trace, sizeof(long long) * (size_t)(n < 4096 ? n : 4096), cudaMemcpyDeviceToHost);
  return err == cudaSuccess ? EBC_OK : ebc_fail(s, EBC_ERR_CUDA, "ebc_debug_trace: %s", cudaGetErrorString(err));
}

int64_t ebc_launch_count(const ebc_sim *s) { return s ? s->launches : 0; }

}  // extern "C"
