/*
 * ebcadrl.h — C ABI of the B200-native batched crowd-navigation hot path.
 *
 * This is the drop-in boundary for ONE path of kolomeytsev/EB-CADRL: the
 * `simulator/env.py` reset/step/onestep_lookahead loop with ORCA humans and the
 * SARL / EB-CADRL one-step lookahead + value network.  Plain pointers and sizes
 * only: no C++ types, no torch types, no exceptions cross this line.
 *
 * Two implementations export (almost) the same entry points:
 *   - libebcadrl.so  (eb-cadrl_b200/csrc, CUDA sm_100a): `ebc_*`, DEVICE pointers.
 *   - libebc_oracle.so (oracle/, plain C, TEST INFRASTRUCTURE ONLY): `ebc_ref_*`,
 *     HOST pointers, same structs, same semantics.  The product never loads it.
 *
 * Every entry point cites the reference code it replaces (paths relative to the
 * reference repository root).
 *
 * Conventions
 *   N      episodes advanced at once (this rank's shard)
 *   Hmax   human slots per episode; humans are stored adults, then bicycles,
 *          then children (the reference's list order, simulator/env.py:392)
 *   Smax   static-disc slots (walls seen by the robot as ADULT_STATIC discs,
 *          simulator/scene/scene_generator.py:380-422)
 *   Rmax   zero-cell rectangles of the occupancy grid (simulator/env.py:227-261
 *          tests a window of scene.map; the grid is a union of rectangles written
 *          by scene_generator.py:888-922)
 *   A      discrete robot actions (rl/policy/cadrl.py:91-116), index 0 = stop
 *   n      entity rows per lookahead state = Hmax + Smax (rows past an episode's
 *          own count are zero-filled and masked)
 *   D      rotated row width: 13, or 17 with the 4-class entity-type one-hot
 *          (rl/policy/cadrl.py:236-337)
 * All calls are asynchronous on the given stream; no hidden synchronisation.
 * Return value: 0 on success, negative `ebc_status` on failure, positive `EBC_WARN_*` when the
 * call succeeded with a documented downgrade; the message is in `ebc_last_error`.
 */
#ifndef EBCADRL_H
#define EBCADRL_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EBC_ABI_VERSION 2

/* simulator/utils/utils.py:9-14 (AgentType IntEnum) */
enum { EBC_ADULT = 0, EBC_BICYCLE = 1, EBC_CHILD = 2, EBC_ADULT_STATIC = 3, EBC_ROBOT = 4 };

/* Event codes = the Info subclass returned by Reward.compute
 * (simulator/utils/reward.py:103-179, simulator/utils/info.py). */
enum {
  EBC_EV_NOTHING = 0,
  EBC_EV_DANGER = 1,
  EBC_EV_REACH_GOAL = 2,
  EBC_EV_COLLISION_ADULT = 3,
  EBC_EV_COLLISION_BICYCLE = 4,
  EBC_EV_COLLISION_CHILD = 5,
  EBC_EV_COLLISION_OBSTACLE = 6,
  EBC_EV_TIMEOUT = 7
};

enum { EBC_KIN_HOLONOMIC = 0, EBC_KIN_UNICYCLE = 1 };   /* agent.py:164-188: any non-"holonomic" string */
enum { EBC_POLICY_ORCA = 0, EBC_POLICY_LINEAR = 1 };    /* simulator/policy/policy_factory.py:10-14 */

typedef enum ebc_status {
  EBC_OK = 0,
  EBC_ERR_INVALID = -1,   /* bad argument / config */
  EBC_ERR_UNBOUND = -2,   /* ebc_bind / ebc_set_actions / ebc_set_weights not called */
  EBC_ERR_CUDA = -3,      /* CUDA runtime error (message has the cudaError string) */
  EBC_ERR_NOMEM = -4,
  /* positive = accepted, with a note in ebc_last_error */
  EBC_WARN_VALUE_FFMA = 1 /* ebc_set_weights: the network's shape misses the tensor-core tiling; K4 runs on the
                             fp32 FFMA kernels (ebc_get_value_mode() == EBC_VALUE_FP32) */
} ebc_status;

/* Per-simulator constants: the env INI ([env] [reward] [map] [robot]) and the
 * policy INI ([rl] [action_space] [sarl]) boiled down to a POD.
 * simulator/env.py:58-87, simulator/utils/reward.py:18-75, rl/policy/cadrl.py:73-82,
 * rl/policy/sarl.py:90-128, simulator/policy/orca.py:57-69. */
typedef struct ebc_config {
  int32_t abi_version;       /* EBC_ABI_VERSION */
  int32_t n_episodes;        /* N */
  int32_t max_humans;        /* Hmax (1..64) */
  int32_t max_statics;       /* Smax (0..64); Hmax + Smax <= 64 */
  int32_t max_rects;         /* Rmax (>=0) */
  int32_t n_actions;         /* A (1..256) */
  int32_t robot_kinematics;  /* EBC_KIN_*: how env/agent code moves the robot */
  int32_t rotate_theta;      /* 1 iff policy kinematics == "unicycle" exactly (cadrl.py:261-265) */
  int32_t with_agent_type;   /* 1: D = 17 (sarl.py:100-108), 0: D = 13 */
  int32_t robot_visible;     /* [robot] visible: humans' ORCA sees the robot (env.py:401-402) */
  int32_t human_policy[3];   /* EBC_POLICY_* for adults, bicycles, children */
  int32_t new_reward;        /* reward.py:19 */
  int32_t has_max_goal_distance; /* reward.py:21-23 (None when absent) */
  int32_t orca_max_neighbors;    /* orca.py:65 (10) */
  double time_step;          /* [env] time_step */
  double time_limit;         /* [env] time_limit (getint in the reference) */
  double time_max, time_good, max_goal_distance, success_reward;
  double collision_penalty_adult, collision_penalty_bicycle;
  double collision_penalty_obstacle, collision_penalty_child;
  double discomfort_dist_adult, discomfort_dist_bicycle, discomfort_dist_child;
  double discomfort_penalty_factor_adult, discomfort_penalty_factor_bicycle;
  double discomfort_penalty_factor_child;
  double rotation_penalty_factor;
  double map_size_m, map_resolution; /* [map] */
  double gamma;                      /* [rl] gamma */
  double orca_safety_space;          /* orca.py:63 (0; IL robot uses 0.15, train.py:126-132) */
  float orca_neighbor_dist;          /* orca.py:64 (10) */
  float orca_time_horizon;           /* orca.py:66 (5) */
  /* ORCA obstacle half-planes (SURVEY 8f-4; spec: RVO2 computeNewVelocity obstacle section, caller
   * simulator/policy/orca_obstacles.py:83-152).  OFF by default = the reference's live behaviour: humans never see
   * walls (orca.py adds no obstacle to its rvo2 sims).  Turned on by this project's env INI key
   * [sim] orca_obstacles = true; the records come from ebc_build_obstacles (the replayed scenes' polygons, on the
   * device) or ebc_pack_obstacles (host). */
  int32_t orca_obstacles;            /* 1: humans (and the ORCA robot) avoid the episode's obstacle polygons */
  int32_t max_obst;                  /* Omax: obstacle-vertex slots per episode (0..64) */
  float orca_time_horizon_obst;      /* orca_obstacles.py:65 (5) */
  float reserved0;
} ebc_config;

/* Structure-of-arrays episode state.  The library BORROWS these arrays (owned by
 * the caller, e.g. torch tensors); it never frees them.  fp32 state, float4-packed
 * per agent so that one warp lane loads one agent with one 16-byte load.
 * Layout follows simulator/utils/state.py:1-92 (FullState / ObservableState).
 * Slots past an episode's hum_count / stat_count / rect_count are neither read nor written by ebc_orca, ebc_robot_orca,
 * ebc_lookahead, ebc_value, ebc_select, ebc_step, ebc_orca_step, ebc_transform or ebc_local_map_grid: the caller may
 * leave anything there (ebc_reset and ebc_generate write whole episodes). */
/* One RVO2 obstacle vertex (Obstacle.h: point_, unitDir_, nextObstacle_, prevObstacle_, isConvex_) plus this vertex's
 * place in RVO2's obstacle kd-tree (KdTree::buildObstacleTreeRecursive: one node per vertex, edges that straddle a
 * splitting line are split), from which every agent derives the tree's near-first visiting order for distance ties.
 * Produced by ebc_build_obstacles on the device or ebc_pack_obstacles on the host (the same function). */
typedef struct ebc_obst_vertex {
  float px, py;         /* point_ */
  float ux, uy;         /* unitDir_ = normalize(next.point_ - point_) */
  int16_t next, prev;   /* vertex indices within the episode */
  int16_t convex;       /* isConvex_ */
  int16_t pad0;
  uint64_t anc;         /* kd-tree ancestors of this node (bit j = vertex j) */
  uint64_t anc_left;    /* the ancestors whose LEFT subtree holds this node */
  uint64_t pad1;
} ebc_obst_vertex;      /* 48 bytes */

typedef struct ebc_state {
  float *hum_pv;        /* [N*Hmax*4]  px, py, vx, vy */
  float *hum_gr;        /* [N*Hmax*4]  gx, gy, v_pref, radius */
  uint8_t *hum_type;    /* [N*Hmax]    EBC_ADULT / EBC_BICYCLE / EBC_CHILD, sorted ascending */
  int32_t *hum_count;   /* [N]         humans in the episode (<= Hmax) */
  float *hum_nv;        /* [N*Hmax*2]  human action of the current step (ORCA output), written by ebc_orca */
  float *stat;          /* [N*Smax*4]  px, py, radius, 0  (static discs, robot-only observation) */
  int32_t *stat_count;  /* [N] */
  int16_t *rect;        /* [N*Rmax*4]  x0, y0, x1, y1: half-open zero-cell rectangle of scene.map */
  int32_t *rect_count;  /* [N] */
  float *rob_pv;        /* [N*4]       px, py, vx, vy */
  float *rob_gr;        /* [N*4]       gx, gy, v_pref, radius */
  float *rob_theta;     /* [N] */
  double *time;         /* [N]         env.global_time */
  ebc_obst_vertex *obst;/* [N*Omax]    obstacle vertices (may be NULL unless cfg.orca_obstacles) */
  int32_t *obst_count;  /* [N] */
} ebc_state;

/* SARL / EB-CADRL value network (rl/policy/sarl.py:9-82).  HOST pointers to the
 * state_dict tensors, PyTorch nn.Linear layout: weight [out][in] row-major, bias [out].
 * Keys: mlp1.{0,2}, mlp2.{0,2}, attention.{0,2,4}, mlp3.{0,2,4,6}.
 * The library copies (and re-lays-out) them; the caller may free them afterwards. */
typedef struct ebc_linear {
  const float *weight;
  const float *bias;
  int32_t in_dim, out_dim;
} ebc_linear;

typedef struct ebc_weights {
  int32_t input_dim;        /* D */
  int32_t self_state_dim;   /* 6 (cadrl.py:55) */
  int32_t with_global_state;/* sarl.py:28-32 */
  ebc_linear mlp1[2];
  ebc_linear mlp2[2];
  ebc_linear attention[3];
  ebc_linear mlp3[4];
} ebc_weights;

typedef struct ebc_sim ebc_sim;   /* opaque */

/* ---- lifetime -------------------------------------------------------------------- */
int ebc_create(const ebc_config *cfg, int device, ebc_sim **out);
void ebc_destroy(ebc_sim *sim);
const char *ebc_last_error(const ebc_sim *sim);   /* sim may be NULL: last create error */
int ebc_abi_version(void);

/* Borrow the caller's device arrays. */
int ebc_bind(ebc_sim *sim, const ebc_state *state);

/* Per-episode running statistics of the explorer's inner loop (rl/utils/explorer.py:33-94,189-193;
 * rl/test_parallel.py:52-130), kept ON THE DEVICE: device arrays of N entries owned by the caller.  While bound,
 * every committed step (ebc_step / ebc_orca_step) of an episode e that is stepped
 *   cum_reward[e] += discount[e] * reward;  discount[e] *= gamma^(time_step * v_pref_robot);  steps[e] += 1;
 *   event == Danger: too_close[e] += 1, min_dist_sum[e] += Danger.min_dist (reward.py:138-166);
 *   done: final_event[e] = event, alive[e] = 0, alive_count[0] -= 1.
 * With `active == NULL` in ebc_step the bound alive[] is the mask, so a whole batch runs to the end of every episode
 * without a host round trip per step (the host reads alive_count[0] when it wants to). */
typedef struct ebc_stats {
  uint8_t *alive;        /* [N] in/out */
  uint8_t *final_event;  /* [N] */
  int32_t *steps;        /* [N] */
  int32_t *too_close;    /* [N] */
  double *cum_reward;    /* [N] */
  double *discount;      /* [N] initialise to 1 */
  double *min_dist_sum;  /* [N] */
  int32_t *alive_count;  /* [1] initialise to the number of alive episodes */
} ebc_stats;
int ebc_bind_stats(ebc_sim *sim, const ebc_stats *stats);   /* NULL unbinds */

/* RVO2 addObstacle (per polygon, counter-clockwise) + processObstacles for ONE episode, on the HOST: `xy` holds the
 * polygons' vertices back to back (x, y pairs, float like the rvo2 boundary), poly_size[i] vertices each (>= 2).
 * Writes at most `cap` (<= 64) records and their number; EBC_ERR_INVALID when the kd-tree's edge splitting needs more.
 * No handle, no device: the result is plain data for state.obst (simulator/policy/orca_obstacles.py:102-107). */
int ebc_pack_obstacles(const float *xy, const int32_t *poly_size, int32_t n_poly, ebc_obst_vertex *out, int32_t cap,
                       int32_t *n_out);

/* Action table, HOST pointer, A x 2 doubles: (vx, vy) for a holonomic robot, (v, r)
 * otherwise; built on the host exactly like rl/policy/cadrl.py:91-116. */
int ebc_set_actions(ebc_sim *sim, const double *actions, int32_t n_actions);

/* Copies and re-lays-out the weights (setup-time call: allocates and synchronises), and reserves K4's scratch
 * for the lookahead batch of n_episodes * n_actions states.  Returns EBC_WARN_VALUE_FFMA (> 0) when the shape does
 * not fit the tensor-core tiling -- the weights are in place, K4 then runs in EBC_VALUE_FP32. */
int ebc_set_weights(ebc_sim *sim, const ebc_weights *w);

/* Reserve K4's private scratch for ebc_value calls of up to n_states states (setup-time call: may allocate and
 * synchronise).  ebc_value itself never allocates: a larger batch than reserved fails with EBC_ERR_UNBOUND. */
int ebc_reserve(ebc_sim *sim, int64_t n_states);

/* Arithmetic of K4 (the value network).  All four are this library's own kernels.
 *   EBC_VALUE_FP32      fp32 FFMA (CUDA cores): the first parity path, kept as a cross-check
 *   EBC_VALUE_TC_FP16X2 tcgen05 tensor cores, every fp32 operand split into two fp16 parts (22 mantissa
 *                       bits; absolute floor 2^-25 per operand) and three MMAs per product (hi*hi + lo*hi +
 *                       hi*lo) into one fp32 TMEM accumulator: fp32-accurate (what argmax parity needs),
 *                       DEFAULT when the network's shape fits the tensor-core tiling.  An activation
 *                       beyond the fp16 range (65504) turns the value into NaN, which ebc_select flags
 *   EBC_VALUE_TC_FP32   same with three bf16 parts (24 bits, fp32 range) and six MMAs per product
 *   EBC_VALUE_TC_BF16   tcgen05, plain bf16 operands, fp32 accumulation: fast mode, NOT argmax-exact
 *                       (rl/policy/sarl.py:38-82 evaluated with bf16 inputs; agreement rate is reported) */
enum { EBC_VALUE_FP32 = 0, EBC_VALUE_TC_FP32 = 1, EBC_VALUE_TC_BF16 = 2, EBC_VALUE_TC_FP16X2 = 3 };
int ebc_set_value_mode(ebc_sim *sim, int32_t mode);
int ebc_get_value_mode(const ebc_sim *sim);

/* ---- the hot path ---------------------------------------------------------------- */

/* K1. Human policy step: state.hum_nv[e,h] <- policy_h(current state).
 * Replaces the per-human loop of simulator/env.py:392-405 -> agents.py:13-30 ->
 * simulator/policy/orca.py:85-157 -> rvo2 PyRVOSimulator.doStep (agent 0 only), and
 * simulator/policy/linear.py:17-23 for `linear` humans. */
int ebc_orca(ebc_sim *sim, void *stream);

/* Robot driven by ORCA (imitation learning, rl/train.py:99-143; reset() returns
 * obstacle_vertices for it, env.py:201-204): robot = agent 0, neighbours = humans then
 * static discs.  out_action: [N*2] doubles (vx, vy). */
int ebc_robot_orca(ebc_sim *sim, double safety_space, double *out_action, void *stream);

/* K3. One-step lookahead for every (episode, action): env.onestep_lookahead
 * (simulator/env.py:207-209 -> step(update=False) :388-466), i.e. collisions
 * (env.py:303-338, utils/collisions.py:4-57, obstacle grid env.py:227-261), reward /
 * done / event (utils/reward.py:80-181), next human states (agent.py:80-93), robot
 * propagate (rl/policy/cadrl.py:118-165) and the rotated joint state
 * (rl/policy/multi_human_rl.py:52-61 + cadrl.py:236-337).  Requires ebc_orca first.
 *   vin    [N*A*n*D] fp32 value-network input, or NULL: the rows are not materialised -- the kernel leaves the robot
 *          part of every (episode, action)'s rows (48 bytes) in the handle's scratch, from which ebc_value(vin = NULL)
 *          builds them itself (SURVEY 7 step 5: the n x D input never touches HBM)
 *   reward [N*A] f64, done [N*A] u8, event [N*A] u8  (any may be NULL) */
int ebc_lookahead(ebc_sim *sim, float *vin, double *reward, uint8_t *done, uint8_t *event,
                  void *stream);

/* K4. Value network forward (rl/policy/sarl.py:38-82) over `n_states` states of n rows
 * each; row_count[s] (<= n) rows are real, the rest are padding (excluded from the
 * mean and the softmax).  vin [n_states*n*D] -> values [n_states].
 * row_count == NULL selects the lookahead batch: n_states must then equal N*A, state i belongs to
 * episode i / A and takes that episode's bound hum_count + stat_count (anything else is EBC_ERR_INVALID).
 * For any other batch (replay samples, target-network evaluation) pass row_count explicitly.
 * n_states must not exceed what ebc_set_weights / ebc_reserve reserved (this call never allocates).
 * n_states == 0 is valid and launches nothing (pointers may then be NULL).
 * vin == NULL (with row_count == NULL, n_states == N*A, a tensor-core value mode) is the FUSED input path: the kernel
 * computes every rotated joint-state row (cadrl.py:236-337) from the bound state and the records of the preceding
 * ebc_lookahead(vin = NULL) on the same state -- bit-identical values, no N*A*n*D buffer.  EBC_ERR_UNBOUND if no such
 * lookahead preceded (or the state has been stepped / reset since), EBC_ERR_INVALID in the FFMA mode. */
int ebc_value(ebc_sim *sim, const float *vin, int64_t n_states, const int32_t *row_count,
              float *values, void *stream);

/* ValueNetwork.attention_weights / SARL.get_attention_weights (rl/policy/sarl.py:36,69-71,130-131): the softmax
 * weights the network pools the entities with.  With a device array set here, every later ebc_value call also stores
 * attn[i * n + r] = the weight of entity row r of state i (0 for rows past the state's row count; NaN like the
 * reference when every score of the state is exactly 0).  The reference keeps the weights of its LAST forward, which
 * in the lookahead is the last action's state: row (e * A + A - 1) of the batch.  NULL (the default) turns the
 * output off.  The pointer is borrowed; it must hold n floats for every state of the largest ebc_value call. */
int ebc_set_attention_output(ebc_sim *sim, float *attn);

/* K5. Action selection (rl/policy/multi_human_rl.py:25-26,72-80):
 * action_values[e,a] = reward[e,a] + gamma^(time_step*v_pref) * values[e,a] (float64),
 * argmax[e] = first maximum (strict '>'), or 0 (the stop action) when the robot is
 * already within `radius` of its goal (policy.py:43-54).  nan_flag[e] = 1 when no action
 * compares greater than -inf ("Value network is not well trained.", :81-82). */
int ebc_select(ebc_sim *sim, const double *reward, const float *values, double *action_values,
               int32_t *argmax, uint8_t *nan_flag, void *stream);

/* K2. Committed step: env.step(action, update=True) (simulator/env.py:388-466 with
 * compute_step_update :340-386 and agent.py:202-228).  Uses state.hum_nv from ebc_orca.
 * Exactly one of action_idx [N] (index into the action table) / action [N*2] f64 is given.
 * Episodes with active[e] == 0 are left untouched (active may be NULL = all).
 * Outputs (any may be NULL): reward [N] f64, done [N] u8, event [N] u8,
 * dmin [N*3] f64 (adult, bicycle, child; +inf when none), dist_to_goal [N] f64. */
int ebc_step(ebc_sim *sim, const int32_t *action_idx, const double *action, const uint8_t *active,
             double *reward, uint8_t *done, uint8_t *event, double *dmin, double *dist_to_goal,
             void *stream);

/* Convenience for the policy-free path (robot action given, e.g. the `linear` robot of
 * tests/test_collisions_simulation.py): ebc_orca + ebc_step in one call -- K1 for the episodes the step will touch,
 * then K2, on the same stream (with ORCA obstacle half-planes: one block-per-episode launch that stages the
 * episode's obstacle vertices in shared memory once for both). */
int ebc_orca_step(ebc_sim *sim, const int32_t *action_idx, const double *action,
                  const uint8_t *active, double *reward, uint8_t *done, uint8_t *event,
                  double *dmin, double *dist_to_goal, void *stream);

/* Rotated CURRENT joint state for the replay memory
 * (rl/policy/multi_human_rl.py:128-149): out [N*n*D]. */
int ebc_transform(ebc_sim *sim, float *out, void *stream);

/* Device-side env.reset (simulator/env.py:128-205) from a pool of pre-generated scenes:
 * for every episode e with mask[e] != 0 (mask NULL = all), copy scene pool_index[e]
 * (pool_index NULL = e) of `pool` -- an ebc_state of `pool_size` episodes with the same
 * Hmax / Smax / Rmax, device arrays -- into the bound state: robot at its start with v = 0,
 * global_time = 0 (whatever the pool holds), hum_nv cleared. */
int ebc_reset(ebc_sim *sim, const ebc_state *pool, int32_t pool_size, const int32_t *pool_index,
              const uint8_t *mask, void *stream);

/* Shape of a generated scene: the distribution of simulator/scene/scene_generator.py (square_crossing
 * :672-712, circle_crossing :593-618, walls :205-290, static discs :380-422, grid rectangles :888-922)
 * driven by a counter-based generator -- every draw is splitmix64(seed, global episode id, stream, draw),
 * so an episode's scene does not depend on the batch or on how episodes are sharded over ranks.  It does
 * NOT replay numpy's MT19937 stream (that is the host parity path of the Python mirror). */
typedef struct ebc_scene_shape {
  int32_t n_types;            /* human groups, in list order (adults, bicycles, children) */
  int32_t type_code[4];       /* EBC_TYPE_* of each group */
  int32_t type_count[4];
  double v_pref_lo[4], v_pref_hi[4], radius_lo[4], radius_hi[4];
  int32_t rule;               /* 0 square_crossing, 1 circle_crossing, 2 mixed (first half circle: the dynamic part of
                                 mixed_20), 3 mixed_20 (scene_generator.py:577-582: randint(20) static adults in a
                                 6 x 8 box, the first at (-0.5, -2.5), then the dynamic mix), 4 one_static
                                 (scene_generator.py:583-589: exactly two agents standing at (-2, -8) and (-3, -8)) */
  int32_t num_walls;
  int32_t wall_len_lo, wall_len_hi;   /* metres, inclusive */
  int32_t discs_per_wall;     /* static discs a wall of wall_len_hi decomposes into */
  int32_t max_tries;          /* rejection-sampling attempts per placement; the last one is accepted */
  double square_width, circle_radius, robot_radius, robot_v_pref;
  double map_size_m, map_resolution, discomfort_dist;
} ebc_scene_shape;

/* env.reset with a freshly generated scene (simulator/env.py:128-205 + scene_generator.py) for the episodes
 * e with mask[e] != 0 (mask NULL = all): episode_ids[e] (device, int64, the GLOBAL episode id that keys the
 * generator) -> humans with rejection sampling against the robot start and same-type agents, walls with
 * start / goal exclusion, their grid rectangles and static discs, robot at (0, -R) -> (0, R), time = 0. */
int ebc_generate(ebc_sim *sim, const ebc_scene_shape *shape, uint64_t seed, const int64_t *episode_ids,
                 const uint8_t *mask, void *stream);

/* The reference's OWN seeded scenes on the device: generate_random_scene(scene_number = seed)
 * (simulator/scene/scene_generator.py:330-378) replayed for every episode e with mask[e] != 0 (mask NULL = all), one
 * thread per episode.  np.random.seed(seeds[e]) (:362) seeds numpy's legacy MT19937 (init_genrand), and every draw
 * follows in the reference's order, rejected tries included: adults by their rule (:503-591; square_crossing :672-712,
 * circle_crossing :593-618, mixed :523-577, mixed_20 :492-501,578-582, one_static :583-589), then bicycles
 * (square_crossing_old :714-761), then children, then circles and walls (:292-328).  Agent attributes are drawn
 * (v_pref, then radius, simulator/agents/agent.py:49-56) when randomize_attributes is set.  The arithmetic is the
 * reference's float64 sequence, narrowed to fp32 at the store.  The one operation not bit-for-bit the host's is
 * circle_crossing's double cos / sin: CUDA's and the host libm's need not round alike.  On the tested seeds they always
 * agreed, but a last-bit difference is not bounded in its effect: it feeds the following too_close tests, can flip an
 * accept / reject decision, and then changes every later draw of that scene.
 * Writes what BatchedEnv.reset_batch loads: humans (adults, bicycles, children, at rest; hum_nv cleared), the static
 * discs (:380-422), the grid's zero cells (:888-922) as rectangles -- an obstacle strictly inside the map is one
 * rectangle; one on the border, where the per-cell path writes the product of two per-axis cell sets (every other cell
 * along an axis of odd size: Python's half-to-even rounding), is one rectangle per pair of per-axis runs --, the robot
 * at (0, -R) -> (0, R) at rest facing +y, time = 0.  Slots past the scene's counts are zeroed; nothing is written past
 * Hmax / Smax / Rmax / max_polys.
 *   poly_xy    [N*max_polys*4*2] f64 (device): scene.obstacle_vertices, circles then walls, 4 vertices each
 *   poly_count [N] i32 (device)
 *   need       [N*5] i32 (device): humans, static discs, rectangles and polygons the scene holds (a count above the
 *              capacity means the scene did not fit), then the adult count: for the mixed rules the one they draw and leave
 *              in SceneGenerator.adult_num (:537,580), otherwise the adult list's configured size
 *   seeds      [N] u32 (device) */
enum {
  EBC_REPLAY_SQUARE_CROSSING = 0,      /* adults, bicycles, children */
  EBC_REPLAY_CIRCLE_CROSSING = 1,      /* adults, bicycles */
  EBC_REPLAY_MIXED = 2,                /* adults */
  EBC_REPLAY_MIXED_20 = 3,             /* adults */
  EBC_REPLAY_ONE_STATIC = 4,           /* adults */
  EBC_REPLAY_SQUARE_CROSSING_OLD = 5   /* bicycles */
};
typedef struct ebc_replay_config {     /* one phase of SceneGenerator (scene_generator.py:26-66) */
  int32_t count[3];                    /* adults, bicycles, children (1 each in train / val without multiagent_training) */
  int32_t rule[3];                     /* EBC_REPLAY_* of each list (the phase's train_val_sim_* or test_sim_*) */
  int32_t randomize_attributes;        /* [env] randomize_attributes */
  int32_t num_circles, num_walls;      /* [map] */
  int32_t min_wall_length, max_wall_length;
  int32_t max_polys;                   /* Pmax: polygon slots per episode in poly_xy */
  int32_t norm_fused;                  /* 1: numpy.linalg.norm((x, y)) of the numpy being matched is
                                          sqrt(fma(y, y, x * x)) (OpenBLAS ddot on FMA-capable x86 cores);
                                          0: sqrt(x * x + y * y) */
  int32_t reserved;
  double v_pref[3], radius[3];         /* [adults] [bicycles] [children] v_pref / radius (used unless drawn) */
  double v_pref_min[3], v_pref_max[3], radius_min[3], radius_max[3];
  double square_width, circle_radius;  /* [sim] */
  double discomfort_dist;              /* [reward] discomfort_dist */
  double robot_radius, robot_v_pref;   /* [robot] */
  double map_size_m, map_resolution;   /* [map] */
} ebc_replay_config;
int ebc_replay_scenes(ebc_sim *sim, const ebc_replay_config *cfg, const uint32_t *seeds, const uint8_t *mask,
                      double *poly_xy, int32_t *poly_count, int32_t *need, void *stream);

/* RVO2 addObstacle (each polygon of poly_xy, counter-clockwise as scene.obstacle_vertices stores them, narrowed to
 * float like the rvo2 boundary) + processObstacles, per episode on the device, with the function ebc_pack_obstacles
 * runs on the host.  For every episode e with mask[e] != 0 (mask NULL = all): writes state.obst[e] and obst_count[e];
 * need[e] = the records the episode needs, or -1 when edge splitting exceeds cfg.max_obst (obst_count[e] = 0 then).
 * Slots past obst_count[e] are left as they are.  EBC_ERR_INVALID unless cfg.orca_obstacles and max_obst >= 1.
 * poly_xy [N*max_polys*4*2] f64, poly_count [N] i32: as ebc_replay_scenes writes them.  need [N] i32 (device). */
int ebc_build_obstacles(ebc_sim *sim, const double *poly_xy, const int32_t *poly_count, int32_t max_polys,
                        const uint8_t *mask, int32_t *need, void *stream);

/* Angular local map of simulator/env.py:468-628 (SURVEY 8f-3): for every episode the distance to the closest
 * obstacle outline in each of `dim` angular sectors around the robot, in the robot's heading frame (angle 0 at
 * the negative x axis as in the reference), clipped to max_range and optionally normalised by it.  What
 * env.step / env.reset return as `local_map` when [map] use_grid_map = false.
 * Obstacle outlines are the reference's scene.obstacle_vertices: quadrilaterals, 4 vertices each in the
 * reference's order; the robot pose (px, py, radius, theta) comes from the bound state (fp32, promoted).
 * All arithmetic is the reference's float64 sequence; sector minima are order-free, so the kernel spreads the
 * (obstacle, robot corner) and (obstacle, vertex) passes of env.py:596-620 over the lanes of a warp. */
typedef struct ebc_angular_map {
  double max_range;      /* [map] angular_map_max_range */
  double min_angle;      /* [map] angle_min * pi */
  double max_angle;      /* [map] angle_max * pi */
  int32_t dim;           /* [map] angular_map_dim (<= 256) */
  int32_t normalize;     /* divide by max_range (env.py:622-623; the reference's default) */
  int32_t max_polys;     /* Pmax: quadrilaterals per episode in poly_xy */
  int32_t reserved;
} ebc_angular_map;
/* poly_xy [N*Pmax*4*2] f64 (device), poly_count [N] i32 (device), out [N*dim] f64 (device). */
int ebc_local_map_angular(ebc_sim *sim, const ebc_angular_map *map, const double *poly_xy, const int32_t *poly_count,
                          double *out, void *stream);

/* Binary grid sub-map of simulator/env.py:630-708 (SURVEY 8f-3): what env.step / env.reset return as `local_map`
 * when [map] use_grid_map = true.  For every episode a size x size window of the occupancy grid (scene.map, given by
 * the bound state's zero-cell rectangles) centred on the robot's cell -- clipped at the map border with the
 * reference's index arithmetic (env.py:637-672; the window's last row and column keep the fill value 1, as there),
 * all ones when the window misses the map (env.py:674-680) -- rotated by (-theta + pi/2) about (size/2, size/2) and
 * thresholded at 0.9 (env.py:685-689).  The rotation is OpenCV's cv2.getRotationMatrix2D + cv2.warpAffine(grid, M,
 * (size, size), borderValue=1) for a float64 image (third-party, opencv-python, not under /root/reference, no
 * pinned version; restated from OpenCV 4.x imgwarp.cpp WarpAffineInvoker + remapBilinear and pinned to cv2 4.13):
 * inverse map in 1/1024 fixed point (AB_BITS 10, cvRound), sample position to 1/32 pixel (INTER_BITS 5), bilinear
 * weights from the float table, constant border 1.  out[e][i][j] in {0, 1}, i = first (x) index of the rotated grid. */
typedef struct ebc_grid_map {
  double submap_size_m;  /* [map] submap_size_m */
  int32_t size;          /* int(round(submap_size_m / map_resolution)), 1..192; must not exceed the map's cells */
  int32_t reserved;
} ebc_grid_map;
/* out [N*size*size] u8 (device), contiguous, at any alignment: the kernel stores 4 cells per 32-bit word only where
 * size*size % 4 == 0 and out is 4-byte aligned, and single bytes otherwise. */
int ebc_local_map_grid(ebc_sim *sim, const ebc_grid_map *map, uint8_t *out, void *stream);

/* ---- diagnostics (exported, but NOT part of the drop-in surface: nothing in the reference binds these;
 *      declared only when the includer asks for them) ---------------------------------------------------------- */
#ifdef EBC_DIAGNOSTICS
/* With EBC_TC_TRACE=1 in the environment the tensor-core K4 kernel records clock64() stamps of CTA 0 (phase
 * boundaries of its first tiles); this copies up to 4096 of them to the host (synchronises). */
int ebc_debug_trace(ebc_sim *sim, long long *out, int32_t n);
/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t ebc_launch_count(const ebc_sim *sim);
/* The scene replay of ebc_replay_scenes on the HOST, same function, for one seed: host arrays of max_humans /
 * max_statics / max_rects / cfg->max_polys slots in the ebc_state layout, need [5].  No handle, no device. */
int ebc_replay_scene_host(const ebc_replay_config *cfg, uint32_t seed, int32_t max_humans, int32_t max_statics,
                          int32_t max_rects, float *hum_pv, float *hum_gr, uint8_t *hum_type, float *stat, int16_t *rect,
                          double *poly_xy, int32_t *need);
/* One numpy primitive of the replay on a given MT19937 state (key [624], pos, as numpy's get_state() holds them),
 * advanced in place: seed(a), random(), uniform(a, b), randint(a, b) (bounds truncated toward zero like numpy's), or
 * choice([1, -1], p=[0.5, 0.5]).  The result goes to *out. */
enum { EBC_REPLAY_RNG_SEED = 0, EBC_REPLAY_RNG_RANDOM = 1, EBC_REPLAY_RNG_UNIFORM = 2, EBC_REPLAY_RNG_RANDINT = 3,
       EBC_REPLAY_RNG_CHOICE_SIGN = 4 };
int ebc_replay_rng_host(uint32_t *key, int32_t *pos, int32_t op, double a, double b, double *out);
#endif

/* ---- CPU twins (oracle/libebc_oracle.so only; HOST pointers; test infrastructure) -- */
int ebc_ref_create(const ebc_config *cfg, ebc_sim **out);
void ebc_ref_destroy(ebc_sim *sim);
const char *ebc_ref_last_error(const ebc_sim *sim);
int ebc_ref_bind(ebc_sim *sim, const ebc_state *state);
int ebc_ref_bind_stats(ebc_sim *sim, const ebc_stats *stats);
int ebc_ref_pack_obstacles(const float *xy, const int32_t *poly_size, int32_t n_poly, ebc_obst_vertex *out, int32_t cap,
                           int32_t *n_out);
int ebc_ref_set_actions(ebc_sim *sim, const double *actions, int32_t n_actions);
int ebc_ref_set_weights(ebc_sim *sim, const ebc_weights *w);
int ebc_ref_orca(ebc_sim *sim);
int ebc_ref_robot_orca(ebc_sim *sim, double safety_space, double *out_action);
int ebc_ref_lookahead(ebc_sim *sim, float *vin, double *reward, uint8_t *done, uint8_t *event);
int ebc_ref_value(ebc_sim *sim, const float *vin, int64_t n_states, const int32_t *row_count,
                  float *values);
int ebc_ref_set_attention_output(ebc_sim *sim, float *attn);
int ebc_ref_select(ebc_sim *sim, const double *reward, const float *values, double *action_values,
                   int32_t *argmax, uint8_t *nan_flag);
int ebc_ref_step(ebc_sim *sim, const int32_t *action_idx, const double *action,
                 const uint8_t *active, double *reward, uint8_t *done, uint8_t *event,
                 double *dmin, double *dist_to_goal);
int ebc_ref_transform(ebc_sim *sim, float *out);
int ebc_ref_reset(ebc_sim *sim, const ebc_state *pool, int32_t pool_size, const int32_t *pool_index,
                  const uint8_t *mask);
int ebc_ref_local_map_angular(ebc_sim *sim, const ebc_angular_map *map, const double *poly_xy, const int32_t *poly_count,
                              double *out);
int ebc_ref_local_map_grid(ebc_sim *sim, const ebc_grid_map *map, uint8_t *out);
void ebc_ref_set_threads(int n);  /* OpenMP threads over episodes (cpu_baseline leg) */

#ifdef __cplusplus
}
#endif
#endif /* EBCADRL_H */
