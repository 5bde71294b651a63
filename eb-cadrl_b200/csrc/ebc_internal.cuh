// Internal declarations shared by the translation units of libebcadrl.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define EBC_DIAGNOSTICS 1
#include "../../include/ebcadrl.h"

#define EBC_WARPS_PER_BLOCK 8
#define EBC_THREADS (EBC_WARPS_PER_BLOCK * 32)

// Value-network geometry, computed once in ebc_set_weights (host) and passed by value.
struct ValueLayer {
  const float *wt;   // transposed + padded weights [in][out_pad] (device)
  const float *bias; // [out_pad] (device)
  int in, out, out_pad;
};

struct ValueNet {
  int D, self_dim, with_global;
  ValueLayer l[11];      // mlp1[2] mlp2[2] att[3] mlp3[4]; att[0] is split: l[4] = local half
  ValueLayer att0_glob;  // global-state half of attention.0 (bias folded here)
};

// ---- tensor-core (tcgen05) value path, ebc_value_tc.cu -------------------------------------------
enum { ST_L0A = 0, ST_L0B = 1, ST_L1A = 2, ST_L1B = 3, ST_L2 = 4, ST_L3 = 5, ST_L4 = 6, ST_L5 = 7, ST_L4G = 8, ST_COUNT = 9 };

struct TcStage {         // one GEMM stage: acc[:, acc_col : acc_col + np] (+)= A[:, 0 : 16*ksteps] . W^T
  int np;                // padded N (multiple of 16, <= 208)
  int ksteps;            // K / 16
  int acc_col;           // first TMEM column of the accumulator
  int accumulate;        // add to the existing accumulator (second K chunk)
  int n_lo;              // first output column of this stage within its layer (bias offset)
  int n_real;            // real output columns of this stage (the rest of np is padding)
  int bias_k;            // >= 0: the bias rides in the GEMM -- column bias_k of this stage's A operand is a constant
                         // one (written by whoever produces that operand) and row bias_k of the weights is the bias
};

struct TcSched {         // one entry of the MMA warp's per-tile schedule
  uint8_t stage;         // ST_*
  uint8_t chase;         // k-step b waits for block b of the A operand (the producing epilogue is still running)
  uint8_t commit_k;      // release block b of the A operand to the next epilogue as soon as its MMAs complete
  uint8_t commit_acc;    // then tell the crew that every MMA issued so far has completed
};

struct TcIssue {         // a schedule entry flattened for the MMA warp: everything it needs at constant parameter offsets
  int np, ksteps, acc_col, accumulate, commit_k, commit_acc;
  uint32_t idesc;        // tcgen05 instruction descriptor (M = 128, N = np, operand format of the splitting mode)
  int pad;
};

struct TcProgram {
  TcStage st[ST_COUNT];
  TcSched sched[12];
  TcIssue issue[12];     // issue[i] = the stage of sched[i] as the MMA warp sees it (filled by ebc_tc_prepare)
  int n_sched;
  int n_wide;                    // 1 or 2 halves of the wide first layer
  const uint8_t *wpack;          // packed bf16 weight slabs (device)
  const uint32_t *slab_off, *slab_bytes;
  int n_slabs;                   // slabs consumed per tile
  const float *bias[6];          // padded fp32 biases (device)
  const float *w6;               // last (N = 1) layer weights, padded
  float w6c[208];                // the same in the kernel's parameter block: warp-uniform constant-bank reads in the
                                 // score / value epilogue instead of dependent global loads
  float b6;
  int with_global, h1d, h2d;
  int early_x;                   // the next tile's input may be staged before this tile's pooling (TMEM ranges disjoint)
};

struct TcPrograms {
  TcProgram entity, mlp3;
  uint8_t *slab;                 // one device allocation
  int ready;
};

struct ebc_sim {
  ebc_config cfg;
  ebc_state st;
  ebc_stats stats;       // running episode statistics (ebc_bind_stats); all-null when unbound
  int device;
  bool bound, have_actions, have_weights;
  double *d_actions;     // [A*2]
  ValueNet net;
  float *d_weights;      // one slab
  float4 *d_la_rec;      // [N * A * 3] robot part of the rotated rows per (episode, action), written by ebc_lookahead for
                         // K4's fused input path (ebc_value with vin == NULL)
  int la_rec_valid;      // the records belong to the current state (set by ebc_lookahead, consumed by ebc_value)
  float *attn_out;       // caller's array for the softmax attention weights (ebc_set_attention_output), or null
  float *d_joint;        // [cap_states * (self_dim + H2)] scratch for mlp3
  int64_t joint_cap;     // states ebc_value may be called with (ebc_reserve)
  size_t joint_floats;   // allocated floats of d_joint
  TcPrograms tc[3];      // indexed by operand parts - 1: [0] bf16, [1] fp16x2, [2] bf16x3
  long long *d_trace;    // EBC_TC_TRACE=1: clock64 stamps of CTA 0 (diagnostics)
  int value_mode;        // EBC_VALUE_*
  int value_mode_forced; // set explicitly by ebc_set_value_mode
  int64_t launches;
  int sm_count;
  int max_smem_optin;
  char err[256];
};

int ebc_fail(ebc_sim *s, int code, const char *fmt, ...);
int ebc_check_launch(ebc_sim *s, const char *what);

// ebc_sim.cu
int ebc_launch_orca(ebc_sim *s, cudaStream_t st);
int ebc_launch_robot_orca(ebc_sim *s, double safety, double *out, cudaStream_t st);
int ebc_launch_lookahead(ebc_sim *s, float *vin, double *reward, uint8_t *done, uint8_t *event,
                         cudaStream_t st);
int ebc_launch_select(ebc_sim *s, const double *reward, const float *values, double *action_values,
                      int32_t *argmax, uint8_t *nan_flag, cudaStream_t st);
int ebc_launch_step(ebc_sim *s, bool fused_orca, const int32_t *action_idx, const double *action,
                    const uint8_t *active, double *reward, uint8_t *done, uint8_t *event, double *dmin,
                    double *dist_to_goal, cudaStream_t st);
int ebc_launch_transform(ebc_sim *s, float *out, cudaStream_t st);
int ebc_launch_reset(ebc_sim *s, const ebc_state *pool, int pool_size, const int32_t *pool_index,
                     const uint8_t *mask, cudaStream_t st);

int ebc_launch_angular_map(ebc_sim *s, const ebc_angular_map *map, const double *poly_xy, const int32_t *poly_count,
                           double *out, cudaStream_t st);
int ebc_launch_grid_map(ebc_sim *s, const ebc_grid_map *map, uint8_t *out, cudaStream_t st);
int ebc_launch_generate(ebc_sim *s, const ebc_scene_shape *shape, uint64_t seed, const int64_t *episode_ids,
                        const uint8_t *mask, cudaStream_t st);

// ebc_replay.cu
int ebc_launch_replay(ebc_sim *s, const ebc_replay_config *cfg, const uint32_t *seeds, const uint8_t *mask,
                      double *poly_xy, int32_t *poly_count, int32_t *need, cudaStream_t st);

// ebc_obstacles.cu
int ebc_launch_build_obstacles(ebc_sim *s, const double *poly_xy, const int32_t *poly_count, int max_polys,
                               const uint8_t *mask, int32_t *need, cudaStream_t st);

// ebc_value.cu
int ebc_value_prepare(ebc_sim *s, const ebc_weights *w);
void ebc_value_release(ebc_sim *s);
int ebc_launch_value(ebc_sim *s, const float *vin, int64_t n_states, const int32_t *row_count,
                     float *values, cudaStream_t st);

// ebc_value_tc.cu
int ebc_tc_prepare(ebc_sim *s, const ebc_weights *w, int mode_index, int nsplit);
void ebc_tc_release(ebc_sim *s);
// vin == NULL: the fused input path (rows built by the kernel from the bound state + s->d_la_rec)
int ebc_launch_value_tc(ebc_sim *s, int mode, const float *vin, int64_t n_states, const int32_t *row_count,
                        float *values, cudaStream_t st);
