// ebc_value.cu — K4, the SARL / EB-CADRL value network (rl/policy/sarl.py:38-82) on sm_100a.
//
// Round-1 path: fp32 SIMT (FFMA) — fp32-accurate by construction, which is what argmax parity
// with the reference needs (SURVEY §7: TF32 / bf16 operands flip 3-49 % of decisions).
// Two kernels share one shared-memory GEMM routine:
//   value_entity_kernel  per tile of <= 64 entity rows (whole states): mlp1, mlp2, attention,
//                        masked softmax pooling -> joint[state][self_dim + H2] (global scratch)
//   value_mlp3_kernel    per tile of 64 states: mlp3 -> V
// Activations live in shared memory, transposed ([feature][row], row stride 68 floats) so that a
// thread's 8 rows are two float4 loads and the epilogue's stores are conflict-minimal.  Weights are
// pre-transposed on the host to [in][out_pad] (out_pad % 32 == 0) and streamed L2 -> shared memory
// with double-buffered cp.async; each thread owns 8 rows x J columns (columns lane + 32 j).
#include <stdio.h>
#include <string.h>

#include <vector>

#include "ebc_internal.cuh"

namespace {

constexpr int LDA = 68;        // row stride of transposed activations (64 rows + 4 pad)
constexpr int TILE_ROWS = 64;
constexpr int KC = 8;          // k-rows per weight stage
constexpr int WSTAGE = KC * 256;   // floats per stage (J <= 8 -> 256 columns)
constexpr int MAX_TS = 16;     // states per entity tile

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

struct Epilogue {
  const float *bias;      // [out_pad]
  const float *gv;        // optional per-state additive term [MAX_TS][gv_ld] (shared memory)
  int gv_ld;
  int n_rows_per_state;   // to map a row to its state (only with gv)
  bool relu;
};

// out_s[col][row] = act( sum_k in_s[k][row] * wt[k][col] + bias[col] (+ gv[state(row)][col]) )
// for cols [colbase, colbase + 32 J), rows 0..63.  All 256 threads participate.
template <int J>
__device__ void gemm_chunk(const float *in_s, int K, const float *__restrict__ wt, int out_pad, int out_real,
                           int colbase, float *wstage, float *out_s, const Epilogue &ep) {
  const int ty = threadIdx.x >> 5, tx = threadIdx.x & 31;
  constexpr int WS = 32 * J;               // floats per staged k-row
  constexpr int V4_PER_ROW = WS / 4;
  float acc[8][J];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < J; ++j) acc[i][j] = 0.0f;

  const int nk = (K + KC - 1) / KC;
  auto load_stage = [&](int buf, int kc) {
    const int k0 = kc * KC;
    const int rows = min(KC, K - k0);
    float *dst = wstage + buf * WSTAGE;
    for (int i = threadIdx.x; i < rows * V4_PER_ROW; i += blockDim.x) {
      const int kk = i / V4_PER_ROW, v = i % V4_PER_ROW;
      cp_async16(dst + kk * WS + v * 4, wt + (size_t)(k0 + kk) * out_pad + colbase + v * 4);
    }
    cp_async_commit();
  };
  load_stage(0, 0);
  for (int kc = 0; kc < nk; ++kc) {
    if (kc + 1 < nk) {
      load_stage((kc + 1) & 1, kc + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float *ws = wstage + (kc & 1) * WSTAGE;
    const int k0 = kc * KC;
    const int rows = min(KC, K - k0);
    if (rows == KC) {
#pragma unroll
      for (int kk = 0; kk < KC; ++kk) {
        const float4 a0 = *reinterpret_cast<const float4 *>(in_s + (k0 + kk) * LDA + ty * 8);
        const float4 a1 = *reinterpret_cast<const float4 *>(in_s + (k0 + kk) * LDA + ty * 8 + 4);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int j = 0; j < J; ++j) {
          const float w = ws[kk * WS + tx + 32 * j];
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[i][j] = fmaf(a[i], w, acc[i][j]);
        }
      }
    } else {
      for (int kk = 0; kk < rows; ++kk) {
        const float4 a0 = *reinterpret_cast<const float4 *>(in_s + (k0 + kk) * LDA + ty * 8);
        const float4 a1 = *reinterpret_cast<const float4 *>(in_s + (k0 + kk) * LDA + ty * 8 + 4);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int j = 0; j < J; ++j) {
          const float w = ws[kk * WS + tx + 32 * j];
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[i][j] = fmaf(a[i], w, acc[i][j]);
        }
      }
    }
    __syncthreads();
  }
  // epilogue
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int col = colbase + tx + 32 * j;
    if (col < out_real) {
      const float b = ep.bias[col];
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float x = acc[i][j] + b;
        // with fewer than 4 rows per state the tile's MAX_TS states end before row 64: the rows past them belong to
        // no state and their outputs are never read, but the index must stay inside GV
        if (ep.gv) x += ep.gv[min((ty * 8 + i) / ep.n_rows_per_state, MAX_TS - 1) * ep.gv_ld + col];
        v[i] = (ep.relu && x < 0.0f) ? 0.0f : x;
      }
      *reinterpret_cast<float4 *>(out_s + col * LDA + ty * 8) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4 *>(out_s + col * LDA + ty * 8 + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
}

__device__ void gemm_layer(const float *in_s, const ValueLayer &L, float *wstage, float *out_s, const Epilogue &ep) {
  const int n32 = L.out_pad / 32;
  const int chunks = (n32 + 7) / 8;
  const int jc = (n32 + chunks - 1) / chunks;
  int done = 0;
  while (done < n32) {
    const int j = min(jc, n32 - done);
    const int colbase = done * 32;
    switch (j) {
      case 1: gemm_chunk<1>(in_s, L.in, L.wt, L.out_pad, L.out, colbase, wstage, out_s, ep); break;
      case 2: gemm_chunk<2>(in_s, L.in, L.wt, L.out_pad, L.out, colbase, wstage, out_s, ep); break;
      case 3: gemm_chunk<3>(in_s, L.in, L.wt, L.out_pad, L.out, colbase, wstage, out_s, ep); break;
      case 4: gemm_chunk<4>(in_s, L.in, L.wt, L.out_pad, L.out, colbase, wstage, out_s, ep); break;
      case 5: gemm_chunk<5>(in_s, L.in, L.wt, L.out_pad, L.out, colbase, wstage, out_s, ep); break;
      case 6: gemm_chunk<6>(in_s, L.in, L.wt, L.out_pad, L.out, colbase, wstage, out_s, ep); break;
      case 7: gemm_chunk<7>(in_s, L.in, L.wt, L.out_pad, L.out, colbase, wstage, out_s, ep); break;
      default: gemm_chunk<8>(in_s, L.in, L.wt, L.out_pad, L.out, colbase, wstage, out_s, ep); break;
    }
    done += j;
  }
  __syncthreads();
}

struct EntityParams {
  ValueNet net;
  const float *vin;          // [n_states][n][D]
  const int32_t *row_count;  // [n_states] or null
  const int32_t *hum_count, *stat_count;   // per-episode counts (used when row_count == null)
  int n_actions;             // states per episode in that mode
  long long n_states;
  int n;                     // rows per state slot
  int ts;                    // states per tile
  float *joint;              // [n_states][self_dim + H2]
  float *attn;               // [n_states][n] softmax attention weights (ebc_set_attention_output), or null
  // shared-memory offsets (floats)
  int off_x, off_t, off_h1, off_h2, off_w, off_g, off_gv, off_sc;
};

__global__ void __launch_bounds__(256, 1) value_entity_kernel(const EntityParams p) {
  extern __shared__ __align__(16) float smem[];
  float *X = smem + p.off_x, *T = smem + p.off_t, *H1 = smem + p.off_h1, *H2 = smem + p.off_h2;
  float *W = smem + p.off_w, *G = smem + p.off_g, *GV = smem + p.off_gv, *SC = smem + p.off_sc;
  __shared__ int cnt[MAX_TS];
  const ValueNet &net = p.net;
  const int D = net.D, n = p.n, ts = p.ts;
  const int h1d = net.l[1].out, h2d = net.l[3].out, a1d = net.l[4].out;
  const int tid = threadIdx.x;

  for (long long tile = blockIdx.x; tile * ts < p.n_states; tile += gridDim.x) {
    const long long s0 = tile * ts;
    const int ns = (int)min((long long)ts, p.n_states - s0);
    const int rows = ns * n;
    // stage the tile's rows: contiguous rows*D floats in global -> X[d][row]
    for (int i = tid; i < TILE_ROWS * D; i += blockDim.x) {
      const int r = i / D, d = i % D;
      X[d * LDA + r] = (r < rows) ? p.vin[(size_t)s0 * n * D + i] : 0.0f;
    }
    if (tid < MAX_TS) {
      int c = 0;
      if (tid < ns) {
        if (p.row_count) c = p.row_count[s0 + tid];
        else {
          const long long e = (s0 + tid) / p.n_actions;
          c = p.hum_count[e] + p.stat_count[e];
        }
        c = min(max(c, 0), n);
      }
      cnt[tid] = c;
    }
    __syncthreads();
    Epilogue ep = {nullptr, nullptr, 0, n, true};
    ep.bias = net.l[0].bias; gemm_layer(X, net.l[0], W, T, ep);     // mlp1.0 + ReLU
    ep.bias = net.l[1].bias; gemm_layer(T, net.l[1], W, H1, ep);    // mlp1.2 + ReLU (last_relu)
    // global state: mean of mlp1 output over the state's real rows (sarl.py:51-60)
    if (net.with_global) {
      for (int i = tid; i < ts * h1d; i += blockDim.x) {
        const int s = i / h1d, k = i % h1d;
        float acc = 0.0f;
        const int c = cnt[s];
        for (int r = 0; r < c; ++r) acc += H1[k * LDA + s * n + r];
        G[s * h1d + k] = c > 0 ? acc / (float)c : 0.0f;
      }
      __syncthreads();
      // GV[s][c] = attention.0.bias[c] + W_att0[:, h1d:] . G[s]
      const ValueLayer &LG = net.att0_glob;
      for (int i = tid; i < ts * a1d; i += blockDim.x) {
        const int s = i / a1d, c = i % a1d;
        float acc = LG.bias[c];
        for (int k = 0; k < h1d; ++k) acc = fmaf(G[s * h1d + k], LG.wt[(size_t)k * LG.out_pad + c], acc);
        GV[s * a1d + c] = acc;
      }
      __syncthreads();
    }
    ep.bias = net.l[2].bias; gemm_layer(H1, net.l[2], W, T, ep);    // mlp2.0 + ReLU
    ep.relu = false;
    ep.bias = net.l[3].bias; gemm_layer(T, net.l[3], W, H2, ep);    // mlp2.2
    ep.relu = true;
    if (net.with_global) {                                          // attention.0 (+ global half) + ReLU
      ep.bias = net.l[4].bias;   // zeros: the real bias is folded into GV
      ep.gv = GV; ep.gv_ld = a1d;
    } else {
      ep.bias = net.l[4].bias;
    }
    gemm_layer(H1, net.l[4], W, T, ep);
    ep.gv = nullptr;
    ep.bias = net.l[5].bias; gemm_layer(T, net.l[5], W, H1, ep);    // attention.2 + ReLU (H1 is dead: reuse)
    // attention.4: one score per row
    {
      const ValueLayer &L6 = net.l[6];
      if (tid < TILE_ROWS) {
        float acc = L6.bias[0];
        for (int k = 0; k < L6.in; ++k) acc = fmaf(H1[k * LDA + tid], L6.wt[(size_t)k * L6.out_pad], acc);
        SC[tid] = acc;
      }
      __syncthreads();
    }
    // masked softmax without max subtraction (sarl.py:69-70)
    if (tid < ts) {
      const int c = cnt[tid];
      float sum = 0.0f;
      for (int r = 0; r < c; ++r) {
        const float sc = SC[tid * n + r];
        const float e = (sc != 0.0f) ? expf(sc) : 0.0f;
        SC[tid * n + r] = e;
        sum += e;
      }
      for (int r = 0; r < c; ++r) SC[tid * n + r] = SC[tid * n + r] / sum;
      if (p.attn && tid < ns)
        for (int r = 0; r < n; ++r) p.attn[(size_t)(s0 + tid) * n + r] = r < c ? SC[tid * n + r] : 0.0f;
    }
    __syncthreads();
    // joint = [self_state, sum_r w_r * mlp2_r]
    const int jd = net.self_dim + h2d;
    for (int i = tid; i < ns * jd; i += blockDim.x) {
      const int s = i / jd, k = i % jd;
      float v;
      if (k < net.self_dim) {
        v = X[k * LDA + s * n];
      } else {
        v = 0.0f;
        const int c = cnt[s];
        for (int r = 0; r < c; ++r) v = fmaf(SC[s * n + r], H2[(k - net.self_dim) * LDA + s * n + r], v);
      }
      p.joint[(size_t)(s0 + s) * jd + k] = v;
    }
    __syncthreads();
  }
}

struct Mlp3Params {
  ValueNet net;
  const float *joint;
  float *values;
  long long n_states;
  int off_x, off_a, off_b, off_w;
};

__global__ void __launch_bounds__(256, 1) value_mlp3_kernel(const Mlp3Params p) {
  extern __shared__ __align__(16) float smem[];
  float *X = smem + p.off_x, *A = smem + p.off_a, *B = smem + p.off_b, *W = smem + p.off_w;
  const ValueNet &net = p.net;
  const int jd = net.l[7].in;
  const int tid = threadIdx.x;
  for (long long tile = blockIdx.x; tile * TILE_ROWS < p.n_states; tile += gridDim.x) {
    const long long s0 = tile * TILE_ROWS;
    const int ns = (int)min((long long)TILE_ROWS, p.n_states - s0);
    for (int i = tid; i < TILE_ROWS * jd; i += blockDim.x) {
      const int r = i / jd, d = i % jd;
      X[d * LDA + r] = (r < ns) ? p.joint[(size_t)s0 * jd + i] : 0.0f;
    }
    __syncthreads();
    Epilogue ep = {nullptr, nullptr, 0, 1, true};
    ep.bias = net.l[7].bias; gemm_layer(X, net.l[7], W, A, ep);
    ep.bias = net.l[8].bias; gemm_layer(A, net.l[8], W, B, ep);
    ep.bias = net.l[9].bias; gemm_layer(B, net.l[9], W, A, ep);
    const ValueLayer &L = net.l[10];
    if (tid < ns) {
      float acc = L.bias[0];
      for (int k = 0; k < L.in; ++k) acc = fmaf(A[k * LDA + tid], L.wt[(size_t)k * L.out_pad], acc);
      p.values[s0 + tid] = acc;
    }
    __syncthreads();
  }
}

int pad32(int x) { return (x + 31) / 32 * 32; }

}  // namespace

// Copy + transpose + pad the state_dict into one device slab (rl/policy/sarl.py:23-36 shapes).
int ebc_value_prepare(ebc_sim *s, const ebc_weights *w) {
  const int D = s->cfg.with_agent_type ? 17 : 13;
  if (w->input_dim != D) return ebc_fail(s, EBC_ERR_INVALID, "ebc_set_weights: input_dim %d != D %d", w->input_dim, D);
  const ebc_linear *src[11] = {&w->mlp1[0], &w->mlp1[1], &w->mlp2[0], &w->mlp2[1], &w->attention[0],
                               &w->attention[1], &w->attention[2], &w->mlp3[0], &w->mlp3[1], &w->mlp3[2],
                               &w->mlp3[3]};
  for (int i = 0; i < 11; ++i)
    if (!src[i]->weight || !src[i]->bias || src[i]->in_dim < 1 || src[i]->out_dim < 1)
      return ebc_fail(s, EBC_ERR_INVALID, "ebc_set_weights: layer %d missing", i);
  const int h1 = src[1]->out_dim;
  const bool wg = w->with_global_state != 0;
  if (src[0]->in_dim != D || src[1]->in_dim != src[0]->out_dim || src[2]->in_dim != h1 ||
      src[3]->in_dim != src[2]->out_dim || src[4]->in_dim != (wg ? 2 * h1 : h1) ||
      src[5]->in_dim != src[4]->out_dim || src[6]->in_dim != src[5]->out_dim || src[6]->out_dim != 1 ||
      src[7]->in_dim != src[3]->out_dim + w->self_state_dim || src[8]->in_dim != src[7]->out_dim ||
      src[9]->in_dim != src[8]->out_dim || src[10]->in_dim != src[9]->out_dim || src[10]->out_dim != 1 ||
      w->self_state_dim > D)
    return ebc_fail(s, EBC_ERR_INVALID, "ebc_set_weights: inconsistent layer shapes");
  for (int i = 0; i < 11; ++i)
    if (src[i]->out_dim > 1024 || src[i]->in_dim > 2048)
      return ebc_fail(s, EBC_ERR_INVALID, "ebc_set_weights: layer %d too wide", i);

  ValueNet net;
  memset(&net, 0, sizeof(net));
  net.D = D; net.self_dim = w->self_state_dim; net.with_global = wg ? 1 : 0;
  std::vector<float> slab;
  auto reserve = [&](size_t nfl) { size_t off = slab.size(); slab.resize(off + ((nfl + 3) / 4 * 4), 0.0f); return off; };
  size_t off_w[12], off_b[12];
  // layer i: wt[k][c] = weight[c][k]
  auto put = [&](int idx, const float *weight, const float *bias, int in, int out, int ld_in, int k_off, bool zero_bias) {
    const int op = pad32(out);
    off_w[idx] = reserve((size_t)in * op);
    off_b[idx] = reserve(op);
    for (int c = 0; c < out; ++c) {
      for (int k = 0; k < in; ++k) slab[off_w[idx] + (size_t)k * op + c] = weight[(size_t)c * ld_in + k_off + k];
      slab[off_b[idx] + c] = zero_bias ? 0.0f : bias[c];
    }
    return op;
  };
  int in_dim[12], out_dim[12], out_pad[12];
  for (int i = 0; i < 11; ++i) {
    if (i == 4 && wg) {   // attention.0 split: local half (no bias) + global half (bias)
      in_dim[4] = h1; out_dim[4] = src[4]->out_dim;
      out_pad[4] = put(4, src[4]->weight, src[4]->bias, h1, src[4]->out_dim, 2 * h1, 0, true);
      in_dim[11] = h1; out_dim[11] = src[4]->out_dim;
      out_pad[11] = put(11, src[4]->weight, src[4]->bias, h1, src[4]->out_dim, 2 * h1, h1, false);
    } else {
      in_dim[i] = src[i]->in_dim; out_dim[i] = src[i]->out_dim;
      out_pad[i] = put(i, src[i]->weight, src[i]->bias, src[i]->in_dim, src[i]->out_dim, src[i]->in_dim, 0, false);
    }
  }
  cudaError_t err;
  if (s->d_weights) { cudaFree(s->d_weights); s->d_weights = nullptr; }
  if ((err = cudaMalloc(&s->d_weights, slab.size() * sizeof(float))) != cudaSuccess)
    return ebc_fail(s, EBC_ERR_NOMEM, "cudaMalloc weights: %s", cudaGetErrorString(err));
  if ((err = cudaMemcpy(s->d_weights, slab.data(), slab.size() * sizeof(float), cudaMemcpyHostToDevice)) != cudaSuccess)
    return ebc_fail(s, EBC_ERR_CUDA, "cudaMemcpy weights: %s", cudaGetErrorString(err));
  for (int i = 0; i < 11; ++i) {
    net.l[i].wt = s->d_weights + off_w[i];
    net.l[i].bias = s->d_weights + off_b[i];
    net.l[i].in = in_dim[i]; net.l[i].out = out_dim[i]; net.l[i].out_pad = out_pad[i];
  }
  if (wg) {
    net.att0_glob.wt = s->d_weights + off_w[11];
    net.att0_glob.bias = s->d_weights + off_b[11];
    net.att0_glob.in = in_dim[11]; net.att0_glob.out = out_dim[11]; net.att0_glob.out_pad = out_pad[11];
  }
  s->net = net;
  s->have_weights = true;
  return EBC_OK;
}

void ebc_value_release(ebc_sim *s) {
  if (s->d_weights) cudaFree(s->d_weights);
  if (s->d_joint) cudaFree(s->d_joint);
  s->d_weights = nullptr;
  s->d_joint = nullptr;
  s->joint_cap = 0;
  s->joint_floats = 0;
}

int ebc_launch_value(ebc_sim *s, const float *vin, int64_t n_states, const int32_t *row_count, float *values,
                     cudaStream_t stream) {
  if (n_states <= 0) return EBC_OK;
  const ValueNet &net = s->net;
  const int n = s->cfg.max_humans + s->cfg.max_statics;
  const int jd = net.self_dim + net.l[3].out;
  EntityParams p;
  p.net = net;
  p.vin = vin; p.row_count = row_count;
  p.hum_count = s->st.hum_count; p.stat_count = s->st.stat_count;
  p.n_actions = s->cfg.n_actions;
  p.n_states = n_states; p.n = n;
  int ts = TILE_ROWS / n;
  if (ts < 1) ts = 1;
  if (ts > MAX_TS) ts = MAX_TS;
  p.ts = ts;
  p.joint = s->d_joint;
  p.attn = s->attn_out;
  const int h1d = net.l[1].out, h2d = net.l[3].out, a1d = net.l[4].out;
  int tmax = net.l[0].out;
  if (net.l[2].out > tmax) tmax = net.l[2].out;
  if (a1d > tmax) tmax = a1d;
  const int h1rows = h1d > net.l[5].out ? h1d : net.l[5].out;
  int off = 0;
  p.off_x = off; off += net.D * LDA;
  p.off_t = off; off += tmax * LDA;
  p.off_h1 = off; off += h1rows * LDA;
  p.off_h2 = off; off += h2d * LDA;
  p.off_w = off; off += 2 * WSTAGE;
  p.off_g = off; off += MAX_TS * h1d;
  p.off_gv = off; off += MAX_TS * a1d;
  p.off_sc = off; off += TILE_ROWS + 4;
  const size_t smem_a = (size_t)off * sizeof(float);
  Mlp3Params q;
  q.net = net; q.joint = s->d_joint; q.values = values; q.n_states = n_states;
  off = 0;
  const int m1 = net.l[7].out > net.l[9].out ? net.l[7].out : net.l[9].out;
  q.off_x = off; off += jd * LDA;
  q.off_a = off; off += m1 * LDA;
  q.off_b = off; off += net.l[8].out * LDA;
  q.off_w = off; off += 2 * WSTAGE;
  const size_t smem_b = (size_t)off * sizeof(float);
  if (smem_a > (size_t)s->max_smem_optin || smem_b > (size_t)s->max_smem_optin)
    return ebc_fail(s, EBC_ERR_INVALID, "value network too wide for shared memory (%zu / %zu B needed)", smem_a, smem_b);
  cudaFuncSetAttribute(value_entity_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_a);
  cudaFuncSetAttribute(value_mlp3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b);
  const long long tiles_a = (n_states + ts - 1) / ts;
  const long long tiles_b = (n_states + TILE_ROWS - 1) / TILE_ROWS;
  const int grid_a = (int)(tiles_a < s->sm_count ? tiles_a : s->sm_count);
  const int grid_b = (int)(tiles_b < s->sm_count ? tiles_b : s->sm_count);
  value_entity_kernel<<<grid_a, 256, smem_a, stream>>>(p);
  int rc = ebc_check_launch(s, "value_entity_kernel");
  if (rc) return rc;
  value_mlp3_kernel<<<grid_b, 256, smem_b, stream>>>(q);
  return ebc_check_launch(s, "value_mlp3_kernel");
}
