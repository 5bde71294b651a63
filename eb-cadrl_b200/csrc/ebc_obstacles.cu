// ebc_obstacles.cu — the ORCA obstacle half-planes' preprocessing (SURVEY 8f-4): RVO2's addObstacle +
// processObstacles for one episode, producing the packed vertex records the kernels stage in shared memory.
//
// Replaces, for the caller simulator/policy/orca_obstacles.py:102-107,
//     for obstacle in global_map: sim.addObstacle(obstacle)
//     sim.processObstacles()
// i.e. RVOSimulator::addObstacle (one Obstacle per polygon vertex: point, unit direction to the next vertex,
// convexity, prev / next links) and KdTree::buildObstacleTree (a BSP over the obstacle edges whose splitting
// line is the edge that best balances the two sides; edges that straddle it are cut in two, which creates new
// vertices).  RVO2 walks that tree per agent, near side first, and keeps the visible edges sorted by distance
// with ties in visiting order.  The kernels do not walk a tree: each vertex record carries the set of its tree
// ancestors and on which side of each it hangs (two 64-bit masks), from which a warp derives both the range
// pruning and the visiting order of any two nodes with a few bit operations (ebc_sim.cu: obstacle_lines_warp).
//
// One __host__ __device__ function (pack_obstacles) does the work: ebc_pack_obstacles runs it on the host,
// build_obstacles_kernel thread per episode on the polygons ebc_replay_scenes wrote.  fp32 like RVO2, compiled
// without contraction on both sides (-fmad=false, -Xcompiler -ffp-contract=off); division and sqrtf are IEEE.
#include <math.h>
#include <string.h>

#include "ebc_internal.cuh"

#define HD __host__ __device__

namespace {

constexpr float kEps = 0.00001f;   // RVO_EPSILON
constexpr int kMaxVtx = 64;        // vertex records per episode: the width of the kd-tree ancestor masks
constexpr int OBST_THREADS = 32;   // each thread builds one episode's tree serially

HD inline float det(float ax, float ay, float bx, float by) { return ax * by - ay * bx; }
// RVO2 leftOf(a, b, c) = det(a - c, b - a)
HD inline float left_of(const ebc_obst_vertex &a, const ebc_obst_vertex &b, const ebc_obst_vertex &c) {
  return det(a.px - c.px, a.py - c.py, b.px - a.px, b.py - a.py);
}

// (max(left, right), min(left, right)) compared as RVO2's std::pair: smaller is better
HD inline bool score_less(int l, int r, int bl, int br) {
  const int a = l > r ? l : r, b = l > r ? r : l, c = bl > br ? bl : br, d = bl > br ? br : bl;
  return a < c || (a == c && b < d);
}

// A pending call of KdTree::buildObstacleTreeRecursive: pool[start, start + len) holds its edge list (vertex ids; edge
// = vertex -> its next), and it hangs below `parent` (-1: the root) on the left side or not.
struct Frame {
  uint8_t start, len;
  int8_t parent;
  uint8_t left;
};

// processObstacles over v[0, n): recursion replaced by an explicit stack that visits the same calls in the same order
// (node, then its left subtree, then its right one), so cut vertices get RVO2's ids.  Pending edge lists are disjoint
// sets of vertex ids: all of them fit one pool of kMaxVtx ids, the lists of the frames on the stack back to back.
// Returns false when a cut would need more than `cap` vertices.
HD inline bool build_tree(ebc_obst_vertex *v, int &n, int cap) {
  uint8_t pool[kMaxVtx], part[kMaxVtx];
  Frame stack[kMaxVtx];
  int top = 0;
  for (int i = 0; i < n; ++i) pool[i] = (uint8_t)i;
  if (n > 0) stack[top++] = Frame{0, (uint8_t)n, -1, 0};
  while (top > 0) {
    const Frame f = stack[--top];
    const uint8_t *edges = pool + f.start;
    const int m = f.len;
    int best = 0, best_l = m, best_r = m;
    for (int i = 0; i < m; ++i) {
      int l = 0, r = 0;
      const ebc_obst_vertex &a = v[edges[i]], &b = v[a.next];
      for (int j = 0; j < m; ++j) {
        if (i == j) continue;
        const ebc_obst_vertex &p = v[edges[j]], &q = v[p.next];
        const float sp = left_of(a, b, p), sq = left_of(a, b, q);
        if (sp >= -kEps && sq >= -kEps) ++l;
        else if (sp <= kEps && sq <= kEps) ++r;
        else { ++l; ++r; }
        if (!score_less(l, r, best_l, best_r)) break;
      }
      if (score_less(l, r, best_l, best_r)) { best_l = l; best_r = r; best = i; }
    }
    const int node = edges[best];
    const ebc_obst_vertex a = v[node], b = v[a.next];
    // lefts fill part[] from the front, rights from the back (reversed); each keeps the edge list's order, and a cut
    // vertex takes its parent edge's place in the other list
    int nl = 0, nr = 0;
    for (int j = 0; j < m; ++j) {
      if (j == best) continue;
      const int pj = edges[j];
      const ebc_obst_vertex &p = v[pj], &q = v[p.next];
      const float sp = left_of(a, b, p), sq = left_of(a, b, q);
      if (sp >= -kEps && sq >= -kEps) part[nl++] = (uint8_t)pj;
      else if (sp <= kEps && sq <= kEps) part[kMaxVtx - 1 - nr++] = (uint8_t)pj;
      else {
        // cut edge p -> q where it meets the line through a -> b
        if (n >= cap) return false;
        const float t = det(b.px - a.px, b.py - a.py, p.px - a.px, p.py - a.py) /
                        det(b.px - a.px, b.py - a.py, p.px - q.px, p.py - q.py);
        const int id = n++;
        ebc_obst_vertex &cut = v[id];
        cut.px = p.px + t * (q.px - p.px);
        cut.py = p.py + t * (q.py - p.py);
        cut.ux = p.ux; cut.uy = p.uy;
        cut.prev = (int16_t)pj; cut.next = p.next;
        cut.convex = 1;
        cut.pad0 = 0;
        cut.anc = cut.anc_left = cut.pad1 = 0;
        v[p.next].prev = (int16_t)id;
        v[pj].next = (int16_t)id;
        if (sp > 0.0f) { part[nl++] = (uint8_t)pj; part[kMaxVtx - 1 - nr++] = (uint8_t)id; }
        else { part[kMaxVtx - 1 - nr++] = (uint8_t)pj; part[nl++] = (uint8_t)id; }
      }
    }
    const uint64_t anc = f.parent < 0 ? 0 : v[f.parent].anc | (uint64_t)1 << f.parent;
    const uint64_t anc_left = f.parent < 0 ? 0 : v[f.parent].anc_left | (f.left ? (uint64_t)1 << f.parent : 0);
    v[node].anc = anc;
    v[node].anc_left = anc_left;
    // the children's lists replace this one in the pool, rights below lefts: the left subtree is built first.  The
    // lists below f.start and these nl + nr ids are disjoint vertex ids, so f.start + nl + nr <= n <= kMaxVtx.
    uint8_t *out = pool + f.start;
    for (int k = 0; k < nr; ++k) out[k] = part[kMaxVtx - 1 - k];
    for (int k = 0; k < nl; ++k) out[nr + k] = part[k];
    if (nr > 0) stack[top++] = Frame{f.start, (uint8_t)nr, (int8_t)node, 0};
    if (nl > 0) stack[top++] = Frame{(uint8_t)(f.start + nr), (uint8_t)nl, (int8_t)node, 1};
  }
  return true;
}

// RVOSimulator::addObstacle for every polygon (xy: vertices back to back, poly_size[p] each) + processObstacles.
// v holds kMaxVtx records; cap <= kMaxVtx.  Returns the number of records, or -1 when a polygon is degenerate
// (fewer than 2 vertices) or the vertices, cut ones included, need more than `cap` records.
HD inline int pack_obstacles(const float *xy, const int32_t *poly_size, int n_poly, int cap, ebc_obst_vertex *v) {
  int n = 0, off = 0;
  for (int p = 0; p < n_poly; ++p) {
    const int m = poly_size[p];
    if (m < 2 || n + m > cap) return -1;
    const float *q = xy + 2 * off;
    for (int i = 0; i < m; ++i) {
      const int nx = (i + 1) % m, pr = (i + m - 1) % m;
      ebc_obst_vertex &o = v[n + i];
      o.px = q[2 * i]; o.py = q[2 * i + 1];
      o.next = (int16_t)(n + nx); o.prev = (int16_t)(n + pr);
      const float dx = q[2 * nx] - o.px, dy = q[2 * nx + 1] - o.py;
      const float inv = 1.0f / sqrtf(dx * dx + dy * dy);
      o.ux = dx * inv; o.uy = dy * inv;
      if (m == 2) o.convex = 1;
      else o.convex = det(q[2 * pr] - q[2 * nx], q[2 * pr + 1] - q[2 * nx + 1], o.px - q[2 * pr], o.py - q[2 * pr + 1]) >= 0.0f;
      o.pad0 = 0;
      o.anc = o.anc_left = o.pad1 = 0;
    }
    n += m;
    off += m;
  }
  return build_tree(v, n, cap) ? n : -1;
}

// Thread per episode: the episode's quadrilaterals (float64, narrowed to float like the rvo2 boundary) -> its records.
__global__ void __launch_bounds__(OBST_THREADS)
build_obstacles_kernel(const ebc_config c, const ebc_state st, const double *poly_xy, const int32_t *poly_count,
                       int max_polys, const uint8_t *mask, int32_t *need) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= c.n_episodes) return;
  if (mask && !mask[e]) return;
  int P = poly_count[e];
  P = P < 0 ? 0 : (P > max_polys ? max_polys : P);
  int n = -1;
  if (4 * P <= c.max_obst) {           // more vertices than slots overflows before any split
    float xy[kMaxVtx * 2];
    int32_t size[kMaxVtx / 4];
    const double *src = poly_xy + (size_t)e * max_polys * 8;
    for (int k = 0; k < 8 * P; ++k) xy[k] = (float)src[k];
    for (int p = 0; p < P; ++p) size[p] = 4;
    __align__(16) ebc_obst_vertex v[kMaxVtx];     // copied out in 16-byte words
    n = pack_obstacles(xy, size, P, c.max_obst, v);
    uint4 *dst = reinterpret_cast<uint4 *>(st.obst + (size_t)e * c.max_obst);
    for (int k = 0; k < n; ++k) {
      const uint4 *w = reinterpret_cast<const uint4 *>(&v[k]);
      dst[3 * k] = w[0]; dst[3 * k + 1] = w[1]; dst[3 * k + 2] = w[2];
    }
  }
  need[e] = n;
  st.obst_count[e] = n < 0 ? 0 : n;
}

}  // namespace

int ebc_launch_build_obstacles(ebc_sim *s, const double *poly_xy, const int32_t *poly_count, int max_polys,
                               const uint8_t *mask, int32_t *need, cudaStream_t stream) {
  s->la_rec_valid = 0;      // the state moves on: the lookahead records no longer describe it
  const int blocks = (s->cfg.n_episodes + OBST_THREADS - 1) / OBST_THREADS;
  build_obstacles_kernel<<<blocks, OBST_THREADS, 0, stream>>>(s->cfg, s->st, poly_xy, poly_count, max_polys, mask, need);
  return ebc_check_launch(s, "build_obstacles_kernel");
}

extern "C" int ebc_pack_obstacles(const float *xy, const int32_t *poly_size, int32_t n_poly, ebc_obst_vertex *out,
                                  int32_t cap, int32_t *n_out) {
  if (!poly_size || !out || !n_out || n_poly < 0 || cap < 0 || (n_poly > 0 && !xy)) return EBC_ERR_INVALID;
  if (cap > kMaxVtx) cap = kMaxVtx;
  ebc_obst_vertex v[kMaxVtx];
  const int n = pack_obstacles(xy, poly_size, n_poly, cap, v);
  if (n < 0) return EBC_ERR_INVALID;
  memcpy(out, v, sizeof(ebc_obst_vertex) * (size_t)n);
  *n_out = n;
  return EBC_OK;
}
