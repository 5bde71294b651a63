// ebc_sim.cu — simulation kernels of the EB-CADRL hot path for sm_100a.
//
//   K1 orca_kernel        warp per human: RVO2 neighbour selection + ORCA half-planes + the
//                         incremental 2-D linear program, lines distributed one per lane
//                         (simulator/policy/orca.py:85-157 -> rvo2 doStep; SURVEY Appendix A)
//   K3 lookahead_kernel   a group of 8, 16 or 32 lanes per (episode, action): swept-disc collisions,
//                         occupancy-grid test, reward/done/event, next states, rotated joint-state rows
//                         (simulator/env.py:207-209,388-466; rl/policy/cadrl.py:118-165,236-337)
//   K5 select_kernel      warp per episode: reward + gamma^(dt v_pref) V, first-max argmax
//                         (rl/policy/multi_human_rl.py:72-82)
//   K2 step_kernel        committed env.step (+ optionally fused ORCA, block per episode)
//                         (simulator/env.py:340-466, simulator/agents/agent.py:202-228)
//
// This translation unit is compiled with -fmad=false: RVO2 is fp32 without contraction and
// the reference's Python float arithmetic is fp64 without contraction; every predicate
// (collision, reach-goal, discomfort, grid index) is evaluated in fp64 from the fp32 state
// in the reference's operation order so that flags are bit-exact against the oracle.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

#include "ebc_internal.cuh"

#define FULL 0xffffffffu
#define RVO_EPSILON 0.00001f

namespace {

struct Line { float px, py, dx, dy; };

__device__ __forceinline__ float det2(float ax, float ay, float bx, float by) { return ax * by - ay * bx; }
__device__ __forceinline__ float dot2(float ax, float ay, float bx, float by) { return ax * bx + ay * by; }

// Lane groups: a group = GW consecutive lanes of a warp (GW = 8, 16 or 32), its first lane `lane & (32 - GW)`.  Every
// ballot / shuffle / reduction below is confined to the group; `m` is the member mask of the lanes taking part (K1: the
// group's own lanes, group_mask; K3: FULL, its groups are the convergent lanes of whole warps).
template <int GW> __device__ __forceinline__ unsigned group_mask() {
  return (FULL >> (32 - GW)) << ((threadIdx.x & 31) & (32 - GW));
}
template <int GW> __device__ __forceinline__ unsigned grp_ballot(unsigned m, bool p) {
  return (__ballot_sync(m, p) >> ((threadIdx.x & 31) & (32 - GW))) & (FULL >> (32 - GW));
}
template <int GW> __device__ __forceinline__ float grp_min_f(unsigned m, float v) {
#pragma unroll
  for (int o = GW / 2; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(m, v, o, GW));
  return v;
}
template <int GW> __device__ __forceinline__ float grp_max_f(unsigned m, float v) {
#pragma unroll
  for (int o = GW / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(m, v, o, GW));
  return v;
}
template <int GW> __device__ __forceinline__ double grp_min_d(unsigned m, double v) {
#pragma unroll
  for (int o = GW / 2; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(m, v, o, GW));
  return v;
}

// The group's ORCA lines: line index = lane + GW * chunk.  A group = the GW lanes that solve one agent's LP: the whole
// warp (GW = 32), or a half warp (GW = 16: two agents per warp, every shuffle / ballot / reduction confined to the
// half through its member mask `m`; `lane` is then the lane index inside the half).  LPL (lines per lane) = 1 on the
// reference's live path (at most max_neighbors agent lines), 3 when obstacle half-planes are enabled (up to 96
// lines: at most 64 obstacle lines first, then at most 32 agent lines; GW = 32 only).  Every function below is the
// same arithmetic for all (GW, LPL).
template <int LPL> struct Lines { Line l[LPL]; };

template <int LPL, int GW>
__device__ __forceinline__ void bcast_line(unsigned m, const Lines<LPL> &L, int i, float &px, float &py, float &dx,
                                           float &dy) {
  const int il = i & (GW - 1), ic = i / GW;
  Line s = L.l[0];
#pragma unroll
  for (int c = 1; c < LPL; ++c)
    if (ic == c) s = L.l[c];
  px = __shfl_sync(m, s.px, il, GW); py = __shfl_sync(m, s.py, il, GW);
  dx = __shfl_sync(m, s.dx, il, GW); dy = __shfl_sync(m, s.dy, il, GW);
}

// RVO2 linearProgram1 with the scan over earlier lines done by the lanes that hold them.
// tLeft only grows and tRight only shrinks along the sequential scan, so "fails at some
// prefix" == "fails at the end", and the parallel-line failure is order-free (Appendix A.3).
template <int LPL, int GW>
__device__ bool lp1_warp(unsigned m, const Lines<LPL> &L, int lane, int i, float radius, float ox, float oy,
                         bool dir_opt, float &rx, float &ry) {
  float pix, piy, dix, diy;
  bcast_line<LPL, GW>(m, L, i, pix, piy, dix, diy);
  const float dp = dot2(pix, piy, dix, diy);
  const float disc = dp * dp + radius * radius - dot2(pix, piy, pix, piy);
  if (disc < 0.0f) return false;
  const float s = sqrtf(disc);
  float tl = -dp - s;
  float tr = -dp + s;
  float cr = INFINITY, cl = -INFINITY;
  bool bad = false;
#pragma unroll
  for (int c = 0; c < LPL; ++c) {
    const Line &M = L.l[c];
    const float den = det2(dix, diy, M.dx, M.dy);
    const float num = det2(M.dx, M.dy, pix - M.px, piy - M.py);
    const bool act = lane + GW * c < i;
    const bool par = fabsf(den) <= RVO_EPSILON;
    bad = bad || (act && par && (num < 0.0f));
    const float t = num / den;
    cr = fminf(cr, (act && !par && den >= 0.0f) ? t : INFINITY);
    cl = fmaxf(cl, (act && !par && den < 0.0f) ? t : -INFINITY);
  }
  cr = grp_min_f<GW>(m, cr);
  cl = grp_max_f<GW>(m, cl);
  tr = fminf(tr, cr);
  tl = fmaxf(tl, cl);
  if (__any_sync(m, bad) || tl > tr) return false;
  float tt;
  if (dir_opt) {
    tt = (dot2(ox, oy, dix, diy) > 0.0f) ? tr : tl;
  } else {
    tt = dot2(dix, diy, ox - pix, oy - piy);
    if (tt < tl) tt = tl;
    else if (tt > tr) tt = tr;
  }
  rx = pix + tt * dix;
  ry = piy + tt * diy;
  return true;
}

// RVO2 linearProgram2: the result only changes inside lp1, so the sequential "first violated
// line at or after i" is one ballot (per chunk).
template <int LPL, int GW>
__device__ int lp2_warp(unsigned m, const Lines<LPL> &L, int lane, int n, float radius, float ox, float oy,
                        bool dir_opt, float &rx, float &ry) {
  if (dir_opt) {
    rx = ox * radius;
    ry = oy * radius;
  } else if (dot2(ox, oy, ox, oy) > radius * radius) {
    const float inv = 1.0f / sqrtf(dot2(ox, oy, ox, oy));
    rx = (ox * inv) * radius;
    ry = (oy * inv) * radius;
  } else {
    rx = ox;
    ry = oy;
  }
  int i = 0;
  for (;;) {
    int first = -1;
#pragma unroll
    for (int c = 0; c < LPL; ++c) {
      const int idx = lane + GW * c;
      const bool viol = idx >= i && idx < n && det2(L.l[c].dx, L.l[c].dy, L.l[c].px - rx, L.l[c].py - ry) > 0.0f;
      const unsigned vm = grp_ballot<GW>(m, viol);
      if (first < 0 && vm != 0u) first = GW * c + __ffs(vm) - 1;
    }
    if (first < 0) return n;
    i = first;
    const float tx = rx, ty = ry;
    if (!lp1_warp<LPL, GW>(m, L, lane, i, radius, ox, oy, dir_opt, rx, ry)) {
      rx = tx;
      ry = ty;
      return i;
    }
    ++i;
  }
}

// RVO2 linearProgram3.  The projected problem keeps the first num_obst (obstacle) lines verbatim and replaces
// lines num_obst .. i-1 by their bisectors with line i (num_obst = 0 on the reference's live path).
template <int LPL, int GW>
__device__ void lp3_warp(unsigned m, const Lines<LPL> &L, int lane, int n, int num_obst, int begin, float radius,
                         float &rx, float &ry) {
  float distance = 0.0f;
  for (int i = begin; i < n; ++i) {
    float pix, piy, dix, diy;
    bcast_line<LPL, GW>(m, L, i, pix, piy, dix, diy);
    if (det2(dix, diy, pix - rx, piy - ry) > distance) {
      Lines<LPL> P;
      unsigned vm[LPL];
#pragma unroll
      for (int c = 0; c < LPL; ++c) {
        const Line &M = L.l[c];
        const int idx = lane + GW * c;
        bool valid = idx < i;
        const float d = det2(dix, diy, M.dx, M.dy);
        if (fabsf(d) <= RVO_EPSILON) {
          if (dot2(dix, diy, M.dx, M.dy) > 0.0f) valid = false;
          P.l[c].px = 0.5f * (pix + M.px);
          P.l[c].py = 0.5f * (piy + M.py);
        } else {
          const float t = det2(M.dx, M.dy, pix - M.px, piy - M.py) / d;
          P.l[c].px = pix + t * dix;
          P.l[c].py = piy + t * diy;
        }
        const float ddx = M.dx - dix, ddy = M.dy - diy;
        const float inv = 1.0f / sqrtf(dot2(ddx, ddy, ddx, ddy));
        P.l[c].dx = ddx * inv;
        P.l[c].dy = ddy * inv;
        if (LPL > 1 && idx < num_obst) {   // std::vector<Line> projLines(lines.begin(), lines.begin() + numObstLines)
          P.l[c] = M;
          valid = true;
        }
        vm[c] = grp_ballot<GW>(m, valid);
      }
      int cnt = 0;
#pragma unroll
      for (int c = 0; c < LPL; ++c) cnt += __popc(vm[c]);
      Lines<LPL> Q;
      if (LPL == 1) {
        int src = (int)__fns(vm[0], 0, lane + 1);   // lane k takes the k-th surviving line (order kept)
        if (lane >= cnt) src = lane;
        Q.l[0].px = __shfl_sync(m, P.l[0].px, src, GW);
        Q.l[0].py = __shfl_sync(m, P.l[0].py, src, GW);
        Q.l[0].dx = __shfl_sync(m, P.l[0].dx, src, GW);
        Q.l[0].dy = __shfl_sync(m, P.l[0].dy, src, GW);
      } else {
#pragma unroll
        for (int c = 0; c < LPL; ++c) {
          const int t = lane + GW * c;                   // target index: the t-th surviving line
          int sc = 0, sl = lane, base = 0;               // it sits in chunk sc, lane sl
#pragma unroll
          for (int k = 0; k < LPL; ++k) {
            const int nk = __popc(vm[k]);
            if (t >= base && t < base + nk) { sc = k; sl = (int)__fns(vm[k], 0, t - base + 1); }
            base += nk;
          }
          Q.l[c] = Line{0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
          for (int k = 0; k < LPL; ++k) {
            const float a = __shfl_sync(m, P.l[k].px, sl, GW), b = __shfl_sync(m, P.l[k].py, sl, GW);
            const float d0 = __shfl_sync(m, P.l[k].dx, sl, GW), d1 = __shfl_sync(m, P.l[k].dy, sl, GW);
            if (sc == k) { Q.l[c].px = a; Q.l[c].py = b; Q.l[c].dx = d0; Q.l[c].dy = d1; }
          }
        }
      }
      const float tx = rx, ty = ry;
      if (lp2_warp<LPL, GW>(m, Q, lane, cnt, radius, -diy, dix, true, rx, ry) < cnt) {
        rx = tx;
        ry = ty;
      }
      distance = det2(dix, diy, pix - rx, piy - ry);
    }
  }
}

// ---- ORCA obstacle half-planes (SURVEY 8f-4): RVO2 Agent::computeNeighbors (obstacle part) + the obstacle
//      section of Agent::computeNewVelocity, one warp per agent.  The episode's obstacle vertices are staged in
//      shared memory by the block; every lane tests two of them, the visible ones in range are ranked by
//      (distSq, RVO2's kd-tree visiting order), lane r builds the candidate line of neighbour r, and the
//      sequential "already covered by an earlier obstacle line" rule is resolved with one ballot per neighbour.
struct ObstV {                      // = ebc_obst_vertex, 48 bytes
  float px, py, ux, uy;
  short next, prev, convex, pad0;
  unsigned long long anc, anc_left, pad1;
};
static_assert(sizeof(ObstV) == sizeof(ebc_obst_vertex), "obstacle record layout");
constexpr int OBST_SCRATCH_FLOATS = 96 * 4 + 16;   // per warp: 96 lines (or 32 x 5 neighbour floats) + 64 sorted ids

__device__ __forceinline__ float left_of(float ax, float ay, float bx, float by, float cx, float cy) {
  return det2(ax - cx, ay - cy, bx - ax, by - ay);
}
__device__ __forceinline__ unsigned long long ballot64(bool p0, bool p1) {
  return (unsigned long long)__ballot_sync(FULL, p0) | ((unsigned long long)__ballot_sync(FULL, p1) << 32);
}
__device__ __forceinline__ unsigned long long shfl64(unsigned long long v, int src) {
  const unsigned lo = __shfl_sync(FULL, (unsigned)v, src), hi = __shfl_sync(FULL, (unsigned)(v >> 32), src);
  return (unsigned long long)lo | ((unsigned long long)hi << 32);
}

struct ObstCand {      // candidate line of one obstacle neighbour + what the cover test needs
  Line ln;
  float r1x, r1y, r2x, r2y;
  bool creates;
};

// the body of the loop of Agent::computeNewVelocity for one obstacle neighbour (everything but "alreadyCovered")
__device__ __forceinline__ void obstacle_candidate(const ObstV *so, int id, float px, float py, float vx, float vy,
                                                   float radius, float inv_th, ObstCand &out) {
  const ObstV &o1 = so[id];
  const ObstV &o2 = so[o1.next];
  const float r1x = o1.px - px, r1y = o1.py - py, r2x = o2.px - px, r2y = o2.py - py;
  out.r1x = r1x; out.r1y = r1y; out.r2x = r2x; out.r2y = r2y;
  out.creates = false;
  out.ln.px = 0.0f; out.ln.py = 0.0f; out.ln.dx = 1.0f; out.ln.dy = 0.0f;
  const float d1 = dot2(r1x, r1y, r1x, r1y), d2 = dot2(r2x, r2y, r2x, r2y);
  const float rsq = radius * radius;
  const float ovx = o2.px - o1.px, ovy = o2.py - o1.py;
  const float s = dot2(-r1x, -r1y, ovx, ovy) / dot2(ovx, ovy, ovx, ovy);
  const float qx = -r1x - s * ovx, qy = -r1y - s * ovy;
  const float dline = dot2(qx, qy, qx, qy);
  Line ln;
  if (s < 0.0f && d1 <= rsq) {
    if (o1.convex) {
      const float inv = 1.0f / sqrtf(dot2(-r1y, r1x, -r1y, r1x));
      ln.px = 0.0f; ln.py = 0.0f; ln.dx = -r1y * inv; ln.dy = r1x * inv;
      out.ln = ln; out.creates = true;
    }
    return;
  } else if (s > 1.0f && d2 <= rsq) {
    if (o2.convex && det2(r2x, r2y, o2.ux, o2.uy) >= 0.0f) {
      const float inv = 1.0f / sqrtf(dot2(-r2y, r2x, -r2y, r2x));
      ln.px = 0.0f; ln.py = 0.0f; ln.dx = -r2y * inv; ln.dy = r2x * inv;
      out.ln = ln; out.creates = true;
    }
    return;
  } else if (s >= 0.0f && s < 1.0f && dline <= rsq) {
    ln.px = 0.0f; ln.py = 0.0f; ln.dx = -o1.ux; ln.dy = -o1.uy;
    out.ln = ln; out.creates = true;
    return;
  }
  float llx, lly, rlx, rly;
  int a1 = id, a2 = o1.next;     // obstacle1 / obstacle2 after the oblique-view reassignment
  if (s < 0.0f && dline <= rsq) {
    if (!o1.convex) return;
    a2 = id;
    const float leg1 = sqrtf(d1 - rsq);
    const float inv = 1.0f / d1;
    llx = (r1x * leg1 - r1y * radius) * inv; lly = (r1x * radius + r1y * leg1) * inv;
    rlx = (r1x * leg1 + r1y * radius) * inv; rly = (-r1x * radius + r1y * leg1) * inv;
  } else if (s > 1.0f && dline <= rsq) {
    if (!o2.convex) return;
    a1 = o1.next;
    const float leg2 = sqrtf(d2 - rsq);
    const float inv = 1.0f / d2;
    llx = (r2x * leg2 - r2y * radius) * inv; lly = (r2x * radius + r2y * leg2) * inv;
    rlx = (r2x * leg2 + r2y * radius) * inv; rly = (-r2x * radius + r2y * leg2) * inv;
  } else {
    if (o1.convex) {
      const float leg1 = sqrtf(d1 - rsq);
      const float inv = 1.0f / d1;
      llx = (r1x * leg1 - r1y * radius) * inv; lly = (r1x * radius + r1y * leg1) * inv;
    } else { llx = -o1.ux; lly = -o1.uy; }
    if (o2.convex) {
      const float leg2 = sqrtf(d2 - rsq);
      const float inv = 1.0f / d2;
      rlx = (r2x * leg2 + r2y * radius) * inv; rly = (-r2x * radius + r2y * leg2) * inv;
    } else { rlx = o1.ux; rly = o1.uy; }
  }
  const ObstV &A1 = so[a1];
  const ObstV &A2 = so[a2];
  const ObstV &LN = so[A1.prev];
  bool left_foreign = false, right_foreign = false;
  if (A1.convex && det2(llx, lly, -LN.ux, -LN.uy) >= 0.0f) {
    llx = -LN.ux; lly = -LN.uy;
    left_foreign = true;
  }
  if (A2.convex && det2(rlx, rly, A2.ux, A2.uy) <= 0.0f) {
    rlx = A2.ux; rly = A2.uy;
    right_foreign = true;
  }
  const float lcx = inv_th * (A1.px - px), lcy = inv_th * (A1.py - py);
  const float rcx = inv_th * (A2.px - px), rcy = inv_th * (A2.py - py);
  const float cvx = rcx - lcx, cvy = rcy - lcy;
  const bool same = a1 == a2;
  const float t = same ? 0.5f : dot2(vx - lcx, vy - lcy, cvx, cvy) / dot2(cvx, cvy, cvx, cvy);
  const float tl = dot2(vx - lcx, vy - lcy, llx, lly);
  const float tr = dot2(vx - rcx, vy - rcy, rlx, rly);
  if ((t < 0.0f && tl < 0.0f) || (same && tl < 0.0f && tr < 0.0f)) {
    const float wx = vx - lcx, wy = vy - lcy;
    const float inv = 1.0f / sqrtf(dot2(wx, wy, wx, wy));
    const float ux = wx * inv, uy = wy * inv;
    ln.dx = uy; ln.dy = -ux;
    ln.px = lcx + radius * inv_th * ux; ln.py = lcy + radius * inv_th * uy;
    out.ln = ln; out.creates = true;
    return;
  } else if (t > 1.0f && tr < 0.0f) {
    const float wx = vx - rcx, wy = vy - rcy;
    const float inv = 1.0f / sqrtf(dot2(wx, wy, wx, wy));
    const float ux = wx * inv, uy = wy * inv;
    ln.dx = uy; ln.dy = -ux;
    ln.px = rcx + radius * inv_th * ux; ln.py = rcy + radius * inv_th * uy;
    out.ln = ln; out.creates = true;
    return;
  }
  float dcut, dleft, dright;
  if (t < 0.0f || t > 1.0f || same) dcut = INFINITY;
  else { const float ax = vx - (lcx + t * cvx), ay = vy - (lcy + t * cvy); dcut = dot2(ax, ay, ax, ay); }
  if (tl < 0.0f) dleft = INFINITY;
  else { const float ax = vx - (lcx + tl * llx), ay = vy - (lcy + tl * lly); dleft = dot2(ax, ay, ax, ay); }
  if (tr < 0.0f) dright = INFINITY;
  else { const float ax = vx - (rcx + tr * rlx), ay = vy - (rcy + tr * rly); dright = dot2(ax, ay, ax, ay); }
  if (dcut <= dleft && dcut <= dright) {
    ln.dx = -A1.ux; ln.dy = -A1.uy;
    ln.px = lcx + radius * inv_th * -ln.dy; ln.py = lcy + radius * inv_th * ln.dx;
    out.ln = ln; out.creates = true;
  } else if (dleft <= dright) {
    if (left_foreign) return;
    ln.dx = llx; ln.dy = lly;
    ln.px = lcx + radius * inv_th * -ln.dy; ln.py = lcy + radius * inv_th * ln.dx;
    out.ln = ln; out.creates = true;
  } else {
    if (right_foreign) return;
    ln.dx = -rlx; ln.dy = -rly;
    ln.px = rcx + radius * inv_th * -ln.dy; ln.py = rcy + radius * inv_th * ln.dx;
    out.ln = ln; out.creates = true;
  }
}

// Obstacle lines of one agent into linebuf[0 .. n) (shared memory, this warp's); returns n = numObstLines.
// `ids` = this warp's 64 bytes for the sorted neighbour list.
__device__ int obstacle_lines_warp(const ObstV *so, int V, int lane, float px, float py, float vx, float vy, float radius,
                                   float max_speed, float th_obst, Line *linebuf, unsigned char *ids) {
  const float rr = th_obst * max_speed + radius;
  const float range_sq = rr * rr;
  float d[2];
  bool vis[2], lok[2], nearl[2];
  unsigned long long anc[2], ancl[2];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int v = lane + 32 * c;
    d[c] = INFINITY; vis[c] = false; lok[c] = false; nearl[c] = false; anc[c] = 0ull; ancl[c] = 0ull;
    if (v < V) {
      const ObstV &o1 = so[v];
      const ObstV &o2 = so[o1.next];
      const float al = left_of(o1.px, o1.py, o2.px, o2.py, px, py);
      const float ex = o2.px - o1.px, ey = o2.py - o1.py;
      const float dsl = al * al / dot2(ex, ey, ex, ey);
      nearl[c] = al >= 0.0f;                 // the kd-tree descends into the left child first
      lok[c] = dsl < range_sq;               // queryObstacleTreeRecursive crosses this node's line
      vis[c] = al < 0.0f;                    // agent on the right side: it can see the edge
      anc[c] = o1.anc; ancl[c] = o1.anc_left;
      // distSqPointLineSegment(o1, o2, p)
      const float r = dot2(px - o1.px, py - o1.py, ex, ey) / dot2(ex, ey, ex, ey);
      if (r < 0.0f) d[c] = dot2(px - o1.px, py - o1.py, px - o1.px, py - o1.py);
      else if (r > 1.0f) d[c] = dot2(px - o2.px, py - o2.py, px - o2.px, py - o2.py);
      else { const float qx = px - (o1.px + r * ex), qy = py - (o1.py + r * ey); d[c] = dot2(qx, qy, qx, qy); }
    }
  }
  const unsigned long long side_l = ballot64(nearl[0], nearl[1]);
  const unsigned long long line_ok = ballot64(lok[0], lok[1]);
  bool sel[2];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    // reached by the traversal: every ancestor whose FAR subtree holds this node has its line within range
    const unsigned long long far_anc = anc[c] & (ancl[c] ^ side_l);
    sel[c] = vis[c] && lok[c] && ((far_anc & ~line_ok) == 0ull) && d[c] < range_sq;
  }
  const unsigned long long selm = ballot64(sel[0], sel[1]);
  const int M = __popcll(selm);
  if (M == 0) return 0;
  // rank by (distSq, visiting order of the near-first in-order traversal)
  int rank[2] = {0, 0};
  unsigned long long m = selm;
  while (m) {
    const int k = __ffsll((long long)m) - 1;
    m &= m - 1;
    const int kl = k & 31;
    const float dk = k < 32 ? __shfl_sync(FULL, d[0], kl) : __shfl_sync(FULL, d[1], kl);
    const unsigned long long ak = k < 32 ? shfl64(anc[0], kl) : shfl64(anc[1], kl);
    const unsigned long long alk = k < 32 ? shfl64(ancl[0], kl) : shfl64(ancl[1], kl);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int x = lane + 32 * c;
      bool before;                            // k is visited before x
      if (x == k) before = false;
      else if ((anc[c] >> k) & 1ull) before = (((ancl[c] ^ side_l) >> k) & 1ull) != 0ull;      // k above x: x in k's far subtree
      else if ((ak >> x) & 1ull) before = (((alk ^ side_l) >> x) & 1ull) == 0ull;             // x above k: k in x's near subtree
      else {
        const unsigned long long diff = (ancl[c] ^ alk) & anc[c] & ak;                        // the lowest common ancestor
        before = ((alk ^ side_l) & diff) == 0ull;                                             // k on its near side
      }
      rank[c] += (dk < d[c] || (dk == d[c] && before)) ? 1 : 0;
    }
  }
  __syncwarp();
#pragma unroll
  for (int c = 0; c < 2; ++c)
    if (sel[c]) ids[rank[c]] = (unsigned char)(lane + 32 * c);
  __syncwarp();
  // candidate lines: lane r (and r + 32) takes neighbour r
  const float inv_th = 1.0f / th_obst;
  ObstCand cand[2];
  bool accepted[2] = {false, false};
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int r = lane + 32 * c;
    cand[c].creates = false;
    cand[c].r1x = cand[c].r1y = cand[c].r2x = cand[c].r2y = 0.0f;
    cand[c].ln.px = cand[c].ln.py = 0.0f; cand[c].ln.dx = 1.0f; cand[c].ln.dy = 0.0f;
    if (r < M) obstacle_candidate(so, ids[r], px, py, vx, vy, radius, inv_th, cand[c]);
  }
  // "already covered by a previously constructed obstacle ORCA line": sequential over the neighbours
  for (int i = 0; i < M; ++i) {
    const int il = i & 31;
    float r1x, r1y, r2x, r2y;
    if (i < 32) {
      r1x = __shfl_sync(FULL, cand[0].r1x, il); r1y = __shfl_sync(FULL, cand[0].r1y, il);
      r2x = __shfl_sync(FULL, cand[0].r2x, il); r2y = __shfl_sync(FULL, cand[0].r2y, il);
    } else {
      r1x = __shfl_sync(FULL, cand[1].r1x, il); r1y = __shfl_sync(FULL, cand[1].r1y, il);
      r2x = __shfl_sync(FULL, cand[1].r2x, il); r2y = __shfl_sync(FULL, cand[1].r2y, il);
    }
    bool cov = false;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const Line &J = cand[c].ln;
      const bool hit = det2(inv_th * r1x - J.px, inv_th * r1y - J.py, J.dx, J.dy) - inv_th * radius >= -RVO_EPSILON &&
                       det2(inv_th * r2x - J.px, inv_th * r2y - J.py, J.dx, J.dy) - inv_th * radius >= -RVO_EPSILON;
      cov = cov || (accepted[c] && hit);     // accepted lines all belong to neighbours before i
    }
    const bool covered = __any_sync(FULL, cov);
    if (!covered) {
      if (i < 32) { if (lane == il && cand[0].creates) accepted[0] = true; }
      else { if (lane == il && cand[1].creates) accepted[1] = true; }
    }
  }
  // compact the accepted lines, in neighbour order, to linebuf[0 .. n)
  const unsigned a0 = __ballot_sync(FULL, accepted[0]), a1 = __ballot_sync(FULL, accepted[1]);
  const unsigned below = (1u << lane) - 1u;
  if (accepted[0]) linebuf[__popc(a0 & below)] = cand[0].ln;
  if (accepted[1]) linebuf[__popc(a0) + __popc(a1 & below)] = cand[1].ln;
  __syncwarp();
  return __popc(a0) + __popc(a1);
}

// One RVO2 agent step by one group of GW lanes (m = its member mask, lane = the index inside it).  Candidates (the other
// agents, in the reference's list order) sit two per lane: index lane and lane + GW.  `scratch` = this warp's shared memory: 32*5 floats, or
// OBST_SCRATCH_FLOATS with obstacle half-planes (so / V: the episode's obstacle vertices in shared memory).
template <bool OBST, int GW>
__device__ void orca_agent_warp(unsigned m, int lane, float px, float py, float vx, float vy, float radius, float max_speed,
                                float prefx, float prefy, const float (&cpx)[2], const float (&cpy)[2],
                                const float (&cvx)[2], const float (&cvy)[2], const float (&crad)[2],
                                const bool (&cval)[2], int n_chunks, float neighbor_dist, int max_nb,
                                float time_horizon, float time_step, float *scratch, float &outx, float &outy,
                                const ObstV *so = nullptr, int V = 0, float th_obst = 0.0f) {
  constexpr int LPL = OBST ? 3 : 1;
  static_assert(!OBST || GW == 32, "obstacle half-planes use the whole warp");
  // Agent::insertAgentNeighbor == keep the max_nb smallest (distSq, arrival index) below range
  float d[2];
  unsigned vmask[2] = {0u, 0u};
  const float range_sq = neighbor_dist * neighbor_dist;
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const float ddx = px - cpx[c], ddy = py - cpy[c];
    d[c] = dot2(ddx, ddy, ddx, ddy);
    const bool ok = (c < n_chunks) && cval[c] && (d[c] < range_sq);
    vmask[c] = grp_ballot<GW>(m, ok);
  }
  int rank[2] = {0, 0};
#pragma unroll
  for (int c2 = 0; c2 < 2; ++c2) {
    if (c2 >= n_chunks) break;
    unsigned rest = vmask[c2];
    while (rest) {
      const int l = __ffs(rest) - 1;
      rest &= rest - 1;
      const float dk = __shfl_sync(m, d[c2], l, GW);
      const int k = l + GW * c2;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int me = lane + GW * c;
        rank[c] += (dk < d[c] || (dk == d[c] && k < me)) ? 1 : 0;
      }
    }
  }
  const int total = __popc(vmask[0]) + __popc(vmask[1]);
  int cnt = total < max_nb ? total : max_nb;
  __syncwarp(m);
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    if ((vmask[c] >> lane) & 1u) {
      if (rank[c] < cnt) {
        float *s = scratch + rank[c] * 5;
        s[0] = cpx[c]; s[1] = cpy[c]; s[2] = cvx[c]; s[3] = cvy[c]; s[4] = crad[c];
      }
    }
  }
  __syncwarp(m);
  Line A = {0.0f, 0.0f, 1.0f, 0.0f};      // agent line `lane`
  if (lane < cnt) {
    const float *s = scratch + lane * 5;
    const float rpx = s[0] - px, rpy = s[1] - py;
    const float rvx = vx - s[2], rvy = vy - s[3];
    const float dist_sq = dot2(rpx, rpy, rpx, rpy);
    const float R = radius + s[4];
    const float R_sq = R * R;
    const float inv_th = 1.0f / time_horizon;
    float ux, uy;
    if (dist_sq > R_sq) {
      const float wx = rvx - inv_th * rpx, wy = rvy - inv_th * rpy;
      const float wlen_sq = dot2(wx, wy, wx, wy);
      const float dp1 = dot2(wx, wy, rpx, rpy);
      if (dp1 < 0.0f && dp1 * dp1 > R_sq * wlen_sq) {
        const float wlen = sqrtf(wlen_sq);
        const float inv = 1.0f / wlen;
        const float uwx = wx * inv, uwy = wy * inv;
        A.dx = uwy;
        A.dy = -uwx;
        const float sc = R * inv_th - wlen;
        ux = sc * uwx;
        uy = sc * uwy;
      } else {
        const float leg = sqrtf(dist_sq - R_sq);
        const float inv = 1.0f / dist_sq;
        if (det2(rpx, rpy, wx, wy) > 0.0f) {
          A.dx = (rpx * leg - rpy * R) * inv;
          A.dy = (rpx * R + rpy * leg) * inv;
        } else {
          A.dx = (-(rpx * leg + rpy * R)) * inv;
          A.dy = (-(-rpx * R + rpy * leg)) * inv;
        }
        const float dp2 = dot2(rvx, rvy, A.dx, A.dy);
        ux = dp2 * A.dx - rvx;
        uy = dp2 * A.dy - rvy;
      }
    } else {
      const float inv_ts = 1.0f / time_step;
      const float wx = rvx - inv_ts * rpx, wy = rvy - inv_ts * rpy;
      const float wlen = sqrtf(dot2(wx, wy, wx, wy));
      const float inv = 1.0f / wlen;
      const float uwx = wx * inv, uwy = wy * inv;
      A.dx = uwy;
      A.dy = -uwx;
      const float sc = R * inv_ts - wlen;
      ux = sc * uwx;
      uy = sc * uwy;
    }
    A.px = vx + 0.5f * ux;
    A.py = vy + 0.5f * uy;
  }
  __syncwarp(m);
  Lines<LPL> L;
  int num_obst = 0;
  if (OBST) {
    // obstacle lines first (Agent::computeNewVelocity), then the agent lines: at most 64 + 32, all of them kept like
    // RVO2 does
    Line *linebuf = reinterpret_cast<Line *>(scratch);
    unsigned char *ids = reinterpret_cast<unsigned char *>(scratch + 96 * 4);
    num_obst = obstacle_lines_warp(so, V, lane, px, py, vx, vy, radius, max_speed, th_obst, linebuf, ids);
    if (lane < cnt) linebuf[num_obst + lane] = A;
    __syncwarp(m);
#pragma unroll
    for (int c = 0; c < LPL; ++c) {
      const int idx = lane + 32 * c;
      const Line Z = {0.0f, 0.0f, 1.0f, 0.0f};
      L.l[c] = idx < num_obst + cnt ? linebuf[idx] : Z;
    }
    __syncwarp(m);
  } else {
    L.l[0] = A;
  }
  const int n_lines = num_obst + cnt;
  float rx, ry;
  const int fail = lp2_warp<LPL, GW>(m, L, lane, n_lines, max_speed, prefx, prefy, false, rx, ry);
  if (fail < n_lines) lp3_warp<LPL, GW>(m, L, lane, n_lines, num_obst, fail, max_speed, rx, ry);
  outx = rx;
  outy = ry;
}

// simulator/policy/orca.py:113-119,136-140 (float64 in Python, narrowed at the rvo2 boundary)
__device__ __forceinline__ void orca_self_params(float px, float py, float gx, float gy, float radius,
                                                 double safety, float &r_out, float &prefx, float &prefy) {
  r_out = (float)((double)radius + 0.01 + safety);
  const double vx = (double)gx - (double)px, vy = (double)gy - (double)py;
  const double speed = sqrt(vx * vx + vy * vy);
  if (speed > 1.0) {
    prefx = (float)(vx / speed);
    prefy = (float)(vy / speed);
  } else {
    prefx = (float)vx;
    prefy = (float)vy;
  }
}

// Stage the episode's obstacle vertices in shared memory (16-byte words; the whole block takes part).
__device__ __forceinline__ int stage_obstacles(const ebc_config &c, const ebc_state &st, int e, ObstV *so, int tid,
                                               int nthreads) {
  int V = st.obst_count[e];
  V = V < 0 ? 0 : (V > c.max_obst ? c.max_obst : V);
  const uint4 *src = reinterpret_cast<const uint4 *>(st.obst + (size_t)e * c.max_obst);
  uint4 *dst = reinterpret_cast<uint4 *>(so);
  for (int i = tid; i < V * 3; i += nthreads) dst[i] = src[i];
  return V;
}

// Policy of human h of episode e, computed by one warp (env.py:392-405).
template <bool OBST, int GW>
__device__ void human_policy_warp(unsigned m, const ebc_config &c, const ebc_state &st, int e, int h, int H, int lane,
                                  float *scratch, float &nvx, float &nvy, const ObstV *so = nullptr, int V = 0) {
  const int Hm = c.max_humans;
  const float4 *pv = reinterpret_cast<const float4 *>(st.hum_pv) + (size_t)e * Hm;
  const float4 *gr = reinterpret_cast<const float4 *>(st.hum_gr) + (size_t)e * Hm;
  const float4 me_pv = pv[h], me_gr = gr[h];
  int ty = st.hum_type[(size_t)e * Hm + h];
  if (ty > 2) ty = 0;
  if (c.human_policy[ty] == EBC_POLICY_LINEAR) {   // simulator/policy/linear.py:17-23
    const double th = atan2((double)me_gr.y - (double)me_pv.y, (double)me_gr.x - (double)me_pv.x);
    nvx = (float)(cos(th) * (double)me_gr.z);
    nvy = (float)(sin(th) * (double)me_gr.z);
    return;
  }
  const int n_cand = H + (c.robot_visible ? 1 : 0);
  const int n_chunks = (n_cand + GW - 1) / GW;
  float cpx[2], cpy[2], cvx[2], cvy[2], crad[2];
  bool cval[2];
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const int j = lane + GW * ch;
    cval[ch] = false;
    cpx[ch] = cpy[ch] = cvx[ch] = cvy[ch] = crad[ch] = 0.0f;
    if (j < H && j != h) {
      const float4 p = pv[j];
      cpx[ch] = p.x; cpy[ch] = p.y; cvx[ch] = p.z; cvy[ch] = p.w;
      crad[ch] = (float)((double)gr[j].w + 0.01 + c.orca_safety_space);
      cval[ch] = true;
    } else if (j == H && c.robot_visible) {   // env.py:401-402: robot appended last
      const float4 p = reinterpret_cast<const float4 *>(st.rob_pv)[e];
      cpx[ch] = p.x; cpy[ch] = p.y; cvx[ch] = p.z; cvy[ch] = p.w;
      crad[ch] = (float)((double)st.rob_gr[(size_t)e * 4 + 3] + 0.01 + c.orca_safety_space);
      cval[ch] = true;
    }
  }
  float r_self, prefx, prefy;
  orca_self_params(me_pv.x, me_pv.y, me_gr.x, me_gr.y, me_gr.w, c.orca_safety_space, r_self, prefx, prefy);
  orca_agent_warp<OBST, GW>(m, lane, me_pv.x, me_pv.y, me_pv.z, me_pv.w, r_self, me_gr.z, prefx, prefy, cpx, cpy, cvx, cvy,
                            crad, cval, n_chunks, c.orca_neighbor_dist, c.orca_max_neighbors, c.orca_time_horizon,
                            (float)c.time_step, scratch, nvx, nvy, so, V, c.orca_time_horizon_obst);
}

// K1, one group of GW lanes per human: the whole warp, or a half warp (two humans per warp) when every human has at
// most 32 candidates and 16 ORCA lines -- same arithmetic, bit-identical results, half the warp-instructions per human.
template <int GW>
__global__ void __launch_bounds__(EBC_THREADS) orca_kernel(const ebc_config c, const ebc_state st,
                                                           const uint8_t *__restrict__ active) {
  constexpr int GPW = 32 / GW;
  __shared__ float scratch[EBC_WARPS_PER_BLOCK * GPW][32 * 5];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, sub = lane / GW, gl = lane % GW;
  const long long w = ((long long)blockIdx.x * EBC_WARPS_PER_BLOCK + warp) * GPW + sub;
  const int e = (int)(w / c.max_humans), h = (int)(w % c.max_humans);
  if (e >= c.n_episodes) return;
  if (active && !active[e]) return;      // episodes the following step leaves untouched (ebc_orca_step)
  const int H = st.hum_count[e];
  if (h >= H) return;
  float nvx, nvy;
  human_policy_warp<false, GW>(group_mask<GW>(), c, st, e, h, H, gl, scratch[warp * GPW + sub], nvx, nvy);
  if (gl == 0)
    reinterpret_cast<float2 *>(st.hum_nv)[(size_t)e * c.max_humans + h] = make_float2(nvx, nvy);
}

// Robot as ORCA agent 0 over humans + static discs (rl/train.py:99-143).  WPB warps (= episodes) per block; with
// obstacle half-planes one episode per block, its obstacle vertices staged in shared memory.
template <bool OBST, int WPB>
__global__ void __launch_bounds__(WPB * 32) robot_orca_kernel(const ebc_config c, const ebc_state st,
                                                              double safety, double *out) {
  __shared__ float scratch[WPB][OBST ? OBST_SCRATCH_FLOATS : 32 * 5];
  __shared__ __align__(16) ObstV so[OBST ? 64 : 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * WPB + warp;
  if (e >= c.n_episodes) return;
  int V = 0;
  if (OBST) {
    V = stage_obstacles(c, st, e, so, threadIdx.x, WPB * 32);
    __syncthreads();
  }
  const int Hm = c.max_humans, Sm = c.max_statics;
  const int H = st.hum_count[e], S = st.stat_count[e];
  const float4 *pv = reinterpret_cast<const float4 *>(st.hum_pv) + (size_t)e * Hm;
  const float4 *gr = reinterpret_cast<const float4 *>(st.hum_gr) + (size_t)e * Hm;
  const float4 *sd = reinterpret_cast<const float4 *>(st.stat) + (size_t)e * Sm;
  float cpx[2], cpy[2], cvx[2], cvy[2], crad[2];
  bool cval[2];
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const int j = lane + 32 * ch;
    cval[ch] = false;
    cpx[ch] = cpy[ch] = cvx[ch] = cvy[ch] = crad[ch] = 0.0f;
    if (j < H) {
      const float4 p = pv[j];
      cpx[ch] = p.x; cpy[ch] = p.y; cvx[ch] = p.z; cvy[ch] = p.w;
      crad[ch] = (float)((double)gr[j].w + 0.01 + safety);
      cval[ch] = true;
    } else if (j < H + S) {
      const float4 p = sd[j - H];
      cpx[ch] = p.x; cpy[ch] = p.y;
      crad[ch] = (float)((double)p.z + 0.01 + safety);
      cval[ch] = true;
    }
  }
  const float4 rp = reinterpret_cast<const float4 *>(st.rob_pv)[e];
  const float4 rg = reinterpret_cast<const float4 *>(st.rob_gr)[e];
  float r_self, prefx, prefy, vx, vy;
  orca_self_params(rp.x, rp.y, rg.x, rg.y, rg.w, safety, r_self, prefx, prefy);
  orca_agent_warp<OBST, 32>(FULL, lane, rp.x, rp.y, rp.z, rp.w, r_self, rg.z, prefx, prefy, cpx, cpy, cvx, cvy, crad, cval,
                            (H + S + 31) >> 5, c.orca_neighbor_dist, c.orca_max_neighbors, c.orca_time_horizon,
                            (float)c.time_step, scratch[warp], vx, vy, so, V, c.orca_time_horizon_obst);
  if (lane == 0) {
    out[(size_t)e * 2] = (double)vx;
    out[(size_t)e * 2 + 1] = (double)vy;
  }
}

// simulator/utils/collisions.py:4-26 with (x3, y3) = (0, 0)
__device__ __forceinline__ double point_to_segment_dist0(double x1, double y1, double x2, double y2) {
  const double px = x2 - x1, py = y2 - y1;
  if (px == 0.0 && py == 0.0) return sqrt((0.0 - x1) * (0.0 - x1) + (0.0 - y1) * (0.0 - y1));
  double u = ((0.0 - x1) * px + (0.0 - y1) * py) / (px * px + py * py);
  if (u > 1.0) u = 1.0;
  else if (u < 0.0) u = 0.0;
  const double x = x1 + u * px, y = y1 + u * py;
  return sqrt((x - 0.0) * (x - 0.0) + (y - 0.0) * (y - 0.0));
}

struct Outcome {
  double dmin[3];
  double end_x, end_y, dist_to_goal, reward;
  double min_dist; // Danger.min_dist (reward.py:138-166): the dmin of the type that triggered it
  double cs, sn;   // cos / sin of the robot's heading after the action (non-holonomic), computed once per action
  int done, event;
};

// The humans of one episode over a group of G lanes: lane l holds humans l + G * chunk, a second chunk only for G = 32
// (K3 gives a smaller group only states of at most G rows).
struct EpisodeHumans {
  float4 pv[2];
  float rad[2];
  int type[2];   // -1 = empty slot
};

// reward.py:80-181 and the Info classes: the priority chain from the three dmin / four collision flags
__device__ __forceinline__ void classify_outcome(const ebc_config &c, const float4 rg, double gt, double a1,
                                                 const bool (&coll)[3], bool coll_obst, Outcome &o) {
  const double rrad = rg.w, dt = c.time_step;
  const double gdx = o.end_x - (double)rg.x, gdy = o.end_y - (double)rg.y;
  const double dist = sqrt(gdx * gdx + gdy * gdy);
  o.dist_to_goal = dist;
  const bool reaching = dist < rrad;
  const double goal_reward = c.has_max_goal_distance ? 1.0 - dist / c.max_goal_distance : 0.0;
  double reward = c.new_reward ? goal_reward : 0.0;
  int done, ev;
  o.min_dist = 0.0;
  if (gt >= c.time_limit) { done = 1; ev = EBC_EV_TIMEOUT; }
  else if (coll[EBC_CHILD]) { reward += c.collision_penalty_child; done = 1; ev = EBC_EV_COLLISION_CHILD; }
  else if (coll[EBC_BICYCLE]) { reward += c.collision_penalty_bicycle; done = 1; ev = EBC_EV_COLLISION_BICYCLE; }
  else if (coll[EBC_ADULT]) { reward += c.collision_penalty_adult; done = 1; ev = EBC_EV_COLLISION_ADULT; }
  else if (coll_obst) { reward += c.collision_penalty_obstacle; done = 1; ev = EBC_EV_COLLISION_OBSTACLE; }
  else if (reaching) {
    if (c.new_reward) {
      double tr;
      if (gt < c.time_good) tr = 1.0;
      else if (gt <= c.time_max) tr = (c.time_max - gt) / (c.time_max - c.time_good);
      else tr = 0.0;
      reward += tr;
    } else {
      reward += c.success_reward;
    }
    done = 1; ev = EBC_EV_REACH_GOAL;
  } else if (o.dmin[EBC_CHILD] < c.discomfort_dist_child) {
    reward = (o.dmin[EBC_CHILD] - c.discomfort_dist_child) * c.discomfort_penalty_factor_child * dt;
    o.min_dist = o.dmin[EBC_CHILD];
    done = 0; ev = EBC_EV_DANGER;
  } else if (o.dmin[EBC_BICYCLE] < c.discomfort_dist_bicycle) {
    reward = (o.dmin[EBC_BICYCLE] - c.discomfort_dist_bicycle) * c.discomfort_penalty_factor_bicycle * dt;
    o.min_dist = o.dmin[EBC_BICYCLE];
    done = 0; ev = EBC_EV_DANGER;
  } else if (o.dmin[EBC_ADULT] < c.discomfort_dist_adult) {
    reward = (o.dmin[EBC_ADULT] - c.discomfort_dist_adult) * c.discomfort_penalty_factor_adult * dt;
    o.min_dist = o.dmin[EBC_ADULT];
    done = 0; ev = EBC_EV_DANGER;
  } else if (c.robot_kinematics != EBC_KIN_HOLONOMIC && fabs(a1) > 0.0 && c.rotation_penalty_factor != 0.0) {
    reward = fabs(a1) * c.rotation_penalty_factor;
    done = 0; ev = EBC_EV_NOTHING;
  } else { reward = 0.0; done = 0; ev = EBC_EV_NOTHING; }
  o.reward = reward; o.done = done; o.event = ev;
}

// env.py:424-444 for one (episode, action) of an episode with H humans, cooperatively by a group of G lanes (lane = the
// index inside it), which load the humans into `hm` (the commit integrates them afterwards); the result is uniform over
// the group.  The group's lanes take part in full warps (member mask FULL).
template <int G>
__device__ void evaluate_action(const ebc_config &c, const ebc_state &st, int e, int lane, int H, const float4 rp,
                                const float4 rg, double theta, double gt, double a0, double a1, EpisodeHumans &hm,
                                Outcome &o) {
  const double rpx = rp.x, rpy = rp.y, rrad = rg.w;
  const double dt = c.time_step;
  double avx, avy;
  if (c.robot_kinematics == EBC_KIN_HOLONOMIC) {   // collisions.py:37-42, agent.py:164-176
    avx = a0;
    avy = a1;
    o.cs = 0.0; o.sn = 0.0;
    o.end_x = rpx + a0 * dt;
    o.end_y = rpy + a1 * dt;
  } else {
    // collisions.py:39-41 uses action.r + theta, agent.py:172-183 theta + action.r: the same double
    const double th = theta + a1;
    o.cs = cos(th);
    o.sn = sin(th);
    avx = a0 * o.cs;
    avy = a0 * o.sn;
    o.end_x = rpx + o.cs * a0 * dt;
    o.end_y = rpy + o.sn * a0 * dt;
  }
  const int Hm = c.max_humans;
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const int h = lane + G * ch;
    hm.type[ch] = -1;
    hm.pv[ch] = make_float4(0.f, 0.f, 0.f, 0.f);
    hm.rad[ch] = 0.f;
    if ((G == 32 || ch == 0) && h < H) {
      hm.pv[ch] = reinterpret_cast<const float4 *>(st.hum_pv)[(size_t)e * Hm + h];
      hm.rad[ch] = st.hum_gr[((size_t)e * Hm + h) * 4 + 3];
      hm.type[ch] = st.hum_type[(size_t)e * Hm + h];
    }
  }
  // env.py:303-338: per type, list order, dmin frozen at the first collision
  double closest[2] = {INFINITY, INFINITY};
  unsigned long long collm = 0ull, typem[3] = {0ull, 0ull, 0ull};
  const int n_ch = G == 32 && c.max_humans > 32 ? 2 : 1;   // lanes hold humans 32..63 only when the batch has that many
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    if (ch >= n_ch) break;
    const bool valid = hm.type[ch] >= 0 && hm.type[ch] <= 2;
    const double px = (double)hm.pv[ch].x - rpx, py = (double)hm.pv[ch].y - rpy;
    const double vx = (double)hm.pv[ch].z - avx, vy = (double)hm.pv[ch].w - avy;
    const double ex = px + vx * dt, ey = py + vy * dt;
    closest[ch] = point_to_segment_dist0(px, py, ex, ey) - (double)hm.rad[ch] - rrad;
    collm |= (unsigned long long)grp_ballot<G>(FULL, valid && closest[ch] < 0.0) << (G * ch);
#pragma unroll
    for (int t = 0; t < 3; ++t)
      typem[t] |= (unsigned long long)grp_ballot<G>(FULL, valid && hm.type[ch] == t) << (G * ch);
  }
  bool coll[3];
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    const unsigned long long cm = collm & typem[t];
    coll[t] = cm != 0ull;
    const unsigned lo = (unsigned)cm, hi = (unsigned)(cm >> 32);   // __ffsll(cm) - 1 by halves: fewer registers
    const int first = lo ? __ffs(lo) - 1 : (hi ? 31 + __ffs(hi) : 64);
    double local = INFINITY;
#pragma unroll
    for (int ch = 0; ch < 2; ++ch)
      if (hm.type[ch] == t && lane + G * ch < first) local = fmin(local, closest[ch]);
    o.dmin[t] = grp_min_d<G>(FULL, local);
  }
  // env.py:227-261 on the rectangle list
  bool coll_obst = false;
  {
    const int ix = (int)rint((o.end_x + c.map_size_m / 2.0) / c.map_resolution);
    const int iy = (int)rint((o.end_y + c.map_size_m / 2.0) / c.map_resolution);
    const int sz = (int)ceil(rrad / sqrt(2.0) / c.map_resolution);
    const int GR = (int)rint(c.map_size_m / c.map_resolution);
    int sx = ix - sz, ex = sx + sz * 2, sy = iy - sz, ey = sy + sz * 2;
    sx = max(sx, 0); ex = min(ex, GR); sy = max(sy, 0); ey = min(ey, GR);
    const int R = st.rect_count[e];
    bool hit = false;
    if (ex > sx && ey > sy) {
      const short4 *rc = reinterpret_cast<const short4 *>(st.rect) + (size_t)e * c.max_rects;
      for (int j = lane; j < R; j += G) {
        const short4 r = rc[j];
        hit |= (sx < r.z && r.x < ex && sy < r.w && r.y < ey);
      }
    }
    coll_obst = grp_ballot<G>(FULL, hit) != 0u;
  }
  classify_outcome(c, rg, gt, a1, coll, coll_obst, o);
}

// rl/policy/cadrl.py:236-337, one row, fp32 (-fmad=false keeps torch's separate mul/add).
// robot = (px, py, vx, vy, radius, gx, gy, v_pref, theta), entity = (px1, py1, vx1, vy1, radius1, type)
struct RobotRow { float px, py, vx, vy, radius, gx, gy, v_pref, theta; };

__device__ __forceinline__ void rotate_row(const RobotRow &r, float px1, float py1, float vx1, float vy1,
                                           float radius1, int type1, int rotate_theta, int D, float *out) {
  const float dx = r.gx - r.px, dy = r.gy - r.py;
  const float rot = atan2f(r.gy - r.py, r.gx - r.px);
  const float cr = cosf(rot), sr = sinf(rot);
  out[0] = sqrtf(dx * dx + dy * dy);
  out[1] = r.v_pref;
  out[2] = rotate_theta ? r.theta - rot : 0.0f;
  out[3] = r.radius;
  out[4] = r.vx * cr + r.vy * sr;
  out[5] = r.vy * cr - r.vx * sr;
  out[6] = (px1 - r.px) * cr + (py1 - r.py) * sr;
  out[7] = (py1 - r.py) * cr - (px1 - r.px) * sr;
  out[8] = vx1 * cr + vy1 * sr;
  out[9] = vy1 * cr - vx1 * sr;
  out[10] = radius1;
  const float ax = r.px - px1, ay = r.py - py1;
  out[11] = sqrtf(ax * ax + ay * ay);
  out[12] = r.radius + radius1;
  if (D == 17) {
#pragma unroll
    for (int k = 0; k < 4; ++k) out[13 + k] = (k == type1) ? 1.0f : 0.0f;
  }
}

// The robot's part of rotate_row for one (episode, action), stored for K4's fused input path (ebc_value with vin ==
// NULL builds the entity part of every row itself): {out0..3}, {out4, out5, px, py}, {cos, sin, 0, 0} -- the very
// expressions of rotate_row above, so the fused rows equal the materialised ones bit for bit.
__device__ __forceinline__ void store_robot_record(const RobotRow &r, int rotate_theta, float4 *rec) {
  const float dx = r.gx - r.px, dy = r.gy - r.py;
  const float rot = atan2f(r.gy - r.py, r.gx - r.px);
  const float cr = cosf(rot), sr = sinf(rot);
  rec[0] = make_float4(sqrtf(dx * dx + dy * dy), r.v_pref, rotate_theta ? r.theta - rot : 0.0f, r.radius);
  rec[1] = make_float4(r.vx * cr + r.vy * sr, r.vy * cr - r.vx * sr, r.px, r.py);
  rec[2] = make_float4(cr, sr, 0.0f, 0.0f);
}

// rl/policy/cadrl.py:118-165 propagate(robot) in fp64, narrowed like torch.Tensor([...])
__device__ __forceinline__ RobotRow propagate_robot(const ebc_config &c, const float4 rp, const float4 rg, double theta,
                                                    double a0, double a1, const Outcome &o) {
  RobotRow rr;
  const double dt = c.time_step;
  if (c.robot_kinematics == EBC_KIN_HOLONOMIC) {
    rr.px = (float)((double)rp.x + a0 * dt);
    rr.py = (float)((double)rp.y + a1 * dt);
    rr.vx = (float)a0;
    rr.vy = (float)a1;
    rr.theta = (float)theta;
  } else {
    const double nth = theta + a1;
    const double nvx = a0 * o.cs, nvy = a0 * o.sn;   // cos / sin of theta + a1, already computed for the collision test
    rr.px = (float)((double)rp.x + nvx * dt);
    rr.py = (float)((double)rp.y + nvy * dt);
    rr.vx = (float)nvx;
    rr.vy = (float)nvy;
    rr.theta = (float)nth;
  }
  rr.radius = rg.w; rr.gx = rg.x; rr.gy = rg.y; rr.v_pref = rg.z;
  return rr;
}

// Build the n x D rows of one state into `tile` (this group's shared-memory staging area; lane l of the group builds
// rows l, l + G, ...), then stream them out with coalesced stores (dst == NULL: an idle group, nothing to store).
// next_state: humans advanced by their ORCA action (agent.py:80-93) when true, current state (multi_human_rl.py:128-149)
// when false.  Every lane of the warp takes part (__syncwarp).
template <int G>
__device__ void build_rows(const ebc_config &c, const ebc_state &st, int e, int lane, int H, int S,
                           const RobotRow &rr, bool next_state, float *tile, float *dst) {
  const int Hm = c.max_humans, Sm = c.max_statics, n = Hm + Sm;
  const int D = c.with_agent_type ? 17 : 13;
  const double dt = c.time_step;
  for (int r = lane; r < n; r += G) {
    float *row = tile + r * D;
    if (r < H) {
      const float4 p = reinterpret_cast<const float4 *>(st.hum_pv)[(size_t)e * Hm + r];
      const float rad = st.hum_gr[((size_t)e * Hm + r) * 4 + 3];
      const int ty = st.hum_type[(size_t)e * Hm + r];
      if (next_state) {
        const float2 nv = reinterpret_cast<const float2 *>(st.hum_nv)[(size_t)e * Hm + r];
        const float npx = (float)((double)p.x + (double)nv.x * dt);
        const float npy = (float)((double)p.y + (double)nv.y * dt);
        rotate_row(rr, npx, npy, nv.x, nv.y, rad, ty, c.rotate_theta, D, row);
      } else {
        rotate_row(rr, p.x, p.y, p.z, p.w, rad, ty, c.rotate_theta, D, row);
      }
    } else if (r < H + S) {   // env.py:457-458 static discs, type 3
      const float4 p = reinterpret_cast<const float4 *>(st.stat)[(size_t)e * Sm + (r - H)];
      rotate_row(rr, p.x, p.y, 0.0f, 0.0f, p.z, EBC_ADULT_STATIC, c.rotate_theta, D, row);
    } else {
      for (int k = 0; k < D; ++k) row[k] = 0.0f;
    }
  }
  __syncwarp();
  if (!dst) return;
  const int total = n * D;
  for (int i = lane; i < total; i += G) dst[i] = tile[i];
}

// K3, a group of G lanes per (episode, action): G = 8 / 16 for states of at most G rows (32 / G pairs per warp), else
// the whole warp.  G < 32 keeps four blocks per SM (64 registers).
template <int G>
__global__ void __launch_bounds__(EBC_THREADS, G < 32 ? 4 : 0)
lookahead_kernel(const ebc_config c, const ebc_state st, const double *__restrict__ actions, float *vin,
                 double *reward, uint8_t *done, uint8_t *event, float4 *rec) {
  extern __shared__ float tiles[];
  constexpr int GPW = 32 / G;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, sub = lane / G, l = lane % G;
  const int A = c.n_actions;
  const long long total = (long long)c.n_episodes * A;
  const long long w0 = ((long long)blockIdx.x * EBC_WARPS_PER_BLOCK + warp) * GPW;
  if (w0 >= total) return;                       // warp-uniform
  const long long w = w0 + sub;
  const bool live = w < total;                   // trailing groups of the last warp idle along (shuffles are warp-wide)
  const long long wc = live ? w : total - 1;
  const int e = (int)(wc / A), a = (int)(wc % A);
  const int n = c.max_humans + c.max_statics, D = c.with_agent_type ? 17 : 13;
  const int H = st.hum_count[e], S = st.stat_count[e];
  const float4 rp = reinterpret_cast<const float4 *>(st.rob_pv)[e];
  const float4 rg = reinterpret_cast<const float4 *>(st.rob_gr)[e];
  const double theta = (double)st.rob_theta[e];
  const double a0 = actions[a * 2], a1 = actions[a * 2 + 1];
  EpisodeHumans hm;
  Outcome o;
  evaluate_action<G>(c, st, e, l, H, rp, rg, theta, st.time[e], a0, a1, hm, o);
  const size_t ea = (size_t)e * A + a;
  if (live && l == 0) {
    if (reward) reward[ea] = o.reward;
    if (done) done[ea] = (uint8_t)o.done;
    if (event) event[ea] = (uint8_t)o.event;
  }
  if (!vin && !rec) return;
  const RobotRow rr = propagate_robot(c, rp, rg, theta, a0, a1, o);
  if (rec && live && l == 0) store_robot_record(rr, c.rotate_theta, rec + ea * 3);
  if (vin)                        // (warp-uniform: a kernel argument)
    build_rows<G>(c, st, e, l, H, S, rr, true, tiles + (size_t)(warp * GPW + sub) * n * D,
                  live ? vin + ea * (size_t)n * D : nullptr);
}

// rl/policy/multi_human_rl.py:128-149
__global__ void __launch_bounds__(EBC_THREADS) transform_kernel(const ebc_config c, const ebc_state st, float *out) {
  extern __shared__ float tiles[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * EBC_WARPS_PER_BLOCK + warp;
  if (e >= c.n_episodes) return;
  const int n = c.max_humans + c.max_statics, D = c.with_agent_type ? 17 : 13;
  const float4 rp = reinterpret_cast<const float4 *>(st.rob_pv)[e];
  const float4 rg = reinterpret_cast<const float4 *>(st.rob_gr)[e];
  RobotRow rr;
  rr.px = rp.x; rr.py = rp.y; rr.vx = rp.z; rr.vy = rp.w;
  rr.radius = rg.w; rr.gx = rg.x; rr.gy = rg.y; rr.v_pref = rg.z; rr.theta = st.rob_theta[e];
  build_rows<32>(c, st, e, lane, st.hum_count[e], st.stat_count[e], rr, false, tiles + (size_t)warp * n * D,
                 out + (size_t)e * n * D);
}

// K5
__global__ void __launch_bounds__(EBC_THREADS)
select_kernel(const ebc_config c, const ebc_state st, const double *__restrict__ reward,
              const float *__restrict__ values, double *action_values, int32_t *argmax, uint8_t *nan_flag) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * EBC_WARPS_PER_BLOCK + warp;
  if (e >= c.n_episodes) return;
  const int A = c.n_actions;
  const float4 rp = reinterpret_cast<const float4 *>(st.rob_pv)[e];
  const float4 rg = reinterpret_cast<const float4 *>(st.rob_gr)[e];
  const double disc = pow(c.gamma, c.time_step * (double)rg.z);
  double best = -INFINITY;
  int arg = 0x7fffffff;
  for (int a = lane; a < A; a += 32) {
    const double v = reward[(size_t)e * A + a] + disc * (double)values[(size_t)e * A + a];
    if (action_values) action_values[(size_t)e * A + a] = v;
    if (v > best) { best = v; arg = a; }   // strict '>' keeps the first maximum of this lane's stride
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(FULL, best, o);
    const int oa = __shfl_xor_sync(FULL, arg, o);
    if (oa != 0x7fffffff && (arg == 0x7fffffff || ob > best || (ob == best && oa < arg))) { best = ob; arg = oa; }
  }
  if (lane == 0) {
    const bool none = arg == 0x7fffffff;
    if (nan_flag) nan_flag[e] = none ? 1 : 0;
    if (none) arg = 0;
    const double dy = (double)rp.y - (double)rg.y, dx = (double)rp.x - (double)rg.x;   // policy.py:43-54
    if (sqrt(dy * dy + dx * dx) < (double)rg.w) arg = 0;
    argmax[e] = arg;
  }
}

// Commit of one episode by one warp (env.py:340-386,424-466; agent.py:202-228).
__device__ void commit_episode_warp(const ebc_config &c, const ebc_state &st, int e, int lane,
                                    const double *actions, const int32_t *action_idx, const double *action,
                                    double *reward, uint8_t *done, uint8_t *event, double *dmin, double *dist_to_goal,
                                    const ebc_stats &sx) {
  const int Hm = c.max_humans;
  const int H = st.hum_count[e];
  double a0, a1;
  if (action_idx) {
    int ai = action_idx[e];
    if (ai < 0 || ai >= c.n_actions) ai = 0;
    a0 = actions[ai * 2];
    a1 = actions[ai * 2 + 1];
  } else {
    a0 = action[(size_t)e * 2];
    a1 = action[(size_t)e * 2 + 1];
  }
  const float4 rp = reinterpret_cast<const float4 *>(st.rob_pv)[e];
  const float4 rg = reinterpret_cast<const float4 *>(st.rob_gr)[e];
  const double theta = (double)st.rob_theta[e];
  const double gt = st.time[e];
  EpisodeHumans hm;
  Outcome o;
  evaluate_action<32>(c, st, e, lane, H, rp, rg, theta, gt, a0, a1, hm, o);
  const double dt = c.time_step;
  // humans: agent.step(ActionXY), holonomic
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const int h = lane + 32 * ch;
    if (h < H) {
      const float2 nv = reinterpret_cast<const float2 *>(st.hum_nv)[(size_t)e * Hm + h];
      float4 p;
      p.x = (float)((double)hm.pv[ch].x + (double)nv.x * dt);
      p.y = (float)((double)hm.pv[ch].y + (double)nv.y * dt);
      p.z = nv.x;
      p.w = nv.y;
      reinterpret_cast<float4 *>(st.hum_pv)[(size_t)e * Hm + h] = p;
    }
  }
  if (lane == 0) {
    if (reward) reward[e] = o.reward;
    if (done) done[e] = (uint8_t)o.done;
    if (event) event[e] = (uint8_t)o.event;
    if (dmin) { dmin[(size_t)e * 3] = o.dmin[0]; dmin[(size_t)e * 3 + 1] = o.dmin[1]; dmin[(size_t)e * 3 + 2] = o.dmin[2]; }
    if (dist_to_goal) dist_to_goal[e] = o.dist_to_goal;
    float4 np;
    np.x = (float)o.end_x;
    np.y = (float)o.end_y;
    if (c.robot_kinematics == EBC_KIN_HOLONOMIC) {
      np.z = (float)a0;
      np.w = (float)a1;
    } else {
      const double two_pi = 2.0 * 3.14159265358979323846;
      double th = fmod(theta + a1, two_pi);
      if (th < 0.0) th += two_pi;   // Python % is non-negative
      st.rob_theta[e] = (float)th;
      np.z = (float)(a0 * cos(th));
      np.w = (float)(a0 * sin(th));
    }
    reinterpret_cast<float4 *>(st.rob_pv)[e] = np;
    st.time[e] = gt + dt;
    if (sx.alive) {   // the explorer's running statistics (explorer.py:33-94,189-193), one writer per episode
      const double disc = sx.discount[e];
      sx.cum_reward[e] += disc * o.reward;
      sx.discount[e] = disc * pow(c.gamma, dt * (double)rg.z);
      sx.steps[e] += 1;
      if (o.event == EBC_EV_DANGER) {
        sx.too_close[e] += 1;
        sx.min_dist_sum[e] += o.min_dist;
      }
      if (o.done) {
        sx.final_event[e] = (uint8_t)o.event;
        sx.alive[e] = 0;
        atomicSub(sx.alive_count, 1);
      }
    }
  }
}

// K2, warp per episode; hum_nv comes from a preceding orca_kernel.
__global__ void __launch_bounds__(EBC_THREADS)
step_kernel(const ebc_config c, const ebc_state st, const double *__restrict__ actions, const int32_t *action_idx,
            const double *action, const uint8_t *active, double *reward, uint8_t *done, uint8_t *event,
            double *dmin, double *dist_to_goal, const ebc_stats sx) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * EBC_WARPS_PER_BLOCK + warp;
  if (e >= c.n_episodes) return;
  if (active && !active[e]) return;
  commit_episode_warp(c, st, e, lane, actions, action_idx, action, reward, done, event, dmin, dist_to_goal, sx);
}

// K1 + K2 fused with ORCA obstacle half-planes, block per episode: the episode's obstacle vertices are staged in
// shared memory next to the neighbour scratch, every warp solves humans' LPs from the untouched state, the block
// synchronises, then warp 0 commits.  COMMIT = false is K1 alone in that shape (ebc_orca with obstacles).
template <bool COMMIT>
__global__ void __launch_bounds__(512)
orca_step_kernel(const ebc_config c, const ebc_state st, const double *__restrict__ actions,
                 const int32_t *action_idx, const double *action, const uint8_t *active, double *reward,
                 uint8_t *done, uint8_t *event, double *dmin, double *dist_to_goal, const ebc_stats sx) {
  __shared__ float scratch[16][OBST_SCRATCH_FLOATS];
  __shared__ __align__(16) ObstV so[64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
  const int e = blockIdx.x;
  if (active && !active[e]) return;
  const int H = st.hum_count[e];
  const int V = stage_obstacles(c, st, e, so, threadIdx.x, blockDim.x);
  __syncthreads();
  for (int h = warp; h < H; h += n_warps) {
    float nvx, nvy;
    human_policy_warp<true, 32>(FULL, c, st, e, h, H, lane, scratch[warp], nvx, nvy, so, V);
    if (lane == 0)
      reinterpret_cast<float2 *>(st.hum_nv)[(size_t)e * c.max_humans + h] = make_float2(nvx, nvy);
  }
  if (!COMMIT) return;
  __syncthreads();   // all reads of the old state are done; hum_nv is visible block-wide
  if (warp == 0)
    commit_episode_warp(c, st, e, lane, actions, action_idx, action, reward, done, event, dmin, dist_to_goal, sx);
}

// env.reset from a device-resident scene pool; one warp per episode, lanes copy 16-byte words.
__global__ void __launch_bounds__(EBC_THREADS)
reset_kernel(const ebc_config c, const ebc_state st, const ebc_state pool, int pool_size,
             const int32_t *pool_index, const uint8_t *mask) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * EBC_WARPS_PER_BLOCK + warp;
  if (e >= c.n_episodes) return;
  if (mask && !mask[e]) return;
  int q = pool_index ? pool_index[e] : e;
  if (q < 0 || q >= pool_size) q = ((q % pool_size) + pool_size) % pool_size;
  const int Hm = c.max_humans, Sm = c.max_statics, Rm = c.max_rects;
  for (int h = lane; h < Hm; h += 32) {
    reinterpret_cast<float4 *>(st.hum_pv)[(size_t)e * Hm + h] = reinterpret_cast<const float4 *>(pool.hum_pv)[(size_t)q * Hm + h];
    reinterpret_cast<float4 *>(st.hum_gr)[(size_t)e * Hm + h] = reinterpret_cast<const float4 *>(pool.hum_gr)[(size_t)q * Hm + h];
    st.hum_type[(size_t)e * Hm + h] = pool.hum_type[(size_t)q * Hm + h];
    reinterpret_cast<float2 *>(st.hum_nv)[(size_t)e * Hm + h] = make_float2(0.f, 0.f);
  }
  for (int k = lane; k < Sm; k += 32)
    reinterpret_cast<float4 *>(st.stat)[(size_t)e * Sm + k] = reinterpret_cast<const float4 *>(pool.stat)[(size_t)q * Sm + k];
  for (int j = lane; j < Rm; j += 32)
    reinterpret_cast<short4 *>(st.rect)[(size_t)e * Rm + j] = reinterpret_cast<const short4 *>(pool.rect)[(size_t)q * Rm + j];
  if (c.max_obst > 0 && st.obst && pool.obst && st.obst_count && pool.obst_count) {
    const uint4 *src = reinterpret_cast<const uint4 *>(pool.obst + (size_t)q * c.max_obst);
    uint4 *dst = reinterpret_cast<uint4 *>(st.obst + (size_t)e * c.max_obst);
    for (int i = lane; i < c.max_obst * 3; i += 32) dst[i] = src[i];
    if (lane == 0) st.obst_count[e] = pool.obst_count[q];
  }
  if (lane == 0) {
    st.hum_count[e] = pool.hum_count[q];
    st.stat_count[e] = pool.stat_count[q];
    st.rect_count[e] = pool.rect_count[q];
    reinterpret_cast<float4 *>(st.rob_pv)[e] = reinterpret_cast<const float4 *>(pool.rob_pv)[q];
    reinterpret_cast<float4 *>(st.rob_gr)[e] = reinterpret_cast<const float4 *>(pool.rob_gr)[q];
    st.rob_theta[e] = pool.rob_theta[q];
    st.time[e] = pool.time[q];
  }
}

// ---- angular local map (SURVEY 8f-3, simulator/env.py:468-628) ------------------------------------------------
// One vertex seen from one robot corner, then the outline towards every earlier vertex of the same sweep
// (env.py:468-568).  Sector minima go to shared memory with a 64-bit atomicMin on the bit pattern of the
// (non-negative) distance: the minimum does not depend on the order, so the reference's sequential sweeps can
// run on different lanes.  fp64 in the reference's operation order (this unit has no FMA contraction).
struct AngularMap { double max_range, min_angle, res; int dim; };

__device__ __forceinline__ void amap_min(unsigned long long *vec, int i, double d) {
  atomicMin(vec + i, (unsigned long long)__double_as_longlong(d));
}

__device__ void amap_calc(const AngularMap &m, double vx, double vy, double ex, double ey, double cs, double sn,
                          unsigned long long *vec, int (&rad_indeces)[4], double (&lx)[4], double (&ly)[4], int &n_seen) {
  double px = (vx - ex) * cs + (vy - ey) * sn;
  double py = (vy - ey) * cs - (vx - ex) * sn;
  const double phi = atan2(py, px);
  const int rad_idx = (int)((phi - m.min_angle) / m.res);          // Python int(): truncation
  if (rad_idx >= 0 && rad_idx < m.dim) amap_min(vec, rad_idx, sqrt(px * px + py * py));
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    if (k >= n_seen) break;
    const int old = rad_indeces[k];
    bool wrapped;
    int idx_diff;
    if ((double)abs(rad_idx - old) > 3.141592653589793 / m.res) {
      wrapped = true;
      idx_diff = rad_idx > old ? m.dim - rad_idx + old : m.dim - old + rad_idx;
    } else {
      wrapped = false;
      idx_diff = abs(rad_idx - old);
    }
    const bool from_vertex = (rad_idx < old && !wrapped) || (rad_idx > old && wrapped);
    const double ax = from_vertex ? vx : lx[k], ay = from_vertex ? vy : ly[k];      // start of the interpolation
    const double bx = from_vertex ? lx[k] : vx, by = from_vertex ? ly[k] : vy;      // its end
    const int first = from_vertex ? rad_idx : old;
    for (int i = 0; i < idx_diff; ++i) {
      if (first + i < 0 || first + i >= m.dim) continue;
      const double t = (double)i / (double)idx_diff;
      const double qx = ax + t * (bx - ax) - ex;
      const double qy = ay + t * (by - ay) - ey;
      px = qx * cs + qy * sn;
      py = qy * cs - qx * sn;
      amap_min(vec, first + i, sqrt(px * px + py * py));
    }
  }
  rad_indeces[n_seen] = rad_idx; lx[n_seen] = vx; ly[n_seen] = vy;
  ++n_seen;
}

// Warp per episode; lane g takes sweep g: sweeps [0, 4P) = (obstacle, robot corner) over the obstacle's four
// vertices (env.py:596-609), sweeps [4P, 8P) = (obstacle, vertex) over the four robot corners (env.py:611-620).
__global__ void __launch_bounds__(EBC_THREADS)
angular_map_kernel(const ebc_config c, const ebc_state st, const ebc_angular_map mp, const double *__restrict__ poly_xy,
                   const int32_t *__restrict__ poly_count, double *__restrict__ out) {
  __shared__ unsigned long long vecs[EBC_WARPS_PER_BLOCK][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * EBC_WARPS_PER_BLOCK + warp;
  if (e >= c.n_episodes) return;
  unsigned long long *vec = vecs[warp];
  AngularMap m;
  m.max_range = mp.max_range; m.min_angle = mp.min_angle; m.dim = mp.dim;
  m.res = (mp.max_angle - mp.min_angle) / (double)mp.dim;
  for (int i = lane; i < m.dim; i += 32) vec[i] = (unsigned long long)__double_as_longlong(m.max_range);
  __syncwarp();
  const float4 rp = reinterpret_cast<const float4 *>(st.rob_pv)[e];
  const double rx = (double)rp.x, ry = (double)rp.y, rad = (double)st.rob_gr[(size_t)e * 4 + 3];
  const double theta = (double)st.rob_theta[e];
  const double cs = cos(theta), sn = sin(theta);
  int P = poly_count[e];
  P = P < 0 ? 0 : (P > mp.max_polys ? mp.max_polys : P);
  for (int g = lane; g < 8 * P; g += 32) {
    const bool by_vertex = g >= 4 * P;
    const int gg = by_vertex ? g - 4 * P : g;
    const int o = gg >> 2, k = gg & 3;
    const double *poly = poly_xy + ((size_t)e * mp.max_polys + o) * 8;
    int idx[4], n_seen = 0;
    double lx[4], ly[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int v = by_vertex ? k : j, corner = by_vertex ? j : k;      // (-1,-1), (1,-1), (-1,1), (1,1): env.py:592-594
      const double ex = rx + ((corner & 1) ? 1.0 : -1.0) * rad, ey = ry + ((corner & 2) ? 1.0 : -1.0) * rad;
      amap_calc(m, poly[2 * v], poly[2 * v + 1], ex, ey, cs, sn, vec, idx, lx, ly, n_seen);
    }
  }
  __syncwarp();
  for (int i = lane; i < m.dim; i += 32) {
    const double d = __longlong_as_double((long long)vec[i]);
    out[(size_t)e * m.dim + i] = mp.normalize ? d / m.max_range : d;
  }
}

// ---- binary grid sub-map (SURVEY 8f-3, simulator/env.py:630-708, [map] use_grid_map = true) ----------------------
// Block per episode.  (1) thread 0: the reference's window / clip index arithmetic and the inverse rotation matrix of
// cv2.getRotationMatrix2D + cv2.warpAffine in float64; (2) the first `size` threads: the per-column and per-row
// fixed-point terms (OpenCV's adelta / bdelta / X0 / Y0, 1/1024 units, cvRound = rint); (3) the window of scene.map is
// rasterised from the episode's zero-cell rectangles into shared memory, one byte per cell, inside a one-cell frame
// of ones (the constant border: a tap outside the window reads 1 without a bounds test); (4) every thread takes four
// consecutive output cells: sample position to 1/32 pixel, four taps from shared memory, threshold, one 32-bit store
// (`packed`: the host's test that every episode's map starts on a 4-byte boundary; four byte stores otherwise).
// The bilinear sum is taken in integers: OpenCV's float weights are (32 - fy)(32 - fx) / 1024 etc. (exact in
// float), the taps are 0 or 1, so its float64 sum equals (integer sum) / 1024 exactly and "> 0.9" is "integer sum >=
// 922" (0.9 * 1024 = 921.6) -- the oracle keeps OpenCV's float / double sequence, the tests demand equal cells.
// HBM traffic = the size x size bytes written per episode + the rectangle list; the rest stays in shared memory.
struct GridMapShared {
  double m[6];
  int sgx, sgy, egx, egy, six, siy, degenerate, pad;
};

__global__ void __launch_bounds__(256)
grid_map_kernel(const ebc_config c, const ebc_state st, const int S, const bool packed, uint8_t *__restrict__ out) {
  extern __shared__ __align__(16) uint8_t gm_smem[];
  __shared__ GridMapShared sh;
  const int e = blockIdx.x, tid = threadIdx.x;
  const int cells = S * S, P = S + 2, framed = P * P;                  // framed grid: [S + 2][S + 2], window at (1, 1)
  uint8_t *grid = gm_smem;
  int *adelta = reinterpret_cast<int *>(gm_smem + ((framed + 15) & ~15));   // [S] each
  int *bdelta = adelta + S, *x0s = bdelta + S, *y0s = x0s + S;
  if (tid == 0) {
    const float4 rp = reinterpret_cast<const float4 *>(st.rob_pv)[e];
    const double px = (double)rp.x, py = (double)rp.y, theta = (double)st.rob_theta[e];
    const int G = (int)rint(c.map_size_m / c.map_resolution);
    const int cx = (int)rint((px + c.map_size_m / 2.0) / c.map_resolution);       // env.py:637-642
    const int cy = (int)rint((py + c.map_size_m / 2.0) / c.map_resolution);
    int six = (int)rint((double)cx - floor((double)S / 2.0));                       // env.py:645-648
    int siy = (int)rint((double)cy - floor((double)S / 2.0));
    int eix = six + S - 1, eiy = siy + S - 1;
    const int max_idx = G - 1;
    int sgx = 0, sgy = 0, egx = S - 1, egy = S - 1;
    if (six < 0) { sgx = -six; six = 0; }                                            // env.py:660-672
    else if (eix > max_idx) { egx = egx - (eix - max_idx); eix = max_idx; }
    if (siy < 0) { sgy = -siy; siy = 0; }
    else if (eiy > max_idx) { egy = egy - (eiy - max_idx); eiy = max_idx; }
    sh.degenerate = (sgy > egy || siy > eiy || six > eix || sgx > egx) ? 1 : 0;      // env.py:674-680
    sh.sgx = sgx; sh.sgy = sgy; sh.egx = egx; sh.egy = egy; sh.six = six; sh.siy = siy;
    const double angle = (-theta + 3.141592653589793 / 2) * 180 / 3.141592653589793;   // env.py:686
    const double a = angle * (3.141592653589793 / 180), alpha = cos(a), beta = sin(a), ctr = (double)S / 2.0;
    double M[6] = {alpha, beta, (1 - alpha) * ctr - beta * ctr, -beta, alpha, beta * ctr + (1 - alpha) * ctr};
    double D = M[0] * M[4] - M[1] * M[3];
    D = D != 0 ? 1. / D : 0;
    const double A11 = M[4] * D, A22 = M[0] * D;
    M[0] = A11; M[1] *= -D; M[3] *= -D; M[4] = A22;
    const double b1 = -M[0] * M[2] - M[1] * M[5], b2 = -M[3] * M[2] - M[4] * M[5];
    M[2] = b1; M[5] = b2;
#pragma unroll
    for (int k = 0; k < 6; ++k) sh.m[k] = M[k];
  }
  for (int i = tid; i < (framed + 3) / 4; i += blockDim.x) reinterpret_cast<uint32_t *>(grid)[i] = 0x01010101u;
  __syncthreads();
  if (sh.degenerate) {
    for (int i = tid; i < cells; i += blockDim.x) out[(size_t)e * cells + i] = 1;
    return;
  }
  for (int i = tid; i < S; i += blockDim.x) {
    adelta[i] = (int)rint(sh.m[0] * i * 1024);
    bdelta[i] = (int)rint(sh.m[3] * i * 1024);
    x0s[i] = (int)rint((sh.m[1] * i + sh.m[2]) * 1024) + 16;
    y0s[i] = (int)rint((sh.m[4] * i + sh.m[5]) * 1024) + 16;
  }
  {   // grid[sgx:egx, sgy:egy] = map[six:eix, siy:eiy]: the zero cells are the rectangles' cells (env.py:682-684)
    const int R = c.max_rects ? min(st.rect_count[e], c.max_rects) : 0;
    const short4 *rc = reinterpret_cast<const short4 *>(st.rect) + (size_t)e * c.max_rects;
    for (int j = 0; j < R; ++j) {
      const short4 r = rc[j];
      const int i0 = max(sh.sgx, (int)r.x - sh.six + sh.sgx), i1 = min(sh.egx, (int)r.z - sh.six + sh.sgx);
      const int j0 = max(sh.sgy, (int)r.y - sh.siy + sh.sgy), j1 = min(sh.egy, (int)r.w - sh.siy + sh.sgy);
      const int w = j1 - j0, n = (i1 - i0) * w;
      if (i1 <= i0 || w <= 0) continue;
      for (int k = tid; k < n; k += blockDim.x) grid[(i0 + 1 + k / w) * P + j0 + 1 + k % w] = 0;
    }
  }
  __syncthreads();
  for (int q = tid; 4 * q < cells; q += blockDim.x) {
    uint32_t word = 0;
    int y = (4 * q) / S, x = 4 * q - y * S;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (4 * q + k >= cells) break;
      const int X = (x0s[y] + adelta[x]) >> 5, Y = (y0s[y] + bdelta[x]) >> 5;
      const int sx = X >> 5, sy = Y >> 5, fx = X & 31, fy = Y & 31;
      uint32_t bit = 1u;                           // all four taps outside the window: the border value
      if ((unsigned)(sx + 1) <= (unsigned)S && (unsigned)(sy + 1) <= (unsigned)S) {     // sx, sy in [-1, S - 1]
        const uint8_t *g = grid + (sy + 1) * P + sx + 1;
        const int sum = (int)g[0] * (32 - fy) * (32 - fx) + (int)g[1] * (32 - fy) * fx + (int)g[P] * fy * (32 - fx) +
                        (int)g[P + 1] * fy * fx;
        bit = sum >= 922 ? 1u : 0u;                // env.py:687-689: > 0.9
      }
      if (packed) word |= bit << (8 * k);
      else out[(size_t)e * cells + 4 * q + k] = (uint8_t)bit;
      if (++x == S) { x = 0; ++y; }
    }
    if (packed) reinterpret_cast<uint32_t *>(out + (size_t)e * cells)[q] = word;
  }
}

// The same map for windows of at most 62 cells (the reference's 5 m and 6 m sub-maps on the 0.1 m grid): a framed row
// of the window is ONE 64-bit word (bit = 1: free cell or border), so rasterising is a thread per row that clears
// the bit range of every rectangle crossing it, the four taps of a sample are two 8-byte loads and two shifts
// (code = t00 | t01 << 1 | t10 << 2 | t11 << 3), and the thresholded bilinear sum is a table lookup: bit fx of
// lut[code * 32 + fy] says whether the integer sum (see above) reaches 922 -- the table is built at compile time.
struct GridLut { uint32_t w[512]; };
constexpr GridLut make_grid_lut() {
  GridLut t{};
  for (int code = 0; code < 16; ++code)
    for (int fy = 0; fy < 32; ++fy) {
      uint32_t bits = 0;
      for (int fx = 0; fx < 32; ++fx) {
        const int sum = ((code & 1) * (32 - fx) + ((code >> 1) & 1) * fx) * (32 - fy) +
                        (((code >> 2) & 1) * (32 - fx) + ((code >> 3) & 1) * fx) * fy;
        if (sum >= 922) bits |= 1u << fx;
      }
      t.w[code * 32 + fy] = bits;
    }
  return t;
}
__device__ const GridLut grid_lut = make_grid_lut();

__global__ void __launch_bounds__(256)
grid_map_bits_kernel(const ebc_config c, const ebc_state st, const int S, const uint32_t magic, uint8_t *__restrict__ out) {
  __shared__ GridMapShared sh;
  __shared__ unsigned long long rows[64];           // framed rows 0 .. S + 1, window cell (i, j) = bit j + 1 of rows[i + 1]
  __shared__ int2 ab[64];                           // {adelta, bdelta} of column x
  __shared__ int2 xy0[64];                          // {X0, Y0} of row y
  __shared__ uint32_t lut[512];
  const int e = blockIdx.x, tid = threadIdx.x;
  const int cells = S * S;
  if (tid == 0) {
    const float4 rp = reinterpret_cast<const float4 *>(st.rob_pv)[e];
    const double px = (double)rp.x, py = (double)rp.y, theta = (double)st.rob_theta[e];
    const int G = (int)rint(c.map_size_m / c.map_resolution);
    const int cx = (int)rint((px + c.map_size_m / 2.0) / c.map_resolution);       // env.py:637-642
    const int cy = (int)rint((py + c.map_size_m / 2.0) / c.map_resolution);
    int six = (int)rint((double)cx - floor((double)S / 2.0));                       // env.py:645-648
    int siy = (int)rint((double)cy - floor((double)S / 2.0));
    int eix = six + S - 1, eiy = siy + S - 1;
    const int max_idx = G - 1;
    int sgx = 0, sgy = 0, egx = S - 1, egy = S - 1;
    if (six < 0) { sgx = -six; six = 0; }                                            // env.py:660-672
    else if (eix > max_idx) { egx = egx - (eix - max_idx); eix = max_idx; }
    if (siy < 0) { sgy = -siy; siy = 0; }
    else if (eiy > max_idx) { egy = egy - (eiy - max_idx); eiy = max_idx; }
    sh.degenerate = (sgy > egy || siy > eiy || six > eix || sgx > egx) ? 1 : 0;      // env.py:674-680
    sh.sgx = sgx; sh.sgy = sgy; sh.egx = egx; sh.egy = egy; sh.six = six; sh.siy = siy;
    const double angle = (-theta + 3.141592653589793 / 2) * 180 / 3.141592653589793;   // env.py:686
    const double a = angle * (3.141592653589793 / 180), alpha = cos(a), beta = sin(a), ctr = (double)S / 2.0;
    double M[6] = {alpha, beta, (1 - alpha) * ctr - beta * ctr, -beta, alpha, beta * ctr + (1 - alpha) * ctr};
    double D = M[0] * M[4] - M[1] * M[3];
    D = D != 0 ? 1. / D : 0;
    const double A11 = M[4] * D, A22 = M[0] * D;
    M[0] = A11; M[1] *= -D; M[3] *= -D; M[4] = A22;
    const double b1 = -M[0] * M[2] - M[1] * M[5], b2 = -M[3] * M[2] - M[4] * M[5];
    M[2] = b1; M[5] = b2;
#pragma unroll
    for (int k = 0; k < 6; ++k) sh.m[k] = M[k];
  }
  for (int i = tid; i < 512; i += blockDim.x) lut[i] = grid_lut.w[i];
  __syncthreads();
  if (sh.degenerate) {
    for (int i = tid; i < cells; i += blockDim.x) out[(size_t)e * cells + i] = 1;
    return;
  }
  if (tid < S) {
    ab[tid] = make_int2((int)rint(sh.m[0] * tid * 1024), (int)rint(sh.m[3] * tid * 1024));
    xy0[tid] = make_int2((int)rint((sh.m[1] * tid + sh.m[2]) * 1024) + 16, (int)rint((sh.m[4] * tid + sh.m[5]) * 1024) + 16);
  } else if (tid >= 64 && tid < 64 + S + 2) {
    // framed row fr of the window (window row gi = fr - 1): grid[sgx:egx, sgy:egy] = map[six:eix, siy:eiy] (env.py:682-684)
    const int fr = tid - 64, gi = fr - 1;
    unsigned long long bits = ~0ull;
    if (gi >= sh.sgx && gi < sh.egx) {
      const int mx = sh.six + gi - sh.sgx;                          // scene.map row of this window row
      const int R = c.max_rects ? min(st.rect_count[e], c.max_rects) : 0;
      const short4 *rc = reinterpret_cast<const short4 *>(st.rect) + (size_t)e * c.max_rects;
      for (int j = 0; j < R; ++j) {
        const short4 r = rc[j];
        if (mx < (int)r.x || mx >= (int)r.z) continue;
        const int j0 = max(sh.sgy, (int)r.y - sh.siy + sh.sgy), j1 = min(sh.egy, (int)r.w - sh.siy + sh.sgy);
        if (j1 > j0) bits &= ~((((1ull << (j1 - j0)) - 1ull)) << (j0 + 1));     // j1 - j0 <= 61
      }
    }
    rows[fr] = bits;
  }
  __syncthreads();
  // 32-bit shared-memory addresses taken once (a generic pointer to static shared memory costs an S2R + LEA per use);
  // no branch per cell: out-of-window samples read a clamped, valid word and are overridden by a select.
  // Consecutive lanes take consecutive cells: the {adelta, bdelta} loads of a warp are one contiguous 256 bytes, most
  // lanes of a warp sample the same one or two source rows (broadcast), and a warp stores 32 consecutive bytes.  (Four
  // consecutive cells per thread and one 32-bit store cost 6 shared-memory wavefronts per {adelta, bdelta} load -- a
  // stride of 32 bytes between lanes -- and the kernel ran at 88-95 % of the shared-memory pipe.)
  const uint32_t rows_s = (uint32_t)__cvta_generic_to_shared(rows), ab_s = (uint32_t)__cvta_generic_to_shared(ab);
  const uint32_t xy0_s = (uint32_t)__cvta_generic_to_shared(xy0), lut_s = (uint32_t)__cvta_generic_to_shared(lut);
  auto lds64 = [](uint32_t a) { unsigned long long v; asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a)); return v; };
  auto lds32x2 = [](uint32_t a) { int2 v; asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v; };
  auto lds32 = [](uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; };
  uint8_t *dst = out + (size_t)e * cells;
  for (int idx = tid; idx < cells; idx += blockDim.x) {     // idx / S = umulhi(idx, magic), magic = ceil(2^32 / S) (host)
    const int y = (int)__umulhi((uint32_t)idx, magic), x = idx - y * S;
    const int2 o = lds32x2(xy0_s + 8u * (uint32_t)y), d = lds32x2(ab_s + 8u * (uint32_t)x);
    const int Xf = o.x + d.x, Yf = o.y + d.y;               // 1/1024 pixel
    const uint32_t cx = (uint32_t)((Xf >> 10) + 1), cy = (uint32_t)((Yf >> 10) + 1);   // framed column / row of tap (0, 0)
    const bool inside = cx <= (uint32_t)S && cy <= (uint32_t)S;                     // sx, sy in [-1, S - 1]
    const uint32_t ccx = min(cx, (uint32_t)S), ccy = min(cy, (uint32_t)S);
    const uint32_t p0 = (uint32_t)(lds64(rows_s + 8u * ccy) >> ccx) & 3u, p1 = (uint32_t)(lds64(rows_s + 8u * ccy + 8u) >> ccx) & 3u;
    const uint32_t lw = lds32(lut_s + (((p0 | (p1 << 2)) << 5) | (((uint32_t)Yf >> 5) & 31u)) * 4u);
    dst[idx] = inside ? (uint8_t)((lw >> (((uint32_t)Xf >> 5) & 31u)) & 1u) : (uint8_t)1;     // env.py:687-689: > 0.9; outside: the border
  }
}

// ---- scene generator (SURVEY 8f-1): thread per episode, counter-based draws, fp64 in the host generator's
//      operation order (this unit is compiled without FMA contraction), narrowed to fp32 at the end ----------
__device__ __forceinline__ unsigned long long gen_mix(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__device__ __forceinline__ double gen_uniform(unsigned long long seed, unsigned long long episode, unsigned long long stream,
                                              unsigned long long draw) {
  unsigned long long h = gen_mix(seed ^ gen_mix(episode));
  h = gen_mix(h ^ (stream * 0xD6E8FEB86659FD93ull));
  h = gen_mix(h ^ (draw * 0xCA5A826395121157ull));
  return (double)(h >> 11) * (1.0 / 9007199254740992.0);
}

__global__ void __launch_bounds__(128)
generate_kernel(const ebc_config c, const ebc_state st, const ebc_scene_shape sh, unsigned long long seed,
                const long long *episode_ids, const uint8_t *mask) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= c.n_episodes) return;
  if (mask && !mask[e]) return;
  const unsigned long long id = (unsigned long long)episode_ids[e];
  const int Hm = c.max_humans, Sm = c.max_statics, Rm = c.max_rects;
  const double R = sh.circle_radius, hw = sh.square_width / 2.0, dd = sh.discomfort_dist;
  double px[64], py[64], gx[64], gy[64], rad[64];
  int H = 0;
  for (int t = 0; t < sh.n_types; ++t) H += sh.type_count[t];
  // rule 3 = mixed_20 (scene_generator.py:577-582): randint(20) static adults in a 6 x 8 box, the rest dynamic
  const int n_static = sh.rule == 3 ? (int)floor(gen_uniform(seed, id, 4000, 0) * 20.0) : 0;
  const int n_dynamic = H - n_static;
  // scene_generator.py:292-328: per-agent preferred speed and radius, group by group
  int h0 = 0;
  for (int t = 0; t < sh.n_types; ++t) {
    int first_of_type = h0;                     // first agent of the same list (groups may repeat a type)
    for (int u = t - 1, hu = h0; u >= 0; --u) {
      hu -= sh.type_count[u];
      if (sh.type_code[u] == sh.type_code[t] && sh.type_count[u] > 0) first_of_type = hu;
    }
    for (int k = 0; k < sh.type_count[t]; ++k) {
      const int h = h0 + k;
      const double vpref = sh.v_pref_lo[t] + (sh.v_pref_hi[t] - sh.v_pref_lo[t]) * gen_uniform(seed, id, 1000 + h, 0);
      rad[h] = sh.radius_lo[t] + (sh.radius_hi[t] - sh.radius_lo[t]) * gen_uniform(seed, id, 1000 + h, 1);
      const int hd = h - n_static;              // index among the dynamic agents
      const bool is_static = h < n_static;
      const bool circle = !is_static && (sh.rule == 1 || ((sh.rule == 2 || sh.rule == 3) && hd < n_dynamic / 2));
      const double md_robot = rad[h] + sh.robot_radius + dd;
      double x = 0, y = 0, tx = 0, ty = 0;
      if (sh.rule == 4) {                       // one_static (scene_generator.py:583-589): two adults standing at (-2, -8), (-3, -8)
        x = -2.0 - (double)h; y = -8.0; tx = x; ty = y;
      } else if (is_static && h == 0) {         // scene_generator.py:463-466: the first static adult is fixed
        x = -0.5; y = -2.5; tx = x; ty = y;
      } else {
        // static adults (:467-487): one side of the y axis for all tries of this adult
        const double sign = gen_uniform(seed, id, 2000 + h, 7) < 0.5 ? 1.0 : -1.0;
        for (int attempt = 0; attempt < sh.max_tries; ++attempt) {
          const unsigned long long d0 = (unsigned long long)attempt * 8ull;
          bool ok;
          if (is_static) {          // a 6 x 8 box; no start closer than the comfort distance to anybody, nor to the robot's goal
            x = gen_uniform(seed, id, 2000 + h, d0) * 6.0 * 0.5 * sign;
            y = (gen_uniform(seed, id, 2000 + h, d0 + 1) - 0.5) * 8.0;
            tx = x; ty = y;
            ok = hypot(x - 0.0, y + R) >= md_robot;
            for (int j = first_of_type; j < h && ok; ++j) ok = hypot(x - px[j], y - py[j]) >= rad[h] + rad[j] + dd;
            // (:480-483 takes the radius of the LAST agent of the list it has just walked)
            ok = ok && hypot(x - 0.0, y - R) >= rad[h] + (h > first_of_type ? rad[h - 1] : sh.robot_radius) + dd;
          } else if (circle) {      // :593-618: start on the circle, goal opposite; clear of everybody's start AND goal
            const double ang = gen_uniform(seed, id, 2000 + h, d0) * 2.0 * 3.141592653589793;
            x = R * cos(ang); y = R * sin(ang);
            tx = -x; ty = -y;
            ok = hypot(x - 0.0, y + R) >= md_robot && hypot(x - 0.0, y - R) >= md_robot;
            for (int j = first_of_type; j < h && ok; ++j)
              ok = hypot(x - px[j], y - py[j]) >= rad[h] + rad[j] + dd && hypot(x - gx[j], y - gy[j]) >= rad[h] + rad[j] + dd;
          } else {                  // :672-712: start on one side of the square, goal on the opposite side; starts only
            const long long side = (long long)floor(gen_uniform(seed, id, 2000 + h, d0) * 4.0);
            const double a = -hw + 2.0 * hw * gen_uniform(seed, id, 2000 + h, d0 + 1);
            const double b = -hw + 2.0 * hw * gen_uniform(seed, id, 2000 + h, d0 + 2);
            x = side == 0 ? a : (side == 1 ? a : (side == 2 ? -hw : hw));
            y = side == 0 ? hw : (side == 1 ? -hw : a);
            tx = side == 0 ? b : (side == 1 ? b : (side == 2 ? hw : -hw));
            ty = side == 0 ? -hw : (side == 1 ? hw : b);
            ok = hypot(x - 0.0, y + R) >= md_robot;
            for (int j = first_of_type; j < h && ok; ++j) ok = hypot(x - px[j], y - py[j]) >= rad[h] + rad[j] + dd;
          }
          if (ok || attempt == sh.max_tries - 1) break;
        }
      }
      px[h] = x; py[h] = y; gx[h] = tx; gy[h] = ty;
      reinterpret_cast<float4 *>(st.hum_pv)[(size_t)e * Hm + h] = make_float4((float)x, (float)y, 0.f, 0.f);
      reinterpret_cast<float4 *>(st.hum_gr)[(size_t)e * Hm + h] = make_float4((float)tx, (float)ty, (float)vpref, (float)rad[h]);
      st.hum_type[(size_t)e * Hm + h] = (uint8_t)sh.type_code[t];
      reinterpret_cast<float2 *>(st.hum_nv)[(size_t)e * Hm + h] = make_float2(0.f, 0.f);
    }
    h0 += sh.type_count[t];
  }
  for (int h = H; h < Hm; ++h) {
    reinterpret_cast<float4 *>(st.hum_pv)[(size_t)e * Hm + h] = make_float4(0.f, 0.f, 0.f, 0.f);
    reinterpret_cast<float4 *>(st.hum_gr)[(size_t)e * Hm + h] = make_float4(0.f, 0.f, 0.f, 0.f);
    st.hum_type[(size_t)e * Hm + h] = 0;
    reinterpret_cast<float2 *>(st.hum_nv)[(size_t)e * Hm + h] = make_float2(0.f, 0.f);
  }
  st.hum_count[e] = H;
  // walls (:205-290) -> grid rectangle (:888-922) + static discs (:380-422)
  const double res = sh.map_resolution;
  const double G = rint(sh.map_size_m / res);
  const double clear = sh.robot_radius + dd;
  int n_stat = 0;
  for (int w = 0; w < sh.num_walls; ++w) {
    double lx = 0, ly = 0, xd = 1, yd = 1;
    for (int attempt = 0; attempt < sh.max_tries; ++attempt) {
      const unsigned long long d0 = (unsigned long long)attempt * 8ull;
      const double cx = floor(-G / 2.0 + G * gen_uniform(seed, id, 3000 + w, d0));
      const double cy = floor(-G / 2.0 + G * gen_uniform(seed, id, 3000 + w, d0 + 1));
      const double length = floor((double)sh.wall_len_lo +
                                  (double)(sh.wall_len_hi - sh.wall_len_lo + 1) * gen_uniform(seed, id, 3000 + w, d0 + 3));
      const bool horiz = gen_uniform(seed, id, 3000 + w, d0 + 2) > 0.5;
      const double xdim = horiz ? length : 1.0, ydim = horiz ? 1.0 : length;
      const double xm = cx * res, ym = cy * res;
      const bool near_start = fabs(xm - 0.0) < xdim / 2 + clear && fabs(ym + R) < ydim / 2 + clear;
      const bool near_goal = fabs(xm - 0.0) < xdim / 2 + clear && fabs(ym - R) < ydim / 2 + clear;
      lx = cx; ly = cy; xd = xdim; yd = ydim;
      if (!(near_start || near_goal) || attempt == sh.max_tries - 1) break;
    }
    const double dimx = rint(xd / res), dimy = rint(yd / res);
    const double locx = rint(lx + G / 2.0), locy = rint(ly + G / 2.0);
    const double x0 = rint(locx - dimx / 2.0), y0 = rint(locy - dimy / 2.0);
    // scene_generator.py:888-922: a wall strictly inside the map is the slice [start, start + dim); one that touches the
    // border goes through the per-cell path, which only writes cells 0 < index < G: [max(start, 1), min(start + dim, G))
    short4 r;
    r.x = (short)fmin(fmax(x0, 1.0), G); r.y = (short)fmin(fmax(y0, 1.0), G);
    r.z = (short)fmin(fmax(x0 + dimx, 1.0), G); r.w = (short)fmin(fmax(y0 + dimy, 1.0), G);
    reinterpret_cast<short4 *>(st.rect)[(size_t)e * Rm + w] = r;
    const double xm = lx * res, ym = ly * res;
    const bool square = xd == yd;               // :383-396: one disc at the centre
    const bool horiz = xd > yd;
    const double rr = (horiz ? yd : xd) / 2.0 * sqrt(2.0);
    const double hi = horiz ? xm + xd / 2.0 : ym + yd / 2.0;
    double pos = (horiz ? xm - xd / 2.0 : ym - yd / 2.0) + rr;
    for (int k = 0; k < sh.discs_per_wall; ++k) {
      const bool live = square ? k == 0 : pos < hi;
      if (live && n_stat < Sm) {
        reinterpret_cast<float4 *>(st.stat)[(size_t)e * Sm + n_stat] =
            make_float4((float)(square ? xm : (horiz ? pos : xm)), (float)(square ? ym : (horiz ? ym : pos)), (float)rr, 0.f);
        ++n_stat;
      }
      pos = pos + 2.0 * rr;
    }
  }
  for (int k = n_stat; k < Sm; ++k) reinterpret_cast<float4 *>(st.stat)[(size_t)e * Sm + k] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int w = sh.num_walls; w < Rm; ++w) reinterpret_cast<short4 *>(st.rect)[(size_t)e * Rm + w] = make_short4(0, 0, 0, 0);
  st.stat_count[e] = n_stat;
  st.rect_count[e] = sh.num_walls;
  // env.py:128-140: robot at (0, -R) facing +y, goal (0, R), at rest; global_time = 0
  reinterpret_cast<float4 *>(st.rob_pv)[e] = make_float4(0.f, (float)(-R), 0.f, 0.f);
  reinterpret_cast<float4 *>(st.rob_gr)[e] = make_float4(0.f, (float)R, (float)sh.robot_v_pref, (float)sh.robot_radius);
  st.rob_theta[e] = (float)(3.141592653589793 / 2);
  st.time[e] = 0.0;
}

}  // namespace

int ebc_launch_generate(ebc_sim *s, const ebc_scene_shape *shape, uint64_t seed, const int64_t *episode_ids,
                        const uint8_t *mask, cudaStream_t stream) {
  s->la_rec_valid = 0;      // the state moves on: the lookahead records no longer describe it
  const int blocks = (s->cfg.n_episodes + 127) / 128;
  generate_kernel<<<blocks, 128, 0, stream>>>(s->cfg, s->st, *shape, (unsigned long long)seed,
                                              reinterpret_cast<const long long *>(episode_ids), mask);
  return ebc_check_launch(s, "generate_kernel");
}

int ebc_launch_reset(ebc_sim *s, const ebc_state *pool, int pool_size, const int32_t *pool_index,
                     const uint8_t *mask, cudaStream_t stream) {
  s->la_rec_valid = 0;      // the state moves on: the lookahead records no longer describe it
  const int blocks = (s->cfg.n_episodes + EBC_WARPS_PER_BLOCK - 1) / EBC_WARPS_PER_BLOCK;
  reset_kernel<<<blocks, EBC_THREADS, 0, stream>>>(s->cfg, s->st, *pool, pool_size, pool_index, mask);
  return ebc_check_launch(s, "reset_kernel");
}

// lanes per human in K1: a half warp when every human has at most 32 candidates and 16 ORCA lines (two humans per
// warp, bit-identical to the whole-warp kernel; EBC_ORCA_GROUP=32 forces one human per warp)
static int orca_group(const ebc_sim *s) {
  const char *env = getenv("EBC_ORCA_GROUP");
  if (env && atoi(env) == 32) return 32;
  if (s->cfg.orca_obstacles) return 32;
  return (s->cfg.max_humans + (s->cfg.robot_visible ? 1 : 0) <= 32 && s->cfg.orca_max_neighbors <= 16) ? 16 : 32;
}
static int fused_warps(const ebc_sim *s) {   // orca_step_kernel: a warp per human, at most 16 warps per block
  const int warps = s->cfg.max_humans < 16 ? s->cfg.max_humans : 16;
  return warps < 1 ? 1 : warps;
}

static int launch_orca_groups(ebc_sim *s, const uint8_t *active, cudaStream_t stream) {
  const int group = orca_group(s);
  const long long groups = (long long)s->cfg.n_episodes * s->cfg.max_humans;
  const long long warps = (groups + (32 / group) - 1) / (32 / group);
  const int blocks = (int)((warps + EBC_WARPS_PER_BLOCK - 1) / EBC_WARPS_PER_BLOCK);
  if (group == 16) orca_kernel<16><<<blocks, EBC_THREADS, 0, stream>>>(s->cfg, s->st, active);
  else orca_kernel<32><<<blocks, EBC_THREADS, 0, stream>>>(s->cfg, s->st, active);
  return ebc_check_launch(s, "orca_kernel");
}

int ebc_launch_orca(ebc_sim *s, cudaStream_t stream) {
  if (s->cfg.orca_obstacles) {   // block per episode: the obstacle vertices are staged once per block
    orca_step_kernel<false><<<s->cfg.n_episodes, fused_warps(s) * 32, 0, stream>>>(
        s->cfg, s->st, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, ebc_stats{});
    return ebc_check_launch(s, "orca_step_kernel<obstacles, no commit>");
  }
  return launch_orca_groups(s, nullptr, stream);
}

int ebc_launch_robot_orca(ebc_sim *s, double safety, double *out, cudaStream_t stream) {
  if (s->cfg.orca_obstacles) {
    robot_orca_kernel<true, 1><<<s->cfg.n_episodes, 32, 0, stream>>>(s->cfg, s->st, safety, out);
    return ebc_check_launch(s, "robot_orca_kernel<obstacles>");
  }
  const int blocks = (s->cfg.n_episodes + EBC_WARPS_PER_BLOCK - 1) / EBC_WARPS_PER_BLOCK;
  robot_orca_kernel<false, EBC_WARPS_PER_BLOCK><<<blocks, EBC_THREADS, 0, stream>>>(s->cfg, s->st, safety, out);
  return ebc_check_launch(s, "robot_orca_kernel");
}

int ebc_launch_lookahead(ebc_sim *s, float *vin, double *reward, uint8_t *done, uint8_t *event,
                         cudaStream_t stream) {
  const long long pairs = (long long)s->cfg.n_episodes * s->cfg.n_actions;
  const int n = s->cfg.max_humans + s->cfg.max_statics, D = s->cfg.with_agent_type ? 17 : 13;
  // lanes per (episode, action): small states put several pairs in one warp
  const int group = n <= 8 ? 8 : (n <= 16 ? 16 : 32);
  const int gpw = 32 / group;
  const long long warps = (pairs + gpw - 1) / gpw;
  const int blocks = (int)((warps + EBC_WARPS_PER_BLOCK - 1) / EBC_WARPS_PER_BLOCK);
  const size_t smem = (size_t)EBC_WARPS_PER_BLOCK * gpw * n * D * sizeof(float);
  // without a destination for the rows the kernel leaves the robot part of every (episode, action) in s->d_la_rec:
  // K4's fused input path builds the rows from it (ebc_value with vin == NULL)
  float4 *rec = vin ? nullptr : s->d_la_rec;
  if (group == 8)
    lookahead_kernel<8><<<blocks, EBC_THREADS, smem, stream>>>(s->cfg, s->st, s->d_actions, vin, reward, done, event, rec);
  else if (group == 16)
    lookahead_kernel<16><<<blocks, EBC_THREADS, smem, stream>>>(s->cfg, s->st, s->d_actions, vin, reward, done, event, rec);
  else
    lookahead_kernel<32><<<blocks, EBC_THREADS, smem, stream>>>(s->cfg, s->st, s->d_actions, vin, reward, done, event, rec);
  s->la_rec_valid = rec != nullptr;
  return ebc_check_launch(s, "lookahead_kernel");
}

int ebc_launch_transform(ebc_sim *s, float *out, cudaStream_t stream) {
  const int blocks = (s->cfg.n_episodes + EBC_WARPS_PER_BLOCK - 1) / EBC_WARPS_PER_BLOCK;
  const int n = s->cfg.max_humans + s->cfg.max_statics, D = s->cfg.with_agent_type ? 17 : 13;
  const size_t smem = (size_t)EBC_WARPS_PER_BLOCK * n * D * sizeof(float);
  transform_kernel<<<blocks, EBC_THREADS, smem, stream>>>(s->cfg, s->st, out);
  return ebc_check_launch(s, "transform_kernel");
}

int ebc_launch_select(ebc_sim *s, const double *reward, const float *values, double *action_values,
                      int32_t *argmax, uint8_t *nan_flag, cudaStream_t stream) {
  const int blocks = (s->cfg.n_episodes + EBC_WARPS_PER_BLOCK - 1) / EBC_WARPS_PER_BLOCK;
  select_kernel<<<blocks, EBC_THREADS, 0, stream>>>(s->cfg, s->st, reward, values, action_values, argmax, nan_flag);
  return ebc_check_launch(s, "select_kernel");
}

int ebc_launch_step(ebc_sim *s, bool fused_orca, const int32_t *action_idx, const double *action,
                    const uint8_t *active, double *reward, uint8_t *done, uint8_t *event, double *dmin,
                    double *dist_to_goal, cudaStream_t stream) {
  s->la_rec_valid = 0;      // the state moves on: the lookahead records no longer describe it
  ebc_stats sx = s->stats;                      // all-null when unbound
  if (!active && sx.alive) active = sx.alive;   // the bound alive[] is the mask (ebc_bind_stats)
  if (fused_orca && s->cfg.orca_obstacles) {
    // block per episode: the obstacle vertices are staged in shared memory once, every warp solves humans' LPs,
    // the block synchronises, warp 0 commits
    const int threads = fused_warps(s) * 32;
    orca_step_kernel<true><<<s->cfg.n_episodes, threads, 0, stream>>>(s->cfg, s->st, s->d_actions, action_idx, action,
                                                                    active, reward, done, event, dmin, dist_to_goal, sx);
    return ebc_check_launch(s, "orca_step_kernel");
  }
  if (fused_orca) {
    // without obstacles the policy-free step is K1 (a warp, or half a warp, per human over the WHOLE batch) followed by
    // K2 on the same stream: measured 0.46 ms against 0.64 ms for the block-per-episode kernel at 65,536 episodes of
    // cfg2 (0.047 against 0.052 ms at 4,096) -- a block that waits for its one committing warp keeps its slot idle
    const int rc = launch_orca_groups(s, active, stream);
    if (rc) return rc;
  }
  const int blocks = (s->cfg.n_episodes + EBC_WARPS_PER_BLOCK - 1) / EBC_WARPS_PER_BLOCK;
  step_kernel<<<blocks, EBC_THREADS, 0, stream>>>(s->cfg, s->st, s->d_actions, action_idx, action, active, reward,
                                                  done, event, dmin, dist_to_goal, sx);
  return ebc_check_launch(s, "step_kernel");
}

int ebc_launch_grid_map(ebc_sim *s, const ebc_grid_map *map, uint8_t *out, cudaStream_t stream) {
  const int S = map->size;
  const size_t smem = (size_t)(((S + 2) * (S + 2) + 15) & ~15) + 4 * sizeof(int) * (size_t)S;
  if (S <= 62 && !getenv("EBC_GRID_MAP_BYTES")) {      // a framed row fits one 64-bit word (EBC_GRID_MAP_BYTES=1: the general kernel)
    const uint32_t magic = (uint32_t)((0x100000000ull + (unsigned)S - 1u) / (unsigned)S);   // idx / S = umulhi(idx, magic): exact for idx * S < 2^32
    grid_map_bits_kernel<<<s->cfg.n_episodes, 256, 0, stream>>>(s->cfg, s->st, S, magic, out);
    return ebc_check_launch(s, "grid_map_bits_kernel");
  }
  // one 32-bit store per four cells only where every episode's map starts on a 4-byte boundary: S * S % 4 == 0 and
  // an aligned `out` (the C API takes any uint8_t *, e.g. a view at an odd offset); byte stores otherwise
  const bool packed = (S * S) % 4 == 0 && (uintptr_t)out % 4 == 0;
  grid_map_kernel<<<s->cfg.n_episodes, 256, smem, stream>>>(s->cfg, s->st, S, packed, out);
  return ebc_check_launch(s, "grid_map_kernel");
}

int ebc_launch_angular_map(ebc_sim *s, const ebc_angular_map *map, const double *poly_xy, const int32_t *poly_count,
                           double *out, cudaStream_t stream) {
  const int blocks = (s->cfg.n_episodes + EBC_WARPS_PER_BLOCK - 1) / EBC_WARPS_PER_BLOCK;
  angular_map_kernel<<<blocks, EBC_THREADS, 0, stream>>>(s->cfg, s->st, *map, poly_xy, poly_count, out);
  return ebc_check_launch(s, "angular_map_kernel");
}
