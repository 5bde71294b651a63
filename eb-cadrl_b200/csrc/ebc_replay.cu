// ebc_replay.cu — the reference's seeded scene stream (simulator/scene/scene_generator.py, generate_random_scene with
// scene_number = seed) replayed per episode: numpy's legacy MT19937 RandomState and the generator's rules, statement by
// statement, in one __host__ __device__ function.  The kernel runs it thread per episode; the diagnostics export runs
// the same function on the host so that the CPU tests can hold it to numpy.
//
// This unit is compiled without FMA contraction on both sides (-fmad=false, -Xcompiler -ffp-contract=off): every fp64
// operation happens as the Python code writes it, and the one fused multiply-add numpy performs (numpy.linalg.norm of a
// 2-vector, see scene_norm) is written out explicitly.
#include <math.h>
#include <string.h>

#include "ebc_internal.cuh"

#define HD __host__ __device__

namespace {

constexpr int MT_N = 624, MT_M = 397;
constexpr int MAX_TRIES = 100000;                // scene_generator.py MAX_TRIES
constexpr int GROUP_CAP = 64;                    // agents of one list (adults / bicycles / children) a scene may hold
// threads per block: each thread replays one whole scene serially, so small blocks spread a batch over more SMs
constexpr int REPLAY_THREADS = 32;

// ---- numpy's legacy RandomState over MT19937 (numpy/random/src/mt19937, legacy distributions) -------------------------
struct Mt19937 {
  uint32_t key[MT_N];
  int pos;
};

// np.random.seed(int): init_genrand (mt19937_seed), not init_by_array
HD inline void mt_seed(Mt19937 &m, uint32_t s) {
  for (int i = 0; i < MT_N; ++i) {
    m.key[i] = s;
    s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)(i + 1);
  }
  m.pos = MT_N;
}

HD inline void mt_refill(Mt19937 &m) {
  int i = 0;
  uint32_t y;
  for (; i < MT_N - MT_M; ++i) {
    y = (m.key[i] & 0x80000000u) | (m.key[i + 1] & 0x7fffffffu);
    m.key[i] = m.key[i + MT_M] ^ (y >> 1) ^ (-(y & 1u) & 0x9908b0dfu);
  }
  for (; i < MT_N - 1; ++i) {
    y = (m.key[i] & 0x80000000u) | (m.key[i + 1] & 0x7fffffffu);
    m.key[i] = m.key[i + (MT_M - MT_N)] ^ (y >> 1) ^ (-(y & 1u) & 0x9908b0dfu);
  }
  y = (m.key[MT_N - 1] & 0x80000000u) | (m.key[0] & 0x7fffffffu);
  m.key[MT_N - 1] = m.key[MT_M - 1] ^ (y >> 1) ^ (-(y & 1u) & 0x9908b0dfu);
  m.pos = 0;
}

HD inline uint32_t mt_next(Mt19937 &m) {
  if (m.pos == MT_N) mt_refill(m);
  uint32_t y = m.key[m.pos++];
  y ^= y >> 11;
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  return y ^ (y >> 18);
}

// random(): 53 bits from two outputs
HD inline double np_random(Mt19937 &m) {
  const int32_t a = (int32_t)(mt_next(m) >> 5), b = (int32_t)(mt_next(m) >> 6);
  return (a * 67108864.0 + b) / 9007199254740992.0;
}

// uniform(lo, hi)
HD inline double np_uniform(Mt19937 &m, double lo, double hi) { return lo + (hi - lo) * np_random(m); }

// randint(lo, hi) with integer bounds (float bounds are truncated toward zero by the caller): masked rejection on single
// 32-bit outputs; an empty range [lo, lo] draws nothing.  Every range here is far below 2^32.
HD inline long long np_randint(Mt19937 &m, long long lo, long long hi) {
  const uint32_t rng = (uint32_t)(hi - 1 - lo);
  if (rng == 0) return lo;
  uint32_t mask = rng;
  mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
  uint32_t v;
  while ((v = (mt_next(m) & mask)) > rng) {
  }
  return lo + (long long)v;
}

// choice([1, -1], p=[0.5, 0.5]): one random(), right-side search in the cumulative sums [0.5, 1.0]
HD inline int np_choice_sign(Mt19937 &m) { return np_random(m) < 0.5 ? 1 : -1; }

// ---- the generator ------------------------------------------------------------------------------------------------
// numpy.linalg.norm((x, y)) is sqrt(dot(v, v)); the dot product goes through OpenBLAS's ddot, which on FMA-capable x86
// cores accumulates the second product with a fused multiply-add.  `fused` says which of the two the host's numpy does.
HD inline double scene_norm(double x, double y, int fused) { return fused ? sqrt(fma(y, y, x * x)) : sqrt(x * x + y * y); }

struct Group {                   // the agents of one list so far: what _too_close walks besides the robot
  double px[GROUP_CAP], py[GROUP_CAP], gx[GROUP_CAP], gy[GROUP_CAP], r[GROUP_CAP];
  int n;
};

struct Agent {
  double px, py, gx, gy, v_pref, radius;
};

struct Replay {
  const ebc_replay_config *c;
  Mt19937 *mt;
  double R;                      // circle_radius: the robot starts at (0, -R) with its goal at (0, R)
};

// _too_close (scene_generator.py): the robot first, then the list
HD inline bool too_close(const Replay &s, double px, double py, double radius, const Group &g, bool with_goals) {
  const ebc_replay_config &c = *s.c;
  {
    const double d = radius + c.robot_radius + c.discomfort_dist;
    if (scene_norm(px - 0.0, py - (-s.R), c.norm_fused) < d) return true;
    if (with_goals && scene_norm(px - 0.0, py - s.R, c.norm_fused) < d) return true;
  }
  for (int j = 0; j < g.n; ++j) {
    const double d = radius + g.r[j] + c.discomfort_dist;
    if (scene_norm(px - g.px[j], py - g.py[j], c.norm_fused) < d) return true;
    if (with_goals && scene_norm(px - g.gx[j], py - g.gy[j], c.norm_fused) < d) return true;
  }
  return false;
}

// Agent.sample_random_attributes: v_pref, then radius
HD inline void sample_attributes(const Replay &s, Agent &a, int t) {
  if (!s.c->randomize_attributes) return;
  a.v_pref = np_uniform(*s.mt, s.c->v_pref_min[t], s.c->v_pref_max[t]);
  a.radius = np_uniform(*s.mt, s.c->radius_min[t], s.c->radius_max[t]);
}

HD inline void square_crossing(const Replay &s, Agent &a, int t, const Group &g) {
  sample_attributes(s, a, t);
  const double hw = s.c->square_width / 2;
  double px = 0, py = 0, gx = 0, gy = 0;
  for (int index = 0; index < MAX_TRIES; ++index) {
    const int side = (int)np_randint(*s.mt, 0, 4);          // choice(["top", "bottom", "left", "right"])
    const double u = np_uniform(*s.mt, -hw, hw);
    px = side == 0 ? u : side == 1 ? u : side == 2 ? -hw : hw;
    py = side == 0 ? hw : side == 1 ? -hw : u;
    if (too_close(s, px, py, a.radius, g, false) && index != MAX_TRIES - 1) continue;
    const double v = np_uniform(*s.mt, -hw, hw);            // the goal is drawn only for an accepted start
    gx = side == 0 ? v : side == 1 ? v : side == 2 ? hw : -hw;
    gy = side == 0 ? -hw : side == 1 ? hw : v;
    break;
  }
  a.px = px; a.py = py; a.gx = gx; a.gy = gy;
}

HD inline void square_crossing_old(const Replay &s, Agent &a, int t, const Group &g) {
  sample_attributes(s, a, t);
  const double sw = s.c->square_width;
  const double sign = (double)np_choice_sign(*s.mt);
  double px = 0, py = 0, gx = 0, gy = 0;
  for (int index = 0; index < MAX_TRIES; ++index) {
    px = np_random(*s.mt) * sw * 0.5 * sign;
    py = sw * 0.5;
    if (np_random(*s.mt) > 0.5) {
      const double tmp = px; px = py; py = tmp;
    }
    if (too_close(s, px, py, a.radius, g, false) && index != MAX_TRIES - 1) continue;
    const int k = (int)np_randint(*s.mt, 0, 3);              // [(-1, 1), (1, -1), (-1, -1)][randint(3)]
    gx = px * (k == 1 ? 1.0 : -1.0);
    gy = py * (k == 0 ? 1.0 : -1.0);
    const double clear = a.radius + s.c->robot_radius + s.c->discomfort_dist;
    if (index == MAX_TRIES - 1 || !(scene_norm(gx - 0.0, gy - s.R, s.c->norm_fused) < clear)) break;
  }
  a.px = px; a.py = py; a.gx = gx; a.gy = gy;
}

HD inline void circle_crossing(const Replay &s, Agent &a, int t, const Group &g) {
  sample_attributes(s, a, t);
  const double R = s.c->circle_radius;
  double px = 0, py = 0;
  for (int i = 0; i < MAX_TRIES; ++i) {                     // the last try is kept when every one fails
    const double angle = np_random(*s.mt) * 3.141592653589793 * 2;
    px = R * cos(angle) + 0.0;
    py = R * sin(angle) + 0.0;
    if (!too_close(s, px, py, a.radius, g, true)) break;
  }
  a.px = px; a.py = py; a.gx = -px; a.gy = -py;
}

HD inline void standing(Agent &a, double x, double y) { a.px = x; a.py = y; a.gx = x; a.gy = y; }

// Where one scene's agents, discs, rectangles and polygons go; capacities bound every store.
struct ReplayOut {
  float4 *hum_pv, *hum_gr;
  uint8_t *hum_type;
  float2 *hum_nv;
  float4 *stat;
  short4 *rect;
  double *poly;                  // [Pm][4][2]
  int Hm, Sm, Rm, Pm;
  int H, S, Rc, P;               // what the scene needs so far
};

HD inline void emit_agent(ReplayOut &o, Group &g, const Agent &a, int type) {
  if (g.n < GROUP_CAP) {
    g.px[g.n] = a.px; g.py[g.n] = a.py; g.gx[g.n] = a.gx; g.gy[g.n] = a.gy; g.r[g.n] = a.radius;
    ++g.n;
  }
  if (o.H < o.Hm) {
    o.hum_pv[o.H] = make_float4((float)a.px, (float)a.py, 0.f, 0.f);
    o.hum_gr[o.H] = make_float4((float)a.gx, (float)a.gy, (float)a.v_pref, (float)a.radius);
    o.hum_type[o.H] = (uint8_t)type;
    o.hum_nv[o.H] = make_float2(0.f, 0.f);
  }
  ++o.H;
}

HD inline Agent fresh(const ebc_replay_config &c, int t) {
  Agent a;
  a.px = a.py = a.gx = a.gy = 0.0;
  a.v_pref = c.v_pref[t];
  a.radius = c.radius[t];
  return a;
}

// the `mixed` rule's tables, in sorted key order: static {0: .05, 1: .2, 2: .2, 3: .3, 4: .1, 5: .15}, dynamic
// {1: .3, 2: .3, 3: .2, 4: .1, 5: .1}
HD inline double mixed_probability(bool is_static, int k) {
  if (is_static) return k == 0 ? 0.05 : k == 1 ? 0.2 : k == 2 ? 0.2 : k == 3 ? 0.3 : k == 4 ? 0.1 : 0.15;
  return k == 0 ? 0.3 : k == 1 ? 0.3 : k == 2 ? 0.2 : k == 3 ? 0.1 : 0.1;
}

// generate_random_adult_position; returns what the rule leaves in SceneGenerator.adult_num
HD inline int replay_adults(const Replay &s, ReplayOut &o, Group &g) {
  const ebc_replay_config &c = *s.c;
  Mt19937 &mt = *s.mt;
  int adult_num = c.count[0];
  g.n = 0;
  switch (c.rule[0]) {
    case EBC_REPLAY_SQUARE_CROSSING:
    case EBC_REPLAY_CIRCLE_CROSSING:
      for (int i = 0; i < adult_num; ++i) {
        Agent a = fresh(c, 0);
        if (c.rule[0] == EBC_REPLAY_SQUARE_CROSSING) square_crossing(s, a, 0, g);
        else circle_crossing(s, a, 0, g);
        emit_agent(o, g, a, EBC_ADULT);
      }
      break;
    case EBC_REPLAY_MIXED: {
      const bool is_static = np_random(mt) < 0.2;
      double prob = np_random(mt);
      const int n_keys = is_static ? 6 : 5, first_key = is_static ? 0 : 1;
      for (int k = 0; k < n_keys; ++k) {
        const double value = mixed_probability(is_static, k);
        if (prob - value <= 0) {
          adult_num = first_key + k;
          break;
        }
        prob -= value;
      }
      if (is_static) {
        if (adult_num == 0) {
          Agent a = fresh(c, 0);
          standing(a, 0, -10);
          emit_agent(o, g, a, EBC_ADULT);
        }
        for (int i = 0; i < adult_num; ++i) {
          Agent a = fresh(c, 0);
          const int sign = np_random(mt) > 0.5 ? -1 : 1;
          double px = 0, py = 0;
          for (int k = 0; k < MAX_TRIES; ++k) {
            px = np_random(mt) * 4 * 0.5 * sign;
            py = (np_random(mt) - 0.5) * 8;
            if (!too_close(s, px, py, a.radius, g, false)) break;
          }
          standing(a, px, py);
          emit_agent(o, g, a, EBC_ADULT);
        }
      } else {
        for (int i = 0; i < adult_num; ++i) {
          Agent a = fresh(c, 0);
          if (i < 2) circle_crossing(s, a, 0, g);
          else square_crossing(s, a, 0, g);
          emit_agent(o, g, a, EBC_ADULT);
        }
      }
      break;
    }
    case EBC_REPLAY_MIXED_20: {
      const int static_num = (int)np_randint(mt, 0, 20);
      const int dynamic_num = 20 - static_num;
      adult_num = 20;
      // _static_adults(static_num, width=6, height=8)
      for (int i = 0; i < static_num; ++i) {
        Agent a = fresh(c, 0);
        if (i == 0) {
          standing(a, -0.5, -2.5);
        } else {
          const double sign = (double)np_choice_sign(mt);
          double px = 0, py = 0;
          for (int k = 0; k < MAX_TRIES; ++k) {
            px = np_random(mt) * 6 * 0.5 * sign;
            py = (np_random(mt) - 0.5) * 8;
            const bool collide = too_close(s, px, py, a.radius, g, false);
            const double last_r = g.r[g.n - 1];               // the list's last adult (i >= 1: never empty)
            const bool near_goal = scene_norm(px - 0.0, py - s.R, c.norm_fused) < a.radius + last_r + c.discomfort_dist;
            if (!collide && !near_goal) break;
          }
          standing(a, px, py);
        }
        emit_agent(o, g, a, EBC_ADULT);
      }
      for (int i = 0; i < dynamic_num; ++i) {
        Agent a = fresh(c, 0);
        if (i < dynamic_num / 2) circle_crossing(s, a, 0, g);
        else square_crossing(s, a, 0, g);
        emit_agent(o, g, a, EBC_ADULT);
      }
      break;
    }
    default: {                   // EBC_REPLAY_ONE_STATIC: two adults standing at (-2, -8) and (-3, -8)
      for (int x = -2; x >= -3; --x) {
        Agent a = fresh(c, 0);
        standing(a, (double)x, -8);
        emit_agent(o, g, a, EBC_ADULT);
      }
      break;
    }
  }
  return adult_num;
}

HD inline void replay_group(const Replay &s, ReplayOut &o, Group &g, int t, int type) {
  g.n = 0;
  for (int i = 0; i < s.c->count[t]; ++i) {
    Agent a = fresh(*s.c, t);
    const int rule = s.c->rule[t];
    if (rule == EBC_REPLAY_CIRCLE_CROSSING) circle_crossing(s, a, t, g);
    else if (rule == EBC_REPLAY_SQUARE_CROSSING_OLD) square_crossing_old(s, a, t, g);
    else square_crossing(s, a, t, g);
    emit_agent(o, g, a, type);
  }
}

// _near_robot: the robot's start (0, -R) and goal (0, R)
HD inline bool near_robot(const Replay &s, double xm, double ym, double half_x, double half_y, bool circle) {
  const double clear = s.c->robot_radius + s.c->discomfort_dist;
  for (int k = 0; k < 2; ++k) {
    const double ry = k == 0 ? -s.R : s.R;
    if (circle) {
      if (scene_norm(xm - 0.0, ym - ry, s.c->norm_fused) < half_x + clear) return true;
    } else if (fabs(xm - 0.0) < half_x + clear && fabs(ym - ry) < half_y + clear) {
      return true;
    }
  }
  return false;
}

// The zero cells place_obstacles_on_map writes along one axis of the per-cell path: {rint(loc + i - dim / 2.0)} for
// i < dim, clipped to 0 < index < grid.  The values are nondecreasing in i, so the maximal runs [lo, hi) come out in
// order: this finds the run that starts at or after index i and returns the index past it (lo = -1: no run left).  An
// odd dim gives every other cell (banker's rounding of half-integers): one run per cell.  Recomputed on every walk, so
// no run count is too large to place.
HD inline int next_run(int loc, int dim, int grid, int i, int &lo, int &hi) {
  lo = hi = -1;
  for (; i < dim; ++i) {
    const int v = (int)rint((double)(loc + i) - dim / 2.0);
    if (!(0 < v && v < grid)) {
      if (lo >= 0) break;
      continue;
    }
    if (lo < 0) {
      lo = v;
      hi = v + 1;
    } else if (v == hi) {
      hi = v + 1;
    } else if (v != hi - 1) {
      break;                                     // a gap: the next run starts at i
    }
  }
  return i;
}

// One obstacle of generate_static_map_input: its grid rectangles, static discs and polygon
HD inline void place_obstacle(const Replay &s, ReplayOut &o, int grid, long long lx, long long ly, double xm, double ym,
                              double half_x, double half_y, int dx, int dy) {
  // add(): location on the grid and the polygon (scene.obstacle_vertices)
  const int loc_x = (int)rint((double)lx + grid / 2.0), loc_y = (int)rint((double)ly + grid / 2.0);
  const double v0x = xm + half_x, v0y = ym + half_y, v1x = xm - half_x, v1y = ym + half_y;
  const double v2x = xm - half_x, v2y = ym - half_y, v3x = xm + half_x, v3y = ym - half_y;
  if (o.P < o.Pm) {
    double *p = o.poly + (size_t)o.P * 8;
    p[0] = v0x; p[1] = v0y; p[2] = v1x; p[3] = v1y; p[4] = v2x; p[5] = v2y; p[6] = v3x; p[7] = v3y;
  }
  ++o.P;
  // place_obstacles_on_map: the slice on the interior path; on the per-cell path the product of the per-axis cell sets
  const bool inside = (dx / 2.0 < loc_x && loc_x < grid - dx / 2.0) && (dy / 2.0 < loc_y && loc_y < grid - dy / 2.0);
  if (inside) {
    if (dx > 0 && dy > 0) {
      const int x0 = (int)rint(loc_x - dx / 2.0), y0 = (int)rint(loc_y - dy / 2.0);
      if (o.Rc < o.Rm)
        o.rect[o.Rc] = make_short4((short)x0, (short)y0, (short)min(x0 + dx, grid), (short)min(y0 + dy, grid));
      ++o.Rc;
    }
  } else {
    int x0, x1, y0, y1;
    for (int ix = next_run(loc_x, dx, grid, 0, x0, x1); x0 >= 0; ix = next_run(loc_x, dx, grid, ix, x0, x1))
      for (int iy = next_run(loc_y, dy, grid, 0, y0, y1); y0 >= 0; iy = next_run(loc_y, dy, grid, iy, y0, y1)) {
        if (o.Rc < o.Rm) o.rect[o.Rc] = make_short4((short)x0, (short)y0, (short)x1, (short)y1);
        ++o.Rc;
      }
  }
  // create_observation_from_static_obstacles: ADULT_STATIC discs along the obstacle
  const double cx = (v0x + v2x) / 2.0, cy = (v0y + v2y) / 2.0;
  const double sqrt2 = sqrt(2.0);
  if (dx == dy) {
    if (o.S < o.Sm) o.stat[o.S] = make_float4((float)cx, (float)cy, (float)((v0x - cx) * sqrt2), 0.f);
    ++o.S;
  } else if (dx > dy) {
    const double r = (v0y - cy) * sqrt2;
    for (double x = v1x + r; x < v0x && r > 0; x = x + 2 * r) {
      if (o.S < o.Sm) o.stat[o.S] = make_float4((float)x, (float)cy, (float)r, 0.f);
      ++o.S;
    }
  } else {
    const double r = (v0x - cx) * sqrt2;
    for (double y = v2y + r; y < v0y && r > 0; y = y + 2 * r) {
      if (o.S < o.Sm) o.stat[o.S] = make_float4((float)cx, (float)y, (float)r, 0.f);
      ++o.S;
    }
  }
}

// generate_static_map_input: circles, then walls
HD inline void replay_static_map(const Replay &s, ReplayOut &o) {
  const ebc_replay_config &c = *s.c;
  Mt19937 &mt = *s.mt;
  const double res = c.map_resolution;
  const int grid = (int)rint(c.map_size_m / res);
  const long long lo = (long long)(-grid / 2.0), hi = (long long)(grid / 2.0);    // randint truncates float bounds
  for (int k = 0; k < c.num_circles; ++k) {
    long long lx = 0, ly = 0;
    double radius = 0;
    for (int t = 0; t < MAX_TRIES; ++t) {
      lx = np_randint(mt, lo, hi);
      ly = np_randint(mt, lo, hi);
      radius = (np_random(mt) + 0.5) * 0.7;
      if (!near_robot(s, lx * res, ly * res, radius, radius, true)) break;
    }
    const int d = (int)rint(2 * radius / res);
    place_obstacle(s, o, grid, lx, ly, lx * res, ly * res, 1 * radius, 1 * radius, d, d);
  }
  for (int k = 0; k < c.num_walls; ++k) {
    long long lx = 0, ly = 0, x_dim = 1, y_dim = 1;
    for (int t = 0; t < MAX_TRIES; ++t) {
      lx = np_randint(mt, lo, hi);
      ly = np_randint(mt, lo, hi);
      if (np_random(mt) > 0.5) {
        x_dim = np_randint(mt, c.min_wall_length, c.max_wall_length + 1);
        y_dim = 1;
      } else {
        y_dim = np_randint(mt, c.min_wall_length, c.max_wall_length + 1);
        x_dim = 1;
      }
      if (!near_robot(s, lx * res, ly * res, x_dim / 2.0, y_dim / 2.0, false)) break;
    }
    place_obstacle(s, o, grid, lx, ly, lx * res, ly * res, 1 * x_dim / 2.0, 1 * y_dim / 2.0, (int)rint(x_dim / res),
                   (int)rint(y_dim / res));
  }
}

// One episode: generate_random_scene(scene_number = seed) -> what BatchedEnv.reset_batch loads.  Slots past the
// scene's counts (up to the capacities) are zeroed; nothing is written past a capacity.  need = (humans, static discs,
// grid rectangles, polygons) the scene holds; the return value is what the scene leaves in SceneGenerator.adult_num.
HD int replay_scene(const ebc_replay_config &c, uint32_t seed, Mt19937 &mt, Group &g, ReplayOut &o, int32_t *need) {
  mt_seed(mt, seed);
  Replay s;
  s.c = &c;
  s.mt = &mt;
  s.R = c.circle_radius;
  o.H = o.S = o.Rc = o.P = 0;
  const int adult_num = replay_adults(s, o, g);
  replay_group(s, o, g, 1, EBC_BICYCLE);
  replay_group(s, o, g, 2, EBC_CHILD);
  replay_static_map(s, o);
  for (int h = o.H; h < o.Hm; ++h) {
    o.hum_pv[h] = make_float4(0.f, 0.f, 0.f, 0.f);
    o.hum_gr[h] = make_float4(0.f, 0.f, 0.f, 0.f);
    o.hum_type[h] = 0;
    o.hum_nv[h] = make_float2(0.f, 0.f);
  }
  for (int k = o.S; k < o.Sm; ++k) o.stat[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = o.Rc; k < o.Rm; ++k) o.rect[k] = make_short4(0, 0, 0, 0);
  for (int k = o.P * 8; k < o.Pm * 8; ++k) o.poly[k] = 0.0;
  need[0] = o.H;
  need[1] = o.S;
  need[2] = o.Rc;
  need[3] = o.P;
  return adult_num;
}

__global__ void __launch_bounds__(REPLAY_THREADS)
replay_scenes_kernel(const ebc_config c, const ebc_state st, const ebc_replay_config rc, const uint32_t *seeds,
                     const uint8_t *mask, double *poly_xy, int32_t *poly_count, int32_t *need) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= c.n_episodes) return;
  if (mask && !mask[e]) return;
  Mt19937 mt;
  Group g;
  ReplayOut o;
  const size_t H = (size_t)e * c.max_humans, S = (size_t)e * c.max_statics, R = (size_t)e * c.max_rects;
  o.hum_pv = reinterpret_cast<float4 *>(st.hum_pv) + H;
  o.hum_gr = reinterpret_cast<float4 *>(st.hum_gr) + H;
  o.hum_type = st.hum_type + H;
  o.hum_nv = reinterpret_cast<float2 *>(st.hum_nv) + H;
  o.stat = reinterpret_cast<float4 *>(st.stat) + S;
  o.rect = reinterpret_cast<short4 *>(st.rect) + R;
  o.poly = poly_xy + (size_t)e * rc.max_polys * 8;
  o.Hm = c.max_humans;
  o.Sm = c.max_statics;
  o.Rm = c.max_rects;
  o.Pm = rc.max_polys;
  int32_t n[4];
  const int adult_num = replay_scene(rc, seeds[e], mt, g, o, n);
  for (int k = 0; k < 4; ++k) need[(size_t)e * 5 + k] = n[k];
  need[(size_t)e * 5 + 4] = adult_num;
  st.hum_count[e] = min(n[0], o.Hm);
  st.stat_count[e] = min(n[1], o.Sm);
  st.rect_count[e] = min(n[2], o.Rm);
  poly_count[e] = min(n[3], o.Pm);
  // env.reset: the robot at (0, -R) facing +y with its goal at (0, R), at rest; global_time = 0
  const double Rr = rc.circle_radius;
  reinterpret_cast<float4 *>(st.rob_pv)[e] = make_float4(0.f, (float)(-Rr), 0.f, 0.f);
  reinterpret_cast<float4 *>(st.rob_gr)[e] = make_float4(0.f, (float)Rr, (float)rc.robot_v_pref, (float)rc.robot_radius);
  st.rob_theta[e] = (float)(3.141592653589793 / 2);
  st.time[e] = 0.0;
}

}  // namespace

int ebc_launch_replay(ebc_sim *s, const ebc_replay_config *cfg, const uint32_t *seeds, const uint8_t *mask,
                      double *poly_xy, int32_t *poly_count, int32_t *need, cudaStream_t stream) {
  s->la_rec_valid = 0;      // the state moves on: the lookahead records no longer describe it
  const int blocks = (s->cfg.n_episodes + REPLAY_THREADS - 1) / REPLAY_THREADS;
  replay_scenes_kernel<<<blocks, REPLAY_THREADS, 0, stream>>>(s->cfg, s->st, *cfg, seeds, mask, poly_xy, poly_count, need);
  return ebc_check_launch(s, "replay_scenes_kernel");
}

extern "C" {

int ebc_replay_scene_host(const ebc_replay_config *cfg, uint32_t seed, int32_t max_humans, int32_t max_statics,
                          int32_t max_rects, float *hum_pv, float *hum_gr, uint8_t *hum_type, float *stat, int16_t *rect,
                          double *poly_xy, int32_t *need) {
  if (!cfg || !need || max_humans < 0 || max_statics < 0 || max_rects < 0 || cfg->max_polys < 0 ||
      (max_humans > 0 && (!hum_pv || !hum_gr || !hum_type)) || (max_statics > 0 && !stat) || (max_rects > 0 && !rect) ||
      (cfg->max_polys > 0 && !poly_xy))
    return EBC_ERR_INVALID;
  Mt19937 *mt = new Mt19937;
  Group *g = new Group;
  float2 *nv = new float2[max_humans > 0 ? max_humans : 1];
  ReplayOut o;
  o.hum_pv = reinterpret_cast<float4 *>(hum_pv);
  o.hum_gr = reinterpret_cast<float4 *>(hum_gr);
  o.hum_type = hum_type;
  o.hum_nv = nv;
  o.stat = reinterpret_cast<float4 *>(stat);
  o.rect = reinterpret_cast<short4 *>(rect);
  o.poly = poly_xy;
  o.Hm = max_humans;
  o.Sm = max_statics;
  o.Rm = max_rects;
  o.Pm = cfg->max_polys;
  int32_t n[4];
  const int adult_num = replay_scene(*cfg, seed, *mt, *g, o, n);
  for (int k = 0; k < 4; ++k) need[k] = n[k];
  need[4] = adult_num;
  delete[] nv;
  delete g;
  delete mt;
  return EBC_OK;
}

int ebc_replay_rng_host(uint32_t *key, int32_t *pos, int32_t op, double a, double b, double *out) {
  if (!key || !pos || !out || *pos < 0 || *pos > MT_N) return EBC_ERR_INVALID;
  Mt19937 m;
  memcpy(m.key, key, sizeof(m.key));
  m.pos = *pos;
  switch (op) {
    case EBC_REPLAY_RNG_SEED: mt_seed(m, (uint32_t)a); *out = 0; break;
    case EBC_REPLAY_RNG_RANDOM: *out = np_random(m); break;
    case EBC_REPLAY_RNG_UNIFORM: *out = np_uniform(m, a, b); break;
    case EBC_REPLAY_RNG_RANDINT: {
      const long long lo = (long long)a, hi = (long long)b;     // numpy truncates float bounds toward zero
      if (hi <= lo || hi - 1 - lo > 0xFFFFFFFFll) return EBC_ERR_INVALID;
      *out = (double)np_randint(m, lo, hi);
      break;
    }
    case EBC_REPLAY_RNG_CHOICE_SIGN: *out = np_choice_sign(m); break;
    default: return EBC_ERR_INVALID;
  }
  memcpy(key, m.key, sizeof(m.key));
  *pos = m.pos;
  return EBC_OK;
}

}  // extern "C"
