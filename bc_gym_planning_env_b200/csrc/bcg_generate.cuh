// Device-side AisleTurnEnv generation (SURVEY.md 8f rank 1).  The reference rebuilds a random aisle turn on the
// host at every reset (envs/synth_turn_env.py:278-291 -> :317-332 -> :110-192 -> cv2.line), about 1 k maps/s per
// core.  Here one CTA regenerates one env inside its fixed-size slots of the map / tile / path arenas: geometry,
// five walls rasterised like cv2.line (previous walls erased pixel by pixel), both tile planes kept in step,
// refined path, chunk bounds and the initial state.  Included by bcg_kernels.cu.
#pragma once
#include "bcg_device.cuh"

namespace bcg {

// uniform in [0, 1) from 53 bits of one Philox block half; draws 2 k and 2 k + 1 share a block
__device__ __forceinline__ double philox_uniform(uint64_t seed, uint64_t env, uint64_t draw, uint32_t k) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)draw, 0x41495345u + (k >> 1), (uint32_t)(draw >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const uint64_t bits = (k & 1) ? (((uint64_t)r.z << 21) | (r.w >> 11)) : (((uint64_t)r.x << 21) | (r.y >> 11));
  return (double)bits * 0x1.0p-53;
}

// RandomAisleTurnEnv._draw_random_turn_params (envs/synth_turn_env.py:317-332): same distributions, same draw order,
// Philox instead of MT19937
__device__ __forceinline__ BcgTurnParams draw_turn_params(uint64_t seed, uint64_t env, uint64_t draw) {
  BcgTurnParams t;
  t.main_corridor_length = 10.0 + 6.0 * philox_uniform(seed, env, draw, 0);
  t.turn_corridor_length = 4.0 + 8.0 * philox_uniform(seed, env, draw, 1);
  const double lim = 3. / 8. * BCG_PI;
  t.turn_corridor_angle = -lim + (2 * lim) * philox_uniform(seed, env, draw, 2);
  t.main_corridor_width = 0.5 + philox_uniform(seed, env, draw, 3);
  t.turn_corridor_width = 0.5 + philox_uniform(seed, env, draw, 4);
  t.margin = 1.0;
  t.flip_arnd_oy = philox_uniform(seed, env, draw, 5) < 0.5;
  t.flip_arnd_ox = philox_uniform(seed, env, draw, 6) < 0.5;
  t.rot_theta = BCG_TWO_PI * philox_uniform(seed, env, draw, 7);
  return t;
}

struct AisleGeometry {
  double wall[5][4];    // world end points (x0, y0, x1, y1) of the walls a-i, c-d, d-e, j-g, g-h
  double way[4][3];     // oriented way points
  double origin_x, origin_y;
  int width, height;    // costmap cells
};

// path_and_costmap_from_config (envs/synth_turn_env.py:41-192): corridor corners, way points, flips, rotation,
// world bounds.  np.dot of the 2 x 2 transform with a point accumulates fused (BLAS), hence the fma.
__device__ __forceinline__ AisleGeometry aisle_geometry(const BcgTurnParams& tp, double inv_res) {
  const double h = tp.main_corridor_length / 2, far = tp.turn_corridor_length / 2;
  const double alpha = tp.turn_corridor_angle, d = tp.main_corridor_width, z = tp.turn_corridor_width;
  const double ta = tan(alpha), ca = cos(alpha);
  const double lower = -z / ca, upper = z / ca;
  // a b c d e f g h i j
  const double cx[10] = {-d, 0, d, d, far, far, d, far, -d, d};
  const double cy[10] = {-h, -h, -h, d * ta + lower, far * ta + lower, far * ta, d * ta + upper, far * ta + upper, h, h};
  double sn, cs;
  sincos(tp.rot_theta, &sn, &cs);
  const double fx = tp.flip_arnd_oy ? -1. : 1., fy = tp.flip_arnd_ox ? -1. : 1.;
  const double t00 = cs * fx, t01 = -sn * fy, t10 = sn * fx, t11 = cs * fy;
  double mx[10], my[10];
  double min_x = 1e300, max_x = -1e300, min_y = 1e300, max_y = -1e300;
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    mx[k] = fma(t01, cy[k], t00 * cx[k]);
    my[k] = fma(t11, cy[k], t10 * cx[k]);
    min_x = fmin(min_x, mx[k]); max_x = fmax(max_x, mx[k]);
    min_y = fmin(min_y, my[k]); max_y = fmax(max_y, my[k]);
  }
  AisleGeometry g;
  const int wa[5] = {0, 2, 3, 9, 6}, wb[5] = {8, 3, 4, 6, 7};
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    g.wall[k][0] = mx[wa[k]]; g.wall[k][1] = my[wa[k]];
    g.wall[k][2] = mx[wb[k]]; g.wall[k][3] = my[wb[k]];
  }
  const double wx[4] = {0, 0, d, far * ca};
  const double wy[4] = {-h, d * ta + lower, d * ta, far * ca * ta};
  const double wt[4] = {BCG_PI / 2, BCG_PI / 2, alpha, alpha};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    g.way[k][0] = fma(t01, wy[k], t00 * wx[k]);
    g.way[k][1] = fma(t11, wy[k], t10 * wx[k]);
    double t = wt[k];
    if (tp.flip_arnd_ox) t = -t;
    if (tp.flip_arnd_oy) t = BCG_PI - t;
    g.way[k][2] = py_mod(t + tp.rot_theta, BCG_TWO_PI);
  }
  const double size_x = fabs(max_x - min_x) + 2 * tp.margin, size_y = fabs(max_y - min_y) + 2 * tp.margin;
  g.origin_x = min_x - tp.margin;
  g.origin_y = min_y - tp.margin;
  g.width = world_to_pixel_1d(size_x, 0.0, inv_res);      // CostMap2D.create_empty -> world_to_pixel(size, (0, 0), res)
  g.height = world_to_pixel_1d(size_y, 0.0, inv_res);
  return g;
}

// layout of one env's map as the drawing code needs it
struct MapLayout {
  uint8_t* data;       // uint8 rows
  uint32_t* tiles;     // lethal tile plane
  uint32_t* occ;       // occupancy plane (same layout)
  uint32_t* sum;       // tile summary of the occupancy plane: [tiles_y][(tiles_x + 31) / 32] words
  uint8_t* ctiles;     // cell tiles
  int pitch, rows, tiles_x, ctiles_x;
};

// cv2.line(thickness 1, 8-connected) = LineIterator(left to right): the major axis advances every step, the
// minor axis after step j has moved ceil((2 d j - D) / (2 D)) times (clamped at 0), D/d = major/minor extent --
// Bresenham with the initial error D - 2 d in closed form, pixel for pixel equal to cv2.line
// (tests/test_host_logic.py::test_line_pixels_match_cv2).  Threads take pixels j = first, first + stride, ...;
// `value` 254 draws, 0 erases; the lethal and occupancy tile planes and the cell tiles are kept in step.
__device__ __forceinline__ void draw_wall(const MapLayout& m, int x0, int y0, int x1, int y1, uint8_t value, int first,
                                          int stride) {
  if (x1 < x0) {
    int t = x0; x0 = x1; x1 = t;
    t = y0; y0 = y1; y1 = t;
  }
  const int dx = x1 - x0, dy = y1 - y0;
  const int sy = dy >= 0 ? 1 : -1;
  const int ady = dy >= 0 ? dy : -dy;
  const bool steep = ady > dx;
  const int D = steep ? ady : dx, dm = steep ? dx : ady;
  for (int j = first; j <= D; j += stride) {
    const long long t = 2ll * dm * j - D;
    const int mv = t > 0 ? (int)((t + 2ll * D - 1) / (2ll * D)) : 0;
    const int x = steep ? x0 + mv : x0 + j;
    const int y = steep ? y0 + j * sy : y0 + mv * sy;
    if (x < 0 || y < 0 || x >= m.pitch || y >= m.rows) continue;      // never for aisle walls (1 m margin); be safe
    m.data[(int64_t)y * m.pitch + x] = value;
    m.ctiles[(((int64_t)(y >> 3) * m.ctiles_x + (x >> 4)) << 7) + ((y & 7) << 4) + (x & 15)] = value;
    const int64_t widx = (((int64_t)(y >> 4) * m.tiles_x + (x >> 5)) << 4) + (y & 15);
    // tile summary: walls are the only cells of a generated world and all of them are erased before any is drawn,
    // so a tile an erased pixel lies in is empty by the time the drawing starts
    // Only the pixel with which the line enters a tile touches the summary (x grows along the line, y moves by sy:
    // a tile is entered through its column 0, its row 0 / 15, the map's last row, or at the line's first pixel).
    const bool enters = j == 0 || (x & 31) == 0 || (y & 15) == (sy > 0 ? 0 : 15) || y == m.rows - 1;
    uint32_t* const sword = m.sum + (y >> 4) * ((m.tiles_x + 31) >> 5) + (x >> 10);
    const uint32_t sbit = 1u << ((x >> 5) & 31);
    if (value == 254) {
      atomicOr(m.tiles + widx, 1u << (x & 31));
      atomicOr(m.occ + widx, 1u << (x & 31));
      if (enters) atomicOr(sword, sbit);                 // result unused: a fire-and-forget reduction
    } else {
      atomicAnd(m.tiles + widx, ~(1u << (x & 31)));
      atomicAnd(m.occ + widx, ~(1u << (x & 31)));
      if (enters) atomicAnd(sword, ~sbit);
    }
  }
}

// what a slot currently holds (BcgAisleSlots.gen_state, 128 bytes per env)
struct __align__(16) AisleGenState {
  int32_t wall[5][4];   // pixel end points of the walls drawn
  int32_t pitch, rows, tiles_x, ctiles_x;
  int32_t valid;
  int32_t pad[7];
};
static_assert(sizeof(AisleGenState) == 128, "AisleGenState is 128 bytes");

// refine_path (utilities/path_tools.py:178-240, angle_delta None) of the 4 way points: a segment longer than delta
// becomes int(d / delta) + 2 np.linspace points (k * step + start, the end point dropped) with the angle of its
// start; the last way point closes the path.
struct RefinedShape {
  int count[3];   // points segment i contributes
  int n;          // total, including the closing point
};

__device__ __forceinline__ RefinedShape refined_shape(const double way[4][3], double delta) {
  RefinedShape s;
  s.n = 1;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double dx = way[i + 1][0] - way[i][0], dy = way[i + 1][1] - way[i][1];
    const double d = sqrt(dx * dx + dy * dy);                 // np.linalg.norm(axis=1)
    s.count[i] = d > delta ? (int)(d / delta) + 1 : 1;       // (int(d / delta) + 2 points)[:-1]
    s.n += s.count[i];
  }
  return s;
}

__device__ __forceinline__ void refined_point(const double way[4][3], const RefinedShape& s, int idx, double& x, double& y,
                                              double& th) {
  int i = 0, k = idx;
  while (i < 3 && k >= s.count[i]) {
    k -= s.count[i];
    ++i;
  }
  if (i == 3) {
    x = way[3][0]; y = way[3][1]; th = way[3][2];
    return;
  }
  th = way[i][2];
  if (s.count[i] == 1) {
    x = way[i][0]; y = way[i][1];
    return;
  }
  const double div = (double)s.count[i];                      // num - 1
  const double sx = (way[i + 1][0] - way[i][0]) / div, sy = (way[i + 1][1] - way[i][1]) / div;
  x = (double)k * sx + way[i][0];
  y = (double)k * sy + way[i][1];
}

// ---- RandomMiniEnv (envs/mini_env.py) -------------------------------------------------------------------------------

// cv::clipLine(Size(w, h), pt1, pt2) (OpenCV imgproc drawing.cpp): the part of the segment inside the image, computed in
// integers with truncation exactly like cv2.line does before it walks the pixels; false when nothing is inside
__device__ __forceinline__ bool clip_line(int w, int h, long long& x1, long long& y1, long long& x2, long long& y2) {
  const long long right = w - 1, bottom = h - 1;
  if (w <= 0 || h <= 0) return false;
  int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
  int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
  if ((c1 & c2) == 0 && (c1 | c2) != 0) {
    long long a;
    if (c1 & 12) {
      a = c1 < 8 ? 0 : bottom;
      x1 += (long long)((double)(a - y1) * (double)(x2 - x1) / (double)(y2 - y1));
      y1 = a;
      c1 = (x1 < 0) + (x1 > right) * 2;
    }
    if (c2 & 12) {
      a = c2 < 8 ? 0 : bottom;
      x2 += (long long)((double)(a - y2) * (double)(x2 - x1) / (double)(y2 - y1));
      y2 = a;
      c2 = (x2 < 0) + (x2 > right) * 2;
    }
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
      if (c1) {
        a = c1 == 1 ? 0 : right;
        y1 += (long long)((double)(a - x1) * (double)(y2 - y1) / (double)(x2 - x1));
        x1 = a;
        c1 = 0;
      }
      if (c2) {
        a = c2 == 1 ? 0 : right;
        y2 += (long long)((double)(a - x2) * (double)(y2 - y1) / (double)(x2 - x1));
        x2 = a;
        c2 = 0;
      }
    }
  }
  return (c1 | c2) == 0;
}

// cv2.line with end points anywhere: clip, then walk (the walker swaps to left-to-right itself)
__device__ __forceinline__ void draw_wall_clipped(const MapLayout& m, int width, int height, int x0, int y0, int x1, int y1,
                                                  uint8_t value, int first, int stride) {
  long long a0 = x0, b0 = y0, a1 = x1, b1 = y1;
  if (!clip_line(width, height, a0, b0, a1, b1)) return;
  draw_wall(m, (int)a0, (int)b0, (int)a1, (int)b1, value, first, stride);
}

// the k-th uniform of (seed; env, draw): as philox_uniform, in a stream of its own ('MINI')
struct MiniRng {
  uint64_t seed, env, draw;
  uint32_t k;
  __device__ __forceinline__ double u01() {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)draw, 0x4d494e49u + (k >> 1), (uint32_t)(draw >> 32)),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint64_t bits = (k & 1) ? (((uint64_t)r.z << 21) | (r.w >> 11)) : (((uint64_t)r.x << 21) | (r.y >> 11));
    ++k;
    return (double)bits * 0x1.0p-53;
  }
  __device__ __forceinline__ double uniform(double a, double b) { return a + (b - a) * u01(); }
};

// not_inside_obstacle (envs/mini_env.py:198-208): the bearing of the point seen from the corner is outside the wedge
__device__ __forceinline__ bool mini_outside_obstacle(double x, double y, double ox, double oy, double start_angle, double angle) {
  const double phi = wrap_angle(atan2(y - oy, x - ox));
  if (phi >= start_angle && phi <= start_angle + angle) return false;
  if (phi + BCG_TWO_PI >= start_angle && phi + BCG_TWO_PI <= start_angle + angle) return false;
  return true;
}

// _sample_mini_env_params_no_final_check (envs/mini_env.py:269-320), same draw order.  Returns 1 = drawn, 0 = the
// circle method ran out of tries (SpaceSeemsEmptyError: the caller draws again), -1 = the square method did (ValueError)
__device__ __noinline__ int draw_mini_params(MiniRng& rng, const BcgMiniGenParams& g, BcgMiniParams& out) {
  const double ox = rng.uniform(-g.inner_w / 2, g.inner_w / 2), oy = rng.uniform(-g.inner_h / 2, g.inner_h / 2);
  const double start_angle = rng.uniform(0, BCG_TWO_PI);
  const double angle = rng.uniform(g.min_obstacle_angle, g.max_obstacle_angle);
  const double r = 3 * (g.inner_h + g.inner_w + g.mid_margin + g.out_margin);
  double sn, cs;
  sincos(start_angle, &sn, &cs);
  out.a[0] = r * cs + ox;
  out.a[1] = r * sn + oy;
  sincos(start_angle + angle, &sn, &cs);
  out.b[0] = r * cs + ox;
  out.b[1] = r * sn + oy;
  out.o[0] = ox;
  out.o[1] = oy;
  out.h = g.inner_h + 2 * g.mid_margin + 2 * g.out_margin;
  out.w = g.inner_w + 2 * g.mid_margin + 2 * g.out_margin;
  double sx = 0, sy = 0, ex = 0, ey = 0, theta = 0;
  if (rng.u01() < 0.7) {
    // circle method (:141-178): two opposite points of a circle, heading along the chord
    bool found = false;
    for (int t = 0; t < 1000 && !found; ++t) {
      const double rc = fmin((g.inner_w + g.inner_h) / 4. + g.mid_margin, g.lim_euc_dist);
      const double phi = rng.uniform(0, BCG_TWO_PI);
      sincos(phi, &sn, &cs);
      const double x = rc * cs, y = rc * sn;
      rng.uniform(0, BCG_TWO_PI);                                    // a heading the reference draws and discards
      if (mini_outside_obstacle(x, y, ox, oy, start_angle, angle) && mini_outside_obstacle(-x, -y, ox, oy, start_angle, angle)) {
        sx = x; sy = y; ex = -x; ey = -y;
        theta = wrap_angle(atan2(-y - y, -x - x));
        found = true;
      }
    }
    if (!found) return 0;
  } else {
    // square method (:181-240): two poses of the middle square, the second not too far in heading / distance
    const double lx = g.inner_w / 2 + g.mid_margin, ly = g.inner_h / 2 + g.mid_margin;
    double st = 0;
    bool found = false;
    for (int t = 0; t < 1000 && !found; ++t) {
      const double x = rng.uniform(-lx, lx), y = rng.uniform(-ly, ly);
      const double th = wrap_angle(rng.uniform(0, BCG_TWO_PI));
      if (mini_outside_obstacle(x, y, ox, oy, start_angle, angle)) {
        sx = x; sy = y; st = th;
        found = true;
      }
    }
    if (!found) return -1;
    found = false;
    for (int t = 0; t < 1000 && !found; ++t) {
      const double x = rng.uniform(-lx, lx), y = rng.uniform(-ly, ly);
      const double th = wrap_angle(rng.uniform(0, BCG_TWO_PI));
      if (mini_outside_obstacle(x, y, ox, oy, start_angle, angle) && py_mod(st - th, BCG_TWO_PI) < g.lim_ang_dist &&
          sqrt((sx - x) * (sx - x) + (sy - y) * (sy - y)) < g.lim_euc_dist) {
        ex = x; ey = y;
        found = true;
      }
    }
    if (!found) return -1;
    theta = wrap_angle(atan2(ey - sy, ex - sx));
  }
  const double n1 = rng.uniform(-g.angular_pose_noise_scale / 2.0, g.angular_pose_noise_scale / 2.0);
  out.start[0] = sx; out.start[1] = sy; out.start[2] = wrap_angle(theta + n1);
  const double n2 = rng.uniform(-g.angular_pose_noise_scale / 2.0, g.angular_pose_noise_scale / 2.0);
  out.end[0] = ex; out.end[1] = ey; out.end[2] = wrap_angle(theta + n2);
  return 1;
}

}  // namespace bcg
