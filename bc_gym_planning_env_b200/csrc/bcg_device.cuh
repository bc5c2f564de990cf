// Device-side building blocks of the batched PlanEnv.step path (sm_100a).
// Compiled with --fmad=false: every fp64 expression rounds operation by operation like the NumPy
// reference; the few places where the reference's BLAS route fuses (np.dot in
// utilities/path_tools.py:145) call fma() explicitly.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bcg_b200.h"

#define BCG_PI 3.141592653589793
#define BCG_TWO_PI 6.283185307179586
#define BCG_FULL 0xffffffffu

namespace bcg {

// ---- scalar helpers -------------------------------------------------------------------------
// Python/NumPy floor-mod for doubles (npy_divmod): result carries the divisor's sign.
__device__ __forceinline__ double py_mod(double a, double b) {
  double m = fmod(a, b);
  if (m != 0.0) {
    if ((b < 0.0) != (m < 0.0)) m += b;
  } else {
    m = copysign(0.0, b);
  }
  return m;
}

// normalize_angle, utilities/coordinate_transformations.py:28-36.  For |z + pi| < 4 pi the floor-mod is
// spelled out: a - 2 pi is exact there (Sterbenz), and a + 2 pi is the very addition NumPy's divmod
// performs after its (exact) fmod, so the result is bit-identical to py_mod without the fmod loop.
__device__ __forceinline__ double wrap_angle(double z) {
  const double a = z + BCG_PI;
  double m;
  if (a >= 0.0 && a < BCG_TWO_PI) m = a;
  else if (a >= BCG_TWO_PI && a < 2 * BCG_TWO_PI) m = a - BCG_TWO_PI;
  else if (a < 0.0 && a >= -BCG_TWO_PI) m = a + BCG_TWO_PI;
  else m = py_mod(a, BCG_TWO_PI);
  return m - BCG_PI;
}

// one axis of world_to_pixel, utilities/coordinate_transformations.py:185-205 (np.round = half-even)
__device__ __forceinline__ int world_to_pixel_1d(double w, double origin, double inv_res) {
  double r = rint((w - origin) * inv_res);
  r = fmin(fmax(r, -1073741824.0), 1073741824.0);  // keep later int arithmetic overflow-free
  return (int)r;
}

__device__ __forceinline__ double clampd(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// ---- Philox4x32-10 + Box-Muller (oracle/plan_env_oracle.py:philox_normals is the CPU twin) ------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// counter = (env id, step index low, block, step index high), key = seed
__device__ __forceinline__ void philox_normals(uint64_t seed, uint64_t env, uint64_t step, uint32_t block,
                                               double& z0, double& z1) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)step, block, (uint32_t)(step >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const uint64_t a = ((uint64_t)r.x << 21) | (r.y >> 11);
  const uint64_t b = ((uint64_t)r.z << 21) | (r.w >> 11);
  const double u1 = (double)(a + 1) * 0x1.0p-53;  // (0, 1]
  const double u2 = (double)b * 0x1.0p-53;        // [0, 1)
  const double rad = sqrt(-2.0 * log(u1));
  double sn, cs;
  sincos(BCG_TWO_PI * u2, &sn, &cs);
  z0 = rad * cs;
  z1 = rad * sn;
}

// ---- kinematics --------------------------------------------------------------------------------
// kinematic_body_pose_motion_step, robot_models/differential_drive.py:21-40
__device__ __forceinline__ void pose_motion_step(double& x, double& y, double& th, double v, double w, double dt) {
  const double h = 0.5 * w * dt;
  const double xs = h / BCG_PI;                       // np.sinc(h / pi)
  const double ys = BCG_PI * (xs == 0.0 ? 1.0e-20 : xs);
  const double f = v * dt * (sin(ys) / ys);
  double sn, cs;
  sincos(th + h, &sn, &cs);
  x = x + f * cs;
  y = y + f * sn;
  th = wrap_angle(th + w * dt);
}

// kinematic_body_pose_motion_step_with_noise, robot_models/differential_drive.py:43-74.
// Normal slots: block 0 = (angular, final rotation), block 1 first half = linear.
// the normals of Philox block 0 (angular velocity, final rotation), drawn ahead of their use: they depend on nothing but
// (seed, env, step), so a caller can take them off the dependent chain of the kinematics
struct NoiseDraws {
  bool have0;
  double n_w, n_g;
};
__device__ __forceinline__ NoiseDraws draw_noise_ahead(const BcgParams& p, uint64_t env, uint64_t step) {
  NoiseDraws nd;
  nd.have0 = false;
  nd.n_w = nd.n_g = 0.0;
  if (p.noise_on && (p.alpha[2] > 0.0 || p.alpha[3] > 0.0 || p.alpha[4] > 0.0 || p.alpha[5] > 0.0)) {
    philox_normals(p.seed, env, step, 0u, nd.n_w, nd.n_g);
    nd.have0 = true;
  }
  return nd;
}

__device__ __forceinline__ void noisy_pose_motion_step(double& x, double& y, double& th, double v, double w,
                                                       const BcgParams& p, uint64_t env, uint64_t step,
                                                       NoiseDraws nd = NoiseDraws{false, 0.0, 0.0}) {
  double n_w = nd.n_w, n_g = nd.n_g;
  bool have0 = nd.have0;
  double var = p.alpha[0] * (v * v) + p.alpha[1] * (w * w);
  if (var > 0.0) {
    double n_v, unused;
    philox_normals(p.seed, env, step, 1u, n_v, unused);
    v = v + sqrt(var) * n_v;
  }
  var = p.alpha[2] * (v * v) + p.alpha[3] * (w * w);
  if (var > 0.0) {
    if (!have0) philox_normals(p.seed, env, step, 0u, n_w, n_g);
    have0 = true;
    w = w + sqrt(var) * n_w;
  }
  var = p.alpha[4] * (v * v) + p.alpha[5] * (w * w);
  double gamma = 0.0;
  if (var > 0.0) {
    if (!have0) philox_normals(p.seed, env, step, 0u, n_w, n_g);
    gamma = sqrt(var) * n_g;
  }
  pose_motion_step(x, y, th, v, w, p.dt);
  th = wrap_angle(th + gamma * p.dt);
}

// path_velocity on the two-row path the robots build, utilities/path_tools.py:298-323
__device__ __forceinline__ void measured_velocity(double x0, double y0, double th0, double x1, double y1,
                                                  double th1, double dt, double& v, double& w) {
  const double dx = x1 - x0, dy = y1 - y0;
  double sn, cs;
  sincos(th0, &sn, &cs);
  const double proj = cs * dx + sn * dy;
  double sign = (proj > 0.0) ? 1.0 : ((proj < 0.0) ? -1.0 : 0.0);
  if (sign == 0.0) {
    const double alt = sn * dy;
    sign = (alt > 0.0) ? 1.0 : ((alt < 0.0) ? -1.0 : 0.0);
  }
  const double ds = sqrt(dx * dx + dy * dy) * sign;
  double dth = th1 - th0;
  if (dth < -BCG_PI) dth += BCG_TWO_PI;
  if (dth > BCG_PI) dth -= BCG_TWO_PI;
  v = ds / dt;
  w = dth / dt;
}

// TricycleRobot.step (robot_models/tricycle_model.py:478-538) / DiffDriveRobot.step
// (robot_models/differential_drive.py:236-265).  s[7] = x,y,th,v,w,steer_cmd,wheel, updated in place.
__device__ __forceinline__ void robot_step(double s[7], double u0, double u1, const BcgParams& p, uint64_t env,
                                           uint64_t step, NoiseDraws nd = NoiseDraws{false, 0.0, 0.0}) {
  const double x0 = s[0], y0 = s[1], th0 = s[2];
  double v_new, w_new;
  if (p.robot_kind == BCG_ROBOT_TRICYCLE) {
    const double wheel = s[6];
    // tricycle_front_wheel_column_step :127-154
    double delta = p.p_gain * (u1 - wheel);
    delta = clampd(delta, -p.max_wheel_delta, p.max_wheel_delta);
    const double new_wheel = clampd(wheel + delta, -p.max_wheel_angle, p.max_wheel_angle);
    // tricycle_velocity_dynamic_model_step :157-188
    double sn, cs;
    sincos(new_wheel, &sn, &cs);
    const double v_des = u0 * cs;
    const double w_des = u0 * sn / p.wheel_base;
    const double a_lin = clampd((v_des - s[3]) / p.dt, -2.0 * p.max_lin_acc, p.max_lin_acc);
    const double a_ang = clampd((w_des - s[4]) / p.dt, -p.max_ang_acc, p.max_ang_acc);
    v_new = s[3] + a_lin * p.dt;
    w_new = s[4] + a_ang * p.dt;
    if (0.0 > v_new) v_new = 0.0;
    s[5] = wheel - u1;  // :532
    s[6] = new_wheel;
  } else {
    v_new = u0;
    w_new = u1;
  }
  double x = x0, y = y0, th = th0;
  if (p.noise_on)
    noisy_pose_motion_step(x, y, th, v_new, w_new, p, env, step, nd);
  else
    pose_motion_step(x, y, th, v_new, w_new, p.dt);
  measured_velocity(x0, y0, th0, x, y, th, p.dt, s[3], s[4]);
  s[0] = x;
  s[1] = y;
  s[2] = th;
}

// _get_element_from_list_with_delay, envs/base/env.py:27-49, as a circular buffer of `d` slots.
// q = head | len << 16.  ring rows are laid out slot-major: row(slot, comp) = slot * ncomp + comp.
template <int NCOMP>
__device__ __forceinline__ void delay_line(double* ring, int64_t stride, int& q, int d, double v[NCOMP]) {
  if (d <= 0) return;
  int head = q & 0xffff, len = q >> 16;
  if (len < d) {
    int slot = head + len;
    if (slot >= d) slot -= d;
    double front[NCOMP];
    if (len > 0) {
#pragma unroll
      for (int c = 0; c < NCOMP; ++c) front[c] = ring[(int64_t)(head * NCOMP + c) * stride];
    }
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) ring[(int64_t)(slot * NCOMP + c) * stride] = v[c];
    if (len > 0) {
#pragma unroll
      for (int c = 0; c < NCOMP; ++c) v[c] = front[c];
    }
    ++len;
  } else {
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) {
      double* slotp = ring + (int64_t)(head * NCOMP + c) * stride;
      const double out = *slotp;
      *slotp = v[c];
      v[c] = out;
    }
    head = (head + 1 == d) ? 0 : head + 1;
  }
  q = head | (len << 16);
}

// delay_line in two halves, so that the loads can be issued at the top of a kernel (they depend on the queue word alone)
// and the stores where the new element is known: delay_front reads the element delay_push will hand back.
template <int NCOMP>
__device__ __forceinline__ void delay_front(const double* ring, int64_t stride, int q, int d, double front[NCOMP]) {
  if (d <= 0) return;
  const int head = q & 0xffff, len = q >> 16;
  if (len == 0) return;                     // warm-up with an empty queue: the element itself comes back
#pragma unroll
  for (int c = 0; c < NCOMP; ++c) front[c] = ring[(int64_t)(head * NCOMP + c) * stride];
}
template <int NCOMP>
__device__ __forceinline__ void delay_push(double* ring, int64_t stride, int& q, int d, double v[NCOMP], const double front[NCOMP]) {
  if (d <= 0) return;
  int head = q & 0xffff, len = q >> 16;
  int slot = head;
  if (len < d) {
    slot = head + len;
    if (slot >= d) slot -= d;
  }
#pragma unroll
  for (int c = 0; c < NCOMP; ++c) ring[(int64_t)(slot * NCOMP + c) * stride] = v[c];
  if (len > 0) {
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) v[c] = front[c];
  }
  if (len < d) ++len;
  else head = (head + 1 == d) ? 0 : head + 1;
  q = head | (len << 16);
}

// What delay_line would hand back for `v`, without touching the ring
template <int NCOMP>
__device__ __forceinline__ void delay_peek(const double* ring, int64_t stride, int q, int d, double v[NCOMP]) {
  if (d <= 0) return;
  const int head = q & 0xffff, len = q >> 16;
  if (len == 0) return;                     // warm-up with an empty queue: the element itself comes back
#pragma unroll
  for (int c = 0; c < NCOMP; ++c) v[c] = ring[(int64_t)(head * NCOMP + c) * stride];
}

// ---- per-env parameters (BcgEnvRows) ---------------------------------------------------------------------------------
// The batch-wide params with env e's own values of the per-env fields in place, so that every device function keeps
// reading one BcgParams.  The delays of `p` are the ring capacities: a row delay is clamped to [0, capacity], so what a
// kernel touches never depends on the row contents.
__device__ __forceinline__ BcgParams with_env_rows(const BcgParams& p, const BcgEnvRows& r, int64_t N, int e) {
  BcgParams q = p;
  const double* f = r.f + e;
  const int32_t* i = r.i + e;
  q.spatial_precision = __ldg(f + BCG_EP_F_SP * N);
  q.angular_precision = __ldg(f + BCG_EP_F_AP * N);
  q.progress_multiplier = __ldg(f + BCG_EP_F_PM * N);
#pragma unroll
  for (int k = 0; k < 6; ++k) q.alpha[k] = __ldg(f + (BCG_EP_F_ALPHA + k) * N);
  q.delay_control = min(max(__ldg(i + BCG_EP_I_DELAY_CONTROL * N), 0), p.delay_control);
  q.delay_pose = min(max(__ldg(i + BCG_EP_I_DELAY_POSE * N), 0), p.delay_pose);
  q.delay_state = min(max(__ldg(i + BCG_EP_I_DELAY_STATE * N), 0), p.delay_state);
  q.iteration_timeout = __ldg(i + BCG_EP_I_TIMEOUT * N);
  q.noise_on = __ldg(i + BCG_EP_I_NOISE_ON * N);
  return q;
}

// ---- footprint table lookup ----------------------------------------------------------------------
// Work records: what the warp-per-env kernels need to know about one env, resolved by the thread-per-env
// kernels (kinematics / pose-prep) and stored array-of-structures so that a warp gets everything with one
// round of 16-byte loads instead of chasing map_id -> map descriptor -> tile address through memory.
struct __align__(16) WorkCollide {   // 48 bytes
  int64_t tile_off;                  // lethal tile plane of the env's map (uint32 offset in the tile arena)
  int64_t data_off;                  // uint8 cells of the env's map (byte offset in the map arena)
  int32_t tiles_x, map_pitch;
  int32_t X0, Y0;                    // map pixel of the footprint mask's top-left corner
  int16_t nrows, fwidth;             // mask bounding box
  int16_t map_w, map_h;
  int32_t bin;                       // footprint angle bin
  int32_t sum_off;                   // tile summary of the env's map (BcgMapDesc.sum_off)
};
static_assert(sizeof(WorkCollide) == 48, "WorkCollide is 48 bytes");

#define BCG_WORK_BYTES 192           // per-env scratch slot: WorkCollide (stand-alone collision) or the step's StepRecord at +0

__device__ __forceinline__ const WorkCollide* work_collide(const void* work, int e) {
  return reinterpret_cast<const WorkCollide*>(reinterpret_cast<const uint8_t*>(work) + (int64_t)e * BCG_WORK_BYTES);
}
// Per-thread.  Picks the angle bin whose stored rounded-vertex tuple equals
// round_half_even(R(th) * footprint / res) (utilities/path_tools.py:140-150), i.e. the bin whose
// cv2.fillPoly mask the reference would have rasterised for this exact angle.  A uniform bucket table
// gives the first candidate; the analytic bin edges are only good to ~1e-15 rad, so the tuple is
// verified and neighbours are probed on a miss.
__device__ __forceinline__ int find_foot_bin(const BcgFootprintLut& lut, double th, uint32_t* status) {
  double sn, cs;
  sincos(th, &sn, &cs);
  double t = th;
  if (!(t >= -BCG_PI && t < BCG_PI)) t = wrap_angle(t);
  int bk = (int)((t + BCG_PI) * lut.bucket_scale);
  bk = min(max(bk, 0), lut.n_buckets - 1);
  int k = __ldg(lut.bucket_first + bk);
  while (k + 1 < lut.n_bins && t >= __ldg(lut.edges + k + 1)) ++k;
  while (k > 0 && t < __ldg(lut.edges + k)) --k;
  for (int probe = 0; probe < 9; ++probe) {
    int kk = k + ((probe & 1) ? ((probe + 1) >> 1) : -(probe >> 1));
    if (kk < 0) kk += lut.n_bins;
    if (kk >= lut.n_bins) kk -= lut.n_bins;
    const int16_t* v = lut.verts + (int64_t)kk * 2 * lut.n_verts;
    bool ok = true;
    if ((lut.n_verts & 3) == 0) {
      // four vertices per 16-byte load (a tuple row is n_verts * 4 bytes, rows of a table with n_verts % 4 == 0 are
      // 16-byte aligned): per-lane bins make every load a separate line, so the tuple is fetched in as few loads as possible
      const uint4* v4 = reinterpret_cast<const uint4*>(v);
      for (int i4 = 0; i4 < lut.n_verts / 4 && ok; ++i4) {
        const uint4 q = __ldg(v4 + i4);
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int i = 4 * i4 + j;
          const double fx = __ldg(lut.fp_pix + 2 * i), fy = __ldg(lut.fp_pix + 2 * i + 1);
          const int vx = (int)rint(fma(fy, -sn, fx * cs));   // np.dot's fused form, see oracle
          const int vy = (int)rint(fma(fy, cs, fx * sn));
          ok = ok && ((int)(int16_t)(w[j] & 0xffffu) == vx) && ((int)(int16_t)(w[j] >> 16) == vy);
        }
      }
    } else {
      for (int i = 0; i < lut.n_verts && ok; ++i) {
        const double fx = __ldg(lut.fp_pix + 2 * i), fy = __ldg(lut.fp_pix + 2 * i + 1);
        const int vx = (int)rint(fma(fy, -sn, fx * cs));   // np.dot's fused form, see oracle
        const int vy = (int)rint(fma(fy, cs, fx * sn));
        ok = (v[2 * i] == vx) && (v[2 * i + 1] == vy);
      }
    }
    if (ok) return kk;
  }
  atomicAdd(status + BCG_STATUS_LUT_MISS, 1u);
  return k;
}

// find_foot_bin + the bin's header in two memory round trips instead of five (bucket -> edges -> edges -> tuple -> header):
// the bucket's first bin and its successor are fetched together from the combined table (`bins`: tuple + header per
// 16-byte aligned row), the rounded vertex tuple of the angle is worked out once and compared with both.  An angle that
// is in neither (two bin edges inside one of the 16 384 buckets, or a pose on an edge) takes the probing path above.
__device__ __forceinline__ int find_foot_bin_header(const BcgFootprintLut& lut, double th, uint32_t* status, short4& header) {
  if (lut.bins != nullptr && lut.n_verts == 16) {
    double sn, cs;
    sincos(th, &sn, &cs);
    double t = th;
    if (!(t >= -BCG_PI && t < BCG_PI)) t = wrap_angle(t);
    int bk = (int)((t + BCG_PI) * lut.bucket_scale);
    bk = min(max(bk, 0), lut.n_buckets - 1);
    const int k0 = __ldg(lut.bucket_first + bk);
    const int k1 = (k0 + 1 == lut.n_bins) ? 0 : k0 + 1;
    const uint4* r0 = reinterpret_cast<const uint4*>(lut.bins + (int64_t)k0 * lut.bin_stride);
    const uint4* r1 = reinterpret_cast<const uint4*>(lut.bins + (int64_t)k1 * lut.bin_stride);
    uint4 q0[5], q1[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      q0[i] = __ldg(r0 + i);
      q1[i] = __ldg(r1 + i);
    }
    bool ok0 = true, ok1 = true;
#pragma unroll
    for (int i4 = 0; i4 < 4; ++i4) {
      const uint32_t a[4] = {q0[i4].x, q0[i4].y, q0[i4].z, q0[i4].w}, c[4] = {q1[i4].x, q1[i4].y, q1[i4].z, q1[i4].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = 4 * i4 + j;
        const double fx = __ldg(lut.fp_pix + 2 * i), fy = __ldg(lut.fp_pix + 2 * i + 1);
        const int vx = (int)rint(fma(fy, -sn, fx * cs));   // np.dot's fused form, see oracle
        const int vy = (int)rint(fma(fy, cs, fx * sn));
        const uint32_t want = ((uint32_t)vx & 0xffffu) | ((uint32_t)vy << 16);
        const bool fits = vx >= -32768 && vx < 32768 && vy >= -32768 && vy < 32768;
        ok0 = ok0 && fits && a[j] == want;
        ok1 = ok1 && fits && c[j] == want;
      }
    }
    if (ok0 || ok1) {
      const uint4 h = ok0 ? q0[4] : q1[4];
      header = make_short4((short)(h.x & 0xffffu), (short)(h.x >> 16), (short)(h.y & 0xffffu), (short)(h.y >> 16));
      return ok0 ? k0 : k1;
    }
  }
  const int bin = find_foot_bin(lut, th, status);
  header = __ldg(reinterpret_cast<const short4*>(lut.header) + bin);
  return bin;
}

// The footprint mask of pose (x, y, th) placed on a map: its angle bin and its box in map pixels.
struct FootBox {
  int X0, Y0;          // map pixel of the mask's top-left corner
  int nrows, fwidth;   // mask bounding box
  int bin;
};

__device__ __forceinline__ FootBox foot_box(const BcgFootprintLut& lut, double origin_x, double origin_y, double inv_res,
                                            double x, double y, double th, uint32_t* status) {
  FootBox f;
  short4 h;                                              // xmin, ymin, nrows, width
  f.bin = find_foot_bin_header(lut, th, status, h);
  f.X0 = world_to_pixel_1d(x, origin_x, inv_res) + h.x;
  f.Y0 = world_to_pixel_1d(y, origin_y, inv_res) + h.y;
  f.nrows = h.z;
  f.fwidth = h.w;
  return f;
}

__device__ __forceinline__ WorkCollide make_work_collide(const BcgParams& p, const BcgBatch& b, int map_id, double x, double y,
                                                         double th) {
  const BcgMapDesc m = b.maps[map_id];
  const FootBox f = foot_box(b.lut, m.origin_x, m.origin_y, p.inv_resolution, x, y, th, b.status);
  WorkCollide w;
  w.bin = f.bin;
  w.X0 = f.X0;
  w.Y0 = f.Y0;
  w.nrows = (int16_t)f.nrows;
  w.fwidth = (int16_t)f.fwidth;
  w.tile_off = m.tile_off;
  w.data_off = m.data_off;
  w.tiles_x = m.tiles_x;
  w.map_pitch = m.pitch;
  w.map_w = (int16_t)m.width;
  w.map_h = (int16_t)m.height;
  w.sum_off = m.sum_off;
  return w;
}

// 32 mask bits starting at bit `rel` of a multi-word row mask (bit b <-> column xmin + b)
__device__ __forceinline__ uint32_t mask_bits32(const uint64_t* row, int wpr, int rel) {
  if (rel <= -32 || rel >= wpr * 64) return 0u;
  if (rel < 0) return (uint32_t)(__ldg(row) << (-rel));
  const int j = rel >> 6, off = rel & 63;
  uint64_t lo = __ldg(row + j) >> off;
  if (off > 32 && j + 1 < wpr) lo |= __ldg(row + j + 1) << (64 - off);
  return (uint32_t)lo;
}

// bits [rel, rel + 32) of a 64-bit row mask (bit b <-> column xmin + b), rel in (-32, 64)
__device__ __forceinline__ uint32_t mask_window32(uint64_t mk, int rel) {
  return rel < 0 ? (uint32_t)(mk << (-rel)) : (uint32_t)(mk >> rel);
}

// pose_collides (envs/base/env.py:464-489) on the lethal tile plane.  Warp-cooperative: a lane owns one
// footprint row (two passes cover the <= 64 rows), loads the row's mask once and walks the <= 3 tiles
// the row crosses; 16 consecutive rows of a tile are one coalesced 64-byte read.  Returns the
// warp-uniform verdict.  If COUNT, *pixels gets the number of in-map footprint pixels.
// COHERENT: read the tile words around L1 (ld.global.cg) -- for callers that changed the plane earlier in the SAME
// kernel (the mini-env generator); everyone else reads through the non-coherent path.
template <bool COUNT, bool COHERENT = false>
__device__ __forceinline__ bool collide_tiles(const BcgBatch& b, const WorkCollide& f, unsigned lane, int* pixels) {
  const int X0 = f.X0, Y0 = f.Y0;
  const int X1 = X0 + f.fwidth - 1;
  const int map_w = f.map_w, map_h = f.map_h;
  unsigned hit = 0;
  int cnt = 0;
  if (!(X1 < 0 || X0 >= map_w)) {
    const int tx0 = max(X0, 0) >> 5, tx1 = min(X1, map_w - 1) >> 5;
    const uint32_t* tiles = b.tile_arena + f.tile_off;
    const int wpr = b.lut.wpr;
    const uint64_t* rows = b.lut.rows + (int64_t)f.bin * b.lut.max_rows * wpr;
    for (int dy = lane; dy < f.nrows; dy += 32) {
      const int Y = Y0 + dy;
      if (Y < 0 || Y >= map_h) continue;
      const uint32_t* trow = tiles + (((int64_t)(Y >> 4) * f.tiles_x) << 4) + (Y & 15);
      const uint64_t* mrow = rows + (int64_t)dy * wpr;
      const uint64_t mk = __ldg(mrow);
      for (int tx = tx0; tx <= tx1; ++tx) {
        const uint32_t word = COHERENT ? __ldcg(trow + (tx << 4)) : __ldg(trow + (tx << 4));
        const int rel = (tx << 5) - X0;
        const uint32_t mbits = (wpr == 1) ? mask_window32(mk, rel) : mask_bits32(mrow, wpr, rel);
        hit |= word & mbits;
        if (COUNT) {
          const int over = (tx << 5) + 32 - map_w;  // columns of this tile beyond the map
          const uint32_t valid = over > 0 ? (0xffffffffu >> over) : 0xffffffffu;
          cnt += __popc(mbits & valid);
        }
      }
    }
  }
  if (COUNT) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(BCG_FULL, cnt, o);
    *pixels = cnt;
  }
  return __any_sync(BCG_FULL, hit != 0u);
}

// pose_collides (envs/base/env.py:464-489) by ONE thread per env (collide_warp_balanced, collide_thread_listed,
// collide_thread), for the thread-per-env kinematics + collision kernels.  The footprint box spans a few bands of 16 rows x
// a few tiles of 32 columns.  A thread-serial gather pays a full memory round trip per dependent load, so the loads are
// batched: (1) the tile-summary words of up to BCG_BANDS bands (`sum`:
// 1 bit per tile of the occupancy plane, a superset of the lethal plane), one round trip; (2) per non-empty tile under the
// footprint -- a corridor is mostly free space: typically 0..3 of the 15 -- its four 16-byte quarters and the 16
// footprint-mask rows of its band, one round trip; early exit on the first hit.  Same verdict as collide_tiles.
constexpr int BCG_BANDS = 6;                             // bands per batch of summary words (a 64-row mask spans <= 5)

// tm[k] = the non-empty-tile bits of band tyb + k over the tile columns tx0 .. tx1 (bit j <-> column tx0 + j), from one or
// two summary words; 0 for the bands past ty1
__device__ __forceinline__ void summary_bands(const uint32_t* __restrict__ sum, int tiles_x, int tyb, int ty1, int tx0, int tx1,
                                              uint32_t (&tm)[BCG_BANDS]) {
  const int sw = (tiles_x + 31) >> 5;
  const uint32_t colmask = (2u << (tx1 - tx0)) - 1u;
#pragma unroll
  for (int k = 0; k < BCG_BANDS; ++k) {
    tm[k] = 0u;
    if (tyb + k <= ty1) {
      const uint32_t* srow = sum + (tyb + k) * sw;
      const int w0 = tx0 >> 5;
      uint64_t two = __ldg(srow + w0);
      if ((tx1 >> 5) != w0) two |= (uint64_t)__ldg(srow + w0 + 1) << 32;
      tm[k] = (uint32_t)(two >> (tx0 & 31)) & colmask;
    }
  }
}

// The 16 mask rows of the band whose first tile row is mask row dy0, for one-word rows whose bins start 16-byte aligned:
// nine aligned 16-byte pairs from the even row at or below dy0 (rows beyond the mask are zero in the table; pairs outside
// the bin's max_rows rows are not loaded).
__device__ __forceinline__ void load_band_rows(const uint64_t* __restrict__ rows, int max_rows, int dy0, uint64_t (&v)[18]) {
  const int base = dy0 & ~1;
#pragma unroll
  for (int jj = 0; jj < 9; ++jj) {
    const int r0 = base + 2 * jj;
    ulonglong2 q = make_ulonglong2(0ull, 0ull);
    if ((unsigned)r0 < (unsigned)max_rows) q = __ldg(reinterpret_cast<const ulonglong2*>(rows + r0));
    v[2 * jj] = q.x;
    v[2 * jj + 1] = q.y;
  }
}

// the 16 rows of the tile at `tile` (bit j of a row <-> its column j), as four 16-byte loads
__device__ __forceinline__ void load_tile(const uint32_t* __restrict__ tile, uint32_t (&ws)[16]) {
  const uint4* tq = reinterpret_cast<const uint4*>(tile);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint4 w = __ldg(tq + q);
    ws[4 * q] = w.x;
    ws[4 * q + 1] = w.y;
    ws[4 * q + 2] = w.z;
    ws[4 * q + 3] = w.w;
  }
}

// whether a tile's 16 rows ws meet the band's mask rows v (load_band_rows with the same dy0); rel = the tile's first
// column - X0.  (The callers load the tile before the rows: both are then in flight together.)
__device__ __forceinline__ bool tile_meets_rows(const uint32_t (&ws)[16], const uint64_t (&v)[18], int dy0, int rel) {
  const int odd = dy0 & 1;
  uint32_t hit = 0u;
#pragma unroll
  for (int r = 0; r < 16; ++r) hit |= ws[r] & mask_window32(odd ? v[r + 1] : v[r], rel);
  return hit != 0u;
}

// The boxes collide_warp_balanced does not take (multi-word mask rows, > 4 tile columns, > 6 bands, rows not in aligned
// pairs): per batch of BCG_BANDS bands the summary words, then the non-empty tiles band by band, each row's 32 mask bits
// by mask_bits32, which is exact for any number of words per row.
__device__ __forceinline__ bool collide_thread(const BcgFootprintLut& lut, const uint32_t* __restrict__ tiles,
                                               const uint32_t* __restrict__ sum, int tiles_x, int map_w, int map_h,
                                               const FootBox& f) {
  const int X0 = f.X0, Y0 = f.Y0;
  const int X1 = X0 + f.fwidth - 1, Y1 = Y0 + f.nrows - 1;
  if (X1 < 0 || X0 >= map_w || Y1 < 0 || Y0 >= map_h) return false;
  const int tx0 = max(X0, 0) >> 5, tx1 = min(X1, map_w - 1) >> 5;
  const int ty0 = max(Y0, 0) >> 4, ty1 = min(Y1, map_h - 1) >> 4;
  const int wpr = lut.wpr;
  const uint64_t* __restrict__ rows = lut.rows + (int64_t)f.bin * lut.max_rows * wpr;
  for (int tyb = ty0; tyb <= ty1; tyb += BCG_BANDS) {
    uint32_t tm[BCG_BANDS];
    summary_bands(sum, tiles_x, tyb, ty1, tx0, tx1, tm);
    // the non-empty tiles of each band's first four columns (all of them under a mask <= 97 px wide) are asked into L2
    // right away (no register, no wait): the walk below then pays one DRAM round trip in all instead of one per tile
    uint32_t ahead = 0u;
#pragma unroll
    for (int k = 0; k < BCG_BANDS; ++k) ahead |= (tm[k] & 15u) << (4 * k);
    for (; ahead != 0u; ahead &= ahead - 1u) {
      const int bit = __ffs((int)ahead) - 1;
      const uint32_t* tp = tiles + ((((int64_t)(tyb + (bit >> 2)) * tiles_x) + tx0 + (bit & 3)) << 4);
      asm volatile("prefetch.global.L2 [%0];" ::"l"(tp));
    }
    int k = 0;
    while (k < BCG_BANDS) {                                // band by band
      uint32_t mk = 0u;                                    // tm[k] by selects: a runtime index would put tm[] in local memory
#pragma unroll
      for (int q = 0; q < BCG_BANDS; ++q) mk = (q == k) ? tm[q] : mk;
      if (mk == 0u) { ++k; continue; }
#pragma unroll
      for (int q = 0; q < BCG_BANDS; ++q) if (q == k) tm[q] &= tm[q] - 1u;
      const int ty = tyb + k, tx = tx0 + __ffs((int)mk) - 1;
      const int dy0 = (ty << 4) - Y0;                      // mask row of the band's first tile row
      uint32_t ws[16];
      load_tile(tiles + ((((int64_t)ty * tiles_x) + tx) << 4), ws);
      const int rel = (tx << 5) - X0;
      uint32_t hit = 0u;
#pragma unroll
      for (int r = 0; r < 16; ++r)                         // (unrolled: a dynamic index would put the tile words in local memory)
        if (ws[r] != 0u && (unsigned)(dy0 + r) < (unsigned)f.nrows) hit |= ws[r] & mask_bits32(rows + (int64_t)(dy0 + r) * wpr, wpr, rel);
      if (hit) return true;
    }
  }
  return false;
}

// The tile loop for a box in the fast shape (one-word mask rows in aligned pairs, <= 4 tile columns, <= 6 bands) whose
// non-empty tiles are already listed in `todo` (4 bits per band from band ty0, bit j <-> column tx0 + j).  The list comes
// band by band, so a band's mask rows are kept for its next tile.
__device__ __forceinline__ bool collide_thread_listed(const BcgFootprintLut& lut, const uint32_t* __restrict__ tiles,
                                                      int tiles_x, const FootBox& f, int ty0, int tx0, uint32_t todo) {
  const uint64_t* __restrict__ rows = lut.rows + (int64_t)f.bin * lut.max_rows;
  int vband = -1;
  uint64_t v[18];
  while (todo != 0u) {
    const int bit = __ffs((int)todo) - 1;
    todo &= todo - 1u;
    const int k = bit >> 2, ty = ty0 + k, tx = tx0 + (bit & 3);
    const int dy0 = (ty << 4) - f.Y0;
    uint32_t ws[16];
    load_tile(tiles + ((((int64_t)ty * tiles_x) + tx) << 4), ws);
    if (k != vband) {
      vband = k;
      load_band_rows(rows, lut.max_rows, dy0, v);
    }
    if (tile_meets_rows(ws, v, dy0, (tx << 5) - f.X0)) return true;
  }
  return false;
}

// collide_thread with the tiles of a WARP's 32 envs dealt out evenly.  In collide_thread_listed a warp walks its tile loop as
// often as its busiest lane has non-empty tiles under the footprint (~9 times for ~3 tiles per lane on the aisle workload), and
// that loop was three quarters of move_kernel's instructions.  Here every lane still reads its own env's summary words and
// lists its tiles (4 bits per band), then the warp's (env, tile) pairs are numbered by a prefix sum and lane l takes pair
// (lanes present) r + l of round r: it finds the owner by binary search over the inclusive counts, gets the owner's box by shuffles,
// loads the tile's four 16-byte quarters and the band's mask rows, and a hit travels back to its owner through a ballot.
// ~3 rounds instead of ~9, no lane idles while another works.  `act` = the lanes of the warp that hold an env (all callers
// are thread-per-env kernels whose tail warp is partly empty; those lanes are contiguous from 0).  Boxes that do not fit the
// fast shape (multi-word mask rows, > 4 tile columns, > 6 bands) are checked by collide_thread afterwards.  Same verdict.
__device__ __forceinline__ bool collide_warp_balanced(const BcgFootprintLut& lut, const uint32_t* __restrict__ tile_arena,
                                                      int64_t tile_off, const uint32_t* __restrict__ sum, int tiles_x,
                                                      int map_w, int map_h, const FootBox& f, unsigned act, unsigned lane) {
  const int X0 = f.X0, Y0 = f.Y0;
  const int X1 = X0 + f.fwidth - 1, Y1 = Y0 + f.nrows - 1;
  const bool inside = !(X1 < 0 || X0 >= map_w || Y1 < 0 || Y0 >= map_h);
  const int tx0 = max(X0, 0) >> 5, tx1 = min(X1, map_w - 1) >> 5;
  const int ty0 = max(Y0, 0) >> 4, ty1 = min(Y1, map_h - 1) >> 4;
  const bool pair_rows = lut.wpr == 1 && (lut.max_rows & 1) == 0 && (reinterpret_cast<uintptr_t>(lut.rows) & 15) == 0;
  const bool fast = inside && pair_rows && (tx1 - tx0) < 4 && (ty1 - ty0) < BCG_BANDS && tiles_x < 2048 && ty0 < 2048 &&
                    tx0 < 1024 && X0 > -32768 && Y0 > -32768;
  uint32_t todo = 0u;
  if (fast) {
    uint32_t tm[BCG_BANDS];
    summary_bands(sum, tiles_x, ty0, ty1, tx0, tx1, tm);
#pragma unroll
    for (int k = 0; k < BCG_BANDS; ++k) todo |= tm[k] << (4 * k);
  }
  const int cnt = __popc(todo);
  int incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int v = __shfl_up_sync(act, incl, d);
    if ((int)lane >= d) incl += v;
  }
  const int last = 31 - __clz((int)act);
  const int total = __shfl_sync(act, incl, last);
  // Dealing pays when the lanes' lists differ in length.  When they do not (Monte-Carlo fan-outs: the rollouts of one
  // start state share a pose for many steps) the per-thread loop is as short and keeps a band's mask rows across its
  // tiles: a dealt round costs about 1.5 of its iterations.
  const int longest = (int)__reduce_max_sync(act, (unsigned)cnt);
  const int rounds = (total + last) / (last + 1);
  bool myhit = false;
  if (3 * rounds >= 2 * longest) {
    if (fast) myhit = collide_thread_listed(lut, tile_arena + tile_off, tiles_x, f, ty0, tx0, todo);
  } else {
    // what a lane needs of a pair's owner, packed for the shuffles
    const uint32_t pk_xy = ((uint32_t)X0 & 0xffffu) | ((uint32_t)Y0 << 16);
    const uint32_t pk_t = (uint32_t)ty0 | ((uint32_t)tx0 << 11) | ((uint32_t)tiles_x << 21);
    const int excl = incl - cnt;
    for (int base = 0; base < total; base += last + 1) {   // a round deals one pair to each lane that is there
      const int i = base + (int)lane;
      const bool has = i < total;
      int o = 0;                                           // owner = the first lane whose inclusive count exceeds i
#pragma unroll
      for (int st = 16; st >= 1; st >>= 1) {
        const int probe = o + st - 1;
        const int t = __shfl_sync(act, incl, min(probe, last));
        if (probe <= last && t <= i) o += st;
      }
      o = min(o, last);
      const uint32_t otodo = __shfl_sync(act, todo, o);
      const int r = i - __shfl_sync(act, excl, o);
      const uint32_t oxy = __shfl_sync(act, pk_xy, o), ot = __shfl_sync(act, pk_t, o);
      const int obin = __shfl_sync(act, f.bin, o);
      const unsigned long long ooff = __shfl_sync(act, (unsigned long long)tile_off, o);
      bool hit = false;
      if (has) {
        uint32_t m = otodo;                                // the pair's tile: set bit number r of the owner's list
        for (int q = 0; q < r; ++q) m &= m - 1u;
        const int bit = __ffs((int)m) - 1;
        const int ty = (int)(ot & 2047u) + (bit >> 2), tx = (int)((ot >> 11) & 1023u) + (bit & 3);
        const int oX0 = (int)(short)(oxy & 0xffffu), oY0 = (int)(short)(oxy >> 16);
        const int dy0 = (ty << 4) - oY0;
        uint32_t ws[16];
        load_tile(tile_arena + (int64_t)ooff + ((((int64_t)ty * (int)(ot >> 21)) + tx) << 4), ws);
        uint64_t v[18];
        load_band_rows(lut.rows + (int64_t)obin * lut.max_rows, lut.max_rows, dy0, v);
        hit = tile_meets_rows(ws, v, dy0, (tx << 5) - oX0);
      }
      const uint32_t hb = __ballot_sync(act, hit);
      for (uint32_t h2 = hb; h2 != 0u; h2 &= h2 - 1u) {    // rare: a collision ends the episode
        const int l = __ffs((int)h2) - 1;
        if (__shfl_sync(act, o, l) == (int)lane) myhit = true;
      }
    }
  }
  // boxes outside the fast shape, after either branch: one call site, so one inlined copy of collide_thread
  if (inside && !fast) myhit = collide_thread(lut, tile_arena + tile_off, sum, tiles_x, map_w, map_h, f);
  return myhit;
}

// the lanes of this warp that hold one of the n items of a thread-per-item kernel (item = global thread index)
__device__ __forceinline__ unsigned warp_item_mask(int first_item_of_warp, int n) {
  const int left = n - first_item_of_warp;
  return left >= 32 ? BCG_FULL : ((1u << left) - 1u);
}

// The same verdict read straight from the uint8 costmap rows: each half-warp owns one footprint row
// per pass, each lane one aligned 4-byte word of it.
__device__ __forceinline__ bool collide_u8(const BcgBatch& b, const WorkCollide& f, unsigned lane) {
  const int X0 = f.X0, Y0 = f.Y0;
  const int X1 = X0 + f.fwidth - 1;
  const int map_w = f.map_w, map_h = f.map_h;
  unsigned hit = 0;
  if (!(X1 < 0 || X0 >= map_w)) {
    const int w0 = max(X0, 0) >> 2, w1 = min(X1, map_w - 1) >> 2;
    const uint8_t* data = b.map_arena + f.data_off;
    const uint64_t* rows = b.lut.rows + (int64_t)f.bin * b.lut.max_rows * b.lut.wpr;
    const int half = lane >> 4, sub = lane & 15;
    for (int dy = half; dy < f.nrows; dy += 2) {
      const int Y = Y0 + dy;
      if (Y < 0 || Y >= map_h) continue;
      const uint32_t* rowp = reinterpret_cast<const uint32_t*>(data + (int64_t)Y * f.map_pitch);
      for (int wi = w0 + sub; wi <= w1; wi += 16) {
        const uint32_t bytes = __ldg(rowp + wi);
        const uint32_t m4 = mask_bits32(rows + (int64_t)dy * b.lut.wpr, b.lut.wpr, (wi << 2) - X0) & 0xfu;
        const uint32_t eq = __vcmpeq4(bytes, 0xFEFEFEFEu);                 // 0xFF where cell == 254
        const uint32_t sel = ((m4 * 0x00204081u) & 0x01010101u) * 0xFFu;  // 0xFF where the mask is set
        hit |= eq & sel;
      }
    }
  }
  return __any_sync(BCG_FULL, hit != 0u);
}

// ---- reward -----------------------------------------------------------------------------------------
// find_last_reached (utilities/path_tools.py:408-448) restricted to indices >= lo (SURVEY.md A.8):
// max i with hypot < sp, |wrap(dth)| < ap, parallel distance >= -sp/9.  Chunks of 32 points whose
// bounding circle is farther than sp from the pose cannot contain a reached point and are skipped.
// Warp-cooperative; returns -1 when nothing is reached.
template <bool COHERENT>
__device__ __forceinline__ double ldro(const double* q) { return COHERENT ? *q : __ldg(q); }

struct PathRef {
  const double* P;   // 5 rows x, y, th, cos th, sin th, each `pitch` long
  const double* C;   // 3 chunk rows cx, cy, radius, each `chunk_pitch` long
  int n, pitch, chunk_pitch;
};

__device__ __forceinline__ PathRef path_ref(const BcgBatch& b, const BcgPathDesc& d) {
  PathRef r;
  r.P = b.path_arena + d.off;
  r.C = b.path_arena + d.chunk_off;
  r.n = d.n;
  r.pitch = d.pitch;
  r.chunk_pitch = d.chunk_pitch;
  return r;
}

// COHERENT: plain loads instead of ld.global.nc -- for callers whose path rows were written earlier in the SAME launch (the
// device generators); the read-only path is only defined for data that is constant for the whole kernel.
template <bool COHERENT = false>
__device__ __forceinline__ int last_reached_from(const BcgParams& p, const PathRef& pd, int lo, double px, double py,
                                                 double pth, unsigned lane) {
  if (lo >= pd.n) return -1;
  const double* P = pd.P;
  const double* C = pd.C;
  const double par_thr = -p.spatial_precision / 9;
  const double sp2 = p.spatial_precision * p.spatial_precision;
  const int c_lo = lo >> 5, c_hi = (pd.n - 1) >> 5;
  for (int g = c_hi >> 5; g >= (c_lo >> 5); --g) {
    const int c = (g << 5) + lane;
    bool near = false;
    if (c >= c_lo && c <= c_hi) {
      const double cx = ldro<COHERENT>(C + c) - px, cy = ldro<COHERENT>(C + pd.chunk_pitch + c) - py;
      const double reach = p.spatial_precision + ldro<COHERENT>(C + 2 * pd.chunk_pitch + c);
      near = (cx * cx + cy * cy) < reach * reach * (1.0 + 1e-12);     // conservative: never drops a reachable chunk
    }
    unsigned bits = __ballot_sync(BCG_FULL, near);
    while (bits) {
      const int cl = 31 - __clz(bits);
      bits &= ~(1u << cl);
      const int i = (((g << 5) + cl) << 5) + lane;
      bool reached = false;
      if (i >= lo && i < pd.n) {
        const double xi = ldro<COHERENT>(P + i), yi = ldro<COHERENT>(P + pd.pitch + i), ti = ldro<COHERENT>(P + 2 * pd.pitch + i);
        const double ci = ldro<COHERENT>(P + 3 * pd.pitch + i), si = ldro<COHERENT>(P + 4 * pd.pitch + i);
        // hypot(dx, dy) < sp, decided from the squared distance unless it is within 1e-12 of the threshold
        const double dx = xi - px, dy = yi - py, d2 = dx * dx + dy * dy;
        bool close = d2 < sp2 * (1.0 - 1e-12);
        if (!close && d2 <= sp2 * (1.0 + 1e-12)) close = hypot(dx, dy) < p.spatial_precision;
        if (close) {
          const double ang = fabs(wrap_angle(pth - ti));
          const double par = ci * (px - xi) + si * (py - yi);
          reached = (ang < p.angular_precision) && (par >= par_thr);
        }
      }
      const unsigned rb = __ballot_sync(BCG_FULL, reached);
      if (rb) return (((g << 5) + cl) << 5) + (31 - __clz(rb));
    }
  }
  return -1;
}

// The same scan by a GROUP of G lanes (G = 8: four envs per warp; reward_kernel).  With a whole warp per env the ~370
// straight-line instructions around the scan (record unpack, chunk test, reward, done, outputs) are paid per env; a group
// of 8 lanes pays a quarter of that and tests a 32-point chunk in four rounds.  Lane gl of a group takes the gl-th highest
// index of a round, so the lowest set ballot bit is the largest index.  Every loop is warp-uniform (exit when all groups
// are done): the ballots are full-warp ballots, each group reads its own G bits.
template <int G>
__device__ __forceinline__ int last_reached_group(const BcgParams& p, const PathRef& pd, int lo, double px, double py,
                                                  double pth, unsigned lane, bool active) {
  const unsigned gl = lane & (G - 1), gbase = lane & ~(unsigned)(G - 1);
  const uint32_t gmask = G == 32 ? 0xffffffffu : ((1u << G) - 1u);
  const double* __restrict__ P = pd.P;
  const double* __restrict__ C = pd.C;
  const double par_thr = -p.spatial_precision / 9;
  const double sp2 = p.spatial_precision * p.spatial_precision;
  bool done = !active || lo >= pd.n;
  const int c_lo = lo >> 5;
  int ctop = (pd.n - 1) >> 5;
  int result = -1;
  while (!__all_sync(BCG_FULL, done)) {
    const int c = ctop - (int)gl;
    bool near = false;
    if (!done && c >= c_lo) {
      const double cx = __ldg(C + c) - px, cy = __ldg(C + pd.chunk_pitch + c) - py;
      const double reach = p.spatial_precision + __ldg(C + 2 * pd.chunk_pitch + c);
      near = (cx * cx + cy * cy) < reach * reach * (1.0 + 1e-12);     // conservative: never drops a reachable chunk
    }
    uint32_t bits = (__ballot_sync(BCG_FULL, near) >> gbase) & gmask;   // bit j <-> chunk ctop - j
    while (true) {
      const bool has = !done && bits != 0u;
      if (!__any_sync(BCG_FULL, has)) break;
      int cc = 0;
      if (has) {
        cc = ctop - (__ffs((int)bits) - 1);
        bits &= bits - 1u;
      }
#pragma unroll 1
      for (int r = 0; r < 32 / G; ++r) {
        const int i = (cc << 5) + 31 - r * G - (int)gl;
        bool reached = false;
        if (has && !done && i >= lo && i < pd.n) {
          const double xi = __ldg(P + i), yi = __ldg(P + pd.pitch + i);
          // hypot(dx, dy) < sp, decided from the squared distance unless it is within 1e-12 of the threshold
          const double dx = xi - px, dy = yi - py, d2 = dx * dx + dy * dy;
          bool close = d2 < sp2 * (1.0 - 1e-12);
          if (!close && d2 <= sp2 * (1.0 + 1e-12)) close = hypot(dx, dy) < p.spatial_precision;
          if (close) {
            const double ti = __ldg(P + 2 * pd.pitch + i), ci = __ldg(P + 3 * pd.pitch + i), si = __ldg(P + 4 * pd.pitch + i);
            const double ang = fabs(wrap_angle(pth - ti));
            const double par = ci * (px - xi) + si * (py - yi);
            reached = (ang < p.angular_precision) && (par >= par_thr);
          }
        }
        const uint32_t rb = (__ballot_sync(BCG_FULL, reached) >> gbase) & gmask;
        if (rb != 0u && !done) {
          result = (cc << 5) + 31 - r * G - (__ffs((int)rb) - 1);
          done = true;
        }
      }
    }
    ctop -= G;
    if (ctop < c_lo) done = true;
  }
  return result;
}

// ContinuousRewardPurePursuitProviderState.update_goal (envs/base/reward.py:126-137): the first way point from `lo` on
// that is more than `radius` from the pose, else the last point -- by a group of G lanes (see last_reached_group)
template <int G>
__device__ __forceinline__ int first_beyond_radius_group(const PathRef& pd, int lo, double px, double py, double radius,
                                                         unsigned lane, bool active) {
  const unsigned gl = lane & (G - 1), gbase = lane & ~(unsigned)(G - 1);
  const uint32_t gmask = G == 32 ? 0xffffffffu : ((1u << G) - 1u);
  int base = max(lo, 0);
  int result = pd.n - 1;
  bool done = !active || base >= pd.n;
  while (!__all_sync(BCG_FULL, done)) {
    const int i = base + (int)gl;
    bool far = false;
    if (!done && i < pd.n) {
      const double dx = __ldg(pd.P + i) - px, dy = __ldg(pd.P + pd.pitch + i) - py;
      far = sqrt(fma(dy, dy, dx * dx)) > radius;        // np.linalg.norm of a 2-vector = sqrt(ddot), fused like the BLAS
    }
    const uint32_t bits = (__ballot_sync(BCG_FULL, far) >> gbase) & gmask;
    if (!done && bits != 0u) {
      result = base + __ffs((int)bits) - 1;
      done = true;
    }
    base += G;
    if (base >= pd.n) done = true;
  }
  return result;
}

}  // namespace bcg
