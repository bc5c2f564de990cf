// Kernels + C-ABI of the batched PlanEnv.step path for B200 (sm_100a).  See include/bcg_b200.h.
//
// One step = three launches on one stream (DESIGN.md has the rooflines and the measurements):
//   move_kernel            1 thread / env    -- control delay ring, robot model, Philox noise, footprint lookup, collision
//                                               on the 1-bit lethal tile plane (batched loads of the non-empty tiles under
//                                               the footprint), rollback, pose / state delay rings, compact observation,
//                                               the 128-byte egocentric record and the 144-byte record of
//   reward_kernel          8 lanes / env     -- chunk-culled reached-index scan of the remaining path, reward, done, episode
//                                               statistics, goal vector, the rare auto-reset
//   ego_sparse_kernel      persistent, 64-thread CTAs x 18 per SM -- cv2.warpAffine(INTER_NEAREST)-exact egocentric crop as a
//                                               scatter of the occupied cells of the source window
//   (ego_tiles_kernel      persistent, 256-thread CTAs -- the dense per-pixel gather: pools of dense maps, and the envs
//                                               the sparse kernel hands over when a batch mixes sparse and dense maps)
//   (regenerate_kernel     fixed grid, between reward_kernel and the egocentric kernels when the batch auto-resets into new
//                                               worlds: the done envs' final crops, new worlds and initial observations)
// plus the set-up kernels (tile planes and summary, cell tiles, initial state), the device-side world generators and
// the stand-alone entry points of the hook seam.
// No tensor cores: nothing here is a dense contraction.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>

#include "bcg_b200.h"
#include "bcg_device.cuh"
#include "bcg_generate.cuh"

using namespace bcg;
namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

#define BCG_CHECK_CUDA(expr)                                                                  \
  do {                                                                                        \
    cudaError_t err__ = (expr);                                                               \
    if (err__ != cudaSuccess)                                                                 \
      return fail(BCG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(err__));       \
  } while (0)

// driver entry points without linking libcuda (the library must load on a box without a driver: tests -m "not gpu")
template <class F>
static int driver_fn(const char* name, F* out) {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  BCG_CHECK_CUDA(cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return fail(BCG_ERR_CUDA, "driver entry point not available");
  *out = reinterpret_cast<F>(fn);
  return BCG_OK;
}
#define BCG_CHECK_CU(x)                                                         \
  do {                                                                          \
    const CUresult r_ = (x);                                                    \
    if (r_ != CUDA_SUCCESS) return fail(BCG_ERR_CUDA, #x " failed");            \
  } while (0)


#define BCG_REQUIRE(cond, msg) \
  do {                         \
    if (!(cond)) return fail(BCG_ERR_INVALID, msg); \
  } while (0)

// Programmatic dependent launch: a step kernel launched with the attribute may start while its predecessor in the stream
// is still draining (launch latency and its own prologue overlap that tail); it calls pdl_wait() before it touches
// anything the predecessor wrote -- the wait returns when the predecessor grid has completed and its writes are visible.
// No kernel triggers its successor early (griddepcontrol.launch_dependents): successor CTAs waiting in pdl_wait() would
// hold the slots of the kernel they wait for, so the trigger is left to CTA exit (DESIGN.md section 3).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

bool g_pdl_refused = false;       // the driver turned a dependent launch down once: classic launches from then on
bool pdl_enabled() {
  static const bool on = [] {
    const char* v = getenv("BCG_PDL");
    return !(v && v[0] == '0');
  }();
  return on && !g_pdl_refused;
}

template <class... KArgs, class... Args>
cudaError_t launch_step_kernel(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t s, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl && pdl_enabled()) ? 1 : 0;
  cudaError_t err = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
  if (err != cudaSuccess && cfg.numAttrs == 1 && (err == cudaErrorNotSupported || err == cudaErrorInvalidValue)) {
    (void)cudaGetLastError();           // a driver without programmatic dependent launch: same kernel, ordinary launch
    g_pdl_refused = true;
    cfg.numAttrs = 0;
    err = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
  }
  return err;
}

BcgStateLayout make_layout(const BcgParams& p) {
  BcgStateLayout L;
  L.ring_control = BCG_F_FIXED;
  L.ring_pose = L.ring_control + 2 * p.delay_control;
  L.ring_state = L.ring_pose + 3 * p.delay_pose;
  L.n_frows = L.ring_state + 7 * p.delay_state;
  L.n_irows = BCG_I_FIXED;
  return L;
}

int check_batch(const BcgParams* p, const BcgBatch* b) {
  BCG_REQUIRE(p && b, "null params/batch");
  BCG_REQUIRE(b->n_envs > 0, "n_envs must be positive");
  BCG_REQUIRE(p->delay_control >= 0 && p->delay_pose >= 0 && p->delay_state >= 0, "negative delay");
  BCG_REQUIRE(p->delay_control < 4096 && p->delay_pose < 4096 && p->delay_state < 4096, "delay too large");
  const BcgStateLayout L = make_layout(*p);
  BCG_REQUIRE(b->n_frows == L.n_frows && b->n_irows == L.n_irows, "state row count does not match bcg_state_layout");
  BCG_REQUIRE(b->state_f && b->state_i && b->init_f && b->init_i && b->cand && b->cand_i && b->work, "null state pointers");
  BCG_REQUIRE(b->map_id && b->path_id && b->maps && b->paths && b->map_arena && b->tile_arena && b->path_arena,
              "null arena pointers");
  BCG_REQUIRE(b->occ_tile_arena, "null occupancy plane (BcgBatch.occ_tile_arena)");
  BCG_REQUIRE(b->occ_sum_arena, "null tile summary (BcgBatch.occ_sum_arena)");
  BCG_REQUIRE(b->lut.edges && b->lut.verts && b->lut.header && b->lut.rows && b->lut.fp_pix && b->lut.bucket_first,
              "null footprint table");
  BCG_REQUIRE(b->lut.n_buckets > 0 && b->lut.bucket_scale > 0, "empty footprint bucket table");
  BCG_REQUIRE(b->lut.n_verts > 0 && b->lut.n_verts <= 32, "footprint must have 1..32 vertices");
  BCG_REQUIRE(b->lut.n_bins > 0 && b->lut.wpr > 0 && b->lut.max_rows > 0, "empty footprint table");
  BCG_REQUIRE(b->status && b->stats, "null status/stats");
  if (p->auto_reset == BCG_AUTO_RESET_NEW_WORLD) {
    BCG_REQUIRE(b->world_gen, "auto_reset BCG_AUTO_RESET_NEW_WORLD needs the world generator (BcgBatch.world_gen)");
    BCG_REQUIRE(b->n_maps == b->n_envs && b->n_paths == b->n_envs && b->cell_tile_arena,
                "auto_reset BCG_AUTO_RESET_NEW_WORLD (BcgBatch.world_gen) needs a batch of per-env world slots: n_maps == n_paths == "
                "n_envs and the cell-tile arena");
  }
  return BCG_OK;
}

// per-env parameter rows: NULL (batch-wide) or both row arrays
int check_rows(const BcgEnvRows* rows) {
  if (rows) BCG_REQUIRE(rows->f && rows->i, "null per-env parameter rows");
  return BCG_OK;
}

// the per-env slots of the device-side world generators (`who` names the entry point in the messages)
int check_slots(const BcgParams* p, const BcgBatch* b, const BcgAisleSlots* slots, double path_delta, const char* who) {
  BCG_REQUIRE(slots && slots->gen_state, "null slots / gen_state");
  BCG_REQUIRE(b->cell_tile_arena, std::string(who) + " needs the cell-tile arena");
  BCG_REQUIRE(b->n_maps == b->n_envs && b->n_paths == b->n_envs, "device-generated envs own one map and one path slot each");
  BCG_REQUIRE(slots->map_slot_bytes > 0 && slots->tile_slot_words > 0 && slots->path_pitch >= 8 && slots->path_pitch % 4 == 0 &&
                  slots->chunk_pitch * 32 >= slots->path_pitch,
              "bad slot sizes");
  BCG_REQUIRE(path_delta > 0, "path_delta must be positive");
  BCG_REQUIRE((int)(0.05 / p->resolution) <= 1, "walls are drawn one pixel thick: resolution must be above 0.025 m");
  return BCG_OK;
}

// ---- kernels -------------------------------------------------------------------------------------

// work records of arbitrary poses [3][n] (stand-alone collision entry points)
__global__ void __launch_bounds__(128) pose_prep_kernel(const BcgParams p, const BcgBatch b,
                                                        const double* __restrict__ poses) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= b.n_envs) return;
  const int64_t N = b.n_envs;
  uint8_t* rec = reinterpret_cast<uint8_t*>(b.work) + (int64_t)e * BCG_WORK_BYTES;
  *reinterpret_cast<WorkCollide*>(rec) = make_work_collide(p, b, b.map_id[e], poses[e], poses[N + e], poses[2 * N + e]);
}

#define BCG_EGO_MAX 256

struct EgoAffine {
  double a11, a12, b1, a21, a22, b2;   // source = A * (u, v) + b, cv::warpAffine's inverted map
};

// costmap_utils.py:42-65 + the fp64 inversion cv::warpAffine applies to the float32 forward matrix
__device__ __forceinline__ EgoAffine ego_affine(const BcgParams& p, const BcgMapDesc& m, double px, double py,
                                                double pth, float* fwd = nullptr) {
  const double cx = (double)world_to_pixel_1d(px, m.origin_x, p.inv_resolution);
  const double cy = (double)world_to_pixel_1d(py, m.origin_y, p.inv_resolution);
  const double deg = 180 * pth / BCG_PI;
  const double rad = deg * (BCG_PI / 180.);
  double bsn, acs;
  sincos(rad, &bsn, &acs);
  const float r00 = (float)acs, r01 = (float)bsn, r02 = (float)((1 - acs) * cx - bsn * cy);
  const float r10 = (float)(-bsn), r11 = (float)acs, r12 = (float)(bsn * cx + (1 - acs) * cy);
  const double dsx = rint((p.ego_x0 - (m.origin_x - px)) * p.inv_resolution);
  const double dsy = rint((p.ego_y0 - (m.origin_y - py)) * p.inv_resolution);
  const double M0 = (double)r00, M1 = (double)r01, M2 = (double)(r02 - (float)dsx);
  const double M3 = (double)r10, M4 = (double)r11, M5 = (double)(r12 - (float)dsy);
  if (fwd) {                           // the float32 forward matrix itself (source pixel -> crop pixel)
    fwd[0] = (float)M0; fwd[1] = (float)M1; fwd[2] = (float)M2;
    fwd[3] = (float)M3; fwd[4] = (float)M4; fwd[5] = (float)M5;
  }
  double D = M0 * M4 - M1 * M3;
  D = (D != 0.0) ? 1. / D : 0.0;
  EgoAffine a;
  a.a11 = M4 * D;
  a.a22 = M0 * D;
  a.a12 = M1 * (-D);
  a.a21 = M3 * (-D);
  a.b1 = -a.a11 * M2 - a.a12 * M5;
  a.b2 = -a.a21 * M2 - a.a22 * M5;
  return a;
}

// The path point goal_n_state points at.  envs/egocentric.py:141-160 takes the first point of Observation.path: path[target:]
// with the continuous reward, so the next way point; path[:target + 1] with pure pursuit (reward.py:120-124), so the first
// point of the path.  The colored variant (synth_turn_env.py:412-418) points at the last path point.
__device__ __forceinline__ int goal_point_index(const BcgParams& p, int n, int target) {
  if (p.ego_variant == 1) return n - 1;
  return p.reward_kind == BCG_REWARD_PURE_PURSUIT ? 0 : target;
}

// goal_n_state (envs/egocentric.py:141-160) by one thread
// `target` and `drobot` (the delayed robot state x, y, th, v, w, steer, wheel) are those of the state being observed
__device__ __forceinline__ void write_goal_n_state(const BcgParams& p, const BcgBatch& b, int e, const BcgPathDesc& pd,
                                                   double px, double py, double pth, int target, const double drobot[7],
                                                   float* __restrict__ goal_n_state) {
  float* g = goal_n_state + (int64_t)e * 9;
  if (target > pd.n - 1) {
#pragma unroll
    for (int k = 0; k < 9; ++k) g[k] = 0.f;
    return;
  }
  // from_global_to_egocentric (coordinate_transformations.py:341-362 -> :57-84 -> :310-328)
  const double* P = b.path_arena + pd.off;
  const int gi = goal_point_index(p, pd.n, target);
  const double gx = P[gi], gy = P[pd.pitch + gi], gt = P[2 * pd.pitch + gi];
  double sn, cs;
  sincos(pth, &sn, &cs);
  const double tx = -px * cs - py * sn;
  const double ty = px * sn - py * cs;
  const double tt = wrap_angle(-pth);
  double st, ct;
  sincos(tt, &st, &ct);
  const double ex = ct * gx - st * gy + tx;
  const double ey = st * gx + ct * gy + ty;
  const double ea = wrap_angle(gt + tt);
  if (p.ego_variant == 1) {
    // synth_turn_env.py:412-418: goal / crop world size, scaled to unit length; then (v, w, wheel)
    const double nx = ex / p.ego_world_w, ny = ey / p.ego_world_h;
    const double nrm = sqrt(nx * nx + ny * ny);
    g[0] = (float)(nx / nrm);
    g[1] = (float)(ny / nrm);
    g[2] = (float)drobot[3];
    g[3] = (float)drobot[4];
    g[4] = (float)drobot[6];
    g[5] = g[6] = g[7] = g[8] = 0.f;
    return;
  }
  g[0] = (float)clampd(ex / p.ego_world_w, -1.0, 1.0);
  g[1] = (float)clampd(ey / p.ego_world_h, -1.0, 1.0);
  g[2] = (float)ea;
  g[3] = (float)drobot[0];
  g[4] = (float)drobot[1];
  g[5] = (float)drobot[2];
  g[6] = (float)drobot[3];
  g[7] = (float)drobot[4];
  g[8] = (float)drobot[6];
}

#define BCG_EGO_MODE_DIRECT 0
#define BCG_EGO_MODE_TILES 3
#define BCG_EGO_WORK_BYTES 128        // stride of the per-env records in BcgBatch.ego_work (EgoTileWork)

// Record of the persistent cell-tile egocentric kernel (ego_tiles_kernel), resolved one thread per env: the
// inverted affine map, the tile-aligned source window and, per row of cell tiles, which tiles the rotated crop
// rectangle touches.  Doing the clipping here (32 envs per warp) instead of in the image kernel (one env per
// CTA) is ~50x cheaper in issued instructions.
#define BCG_EGT_MAX_TILE_ROWS 64
struct __align__(16) EgoTileWork {   // 128 bytes
  EgoAffine aff;                     // 48
  int32_t X0, Y0;                    // window origin in map pixels, multiples of (16, 8); 0 in direct mode
  int32_t ntx, nty;                  // window size in cell tiles
  int32_t mode, map_id;              // BCG_EGO_MODE_TILES or BCG_EGO_MODE_DIRECT
  int32_t ctiles_x, ctiles_y;        // cell-tile grid of the env's map
  int64_t ctile_off;                 // byte offset of the map's cell tiles in the cell-tile arena
  int32_t fwd[6];                    // cv::warpAffine's forward matrix (source -> crop) in 16.16 fixed point, translation
                                     // relative to the window origin (X0, Y0): the sparse kernel's candidate pixels
  int32_t dense_map;                 // bit 0: more than 1 cell in 20 of the map is occupied (skip the sparse kernel's
                                     // scan); bit 1: every occupied cell is 254 (BCG_MAP_ONLY_LETHAL); bit 2: the map's
                                     // cell index is exact (BCG_MAP_CELL_INDEX)
  // what the sparse kernel needs of the map descriptor, so that its loads start from the record alone
  int32_t sum_off;                   // BcgMapDesc.sum_off
  uint32_t tiles_xy;                 // tiles_x | tiles_y << 16
  uint32_t tile_off16;               // BcgMapDesc.tile_off / 16 (a plane is a whole number of 16-word tiles)
};
static_assert(sizeof(EgoTileWork) == BCG_EGO_WORK_BYTES, "EgoTileWork records are 128 bytes");

// shared-memory bytes of one window buffer of ego_tiles_kernel: worst-case tile-aligned window of the crop
__host__ __device__ inline int ego_window_capacity(const BcgParams& p) {
  const int side = (int)ceil(sqrt((double)p.ego_w * p.ego_w + (double)p.ego_h * p.ego_h)) + 2;
  const int nty = (side + 1 + 7) / 8 + 1, ntx = (side + 1 + 15) / 16 + 1;
  long long cap = (long long)nty * 128 * (ntx | 1);
  if (cap > 52 * 1024) cap = 52 * 1024;     // two buffers x two CTAs per SM must fit; larger crops gather from global
  return (int)cap;
}

// corners of the crop rectangle in source pixels (the image of the crop's corner pixels under the inverted map)
struct EgoQuad {
  double qx[4], qy[4], xlo, xhi, ylo, yhi;
};
__device__ __forceinline__ EgoQuad ego_quad(const EgoAffine& A, int ego_w, int ego_h) {
  EgoQuad q;
  const double uw = (double)(ego_w - 1), vh = (double)(ego_h - 1);
  q.qx[0] = A.b1; q.qx[1] = A.a11 * uw + A.b1; q.qx[2] = A.a11 * uw + A.a12 * vh + A.b1; q.qx[3] = A.a12 * vh + A.b1;
  q.qy[0] = A.b2; q.qy[1] = A.a21 * uw + A.b2; q.qy[2] = A.a21 * uw + A.a22 * vh + A.b2; q.qy[3] = A.a22 * vh + A.b2;
  q.xlo = fmin(fmin(q.qx[0], q.qx[1]), fmin(q.qx[2], q.qx[3]));
  q.xhi = fmax(fmax(q.qx[0], q.qx[1]), fmax(q.qx[2], q.qx[3]));
  q.ylo = fmin(fmin(q.qy[0], q.qy[1]), fmin(q.qy[2], q.qy[3]));
  q.yhi = fmax(fmax(q.qy[0], q.qy[1]), fmax(q.qy[2], q.qy[3]));
  return q;
}

__device__ __forceinline__ void write_ego_tile_record(const BcgParams& p, const BcgBatch& b, int e, int map_id,
                                                      const BcgMapDesc& m, double px, double py, double pth, int win_capacity) {
  EgoTileWork* rec = reinterpret_cast<EgoTileWork*>(reinterpret_cast<uint8_t*>(b.ego_work) + (int64_t)e * BCG_EGO_WORK_BYTES);
  EgoTileWork w;
  float fwd[6];
  w.aff = ego_affine(p, m, px, py, pth, fwd);
#pragma unroll
  for (int k = 0; k < 6; ++k) w.fwd[k] = 0;
  w.X0 = w.Y0 = w.ntx = w.nty = 0;
  w.mode = BCG_EGO_MODE_DIRECT;
  w.map_id = map_id;
  w.dense_map = (((int64_t)m.occupied * 20 > (int64_t)m.width * m.height) ? 1 : 0) | ((m.flags & BCG_MAP_ONLY_LETHAL) ? 2 : 0) |
                (m.flags & BCG_MAP_CELL_INDEX);
  w.sum_off = m.sum_off;
  w.tiles_xy = (uint32_t)m.tiles_x | ((uint32_t)m.tiles_y << 16);
  w.tile_off16 = (uint32_t)(m.tile_off >> 4);
  w.ctiles_x = m.ctiles_x;
  w.ctiles_y = m.ctiles_y;
  w.ctile_off = m.cell_tile_off;
  // every sample is X = floor(x + 0.5 + d), |d| <= 2^-10, of a point x of the rotated crop rectangle: the
  // rectangle grown by 0.51 px bounds all samples
  const EgoQuad q = ego_quad(w.aff, p.ego_w, p.ego_h);
  const double lim = 1048576.0;
  const bool sane = q.xlo > -lim && q.xhi < lim && q.ylo > -lim && q.yhi < lim;   // false for NaN too
  if (sane) {
    const int x0 = (int)floor(q.xlo - 0.51) & ~15, y0 = (int)floor(q.ylo - 0.51) & ~7;
    const int x1 = (int)ceil(q.xhi + 0.51), y1 = (int)ceil(q.yhi + 0.51);
    const int ntx = (x1 >> 4) - (x0 >> 4) + 1, nty = (y1 >> 3) - (y0 >> 3) + 1;
    if (ntx <= 16 && nty <= BCG_EGT_MAX_TILE_ROWS && nty * 128 * (ntx | 1) <= win_capacity) {   // 16: one staging pass per tile row
      w.mode = BCG_EGO_MODE_TILES;
      w.X0 = x0;
      w.Y0 = y0;
      w.ntx = ntx;
      w.nty = nty;
      // crop pixel of window cell (xr, yr): floor((fwd0 xr + fwd1 yr + fwd2) >> 16), same for v.  Candidates only (the
      // exact fixed-point rule decides): 2^-17 per coefficient x 255 cells is far inside the 0.29 px the rule leaves
      const double c0 = (double)fwd[0] * x0 + (double)fwd[1] * y0 + (double)fwd[2];
      const double c1 = (double)fwd[3] * x0 + (double)fwd[4] * y0 + (double)fwd[5];
      w.fwd[0] = __double2int_rn((double)fwd[0] * 65536.0);
      w.fwd[1] = __double2int_rn((double)fwd[1] * 65536.0);
      w.fwd[2] = __double2int_rn(fmin(fmax(c0, -16000.0), 16000.0) * 65536.0);
      w.fwd[3] = __double2int_rn((double)fwd[3] * 65536.0);
      w.fwd[4] = __double2int_rn((double)fwd[4] * 65536.0);
      w.fwd[5] = __double2int_rn(fmin(fmax(c1, -16000.0), 16000.0) * 65536.0);
    }
  }
  uint4* dst = reinterpret_cast<uint4*>(rec);
  const uint4* src = reinterpret_cast<const uint4*>(&w);
#pragma unroll
  for (int k = 0; k < 8; ++k) dst[k] = src[k];
}

// Which cell tiles of row t of the window (8 source rows) the rotated crop rectangle touches: first | last << 8 window
// tile column (first > last: none).  Evaluated by the egocentric kernels themselves, lane <-> tile row, one env ahead
// of its use: for a thread-per-env kernel this loop was 4 k serial fp64 instructions per env, for a warp with one band
// per lane it is ~100.  The rectangle is convex, so over a band of rows its left boundary is the maximum of the lines
// through its left edges (a convex function of y: smallest at a band end or at the leftmost vertex) and its right
// boundary the minimum of the lines through its right edges.  A span only has to COVER the samples (the exact
// fixed-point rule decides every pixel later), so it is worked out in float32 on window-relative coordinates (< 1024,
// rounding errors ~1e-4 px) with the 0.51 px sample margin widened to 0.53.
__device__ __forceinline__ uint32_t ego_band_span(const EgoAffine& A, int ego_w, int ego_h, int X0, int Y0, int ntx, int nty,
                                                  int t) {
  // corners q0 = b, q1 = q0 + U, q2 = q1 + V, q3 = q0 + V with U = (w - 1)(a11, a21), V = (h - 1)(a12, a22); the edges
  // q0q1 and q2q3 share the slope U.x / U.y, the other two V.x / V.y: two approximate divisions (2 ulp) per env
  const float bx = (float)(A.b1 - (double)X0), by = (float)(A.b2 - (double)Y0);
  const float uwf = (float)(ego_w - 1), vhf = (float)(ego_h - 1);
  const float ux = (float)A.a11 * uwf, uy = (float)A.a21 * uwf, vx = (float)A.a12 * vhf, vy = (float)A.a22 * vhf;
  const float qx[4] = {bx, bx + ux, bx + ux + vx, bx + vx};
  const float qy[4] = {by, by + uy, by + uy + vy, by + vy};
  const float edy[4] = {uy, vy, -uy, -vy};
  const float inv_u = uy != 0.f ? __fdividef(ux, uy) : 0.f, inv_v = vy != 0.f ? __fdividef(vx, vy) : 0.f;
  const float xlo = fminf(fminf(qx[0], qx[1]), fminf(qx[2], qx[3])), xhi = fmaxf(fmaxf(qx[0], qx[1]), fmaxf(qx[2], qx[3]));
  const float ylo = fminf(fminf(qy[0], qy[1]), fminf(qy[2], qy[3])), yhi = fmaxf(fmaxf(qy[0], qy[1]), fmaxf(qy[2], qy[3]));
  const bool ccw = ux * vy - uy * vx > 0.f;
  const float BIG = 1e30f, M = 0.53f;
  const float y0 = fmaxf((float)(8 * t) - M, ylo), y1 = fminf((float)(8 * t + 7) + M, yhi);
  int ts = 1, te = 0;
  if (t < nty && y0 <= y1) {
    float l0 = -BIG, l1 = -BIG, r0 = BIG, r1 = BIG;
    float y_at_xlo = qy[0], y_at_xhi = qy[0];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float dy = edy[k];
      const float inv = (k & 1) ? inv_v : inv_u;
      const bool is_left = ccw ? dy < 0.f : dy > 0.f, is_right = ccw ? dy > 0.f : dy < 0.f;   // horizontal edges: neither
      const float v0 = qx[k] + (y0 - qy[k]) * inv, v1 = qx[k] + (y1 - qy[k]) * inv;
      if (is_left) { l0 = fmaxf(l0, v0); l1 = fmaxf(l1, v1); }
      if (is_right) { r0 = fminf(r0, v0); r1 = fminf(r1, v1); }
      if (qx[k] == xlo) y_at_xlo = qy[k];
      if (qx[k] == xhi) y_at_xhi = qy[k];
    }
    float xmin = fminf(l0, l1), xmax = fmaxf(r0, r1);
    if (y_at_xlo >= y0 && y_at_xlo <= y1) xmin = xlo;
    if (y_at_xhi >= y0 && y_at_xhi <= y1) xmax = xhi;
    xmin = fmaxf(xmin, xlo);                // rounding of nearly horizontal edges must not leave the rectangle
    xmax = fminf(xmax, xhi);
    ts = max((int)floorf(xmin - M) >> 4, 0);
    te = min((int)ceilf(xmax + M) >> 4, ntx - 1);
  }
  return (uint32_t)(ts | (te << 8));
}

// ---- the two state kernels of a step --------------------------------------------------------------------------------
// PlanEnv.step (envs/base/env.py:334-361) up to the observation is two launches, split by the shape of the work:
//
//   move_kernel    one THREAD per env.  Everything that is scalar per env and one long dependent chain: control delay
//                  (:371-373), robot model (tricycle_model.py:478-538 / differential_drive.py:236-265) with Philox
//                  noise, footprint lookup, pose_collides (env.py:464-489; collide_warp_balanced: batched loads of the
//                  non-empty lethal tiles under the footprint only), rollback (:458-459), pose / robot-state delay lines
//                  (:377-389), time / iter / sticky collision (:383-393), the compact observation and the 128-byte
//                  record of the egocentric kernel.  Every state access is a coalesced SoA row.  It leaves a 144-byte
//                  StepRecord per env for
//   reward_kernel  eight LANES per env.  The one gather that wants lanes: find_last_reached (path_tools.py:408-448) over
//                  the remaining path, lanes <-> points, chunk-culled; then the group's first lane finishes the step: reward
//                  (reward.py:214-259 / :331-350), done (env.py:407-419), episode statistics, goal_n_state
//                  (egocentric.py:152-159; the pose's inverse transform comes precomputed in the record), and the rare
//                  auto-reset (env.py:293-303), which rewrites the env's rows and its egocentric record from the
//                  initial state.
//
// Round 1 ran three kernels (kin: thread, collide + reward: warp, commit: two threads per env; 0.158 ms per 65 536
// envs): the collision gather sat in the warp kernel (617 warp instructions per env at 49 % issue), and the commit
// kernel repeated the loads of the first.  A fully fused thread-per-env kernel was built and measured first
// (profiles/r2_notes.md): bit-identical, but its thread-serial reached-index scan pays one memory round trip per
// loop iteration -- 0.090 ms at 256 envs against 0.037 for the three kernels.
struct __align__(16) StepRecord {     // 144 bytes, at the start of the env's slot in BcgBatch.work
  double pose[3];                    // State.pose after this step: the pose the reward sees
  double min_dist;                   // ContinuousRewardProviderState.min_spat_dist_so_far before this step
  double ep_return;                  // before this step's reward
  double ct, st, tx, ty, tt;         // inverse transform of the observed pose (coordinate_transformations.py:57-84)
  int64_t path_off;                  // fp64 offset of the env's path rows
  int32_t path_n, path_pitch, chunk_pitch, target;
  int32_t flags, iter_after;
  float drobot[6];                   // delayed robot state x, y, th, v, w, wheel (goal_n_state's tail)
};
static_assert(sizeof(StepRecord) == 144 && sizeof(StepRecord) <= BCG_WORK_BYTES, "StepRecord is 144 bytes");
static_assert(offsetof(StepRecord, path_off) == 80 && offsetof(StepRecord, chunk_pitch) == 96 && offsetof(StepRecord, drobot) == 112,
              "move_kernel stores the record field by field");
// batches with per-env parameters: env e's spatial / angular precision and progress multiplier (3 doubles), written by
// move_kernel behind the StepRecord so that reward_kernel's lane groups read them with the record, not from the rows
#define BCG_SR_ENV_OFF 144
static_assert(BCG_SR_ENV_OFF >= sizeof(StepRecord) && BCG_SR_ENV_OFF + 24 <= BCG_WORK_BYTES, "per-env fields fit the work slot");
__device__ __forceinline__ BcgParams with_slot_precision(const BcgParams& p, const uint8_t* fields) {
  BcgParams q = p;
  const double2 prec = reinterpret_cast<const double2*>(fields)[0];
  q.spatial_precision = prec.x;
  q.angular_precision = prec.y;
  q.progress_multiplier = reinterpret_cast<const double*>(fields)[2];
  return q;
}
#define BCG_SR_HIT 1
#define BCG_SR_COLLIDED_AFTER 2
#define BCG_SR_TIMED_OUT 4
#define BCG_SR_DONE_BEFORE 8
#define BCG_SR_GOAL_BEFORE 16

#ifndef BCG_MOVE_THREADS
#define BCG_MOVE_THREADS 64
#endif
#ifndef BCG_MOVE_MIN_BLOCKS
#define BCG_MOVE_MIN_BLOCKS 8         // register budget: 65536 / (threads x blocks) = 128
#endif
#ifndef BCG_MOVE_FEW_BLOCKS
#define BCG_MOVE_FEW_BLOCKS 6         // the build used when the batch fits one wave of it: 168 registers
#endif
#ifndef BCG_MOVE_FEWER_BLOCKS
#define BCG_MOVE_FEWER_BLOCKS 4       // ... and when it fits one wave of 256 per SM: 230 registers, nothing spilled
#endif
#ifndef BCG_REWARD_THREADS
#define BCG_REWARD_THREADS 64
#endif
#ifndef BCG_REWARD_RESIDENT
#define BCG_REWARD_RESIDENT 1024      // threads per SM the reward kernel is compiled for (register budget 64)
#endif

// the inverse transform of pose (px, py, pth), as write_goal_n_state evaluates it
__device__ __forceinline__ void inverse_transform(double px, double py, double pth, double& ct, double& st, double& tx,
                                                  double& ty, double& tt) {
  double sn, cs;
  sincos(pth, &sn, &cs);
  tx = -px * cs - py * sn;
  ty = px * sn - py * cs;
  tt = wrap_angle(-pth);
  sincos(tt, &st, &ct);
}

// goal_n_state (envs/egocentric.py:141-160) from the precomputed inverse transform; same arithmetic as write_goal_n_state
__device__ __forceinline__ void write_goal_from_transform(const BcgParams& p, const double* __restrict__ P, int pitch, int n,
                                                          int target, double ct, double st, double tx, double ty, double tt,
                                                          const float drobot[6], float* __restrict__ g) {
  if (target > n - 1) {
#pragma unroll
    for (int k = 0; k < 9; ++k) g[k] = 0.f;
    return;
  }
  const int gi = goal_point_index(p, n, target);
  const double gx = P[gi], gy = P[pitch + gi], gt = P[2 * pitch + gi];
  const double ex = ct * gx - st * gy + tx;
  const double ey = st * gx + ct * gy + ty;
  const double ea = wrap_angle(gt + tt);
  if (p.ego_variant == 1) {
    const double nx = ex / p.ego_world_w, ny = ey / p.ego_world_h;
    const double nrm = sqrt(nx * nx + ny * ny);
    g[0] = (float)(nx / nrm);
    g[1] = (float)(ny / nrm);
    g[2] = drobot[3];
    g[3] = drobot[4];
    g[4] = drobot[5];
    g[5] = g[6] = g[7] = g[8] = 0.f;
    return;
  }
  g[0] = (float)clampd(ex / p.ego_world_w, -1.0, 1.0);
  g[1] = (float)clampd(ey / p.ego_world_h, -1.0, 1.0);
  g[2] = (float)ea;
#pragma unroll
  for (int k = 0; k < 6; ++k) g[3 + k] = drobot[k];
}

// MIN_BLOCKS is the register budget: 8 CTAs per SM = 128 registers (1 024 envs in flight per SM: the large batch needs
// the warps), 6 = 168 registers (no spills; ~3.5 us less on the chain when the whole batch fits one wave of 384 per SM).
// ROWS: the batch has per-env parameters (`rows`, unused otherwise).  `p` then carries env e's own values, loaded with
// the env's other top-of-kernel loads, and the goal tolerances and the progress multiplier are forwarded to
// reward_kernel at BCG_SR_ENV_OFF of the work slot.  (The copy is kept in the kernel body, not behind a function call:
// that way the instantiation without rows compiles to the same instructions as before rows existed.)
// ENDS: the step reports episode ends (BcgEpisodeEnds, appended behind the other parameters so that their offsets, and
// the instructions of the instantiation without it, stay as they were).  Its counters are zeroed here, after the wait:
// the previous step's egocentric kernel reads them, and the caller reads them after this step.
template <int MIN_BLOCKS, bool ROWS, bool ENDS>
__global__ void __launch_bounds__(BCG_MOVE_THREADS, MIN_BLOCKS)
move_kernel(const BcgParams p_batch, const BcgBatch b, const BcgStateLayout L, const void* __restrict__ actions,
            const int action_is_f64, const uint64_t step_index_arg, const BcgStepOut out, const int ego_cap,
            const BcgEnvRows rows, int32_t* const ends_count) {
  pdl_wait();                                            // the previous step's kernels are done with the records and rows
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= b.n_envs) return;
  const BcgParams p = ROWS ? with_env_rows(p_batch, rows, b.n_envs, e) : p_batch;
  const int64_t N = b.n_envs;
  const uint64_t step_index = b.step_counter ? *reinterpret_cast<const volatile uint64_t*>(b.step_counter) : step_index_arg;
  if (e == 0 && b.ego_list) b.ego_list[N] = b.ego_list[N + 1] = 0;       // hand-over count, env counter of the sparse kernel
  if (ENDS && e == 0) ends_count[0] = ends_count[1] = 0;                 // episode ends, their hand-over count
  double* const sf = b.state_f + e;
  int32_t* const si = b.state_i + e;
  // ---- everything that is read from rows (independent loads, issued together) ----------------------------------------
  double u[2];
  if (action_is_f64) {
    const double2 a = reinterpret_cast<const double2*>(actions)[e];
    u[0] = a.x;
    u[1] = a.y;
  } else {
    const float2 a = reinterpret_cast<const float2*>(actions)[e];
    u[0] = (double)a.x;
    u[1] = (double)a.y;
  }
  double s[7];
#pragma unroll
  for (int r = 0; r < 7; ++r) s[r] = sf[(BCG_F_ROBOT + r) * N];
  const int map_id = b.map_id[e], path_id = b.path_id[e];
  // the step's normal draws depend on (seed, env, step) alone: Philox + Box-Muller run under the loads above instead of in
  // the middle of the kinematic chain
  const NoiseDraws noise = draw_noise_ahead(p, p.env_id_base + (uint64_t)e, step_index);
  const double time = sf[BCG_F_TIME * N] + p.dt;
  const int target = si[BCG_I_TARGET * N];
  const int collided = si[BCG_I_COLLIDED * N], iter = si[BCG_I_ITER * N];
  int qp = si[BCG_I_QP * N], qs = si[BCG_I_QS * N];
  // the fronts of the pose and robot-state queues (what the delay lines will hand back): loaded here, a round trip early
  double pose_front[3], state_front[7];
  delay_front<3>(sf + (int64_t)L.ring_pose * N, N, qp, p.delay_pose, pose_front);
  delay_front<7>(sf + (int64_t)L.ring_state * N, N, qs, p.delay_state, state_front);
  StepRecord rec;
  rec.min_dist = sf[BCG_F_MIN_DIST * N];
  rec.ep_return = sf[BCG_F_EP_RETURN * N];
  const BcgMapDesc m = b.maps[map_id];
  const BcgPathDesc pdsc = b.paths[path_id];
  bool goal_before = target > pdsc.n - 1;
  if (p.reward_kind == BCG_REWARD_PURE_PURSUIT) {        // reward.py:139-149 on the pose observed before this step
    const double* P = b.path_arena + pdsc.off;
    const double gx = __ldg(P + pdsc.n - 1), gy = __ldg(P + pdsc.pitch + pdsc.n - 1);
    goal_before = hypot(gx - sf[(BCG_F_DPOSE + 0) * N], gy - sf[(BCG_F_DPOSE + 1) * N]) < 1.0;
  }
  const double old_pose[3] = {s[0], s[1], s[2]};
  // ---- env.py:371-373 control delay, then the robot model ------------------------------------------------------------------
  if (p.delay_control > 0) {
    int q = si[BCG_I_QC * N];
    delay_line<2>(sf + (int64_t)L.ring_control * N, N, q, p.delay_control, u);
    si[BCG_I_QC * N] = q;
  }
  robot_step(s, u[0], u[1], p, p.env_id_base + (uint64_t)e, step_index, noise);
  if (b.cand) {                                          // the proposed pose, for the stand-alone collision entry points
#pragma unroll
    for (int r = 0; r < 3; ++r) b.cand[r * N + e] = s[r];
  }
  // ---- env.py:455 pose_collides of the proposed pose --------------------------------------------------------------------------
  const FootBox fb = foot_box(b.lut, m.origin_x, m.origin_y, p.inv_resolution, s[0], s[1], s[2], b.status);
  const bool hit = collide_warp_balanced(b.lut, b.tile_arena, m.tile_off, b.occ_sum_arena + m.sum_off, m.tiles_x, m.width,
                                         m.height, fb, warp_item_mask(e - (int)(threadIdx.x & 31), b.n_envs), threadIdx.x & 31);
  if (hit) {  // env.py:458-459 + tricycle_model.py:471-476: pose restored, v = w = 0, wheel / steer command kept
    s[0] = old_pose[0];
    s[1] = old_pose[1];
    s[2] = old_pose[2];
    s[3] = 0.0;
    s[4] = 0.0;
  }
  // ---- env.py:377-389 pose and robot-state delay lines ------------------------------------------------------------------------
  double dpose[3] = {s[0], s[1], s[2]};
  double dstate[7];
#pragma unroll
  for (int r = 0; r < 7; ++r) dstate[r] = s[r];
  delay_push<3>(sf + (int64_t)L.ring_pose * N, N, qp, p.delay_pose, dpose, pose_front);
  delay_push<7>(sf + (int64_t)L.ring_state * N, N, qs, p.delay_state, dstate, state_front);
  // ---- env.py:383-393: the state rows that do not depend on the reward (reward_kernel writes target, min_dist, return) ---
  const int iter_after = iter + 1;
  const int collided_after = collided | (hit ? 1 : 0);
#pragma unroll
  for (int r = 0; r < 7; ++r) sf[(BCG_F_ROBOT + r) * N] = s[r];
#pragma unroll
  for (int r = 0; r < 7; ++r) sf[(BCG_F_DROBOT + r) * N] = dstate[r];
#pragma unroll
  for (int r = 0; r < 3; ++r) sf[(BCG_F_DPOSE + r) * N] = dpose[r];
  sf[BCG_F_TIME * N] = time;
  si[BCG_I_ITER * N] = iter_after;
  si[BCG_I_COLLIDED * N] = collided_after;
  si[BCG_I_QP * N] = qp;
  si[BCG_I_QS * N] = qs;
  if (out.hit) out.hit[e] = hit ? 1 : 0;
  if (out.obs_vec) {                                     // [11] = target index: reward_kernel
    float* o = out.obs_vec + (int64_t)e * 12;
    reinterpret_cast<float4*>(o)[0] = make_float4((float)dpose[0], (float)dpose[1], (float)dpose[2], (float)dstate[0]);
    reinterpret_cast<float4*>(o)[1] = make_float4((float)dstate[1], (float)dstate[2], (float)dstate[3], (float)dstate[4]);
    o[8] = (float)dstate[5];
    o[9] = (float)dstate[6];
    o[10] = (float)time;
  }
  // ---- what reward_kernel starts from ----------------------------------------------------------------------------------------
  const bool true_pose = p.ego_variant == 1;             // observation about the true robot pose vs the observed (delayed) pose
  const double opx = true_pose ? s[0] : dpose[0], opy = true_pose ? s[1] : dpose[1], opth = true_pose ? s[2] : dpose[2];
  if (out.ego_image) write_ego_tile_record(p, b, e, map_id, m, opx, opy, opth, ego_cap);
  rec.ct = rec.st = rec.tx = rec.ty = rec.tt = 0.0;
  if (out.goal_n_state) inverse_transform(opx, opy, opth, rec.ct, rec.st, rec.tx, rec.ty, rec.tt);
#pragma unroll
  for (int r = 0; r < 3; ++r) rec.pose[r] = dpose[r];
  rec.path_off = pdsc.off;
  rec.path_n = pdsc.n;
  rec.path_pitch = pdsc.pitch;
  rec.chunk_pitch = pdsc.chunk_pitch;
  rec.target = target;
  rec.iter_after = iter_after;
  const bool done_before = goal_before || (iter >= p.iteration_timeout) || (collided != 0);
  rec.flags = (hit ? BCG_SR_HIT : 0) | (collided_after ? BCG_SR_COLLIDED_AFTER : 0) |
              (iter_after >= p.iteration_timeout ? BCG_SR_TIMED_OUT : 0) | (done_before ? BCG_SR_DONE_BEFORE : 0) |
              (goal_before ? BCG_SR_GOAL_BEFORE : 0);
  rec.drobot[0] = (float)dstate[0];
  rec.drobot[1] = (float)dstate[1];
  rec.drobot[2] = (float)dstate[2];
  rec.drobot[3] = (float)dstate[3];
  rec.drobot[4] = (float)dstate[4];
  rec.drobot[5] = (float)dstate[6];
  // (field by field: copying the struct through a uint4 pointer would force it into local memory)
  uint8_t* const dst = reinterpret_cast<uint8_t*>(b.work) + (int64_t)e * BCG_WORK_BYTES;
  double2* d2 = reinterpret_cast<double2*>(dst);
  d2[0] = make_double2(rec.pose[0], rec.pose[1]);
  d2[1] = make_double2(rec.pose[2], rec.min_dist);
  d2[2] = make_double2(rec.ep_return, rec.ct);
  d2[3] = make_double2(rec.st, rec.tx);
  d2[4] = make_double2(rec.ty, rec.tt);
  reinterpret_cast<int4*>(dst + 80)[0] = make_int4((int)(rec.path_off & 0xffffffffll), (int)(rec.path_off >> 32), rec.path_n, rec.path_pitch);
  reinterpret_cast<int4*>(dst + 96)[0] = make_int4(rec.chunk_pitch, rec.target, rec.flags, rec.iter_after);
  reinterpret_cast<float4*>(dst + 112)[0] = make_float4(rec.drobot[0], rec.drobot[1], rec.drobot[2], rec.drobot[3]);
  reinterpret_cast<float2*>(dst + 128)[0] = make_float2(rec.drobot[4], rec.drobot[5]);
  if (ROWS) {
    reinterpret_cast<double2*>(dst + BCG_SR_ENV_OFF)[0] = make_double2(p.spatial_precision, p.angular_precision);
    reinterpret_cast<double*>(dst + BCG_SR_ENV_OFF)[2] = p.progress_multiplier;
  }
}

// auto-reset of env e (env.py:293-303) by its lane group: the rows, the observation and the egocentric record of the
// initial state
// the observation of env e's initial state (init_f / init_i) by one thread: obs_vec, goal_n_state and the egocentric record
__device__ __forceinline__ void write_initial_observation(const BcgParams& p, const BcgBatch& b, const BcgStepOut& out, int e,
                                                          int ego_cap) {
  const int64_t N = b.n_envs;
  double dpose[3], dstate[7], c[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) dpose[r] = b.init_f[(int64_t)(BCG_F_DPOSE + r) * N + e];
#pragma unroll
  for (int r = 0; r < 7; ++r) dstate[r] = b.init_f[(int64_t)(BCG_F_DROBOT + r) * N + e];
#pragma unroll
  for (int r = 0; r < 3; ++r) c[r] = b.init_f[(int64_t)(BCG_F_ROBOT + r) * N + e];
  const int target = b.init_i[(int64_t)BCG_I_TARGET * N + e];
  if (out.obs_vec) {
    float4* o = reinterpret_cast<float4*>(out.obs_vec + (int64_t)e * 12);
    o[0] = make_float4((float)dpose[0], (float)dpose[1], (float)dpose[2], (float)dstate[0]);
    o[1] = make_float4((float)dstate[1], (float)dstate[2], (float)dstate[3], (float)dstate[4]);
    o[2] = make_float4((float)dstate[5], (float)dstate[6], (float)b.init_f[(int64_t)BCG_F_TIME * N + e], (float)target);
  }
  if (out.ego_image || out.goal_n_state) {
    const bool true_pose = p.ego_variant == 1;
    const double opx = true_pose ? c[0] : dpose[0], opy = true_pose ? c[1] : dpose[1], opth = true_pose ? c[2] : dpose[2];
    if (out.ego_image) {
      const int map_id = b.map_id[e];
      write_ego_tile_record(p, b, e, map_id, b.maps[map_id], opx, opy, opth, ego_cap);
    }
    if (out.goal_n_state) write_goal_n_state(p, b, e, b.paths[b.path_id[e]], opx, opy, opth, target, dstate, out.goal_n_state);
  }
}

template <int G>
__device__ __forceinline__ void reset_env_rows(const BcgParams& p, const BcgBatch& b, const BcgStepOut& out, int e, int ego_cap,
                                               unsigned gl) {
  const int64_t N = b.n_envs;
  for (int r = gl; r < b.n_frows; r += G) b.state_f[(int64_t)r * N + e] = b.init_f[(int64_t)r * N + e];
  for (int r = gl; r < b.n_irows; r += G) b.state_i[(int64_t)r * N + e] = b.init_i[(int64_t)r * N + e];
  if (gl != 0) return;
  write_initial_observation(p, b, out, e, ego_cap);
}

// G lanes per env (power of two, 1 < G <= 32): 32 / G envs per warp.  Measured (profiles/r2_notes.md): 65 536 envs G = 8
// 0.045 ms, 16: 0.050, 32: 0.065; 8 192 envs 0.022 / 0.018 / 0.019; 256 envs 0.0147 / 0.0121 / 0.0108 -- a large batch
// wants few warps (the straight-line code is paid per warp), a small one a short chain (a chunk in one round).
// ROWS: the batch has per-env parameters; env e's goal tolerances and progress multiplier come from its work slot, where
// move_kernel left them (in the kernel body for the reason given at move_kernel)
// ENDS: the step reports episode ends (BcgEpisodeEnds): the reason byte of every env and the final record of every env
// whose episode ends now, taken before the auto-reset overwrites its rows and its egocentric record
// With auto_reset == BCG_AUTO_RESET_NEW_WORLD a done env is not reset here: it is appended to BcgWorldGen.list, and
// regenerate_kernel gives it a new world, its initial state and its initial observation.
template <int G, bool ROWS, bool ENDS>
__global__ void __launch_bounds__(BCG_REWARD_THREADS, BCG_REWARD_RESIDENT / BCG_REWARD_THREADS)
reward_kernel(const BcgParams p_batch, const BcgBatch b, const BcgStepOut out, const int ego_cap, const BcgEpisodeEnds ends) {
  pdl_wait();                                            // move_kernel's records
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  const unsigned lane = threadIdx.x & 31, gl = lane & (G - 1);
  const bool active = e < b.n_envs;
  const int64_t N = b.n_envs;
  {
    // the env's record: a group-uniform 144-byte read (env 0's for the idle groups of the last warp)
    const uint8_t* const slot = reinterpret_cast<const uint8_t*>(b.work) + (int64_t)(active ? e : 0) * BCG_WORK_BYTES;
    const StepRecord rec = *reinterpret_cast<const StepRecord*>(slot);
    const BcgParams p = ROWS ? with_slot_precision(p_batch, slot + BCG_SR_ENV_OFF) : p_batch;
    PathRef pd;
    pd.P = b.path_arena + rec.path_off;
    pd.C = pd.P + 5 * (int64_t)rec.path_pitch;
    pd.n = rec.path_n;
    pd.pitch = rec.path_pitch;
    pd.chunk_pitch = rec.chunk_pitch;
    int target = rec.target;
    double min_dist = rec.min_dist;
    const bool pursuit = p.reward_kind == BCG_REWARD_PURE_PURSUIT;
    const bool goal_before = (rec.flags & BCG_SR_GOAL_BEFORE) != 0;
    // issued before the scan needs them: the goal point the reward most likely uses
    double gx = 0.0, gy = 0.0;
    if (pursuit || !goal_before) {
      const int gi = pursuit ? pd.n - 1 : target;
      gx = __ldg(pd.P + gi);
      gy = __ldg(pd.P + pd.pitch + gi);
    }
    double reward = 0.0;
    bool goal;
    if (pursuit) {
      // ContinuousRewardPurePursuitProvider.reward (reward.py:331-350)
      target = first_beyond_radius_group<G>(pd, target, rec.pose[0], rec.pose[1], 2.0, lane, active);
      const double d = hypot(gx - rec.pose[0], gy - rec.pose[1]);
      reward = -0.05;
      reward += min_dist - d;
      if (rec.flags & BCG_SR_COLLIDED_AFTER) reward -= 100;
      min_dist = d;
      goal = d < 1.0;
    } else {
      // (every group of the warp calls the scan: its loops and ballots are warp-uniform)
      const int last = last_reached_group<G>(p, pd, target, rec.pose[0], rec.pose[1], rec.pose[2], lane, active && !goal_before);
      if (!goal_before) {
        if (last >= target) {
          target = last + 1;
          if (target > pd.n - 1) {
            min_dist = 0.0;
          } else {
            min_dist = hypot(__ldg(pd.P + target) - rec.pose[0], __ldg(pd.P + pd.pitch + target) - rec.pose[1]);
          }
          reward = 1.0;
        } else {
          const double d = hypot(gx - rec.pose[0], gy - rec.pose[1]);
          if (d < min_dist) {
            reward = (min_dist - d) * p.progress_multiplier;
            min_dist = d;
          }
        }
      }
      goal = target > pd.n - 1;
    }
    // ---- env.py:407-419 done, statistics, outputs ---------------------------------------------------------------------------
    const bool timed_out = (rec.flags & BCG_SR_TIMED_OUT) != 0, collided_after = (rec.flags & BCG_SR_COLLIDED_AFTER) != 0;
    const bool done = goal || timed_out || collided_after;
    const double ep_return = rec.ep_return + reward;
    if (active && gl == 0) {
      if (out.reward) out.reward[e] = reward;
      if (out.done) out.done[e] = done ? 1 : 0;
      if (done && !(rec.flags & BCG_SR_DONE_BEFORE)) {
        atomicAdd(b.stats + BCG_STAT_EPISODES, 1.0);
        atomicAdd(b.stats + BCG_STAT_RETURN, ep_return);
        atomicAdd(b.stats + BCG_STAT_LENGTH, (double)rec.iter_after);
        if (collided_after) atomicAdd(b.stats + BCG_STAT_COLLIDED, 1.0);
        if (goal) atomicAdd(b.stats + BCG_STAT_GOAL, 1.0);
        if (timed_out) atomicAdd(b.stats + BCG_STAT_TIMEOUT, 1.0);
      }
    }
    if (ENDS && active) {
      // (done, and with it `ended`, is uniform over the env's lane group)
      const bool ended = done && !(rec.flags & BCG_SR_DONE_BEFORE);
      int slot = -1;
      if (gl == 0) {
        const int causes = (goal ? BCG_END_GOAL : 0) | (collided_after ? BCG_END_COLLIDED : 0) | (timed_out ? BCG_END_TIMEOUT : 0);
        ends.reason[e] = (uint8_t)((done ? causes : 0) | (ended ? BCG_END_NOW : 0));
        if (ended) {
          const int k = atomicAdd(ends.count, 1);
          slot = k < ends.capacity ? k : -1;
          // the observation as move_kernel left it in the rows (the obs_vec fields) and the post-step target
          const double* const sf = b.state_f + e;
          float4* const o = reinterpret_cast<float4*>(ends.final_obs_vec + (int64_t)e * 12);
          o[0] = make_float4((float)sf[(BCG_F_DPOSE + 0) * N], (float)sf[(BCG_F_DPOSE + 1) * N], (float)sf[(BCG_F_DPOSE + 2) * N],
                             (float)sf[(BCG_F_DROBOT + 0) * N]);
          o[1] = make_float4((float)sf[(BCG_F_DROBOT + 1) * N], (float)sf[(BCG_F_DROBOT + 2) * N], (float)sf[(BCG_F_DROBOT + 3) * N],
                             (float)sf[(BCG_F_DROBOT + 4) * N]);
          o[2] = make_float4((float)sf[(BCG_F_DROBOT + 5) * N], (float)sf[(BCG_F_DROBOT + 6) * N], (float)sf[BCG_F_TIME * N], (float)target);
          if (out.goal_n_state)
            write_goal_from_transform(p, pd.P, pd.pitch, pd.n, target, rec.ct, rec.st, rec.tx, rec.ty, rec.tt, rec.drobot,
                                      ends.final_goal_n_state + (int64_t)e * 9);
          ends.final_return[e] = ep_return;
          ends.final_length[e] = rec.iter_after;
        }
        ends.final_slot[e] = slot;
      }
      if (ended) {
        const unsigned gmask = (0xffffffffu >> (32 - G)) << (lane & ~(unsigned)(G - 1));
        if (out.ego_image) {
          // the env's egocentric record, 16 bytes per lane, into its slot
          slot = __shfl_sync(gmask, slot, (int)(lane & ~(unsigned)(G - 1)));
          if (slot >= 0) {
            const uint4* const src = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(b.ego_work) + (int64_t)e * BCG_EGO_WORK_BYTES);
            uint4* const dst = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(ends.final_ego_work) + (int64_t)slot * BCG_EGO_WORK_BYTES);
            for (int k = gl; k < BCG_EGO_WORK_BYTES / 16; k += G) dst[k] = src[k];
          }
        }
        __syncwarp(gmask);                               // the record and the rows are read before the reset rewrites them
      }
    }
    if (active && done && p.auto_reset) {
      if (p.auto_reset != BCG_AUTO_RESET_NEW_WORLD) {
        reset_env_rows<G>(p, b, out, e, ego_cap, gl);
      } else if (gl == 0) {
        // a new world: regenerate_kernel, launched behind this kernel, rewrites the rows and the observation (the final
        // record above still read the old episode)
        const BcgWorldGen* const wg = b.world_gen;
        wg->list[atomicAdd(wg->count, 1)] = e;
      }
    } else if (active && gl == 0) {
      b.state_f[BCG_F_MIN_DIST * N + e] = min_dist;
      b.state_f[BCG_F_EP_RETURN * N + e] = ep_return;
      b.state_i[BCG_I_TARGET * N + e] = target;
      if (out.obs_vec) out.obs_vec[(int64_t)e * 12 + 11] = (float)target;
      if (out.goal_n_state)
        write_goal_from_transform(p, pd.P, pd.pitch, pd.n, target, rec.ct, rec.st, rec.tx, rec.ty, rec.tt, rec.drobot,
                                  out.goal_n_state + (int64_t)e * 9);
    }
  }
  // device-side step counter (CUDA-graph replays cannot change a kernel argument): the last CTA to finish bumps it
  if (b.step_counter) {
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      unsigned long long* const ctr = reinterpret_cast<unsigned long long*>(b.step_counter);
      const unsigned long long ticket = atomicAdd(ctr + 1, 1ull);
      if (ticket == (unsigned long long)gridDim.x - 1ull) {
        ctr[1] = 0ull;
        ctr[0] = ctr[0] + 1ull;
      }
    }
  }
}

// make_initial_state (env.py:179-214) + generate_initial_state (reward.py:261-288) of env e by one warp
__device__ __forceinline__ void init_env_state(const BcgParams& p, const BcgBatch& b, const BcgStateLayout& L, int e,
                                               const PathRef& pd, unsigned lane) {
  const int64_t N = b.n_envs;
  const double* P = pd.P;
  const double x0 = P[0], y0 = P[pd.pitch], t0 = P[2 * pd.pitch];
  int target;
  double min_dist = 0.0;
  if (p.reward_kind == BCG_REWARD_PURE_PURSUIT) {        // reward.py:352-371
    target = 1;
    min_dist = hypot(P[pd.n - 1] - x0, P[pd.pitch + pd.n - 1] - y0);
  } else {
    const int last = last_reached_from<true>(p, pd, 0, x0, y0, t0, lane);   // the generators wrote the rows in this launch
    target = last + 1;
    if (target > pd.n - 1) {
      if (lane == 0) atomicAdd(b.status + BCG_STATUS_PATH_EXHAUSTED, 1u);
    } else {
      min_dist = hypot(P[target] - x0, P[pd.pitch + target] - y0);
    }
  }
  for (int r = lane; r < L.n_frows; r += 32) {
    double v = 0.0;
    if (r == BCG_F_ROBOT + 0 || r == BCG_F_DROBOT + 0 || r == BCG_F_DPOSE + 0) v = x0;
    if (r == BCG_F_ROBOT + 1 || r == BCG_F_DROBOT + 1 || r == BCG_F_DPOSE + 1) v = y0;
    if (r == BCG_F_ROBOT + 2 || r == BCG_F_DROBOT + 2 || r == BCG_F_DPOSE + 2) v = t0;
    if (r == BCG_F_MIN_DIST) v = min_dist;
    b.init_f[(int64_t)r * N + e] = v;
    b.state_f[(int64_t)r * N + e] = v;
  }
  for (int r = lane; r < L.n_irows; r += 32) {
    const int v = (r == BCG_I_TARGET) ? target : 0;
    b.init_i[(int64_t)r * N + e] = v;
    b.state_i[(int64_t)r * N + e] = v;
  }
}

// one warp per env; ROWS: the env's own goal tolerances from `rows`
template <bool ROWS>
__global__ void __launch_bounds__(256) init_kernel(const BcgParams p, const BcgBatch b, const BcgStateLayout L, const BcgEnvRows rows) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned lane = threadIdx.x & 31;
  if (e >= b.n_envs) return;
  if (ROWS)
    init_env_state(with_env_rows(p, rows, b.n_envs, e), b, L, e, path_ref(b, b.paths[b.path_id[e]]), lane);
  else
    init_env_state(p, b, L, e, path_ref(b, b.paths[b.path_id[e]]), lane);
}

// env e of bcg_generate_aisles by the whole CTA (see bcg_generate.cuh): the world of turn `tp` in the env's slots, its path,
// chunk bounds and initial state.  Returns false (CTA-uniform) when the world does not fit the slots: the env is left
// exactly as it was.  ROWS: the initial state uses the env's own goal tolerances
template <bool ROWS>
__device__ __forceinline__ bool aisle_world(const BcgParams& p, const BcgBatch& b, const BcgStateLayout& L, const BcgAisleSlots& slots,
                                            const BcgEnvRows& rows, const int e, const BcgTurnParams& tp, const double path_delta) {
  const int tid = threadIdx.x, nthr = blockDim.x;
  // every thread works the geometry out for itself (a few hundred flops; no broadcast, no barrier)
  const AisleGeometry g = aisle_geometry(tp, p.inv_resolution);
  const RefinedShape shape = refined_shape(g.way, path_delta);
  BcgMapDesc* md = const_cast<BcgMapDesc*>(b.maps) + e;
  BcgPathDesc* pdsc = const_cast<BcgPathDesc*>(b.paths) + e;
  const int pitch = (g.width + 31) & ~31;
  const int tiles_x = pitch >> 5, tiles_y = (g.height + 15) >> 4, ctiles_x = pitch >> 4, ctiles_y = (g.height + 7) >> 3;
  const bool fits = g.width > 0 && g.height > 0 && g.width < 32768 && g.height < 32768 &&
                    (int64_t)g.height * pitch <= slots.map_slot_bytes &&
                    (int64_t)ctiles_x * ctiles_y * 128 <= slots.map_slot_bytes &&
                    (int64_t)tiles_x * tiles_y * 16 <= slots.tile_slot_words && shape.n <= slots.path_pitch &&
                    (shape.n + 31) / 32 <= slots.chunk_pitch;
  if (!fits) {                                  // leave the env exactly as it was
    if (tid == 0) atomicAdd(b.status + BCG_STATUS_SLOT_OVERFLOW, 1u);
    return false;
  }
  AisleGenState* gs = reinterpret_cast<AisleGenState*>(slots.gen_state) + e;
  MapLayout m;
  m.data = const_cast<uint8_t*>(b.map_arena) + md->data_off;
  m.tiles = const_cast<uint32_t*>(b.tile_arena) + md->tile_off;
  m.occ = const_cast<uint32_t*>(b.occ_tile_arena) + md->tile_off;
  m.sum = const_cast<uint32_t*>(b.occ_sum_arena) + md->sum_off;
  m.ctiles = const_cast<uint8_t*>(b.cell_tile_arena) + md->cell_tile_off;
  // ---- erase what the slot holds (with the layout it was drawn in) -------------------------------------------
  if (gs->valid) {
    MapLayout old = m;
    old.pitch = gs->pitch; old.rows = gs->rows; old.tiles_x = gs->tiles_x; old.ctiles_x = gs->ctiles_x;
    for (int k = 0; k < 5; ++k) draw_wall(old, gs->wall[k][0], gs->wall[k][1], gs->wall[k][2], gs->wall[k][3], 0, tid, nthr);
  }
  __syncthreads();                              // erased pixels may be drawn again; gs is about to be rewritten
  // ---- draw the new walls: Wall.render (envs/base/maps.py:27-42), thickness max(1, int(0.05 / res)) = 1 px -------
  m.pitch = pitch; m.rows = g.height; m.tiles_x = tiles_x; m.ctiles_x = ctiles_x;
  int wpx[5][4];
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    wpx[k][0] = world_to_pixel_1d(g.wall[k][0], g.origin_x, p.inv_resolution);
    wpx[k][1] = world_to_pixel_1d(g.wall[k][1], g.origin_y, p.inv_resolution);
    wpx[k][2] = world_to_pixel_1d(g.wall[k][2], g.origin_x, p.inv_resolution);
    wpx[k][3] = world_to_pixel_1d(g.wall[k][3], g.origin_y, p.inv_resolution);
    draw_wall(m, wpx[k][0], wpx[k][1], wpx[k][2], wpx[k][3], 254, tid, nthr);
  }
  if (tid == 0) {
    AisleGenState ns;
    for (int k = 0; k < 5; ++k)
      for (int c = 0; c < 4; ++c) ns.wall[k][c] = wpx[k][c];
    ns.pitch = pitch; ns.rows = g.height; ns.tiles_x = tiles_x; ns.ctiles_x = ctiles_x;
    ns.valid = 1;
    for (int k = 0; k < 7; ++k) ns.pad[k] = 0;
    *gs = ns;
    md->origin_x = g.origin_x; md->origin_y = g.origin_y;
    md->height = g.height; md->width = g.width; md->pitch = pitch;
    md->tiles_x = tiles_x; md->tiles_y = tiles_y; md->ctiles_x = ctiles_x; md->ctiles_y = ctiles_y;
    md->flags = BCG_MAP_ONLY_LETHAL;           // walls are the only occupied cells
    md->occupied = 0;                          // (a few hundred: far below the dense threshold)
    pdsc->n = shape.n;
    pdsc->pitch = slots.path_pitch;
    pdsc->n_chunks = (shape.n + 31) / 32;
    pdsc->chunk_pitch = slots.chunk_pitch;
    pdsc->chunk_off = pdsc->off + 5 * (int64_t)slots.path_pitch;
    if (slots.params_out) slots.params_out[e] = tp;
  }
  // ---- refined path rows x, y, th, cos th, sin th ------------------------------------------------------------------
  double* P = const_cast<double*>(b.path_arena) + pdsc->off;
  const int pp = slots.path_pitch;
  for (int i = tid; i < shape.n; i += nthr) {
    double x, y, th, sn, cs;
    refined_point(g.way, shape, i, x, y, th);
    sincos(th, &sn, &cs);
    P[i] = x; P[pp + i] = y; P[2 * pp + i] = th; P[3 * pp + i] = cs; P[4 * pp + i] = sn;
  }
  __syncthreads();                              // the path rows are visible to the whole CTA
  // ---- bounding circles of 32-point chunks (conservative; see last_reached_from) ----------------------------------
  double* Cb = P + 5 * (int64_t)pp;
  const int warp = tid >> 5, lane = tid & 31, nwarp = nthr >> 5;
  for (int c = warp; c * 32 < shape.n; c += nwarp) {
    const int i = min(c * 32 + lane, shape.n - 1);
    const double x = P[i], y = P[pp + i];
    double xlo = x, xhi = x, ylo = y, yhi = y;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      xlo = fmin(xlo, __shfl_xor_sync(BCG_FULL, xlo, o)); xhi = fmax(xhi, __shfl_xor_sync(BCG_FULL, xhi, o));
      ylo = fmin(ylo, __shfl_xor_sync(BCG_FULL, ylo, o)); yhi = fmax(yhi, __shfl_xor_sync(BCG_FULL, yhi, o));
    }
    const double ctx = 0.5 * (xlo + xhi), cty = 0.5 * (ylo + yhi);
    double rad = hypot(x - ctx, y - cty);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rad = fmax(rad, __shfl_xor_sync(BCG_FULL, rad, o));
    if (lane == 0) {
      Cb[c] = ctx; Cb[slots.chunk_pitch + c] = cty; Cb[2 * slots.chunk_pitch + c] = rad * (1 + 1e-12) + 1e-9;
    }
  }
  __syncthreads();
  // ---- initial state ----------------------------------------------------------------------------------------------
  if (warp == 0) {
    PathRef pr;
    pr.P = P; pr.C = Cb; pr.n = shape.n; pr.pitch = pp; pr.chunk_pitch = slots.chunk_pitch;
    if (ROWS)
      init_env_state(with_env_rows(p, rows, b.n_envs, e), b, L, e, pr, lane);
    else
      init_env_state(p, b, L, e, pr, lane);
  }
  return true;
}

// bcg_generate_aisles: one CTA per env
template <bool ROWS>
__global__ void __launch_bounds__(256) generate_aisles_kernel(const BcgParams p, const BcgBatch b, const BcgStateLayout L,
                                                              const BcgAisleSlots slots, const uint8_t* __restrict__ mask,
                                                              const BcgTurnParams* __restrict__ turn_params,
                                                              const uint64_t draw_index, const double path_delta,
                                                              const BcgEnvRows rows) {
  const int e = blockIdx.x;
  if (mask && !mask[e]) return;
  const BcgTurnParams tp = turn_params ? turn_params[e] : draw_turn_params(p.seed, p.env_id_base + (uint64_t)e, draw_index);
  aisle_world<ROWS>(p, b, L, slots, rows, e, tp, path_delta);
}

// env e of bcg_generate_minis by the whole CTA.  Thread 0 samples (the draw count depends on the data), the CTA rasterises
// the two walls, warp 0 checks the two end poses against them; accepted parameters get their path and initial state.
// Returns (CTA-uniform) 1 when a world was accepted, 0 when a world did not fit the slots, -1 when the sampler ran out of
// tries; the status word of either failure is counted.
__device__ __forceinline__ int mini_world(const BcgParams& p, const BcgBatch& b, const BcgStateLayout& L, const BcgAisleSlots& slots,
                                          const BcgMiniGenParams& g, const BcgMiniParams* __restrict__ explicit_params,
                                          BcgMiniParams* __restrict__ params_out, const int e, const uint64_t draw_index,
                                          const double path_delta) {
  const int tid = threadIdx.x, nthr = blockDim.x, warp = tid >> 5, lane = tid & 31;
  __shared__ BcgMiniParams mp_s;
  __shared__ int verdict_s;          // 1 drawn / accepted, 0 draw again, -1 give up
  BcgMapDesc* md = const_cast<BcgMapDesc*>(b.maps) + e;
  BcgPathDesc* pdsc = const_cast<BcgPathDesc*>(b.paths) + e;
  AisleGenState* gs = reinterpret_cast<AisleGenState*>(slots.gen_state) + e;
  MapLayout m;
  m.data = const_cast<uint8_t*>(b.map_arena) + md->data_off;
  m.tiles = const_cast<uint32_t*>(b.tile_arena) + md->tile_off;
  m.occ = const_cast<uint32_t*>(b.occ_tile_arena) + md->tile_off;
  m.sum = const_cast<uint32_t*>(b.occ_sum_arena) + md->sum_off;
  m.ctiles = const_cast<uint8_t*>(b.cell_tile_arena) + md->cell_tile_off;
  MiniRng rng = {p.seed, p.env_id_base + (uint64_t)e, draw_index, 0u};
  bool accepted = false;
  for (int attempt = 0; attempt < 1000 && !accepted; ++attempt) {
    if (tid == 0) {
      int rc = 1;
      if (explicit_params) mp_s = explicit_params[e];
      else rc = draw_mini_params(rng, g, mp_s);
      verdict_s = rc;
    }
    __syncthreads();
    const int drawn = verdict_s;
    __syncthreads();                              // verdict_s is rewritten below
    if (drawn < 0) break;                         // the square method found no pose: "the sampling space looks empty"
    if (drawn == 0) continue;                     // SpaceSeemsEmptyError of the circle method: draw again
    // ---- CostMap2D.create_empty(world_size=(h, w), origin=(-h/2, -w/2)) and the two walls (mini_env.py:364-389) ----
    const double origin_x = -mp_s.h / 2., origin_y = -mp_s.w / 2.;
    const int width = world_to_pixel_1d(mp_s.h, 0.0, p.inv_resolution), height = world_to_pixel_1d(mp_s.w, 0.0, p.inv_resolution);
    const int pitch = (width + 31) & ~31;
    const int tiles_x = pitch >> 5, tiles_y = (height + 15) >> 4, ctiles_x = pitch >> 4, ctiles_y = (height + 7) >> 3;
    const double dxp = mp_s.end[0] - mp_s.start[0], dyp = mp_s.end[1] - mp_s.start[1];
    const double dist = sqrt(dxp * dxp + dyp * dyp);
    const int n_path = dist > path_delta ? (int)(dist / path_delta) + 2 : 2;        // refine_path of a two-point path
    const bool fits = width > 0 && height > 0 && width < 32768 && height < 32768 &&
                      (int64_t)height * pitch <= slots.map_slot_bytes && (int64_t)ctiles_x * ctiles_y * 128 <= slots.map_slot_bytes &&
                      (int64_t)tiles_x * tiles_y * 16 <= slots.tile_slot_words && n_path <= slots.path_pitch &&
                      (n_path + 31) / 32 <= slots.chunk_pitch;
    if (!fits) {
      if (tid == 0) atomicAdd(b.status + BCG_STATUS_SLOT_OVERFLOW, 1u);
      return 0;                                   // (before anything of the slot was touched in this attempt)
    }
    if (gs->valid) {                              // erase what the slot holds, with the layout it was drawn in
      MapLayout old = m;
      old.pitch = gs->pitch; old.rows = gs->rows; old.tiles_x = gs->tiles_x; old.ctiles_x = gs->ctiles_x;
      for (int k = 0; k < 5; ++k)
        draw_wall_clipped(old, gs->pad[0], gs->rows, gs->wall[k][0], gs->wall[k][1], gs->wall[k][2], gs->wall[k][3], 0, tid, nthr);
    }
    __syncthreads();
    m.pitch = pitch; m.rows = height; m.tiles_x = tiles_x; m.ctiles_x = ctiles_x;
    int wpx[2][4];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const double* far = k == 0 ? mp_s.a : mp_s.b;
      wpx[k][0] = world_to_pixel_1d(mp_s.o[0], origin_x, p.inv_resolution);
      wpx[k][1] = world_to_pixel_1d(mp_s.o[1], origin_y, p.inv_resolution);
      wpx[k][2] = world_to_pixel_1d(far[0], origin_x, p.inv_resolution);
      wpx[k][3] = world_to_pixel_1d(far[1], origin_y, p.inv_resolution);
      draw_wall_clipped(m, width, height, wpx[k][0], wpx[k][1], wpx[k][2], wpx[k][3], 254, tid, nthr);
    }
    if (tid == 0) {
      AisleGenState ns;
      for (int k = 0; k < 5; ++k)
        for (int c = 0; c < 4; ++c) ns.wall[k][c] = k < 2 ? wpx[k][c] : -1;      // (-1, -1)-(-1, -1) clips to nothing
      ns.pitch = pitch; ns.rows = height; ns.tiles_x = tiles_x; ns.ctiles_x = ctiles_x;
      ns.valid = 1;
      for (int k = 0; k < 7; ++k) ns.pad[k] = 0;
      ns.pad[0] = width;                          // the clip rectangle of the walls drawn
      *gs = ns;
      md->origin_x = origin_x; md->origin_y = origin_y;
      md->height = height; md->width = width; md->pitch = pitch;
      md->tiles_x = tiles_x; md->tiles_y = tiles_y; md->ctiles_x = ctiles_x; md->ctiles_y = ctiles_y;
      md->flags = BCG_MAP_ONLY_LETHAL;
      md->occupied = 0;
    }
    __syncthreads();                              // walls, planes and the descriptor are visible to the CTA
    // ---- the final check of _sample_mini_env_params (:336-358): both end poses free, not within the goal tolerances ----
    if (warp == 0) {
      bool ok = true;
      if (!explicit_params) {
        const WorkCollide w0 = make_work_collide(p, b, e, mp_s.start[0], mp_s.start[1], mp_s.start[2]);
        const WorkCollide w1 = make_work_collide(p, b, e, mp_s.end[0], mp_s.end[1], mp_s.end[2]);
        const bool hit0 = collide_tiles<false, true>(b, w0, lane, nullptr);
        const bool hit1 = collide_tiles<false, true>(b, w1, lane, nullptr);
        const double cart = hypot(mp_s.start[0] - mp_s.end[0], mp_s.start[1] - mp_s.end[1]);
        const double ang = fabs(wrap_angle(mp_s.start[2] - mp_s.end[2]));
        const bool too_close = cart < g.goal_spat_dist && ang < g.goal_ang_dist;
        ok = !(hit0 || hit1) && !too_close;
      }
      if (lane == 0) verdict_s = ok ? 1 : 0;
    }
    __syncthreads();
    accepted = verdict_s == 1;
    __syncthreads();
    if (!accepted) continue;
    // ---- accepted: refined path (path_tools.py:178-240 for two way points), chunk bounds, initial state ----------------
    double* P = const_cast<double*>(b.path_arena) + pdsc->off;
    const int pp = slots.path_pitch;
    if (tid == 0) {
      pdsc->n = n_path;
      pdsc->pitch = pp;
      pdsc->n_chunks = (n_path + 31) / 32;
      pdsc->chunk_pitch = slots.chunk_pitch;
      pdsc->chunk_off = pdsc->off + 5 * (int64_t)pp;
      if (params_out) params_out[e] = mp_s;
    }
    {
      const double div = (double)(n_path - 1);    // np.linspace(start, end, num)[:-1] then the end point itself
      const double sx = dxp / div, sy = dyp / div;
      double sn0, cs0, sn1, cs1;
      sincos(mp_s.start[2], &sn0, &cs0);
      sincos(mp_s.end[2], &sn1, &cs1);
      for (int i = tid; i < n_path; i += nthr) {
        const bool last = i == n_path - 1;
        const bool refined = dist > path_delta;
        const double x = last ? mp_s.end[0] : (refined ? (double)i * sx + mp_s.start[0] : mp_s.start[0]);
        const double y = last ? mp_s.end[1] : (refined ? (double)i * sy + mp_s.start[1] : mp_s.start[1]);
        P[i] = x; P[pp + i] = y;
        P[2 * pp + i] = last ? mp_s.end[2] : mp_s.start[2];
        P[3 * pp + i] = last ? cs1 : cs0;
        P[4 * pp + i] = last ? sn1 : sn0;
      }
    }
    __syncthreads();
    double* Cb = P + 5 * (int64_t)pp;
    const int nwarp = nthr >> 5;
    for (int c = warp; c * 32 < n_path; c += nwarp) {
      const int i = min(c * 32 + lane, n_path - 1);
      const double x = P[i], y = P[pp + i];
      double xlo = x, xhi = x, ylo = y, yhi = y;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        xlo = fmin(xlo, __shfl_xor_sync(BCG_FULL, xlo, o)); xhi = fmax(xhi, __shfl_xor_sync(BCG_FULL, xhi, o));
        ylo = fmin(ylo, __shfl_xor_sync(BCG_FULL, ylo, o)); yhi = fmax(yhi, __shfl_xor_sync(BCG_FULL, yhi, o));
      }
      const double ctx = 0.5 * (xlo + xhi), cty = 0.5 * (ylo + yhi);
      double rad = hypot(x - ctx, y - cty);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) rad = fmax(rad, __shfl_xor_sync(BCG_FULL, rad, o));
      if (lane == 0) {
        Cb[c] = ctx; Cb[slots.chunk_pitch + c] = cty; Cb[2 * slots.chunk_pitch + c] = rad * (1 + 1e-12) + 1e-9;
      }
    }
    __syncthreads();
    if (warp == 0) {
      PathRef pr;
      pr.P = P; pr.C = Cb; pr.n = n_path; pr.pitch = pp; pr.chunk_pitch = slots.chunk_pitch;
      init_env_state(p, b, L, e, pr, lane);
    }
  }
  if (!accepted && tid == 0) atomicAdd(b.status + BCG_STATUS_SAMPLER_EMPTY, 1u);
  return accepted ? 1 : -1;
}

// bcg_generate_minis: one CTA per env
__global__ void __launch_bounds__(128) generate_minis_kernel(const BcgParams p, const BcgBatch b, const BcgStateLayout L,
                                                             const BcgAisleSlots slots, const uint8_t* __restrict__ mask,
                                                             const BcgMiniGenParams g, const BcgMiniParams* __restrict__ explicit_params,
                                                             BcgMiniParams* __restrict__ params_out, const uint64_t draw_index,
                                                             const double path_delta) {
  const int e = blockIdx.x;
  if (mask && !mask[e]) return;
  mini_world(p, b, L, slots, g, explicit_params, params_out, e, draw_index, path_delta);
}

__global__ void __launch_bounds__(256) reset_kernel(const BcgBatch b, const uint8_t* __restrict__ mask) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= b.n_envs) return;
  if (mask && !mask[e]) return;
  const int64_t N = b.n_envs;
  for (int r = 0; r < b.n_frows; ++r) b.state_f[(int64_t)r * N + e] = b.init_f[(int64_t)r * N + e];
  for (int r = 0; r < b.n_irows; ++r) b.state_i[(int64_t)r * N + e] = b.init_i[(int64_t)r * N + e];
}

// lethal bit-plane: bit x&31 of word ((ty*tiles_x + tx)*16 + (y&15)) <-> costmap[y][x] == 254
__global__ void __launch_bounds__(256) tiles_kernel(const BcgBatch b, const int first) {
  const BcgMapDesc m = b.maps[first + blockIdx.y];
  const int words = m.tiles_x * m.tiles_y * 16;
  uint32_t* dst = const_cast<uint32_t*>(b.tile_arena) + m.tile_off;
  uint32_t* occ = const_cast<uint32_t*>(b.occ_tile_arena) + m.tile_off;
  uint32_t* sum = const_cast<uint32_t*>(b.occ_sum_arena) + m.sum_off;
  const uint8_t* src = b.map_arena + m.data_off;
  bool other = false;                      // a cell that is neither free (0) nor lethal (254)
  int occupied = 0;
  for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < words; w += gridDim.x * blockDim.x) {
    const int tile = w >> 4, r = w & 15;
    const int ty = tile / m.tiles_x, tx = tile - ty * m.tiles_x;
    const int y = (ty << 4) + r;
    uint32_t bits = 0, obits = 0;
    if (y < m.height) {
      const uint4* row = reinterpret_cast<const uint4*>(src + (int64_t)y * m.pitch + (tx << 5));
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint4 v = row[h];
        const uint32_t ws[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t eq = __vcmpeq4(ws[k], 0xFEFEFEFEu) & 0x01010101u;  // bit 0 of each byte
          const uint32_t nz = __vcmpne4(ws[k], 0u) & 0x01010101u;
          const uint32_t nib = (eq * 0x10204080u) >> 28;                    // gather to 4 bits
          const uint32_t onib = (nz * 0x10204080u) >> 28;
          bits |= nib << (h * 16 + k * 4);
          obits |= onib << (h * 16 + k * 4);
        }
      }
      const int over = (tx << 5) + 32 - m.width;
      if (over > 0) {
        const uint32_t keep = (over >= 32) ? 0u : (0xffffffffu >> over);
        bits &= keep;
        obits &= keep;
      }
      other |= (obits != bits);
      occupied += __popc(obits);
    }
    dst[w] = bits;
    occ[w] = obits;
    if (obits) {                             // the tile holds a cell (rows race for the same bit: test before the atomic)
      uint32_t* const sw = sum + ty * ((m.tiles_x + 31) >> 5) + (tx >> 5);
      if ((*(volatile uint32_t*)sw & (1u << (tx & 31))) == 0u) atomicOr(sw, 1u << (tx & 31));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) occupied += __shfl_xor_sync(BCG_FULL, occupied, o);
  if ((threadIdx.x & 31) == 0 && occupied) atomicAdd(&const_cast<BcgMapDesc*>(b.maps)[first + blockIdx.y].occupied, occupied);
  if (__any_sync(BCG_FULL, other) && (threadIdx.x & 31) == 0)
    atomicAnd(&const_cast<BcgMapDesc*>(b.maps)[first + blockIdx.y].flags, ~BCG_MAP_ONLY_LETHAL);
}

__global__ void __launch_bounds__(256) zero_occupied_kernel(const BcgBatch b, const int first, const int count) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  BcgMapDesc* m = const_cast<BcgMapDesc*>(b.maps) + first + k;
  m->occupied = 0;
  m->flags &= ~BCG_MAP_CELL_INDEX;                      // set again by cell_index_kernel once the index matches the plane
  uint32_t* sum = const_cast<uint32_t*>(b.occ_sum_arena) + m->sum_off;     // tiles_kernel only sets summary bits
  const int words = m->tiles_y * ((m->tiles_x + 31) >> 5);
  for (int i = 0; i < words; ++i) sum[i] = 0u;
}

// Cell index of one map per CTA (BCG_BATCH_CELL_INDEX trailer, after tiles_kernel): per 32 x 16 tile of the occupancy
// plane its cell count, an exclusive block scan of the counts in row-major tile order (prefix), and the cells themselves,
// row-major inside each tile, at their tile's prefix.  Dense maps get no trailer; a map whose cells exceed the trailer's
// capacity keeps BCG_MAP_CELL_INDEX clear (nothing is written past the capacity).
#define BCG_CIX_THREADS 256
__global__ void __launch_bounds__(BCG_CIX_THREADS) cell_index_kernel(const BcgBatch b, const int first) {
  __shared__ int warp_sum[BCG_CIX_THREADS / 32];
  const BcgMapDesc m = b.maps[first + blockIdx.x];
  if ((int64_t)m.occupied * 20 > (int64_t)m.width * m.height) return;
  const int ntiles = m.tiles_x * m.tiles_y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t* const occ = b.occ_tile_arena + m.tile_off;
  uint32_t* const trailer = const_cast<uint32_t*>(b.occ_sum_arena) + m.sum_off + m.tiles_y * ((m.tiles_x + 31) >> 5);
  uint32_t* const prefix = trailer + 2;
  uint32_t* const cells = prefix + ntiles + 1;
  const uint32_t cap = trailer[0];
  uint32_t running = 0u;
  for (int t0 = 0; t0 < ntiles; t0 += BCG_CIX_THREADS) {
    const int t = t0 + tid;
    int cnt = 0;
    if (t < ntiles)
      for (int r = 0; r < 16; ++r) cnt += __popc(occ[t * 16 + r]);
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(BCG_FULL, incl, d);
      if (lane >= d) incl += v;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    int before = 0, chunk = 0;
    for (int w = 0; w < BCG_CIX_THREADS / 32; ++w) {
      const int s = warp_sum[w];
      if (w < warp) before += s;
      chunk += s;
    }
    __syncthreads();                        // warp_sum is rewritten by the next chunk
    if (t < ntiles) {
      uint32_t at = running + (uint32_t)(before + incl - cnt);
      prefix[t] = at;
      const int ty = t / m.tiles_x, tx = t - ty * m.tiles_x;
      for (int r = 0; r < 16; ++r) {
        uint32_t w = occ[t * 16 + r];
        while (w) {
          const int bit = __ffs((int)w) - 1;
          w &= w - 1u;
          if (at < cap) cells[at] = (uint32_t)((tx << 5) + bit) | ((uint32_t)((ty << 4) + r) << 16);
          ++at;
        }
      }
    }
    running += (uint32_t)chunk;
  }
  if (tid == 0) {
    prefix[ntiles] = running;
    trailer[1] = running;
    if (running <= cap) atomicOr(&const_cast<BcgMapDesc*>(b.maps)[first + blockIdx.x].flags, BCG_MAP_CELL_INDEX);
  }
}

__global__ void __launch_bounds__(256) cell_tiles_kernel(const BcgBatch b, const int first) {
  const BcgMapDesc m = b.maps[first + blockIdx.y];
  const int pieces = m.ctiles_x * m.ctiles_y * 8;
  uint4* dst = reinterpret_cast<uint4*>(const_cast<uint8_t*>(b.cell_tile_arena) + m.cell_tile_off);
  const uint8_t* src = b.map_arena + m.data_off;
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < pieces; q += gridDim.x * blockDim.x) {
    const int tile = q >> 3, r = q & 7;
    const int ty = tile / m.ctiles_x, tx = tile - ty * m.ctiles_x;
    const int y = (ty << 3) + r;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (y < m.height && (tx << 4) < m.pitch) v = *reinterpret_cast<const uint4*>(src + (int64_t)y * m.pitch + (tx << 4));
    dst[q] = v;
  }
}

// pose_collides of the poses whose work records are in b.work; one warp per env.  MODE 1: lethal tile plane + in-map
// pixel count, 2: raw uint8 rows.
template <int MODE>
__global__ void __launch_bounds__(256, 6) collision_kernel(const BcgBatch b, uint8_t* __restrict__ flags,
                                                        int32_t* __restrict__ pixels) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned lane = threadIdx.x & 31;
  if (e >= b.n_envs) return;
  const WorkCollide f = *work_collide(b.work, e);
  bool hit;
  int cnt = 0;
  if (MODE == 2) hit = collide_u8(b, f, lane);
  else hit = collide_tiles<true>(b, f, lane, &cnt);
  if (lane == 0) {
    flags[e] = hit ? 1 : 0;
    if (MODE == 1) pixels[e] = cnt;
  }
}

// pose_collides of the poses whose work records are in b.work, one THREAD per env (collide_warp_balanced): the form the
// state kernel uses, and the one the collision roofline is measured on.  Per env it reads the 48-byte record, one or two tile
// summary words per 16-row band and 16-byte quarters of the non-empty tiles under the footprint only.
__global__ void __launch_bounds__(64) collision_thread_kernel(const BcgBatch b, uint8_t* __restrict__ flags) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= b.n_envs) return;
  const uint4* rec = reinterpret_cast<const uint4*>(work_collide(b.work, e));
  WorkCollide f;
  uint4* fw = reinterpret_cast<uint4*>(&f);
#pragma unroll
  for (int k = 0; k < 3; ++k) fw[k] = __ldg(rec + k);
  const FootBox fb = {f.X0, f.Y0, f.nrows, f.fwidth, f.bin};
  flags[e] = collide_warp_balanced(b.lut, b.tile_arena, f.tile_off, b.occ_sum_arena + f.sum_off, f.tiles_x, f.map_w, f.map_h,
                                   fb, warp_item_mask(e - (int)(threadIdx.x & 31), b.n_envs), threadIdx.x & 31) ? 1 : 0;
}

// ---- shared-memory and cp.async primitives ----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 16 bytes global -> shared without passing through registers (SASS: LDGSTS); src_bytes 0 writes zeros
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_group_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}

// ---- cell-tile egocentric kernel ----------------------------------------------------------------------------
// EgocentricCostmap.observation (envs/egocentric.py:125-160): extract_egocentric_costmap (utilities/costmap_utils.py:25-75)
// = cv2.getRotationMatrix2D composed in float32 with the crop shift, then cv2.warpAffine(INTER_NEAREST, borderValue=0):
// fp64 inverse and 10-bit fixed-point source coordinates X = (rint(A11 u 2^10) + rint((A12 v + b1) 2^10) + 512) >> 10
// (SURVEY.md A.9).  The source window is staged from the cell tiles (BcgMapDesc), and only the 128-byte tiles the
// rotated crop rectangle touches are read (the per-row tile spans come with the env's EgoTileWork record).
// Persistent CTAs, 5 per SM for the 133 x 117 crop (one 39 KB window each), walking envs blockIdx.x, + gridDim.x, ...;
// the CTAs of an SM overlap each other's load and gather phases.  Per env: 16-byte pieces of the tiles -> registers ->
// the row-major shared-memory window (zeros outside the map = borderValue), fixed-point tables, barrier, rotated
// gather out of shared memory, barrier.  Records are prefetched a few envs ahead with cp.async.
// Measured (profiles/r1_notes.md): the L1 data pipe (byte gathers from shared memory + byte stores) bounds it,
// not HBM; cp.async staging, TMA boxes of the tile view, double-buffered windows and L2 prefetch were all slower.
#define BCG_EGT_THREADS 256
#define BCG_EGT_CTAS 5
#define BCG_EGT_MAX_W 160
#define BCG_EGT_REC_SLOTS 8
struct EgoTab {
  int adx[BCG_EGT_MAX_W], ady[BCG_EGT_MAX_W];   // rint(a11 u 2^10), rint(a21 u 2^10)
  int2 bxy[BCG_EGO_MAX];                        // rint((a12 v + b1) 2^10) + 512 - (X0 << 10), same for y
  int pitch_b, mode, map_id, pad;
};

__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ENDS: after its envs the kernel renders the final crops of the step's episode ends (BcgEpisodeEnds): with env_list the
// slots the sparse kernel handed over (final_list[0 .. count[1] - 1]), without it every slot in use
template <int NG, bool ENDS>
__global__ void __launch_bounds__(BCG_EGT_THREADS, BCG_EGT_CTAS) ego_tiles_kernel(const BcgParams p, const BcgBatch b,
                                                                                  uint8_t* __restrict__ image,
                                                                                  const int win_bytes,
                                                                                  const int* __restrict__ env_list,
                                                                                  const BcgEpisodeEnds ends) {
  extern __shared__ __align__(128) uint8_t egt_smem[];
  constexpr int NT = BCG_EGT_THREADS, NW = NT / 32;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  EgoTab& T = *reinterpret_cast<EgoTab*>(egt_smem + win_bytes);
  uint8_t* const rec_s = egt_smem + win_bytes + sizeof(EgoTab);
  const uint32_t win_u32 = smem_u32(egt_smem), rec_u32 = smem_u32(rec_s);
  const uint8_t* const recs = reinterpret_cast<const uint8_t*>(b.ego_work);
  // env_list (optional): render only the envs env_list[0 .. env_list[n_envs] - 1] (what the sparse kernel left over)
  const int n_env_items = env_list ? env_list[b.n_envs] : b.n_envs, G = gridDim.x;
  // items n_env_items .. n - 1 are final crops
  const int n = ENDS ? n_env_items + (env_list ? ends.count[1] : min(ends.count[0], ends.capacity)) : n_env_items;
  const int ego_w = p.ego_w, ego_h = p.ego_h, npx = ego_w * ego_h;
  const int e0 = blockIdx.x;
  if (e0 >= n) return;
  auto env_of = [&](int i) { return env_list ? env_list[i] : i; };
  auto slot_of = [&](int i) { return env_list ? ends.final_list[i - n_env_items] : i - n_env_items; };

  // record of item `en` -> ring slot `slot` (the first 16 threads move 16 bytes each)
  auto fetch_record = [&](int en, int slot) {
    if (en < n && tid < BCG_EGO_WORK_BYTES / 16) {
      const uint8_t* const src = ENDS && en >= n_env_items
                                     ? reinterpret_cast<const uint8_t*>(ends.final_ego_work) + (int64_t)slot_of(en) * BCG_EGO_WORK_BYTES
                                     : recs + (int64_t)env_of(en) * BCG_EGO_WORK_BYTES;
      cp_async_16(rec_u32 + slot * BCG_EGO_WORK_BYTES + tid * 16, src + tid * 16, 16u);
    }
  };

  // The newest record fetch may still be in flight after a wait, so records are fetched RD envs ahead.
  constexpr int RD = 3;
  static_assert(RD < BCG_EGT_REC_SLOTS, "record ring too small");
#pragma unroll
  for (int k = 0; k < RD; ++k) fetch_record(e0 + k * G, k);
  cp_async_commit();
  cp_async_wait_all();
  __syncthreads();
  // tile spans of the window rows (ego_band_span), thread <-> tile row, computed one env ahead of their use
  __shared__ uint16_t span_s[2][BCG_EGT_MAX_TILE_ROWS];
  auto make_spans = [&](int slot, int buf) {
    const int t = tid - (NT - BCG_EGT_MAX_TILE_ROWS);          // the last two warps
    if (t < 0) return;
    const EgoTileWork* q = reinterpret_cast<const EgoTileWork*>(rec_s + slot * BCG_EGO_WORK_BYTES);
    if (q->mode != BCG_EGO_MODE_TILES || t >= q->nty) return;
    span_s[buf][t] = (uint16_t)ego_band_span(q->aff, ego_w, ego_h, q->X0, q->Y0, q->ntx, q->nty, t);
  };
  make_spans(0, 0);
  __syncthreads();

  int e = e0;
  for (int it = 0; e < n; e += G, ++it) {
    const int slot = it & (BCG_EGT_REC_SLOTS - 1);
    fetch_record(e + RD * G, (it + RD) & (BCG_EGT_REC_SLOTS - 1));
    cp_async_commit();
    if (e + G < n) make_spans((it + 1) & (BCG_EGT_REC_SLOTS - 1), (it + 1) & 1);   // its record landed an iteration ago
    const EgoTileWork* r = reinterpret_cast<const EgoTileWork*>(rec_s + slot * BCG_EGO_WORK_BYTES);
    const int mode = r->mode, X0 = r->X0, Y0 = r->Y0, ntx = r->ntx, nty = r->nty;
    const int pitch_b = 16 * (ntx | 1);          // 16 * odd: staging writes and rotated reads spread over the banks
    if (mode == BCG_EGO_MODE_TILES) {
      // ---- stage: warp w moves the rows of tiles w, w + 8, ...; a lane moves row `piece` of every 4th tile ----------
      const int ctx = r->ctiles_x, cty = r->ctiles_y;
      const int ttx0 = X0 >> 4, tty0 = Y0 >> 3;
      const int piece = lane & 7, sub = lane >> 3;
      // the tile (tty0 + t, ttx0 + tx) adds ((tty0 + t) * ctx + tx) * 128 to src and (8 t pitch + 16 tx) to dst
      const uint8_t* const src_lane = b.cell_tile_arena + r->ctile_off + piece * 16 + ((int64_t)ttx0 + sub) * 128;
      const uint32_t dst_lane = win_u32 + piece * pitch_b + sub * 16;
      const int lo_map = -ttx0, hi_map = ctx - 1 - ttx0;       // window tile columns that exist in the map
      const uint32_t span_u32 = smem_u32(span_s[it & 1]);
      for (int t = warp; t < nty; t += NW) {
        const uint32_t sp = lds_u16(span_u32 + 2 * t);
        const int ts = sp & 0xff, te = sp >> 8;
        const int ty = tty0 + t;
        const int lo = (unsigned)ty < (unsigned)cty ? max(ts, lo_map) : 0x7fffffff;   // rows outside the map: all zero
        const int hi = min(te, hi_map);
        const uint8_t* src = src_lane + ((int64_t)ty * ctx + ts) * 128;
        const uint32_t dst = dst_lane + (uint32_t)(t * 8 * pitch_b + ts * 16);
        uint4 val[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {                        // 16 tile columns >= any span (the record writer checks)
          const int tx = ts + sub + 4 * j;
          val[j] = make_uint4(0u, 0u, 0u, 0u);               // zeros = borderValue
          if (tx <= te && tx >= lo && tx <= hi) val[j] = __ldcg(reinterpret_cast<const uint4*>(src + 512 * j));
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (ts + sub + 4 * j <= te) sts_v4(dst + 64 * j, val[j]);
      }
    }
    // ---- fixed-point tables of the crop (cv::warpAffine: saturate_cast<int> == cvt.rni with saturation) -------------
    {
      const EgoAffine A = r->aff;
      for (int t = tid; t < min(ego_w, BCG_EGT_MAX_W); t += NT) {     // wider crops: direct mode, which needs no column table
        T.adx[t] = __double2int_rn(A.a11 * t * 1024);
        T.ady[t] = __double2int_rn(A.a21 * t * 1024);
      }
      for (int t = tid; t < ego_h; t += NT)
        T.bxy[t] = make_int2(__double2int_rn((A.a12 * t + A.b1) * 1024) + 512 - (X0 << 10),
                             __double2int_rn((A.a22 * t + A.b2) * 1024) + 512 - (Y0 << 10));
    }
    const int map_id = r->map_id;
    cp_async_wait_group_1();                  // the record needed next iteration has landed (the newest may not have)
    __syncthreads();                          // window, tables and that record are visible to every warp
    uint8_t* const dst = ENDS && e >= n_env_items ? ends.final_ego_image + (int64_t)slot_of(e) * npx : image + (int64_t)env_of(e) * npx;
    if (mode == BCG_EGO_MODE_TILES) {
      // ---- gather: warp w takes crop rows w, w + 8, ...; lane l takes columns l, l + 32, ...  (NG = ceil(ego_w / 32):
      // only the last column group can be partial) -----------------------------------------------------------------
      int ax[NG], ay[NG];
#pragma unroll
      for (int k = 0; k < NG; ++k) {
        const int u = min(lane + 32 * k, ego_w - 1);
        ax[k] = T.adx[u];
        ay[k] = T.ady[u];
      }
      const bool last_live = lane + 32 * (NG - 1) < ego_w;
      const int64_t row_step = (int64_t)NW * ego_w;
      uint8_t* d0 = dst + warp * ego_w + lane;
      const int2* brow = T.bxy + warp;
      for (int v = warp; v < ego_h; v += NW, brow += NW, d0 += row_step) {
        const int2 b0 = brow[0];
        uint32_t v0[NG];
#pragma unroll
        for (int k = 0; k < NG; ++k) v0[k] = lds_u8(win_u32 + ((ay[k] + b0.y) >> 10) * pitch_b + ((ax[k] + b0.x) >> 10));
#pragma unroll
        for (int k = 0; k < NG - 1; ++k) d0[32 * k] = (uint8_t)v0[k];
        if (last_live) d0[32 * (NG - 1)] = (uint8_t)v0[NG - 1];
      }
    } else {
      // crops too large for the window / poses far outside any sane range: bounds-checked global gather, with the column
      // terms computed in place (crops wider than the column table come this way)
      const BcgMapDesc m = b.maps[map_id];
      const uint8_t* src = b.map_arena + m.data_off;
      const double a11 = r->aff.a11, a21 = r->aff.a21;
      for (int i = tid; i < npx; i += NT) {
        const int vv = i / ego_w, u = i - vv * ego_w;
        const int2 bb = T.bxy[vv];
        const long long X = ((long long)__double2int_rn(a11 * u * 1024) + bb.x) >> 10;
        const long long Y = ((long long)__double2int_rn(a21 * u * 1024) + bb.y) >> 10;
        uint8_t val = 0;
        if (X >= 0 && X < m.width && Y >= 0 && Y < m.height) val = __ldg(src + Y * m.pitch + X);
        dst[i] = val;
      }
    }
    __syncthreads();                          // every warp is done with the window, the tables and record `it`
  }
}

// ---- ego_sparse_kernel: scatter instead of gather ----------------------------------------------------------------
// A costmap is mostly free space (an aisle turn: five one-pixel walls), so almost every pixel of the crop is 0.  Instead
// of sampling all ego_w x ego_h pixels through a staged copy of the source window (ego_tiles_kernel: 463 M warp
// instructions and 112 M shared-memory wavefronts per launch, profiles/r1b_ncu_summary.txt), one small CTA per env
//   1. zeroes the crop in global memory: one thread hands the 16-byte aligned body to the bulk-copy engine
//      (cp.async.bulk.global.shared::cta from a shared page of zeros), lanes store the < 16 head / tail bytes,
//   2. reads the OCCUPANCY plane (1 bit per cell != 0, bcg_build_lethal_tiles) of the window -- 1/8 of the bytes, and with
//      the tile summary (1 bit per 32 x 16 tile, ego_sparse_kernel<true>) only the tiles that hold a cell at all -- and
//      lists the occupied cells inside the tile spans the rotated crop touches: each warp queues its non-empty 16-byte
//      pieces in a shared ring and expands them 32 at a time, one piece per lane,
//   3. maps every listed cell forward with cv::warpAffine's float32 matrix and tests the <= 4 crop pixels around the
//      image point with the exact fixed-point inverse rule (the one the dense kernel applies to every pixel); a crop
//      pixel samples cell (X, Y) iff that test holds, so the result is bit-identical.  Hits are single-byte stores on
//      top of the zeros (the bulk stores are waited for before the barrier that precedes this phase).
// Why <= 4 candidates: the sample of pixel (u, v) is X = floor(x + 1/2 + d), |d| <= 2^-10, with (x, y) = A (u, v) + b and A
// a rotation, so the pixels sampling (X, Y) lie within 0.501 (|cos| + |sin|) <= 0.709 of the forward image of (X, Y).
// No image lives in shared memory, so a CTA needs ~11.6 KB (2 KB of them the crop's tables, in dynamic shared memory) and
// 18 run per SM: the kernel is bound by its ~2.3 k warp instructions per env and by latency (two dependent DRAM round
// trips -- summary, occupancy words -- and two barriers), then by the image write (profiles/r1_notes.md has the
// ablations).
// Envs whose window holds more than BCG_EGS_LIST occupied cells (filled regions of real costmaps), or whose record is
// in direct mode, are appended to ego_list and rendered by the dense kernel right after.
// shape chosen by measurement (profiles/probes/egs_variants.py, profiles/r1_notes.md): 64 threads x 16 CTAs 0.292 ms,
// 128 x 12 0.303, 256 x 6 0.371, 32 x 24 0.578; with today's 48 registers 64 x 18 0.237 against 0.246 for 64 x 16
#ifndef BCG_EGS_THREADS
#define BCG_EGS_THREADS 64
#endif
#ifndef BCG_EGS_CTAS
#define BCG_EGS_CTAS 18              // register budget (launch bound); the launch asks the occupancy calculator
#endif
#ifndef BCG_EGS_LIST
#define BCG_EGS_LIST 896             // cells of one window; with the crop's 2 KB of tables 18 CTAs share an SM
#endif
#ifndef BCG_EGS_REC_SLOTS
#define BCG_EGS_REC_SLOTS 4          // record ring (power of two, > the prefetch distance 3)
#endif
#define BCG_EGS_MAX_TILES 128        // 32 x 16 bit tiles a window may span (sparse path); more -> dense kernel
#ifndef BCG_EGS_ZERO_BYTES
#define BCG_EGS_ZERO_BYTES 2048      // shared page of zeros the bulk stores read
#endif
#ifndef BCG_EGS_SUM_ROUNDS
#define BCG_EGS_SUM_ROUNDS 3         // rounds of 16 non-empty tiles loaded per pass (2: 0.2454 ms, 3: 0.2457, 4: 0.2488)
#endif
#define BCG_EGS_QCAP 64              // ring slots per warp: a push adds <= 32 to <= 31 left over
#ifndef BCG_EGS_CELL_ROUNDS
#define BCG_EGS_CELL_ROUNDS 8        // with a cell index: cells loaded per thread before the first is resolved (65 536
                                     // envs: 2: 0.2884 ms per step, 4: 0.2792, 8: 0.2773; profiles/r3b_notes.md)
#endif
// The fixed-point tables of the crop live in dynamic shared memory, sized by the crop: adxy[ego_w] = (rint(a11 u 2^10),
// rint(a21 u 2^10)), then bxy[ego_h] = rint((a12 v + b1) 2^10) + 512 - (X0 << 10), same for y (2 KB for a 117 x 133 crop)
struct EgoSparseTab {
  uint32_t list[BCG_EGS_LIST];                  // occupied window cells: y_rel << 16 | x_rel
  uint32_t count[2];
  uint32_t hits[2];                             // compact output: non-zero crop pixels recorded so far (same parity scheme)
};

__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_u16(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint2 lds_v2(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ void bulk_store(void* gdst, uint32_t ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
}
// the same with an L2 evict-first policy: the lines leave L2 early instead of lingering as dirty lines
__device__ __forceinline__ void bulk_store_evict_first(void* gdst, uint32_t ssrc, uint32_t bytes) {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst), "r"(ssrc), "r"(bytes), "l"(pol) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// cv2.warpAffine(INTER_NEAREST) of one crop (record affine map A, map `map_id`) as a bounds-checked per-pixel gather from
// the map's uint8 rows by the CTA's `nthr` threads: fixed-point tables in `tab` (ego_w + ego_h entries of shared memory),
// then every crop pixel samples its cell, 0 outside the map.  Exact for any window; it holds a barrier, so every thread of
// the CTA calls it.
__device__ __forceinline__ void ego_gather_crop(const BcgBatch& b, const EgoAffine& A, const int map_id, const int ego_w, const int ego_h,
                                                uint8_t* __restrict__ dst, int2* tab, const int tid, const int nthr) {
  for (int i = tid; i < ego_w + ego_h; i += nthr) {
    if (i < ego_w) {
      tab[i] = make_int2(__double2int_rn(A.a11 * i * 1024), __double2int_rn(A.a21 * i * 1024));
    } else {
      const int t = i - ego_w;
      tab[i] = make_int2(__double2int_rn((A.a12 * t + A.b1) * 1024) + 512, __double2int_rn((A.a22 * t + A.b2) * 1024) + 512);
    }
  }
  __syncthreads();
  const BcgMapDesc* md = b.maps + map_id;
  const uint8_t* src = b.map_arena + md->data_off;
  const int mw = md->width, mh = md->height, mpitch = md->pitch, npx = ego_w * ego_h;
  for (int i = tid; i < npx; i += nthr) {
    const int vv = i / ego_w, uu = i - vv * ego_w;
    const int2 aa = tab[uu], bb = tab[ego_w + vv];
    const long long X = ((long long)aa.x + bb.x) >> 10, Y = ((long long)aa.y + bb.y) >> 10;
    uint8_t val = 0;
    if (X >= 0 && X < mw && Y >= 0 && Y < mh) val = __ldg(src + Y * mpitch + X);
    dst[i] = val;
  }
}

// ENDS: items n_envs .. n_envs + min(count[0], capacity) - 1 are the final crops of the step's episode ends
// (BcgEpisodeEnds): item n_envs + s renders the record final_ego_work[s] into final_ego_image[s], hands slot s over to the
// dense kernel through final_list, and records no compact hit list
template <bool HITS, bool ENDS>
__global__ void __launch_bounds__(BCG_EGS_THREADS, BCG_EGS_CTAS) ego_sparse_kernel(const BcgParams p, const BcgBatch b,
                                                                                   uint8_t* __restrict__ image,
                                                                                   uint32_t* __restrict__ hit_list,
                                                                                   int32_t* __restrict__ hit_count,
                                                                                   const int hit_cap, const int evict_from,
                                                                                   const BcgEpisodeEnds ends) {
  constexpr int NT = BCG_EGS_THREADS;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // All static shared memory is ONE struct, and its shared-window address is kept in one register (the empty asm hides
  // where it came from): every other address is that register plus a compile-time offset, i.e. an immediate of the
  // load / store.  With separate __shared__ arrays the compiler re-derived each address from the CTA's window (four
  // uniform instructions) at ~20 places of the scan and expand phases instead of spending registers on them.
  struct EgsShared {
    alignas(128) uint8_t zero[BCG_EGS_ZERO_BYTES];
    alignas(128) uint8_t rec[BCG_EGS_REC_SLOTS * BCG_EGO_WORK_BYTES];
    alignas(16) EgoSparseTab T;
    alignas(16) uint4 qword[NT / 32][BCG_EGS_QCAP];
    uint32_t qtag[NT / 32][BCG_EGS_QCAP];
    uint16_t tlist[BCG_EGS_MAX_TILES];                          // non-empty tiles of the window (every warp writes the same values)
    uint16_t span[2][BCG_EGT_MAX_TILE_ROWS];                    // tile spans of the window rows, double buffered
    int ids[8];                                                 // envs this CTA renders next
  };
  __shared__ EgsShared S;
  auto& zero_s = S.zero;
  auto& rec_s = S.rec;
  EgoSparseTab& T = S.T;
  auto& span_s = S.span;
  auto& ids_s = S.ids;
  uint32_t sbase = smem_u32(&S);
  asm volatile("" : "+r"(sbase));
  const uint32_t qword_u32 = sbase + (uint32_t)offsetof(EgsShared, qword) + (uint32_t)warp * (uint32_t)sizeof(S.qword[0]);
  const uint32_t qtag_u32 = sbase + (uint32_t)offsetof(EgsShared, qtag) + (uint32_t)warp * (uint32_t)sizeof(S.qtag[0]);
  const uint32_t tlist_u32 = sbase + (uint32_t)offsetof(EgsShared, tlist);
  const uint32_t zero_u32 = sbase + (uint32_t)offsetof(EgsShared, zero), rec_u32 = sbase + (uint32_t)offsetof(EgsShared, rec);
  // fixed-point tables of the crop with one sentinel entry before and after each: adxy[-1 .. ego_w], bxy[-1 .. ego_h].  A
  // candidate pixel one step outside the crop reads a sentinel, fails the test and is never stored: no clamping, and the
  // four candidates of a cell are the table entries / image bytes at fixed offsets from the first
  extern __shared__ __align__(16) int2 egs_tab[];
  const uint32_t adxy_u32 = smem_u32(egs_tab) + 8u, bxy_u32 = adxy_u32 + 8u * (uint32_t)(p.ego_w + 2);
  const uint32_t list_u32 = sbase + (uint32_t)(offsetof(EgsShared, T) + offsetof(EgoSparseTab, list));
  const uint8_t* const recs = reinterpret_cast<const uint8_t*>(b.ego_work);
  const int n = b.n_envs, G = gridDim.x;
  const int ego_w = p.ego_w, ego_h = p.ego_h, npx = ego_w * ego_h;
  const int e0 = blockIdx.x;
  if (e0 >= n) return;
  int n_items = n;                              // + the final crops (ENDS), counted by reward_kernel: set after the wait

  auto fetch_record = [&](int en, int slot) {
    if (en < n_items && tid < BCG_EGO_WORK_BYTES / 16) {
      const uint8_t* const src = ENDS && en >= n ? reinterpret_cast<const uint8_t*>(ends.final_ego_work) + (int64_t)(en - n) * BCG_EGO_WORK_BYTES
                                                 : recs + (int64_t)en * BCG_EGO_WORK_BYTES;
      cp_async_16(rec_u32 + slot * BCG_EGO_WORK_BYTES + tid * 16, src + tid * 16, 16u);
    }
  };
  const bool cix_batch = (b.flags & BCG_BATCH_CELL_INDEX) != 0;
  // Tile-summary words of the window of record `q`, lane <-> band of 16 rows (zero where the band or the word lies
  // outside the map, or the env will not take the sparse path).  With a cell index (BCG_BATCH_CELL_INDEX) they are the
  // band's prefix counts at the window's first tile column and one past its last instead: the band's cells are
  // cells[lo .. hi).  Loaded one env ahead of their use, so that an env's chain of dependent DRAM round trips is the
  // occupancy words (or cells) alone.
  auto summary_words = [&](const EgoTileWork* q, uint32_t& lo, uint32_t& hi, const bool use_index) {
    lo = hi = 0u;
    if (q->mode != BCG_EGO_MODE_TILES || (q->dense_map & 1)) return;
    const int qby0 = q->Y0 >> 4, qnby = ((q->Y0 + 8 * q->nty - 1) >> 4) - qby0 + 1;
    const int qtx = (int)(q->tiles_xy & 0xffffu), qty = (int)(q->tiles_xy >> 16), sw = (qtx + 31) >> 5;
    const int ty = qby0 + lane, w0 = q->X0 >> 10;                            // X0 >> 5 may be negative: w0 = -1
    if (lane < qnby && (unsigned)ty < (unsigned)qty) {
      if (use_index && cix_batch && (q->dense_map & 4)) {
        const uint32_t* const prow = b.occ_sum_arena + q->sum_off + qty * sw + 2 + ty * qtx;
        const int c0 = min(max(q->X0 >> 5, 0), qtx), c1 = min(max(((q->X0 + 16 * q->ntx - 1) >> 5) + 1, c0), qtx);
        lo = __ldg(prow + c0);
        hi = __ldg(prow + c1);
        return;
      }
      const uint32_t* const srow = b.occ_sum_arena + q->sum_off + ty * sw;
      if ((unsigned)w0 < (unsigned)sw) lo = __ldg(srow + w0);
      if ((unsigned)(w0 + 1) < (unsigned)sw) hi = __ldg(srow + w0 + 1);
    }
  };
  constexpr int RD = 3;
  static_assert(RD < BCG_EGS_REC_SLOTS, "record ring too small");
  for (int i = tid * 16; i < BCG_EGS_ZERO_BYTES; i += NT * 16) *reinterpret_cast<uint4*>(zero_s + i) = make_uint4(0u, 0u, 0u, 0u);
  if (tid < 2) T.count[tid] = T.hits[tid] = 0;
  pdl_wait();                                 // the records (and, on a reset, the state) are reward_kernel's
  if (ENDS) n_items = n + min(ends.count[0], ends.capacity);
#pragma unroll
  for (int k = 0; k < RD; ++k) fetch_record(e0 + k * G, k);
  cp_async_commit();
  // Which envs a CTA renders: its first RD + 1 are blockIdx.x + k G; the later ones come from a global counter
  // (ego_list[n + 1], zeroed with the hand-over count), drawn RD + 1 iterations ahead so that the record can be
  // prefetched -- CTAs whose windows are light take more envs, and the 24-or-25 envs per CTA quantisation goes away.
  if (tid <= RD) ids_s[tid] = e0 + tid * G;
  fence_async_smem();                         // the zeros are visible to the bulk-copy engine
  cp_async_wait_all();
  __syncthreads();

  // tile spans of the window rows (ego_band_span), lane <-> tile row, computed by the last warp one env ahead of their use
  auto make_spans = [&](int slot, int buf) {
    if (warp != NT / 32 - 1) return;
    const EgoTileWork* q = reinterpret_cast<const EgoTileWork*>(rec_s + slot * BCG_EGO_WORK_BYTES);
    if (q->mode != BCG_EGO_MODE_TILES || (q->dense_map & 1)) return;
    for (int t = lane; t < q->nty; t += 32)
      span_s[buf][t] = (uint16_t)ego_band_span(q->aff, ego_w, ego_h, q->X0, q->Y0, q->ntx, q->nty, t);
  };
  make_spans(0, 0);
  __syncthreads();
  uint32_t pf_lo = 0u, pf_hi = 0u;              // summary words of the env about to be rendered
  summary_words(reinterpret_cast<const EgoTileWork*>(rec_s), pf_lo, pf_hi, true);
  for (int it = 0;; ++it) {
    const int e = ids_s[it & 7];
    if (e >= n_items) break;
    int drawn = 0;
    if (tid == 0) drawn = (RD + 1) * G + atomicAdd(b.ego_list + n + 1, 1);       // stored at the end of the iteration
    const int slot = it & (BCG_EGS_REC_SLOTS - 1), par = it & 1;
    fetch_record(ids_s[(it + RD) & 7], (it + RD) & (BCG_EGS_REC_SLOTS - 1));
    cp_async_commit();
    const int e_next = ids_s[(it + 1) & 7];
    // record it + 1 has landed (only the newest fetch may still be in flight): start its summary loads now
    const uint32_t cur_lo = pf_lo, cur_hi = pf_hi;
    if (e_next < n_items)
      summary_words(reinterpret_cast<const EgoTileWork*>(rec_s + ((it + 1) & (BCG_EGS_REC_SLOTS - 1)) * BCG_EGO_WORK_BYTES), pf_lo, pf_hi, true);
    if (e_next < n_items) make_spans((it + 1) & (BCG_EGS_REC_SLOTS - 1), (it + 1) & 1);
    const EgoTileWork* r = reinterpret_cast<const EgoTileWork*>(rec_s + slot * BCG_EGO_WORK_BYTES);
    const int mode = r->mode, X0 = r->X0, Y0 = r->Y0, ntx = r->ntx, nty = r->nty;
    const bool final_crop = ENDS && e >= n;             // a final crop: no compact hit list, its own image and hand-over
    uint8_t* const dst = final_crop ? ends.final_ego_image + (int64_t)(e - n) * npx : image + (int64_t)e * npx;
    const int wx0 = X0 >> 5, nwx = ((X0 + 16 * ntx - 1) >> 5) - wx0 + 1;        // <= 9 columns of 32-cell words
    const int by0 = Y0 >> 4, nby = ((Y0 + 8 * nty - 1) >> 4) - by0 + 1;         // bands of 16 rows
    const int ntile = nby * nwx;
    // maps with more than one cell in 20 occupied (filled regions, inflation gradients) overflow the cell list in
    // almost every window: they go straight to the dense kernel instead of paying for a scan that is thrown away
    const bool dense_map = (r->dense_map & 1) != 0;     // decided by the record writer, which holds the map descriptor
    // (<= 32 bands and <= 32 word columns: a band's summary bits are one lane's, a band's tile mask one word)
    const bool try_sparse = mode == BCG_EGO_MODE_TILES && ntile <= BCG_EGS_MAX_TILES && !dense_map && (nby <= 32 && nwx <= 32);
    // With a cell index (BCG_BATCH_CELL_INDEX, map bit in the record) band b's cells are cells[lo_b .. hi_b) (the words
    // `summary_words` loaded, lane <-> band).  An inclusive warp scan of the band counts numbers the window's cells
    // 0 .. total - 1, and cell j of band b is cells[j + lo_b - start_b]: the scatter reads them straight from there.
    // Nothing is listed or staged; the cells of the bands outside the rotated crop fail the scatter's candidate test like
    // any other.  A window with more than BCG_EGS_LIST cells in its bands (whose cells inside the crop's tile spans may
    // or may not overflow the list) is listed from the occupancy plane instead, so that the overflow rule -- and with it
    // which envs report a compact hit list -- stays exactly that of the listing.
    const bool has_index = cix_batch && try_sparse && (r->dense_map & 4);
    int bincl = 0, boff = 0, total = 0;
    const uint32_t* cells = nullptr;
    if (has_index) {
      const int bcnt = (int)(cur_hi - cur_lo);
      bincl = bcnt;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(BCG_FULL, bincl, d);
        if (lane >= d) bincl += v;
      }
      total = __shfl_sync(BCG_FULL, bincl, 31);
      boff = (int)cur_lo - (bincl - bcnt);
      const int tx_ = (int)(r->tiles_xy & 0xffffu), ty_ = (int)(r->tiles_xy >> 16);
      cells = b.occ_sum_arena + r->sum_off + ty_ * ((tx_ + 31) >> 5) + 3 + tx_ * ty_;
    }
    const bool cix = has_index && total <= BCG_EGS_LIST;
    if (try_sparse) {
      // ---- 1. zero the crop in global memory ----------------------------------------------------------------------
      {
        const int head = min((int)((16u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u), npx);
        const int body = (npx - head) & ~15, tail = npx - head - body;
        // one bulk store of the zero page per lane of warp 0 (a loop in one thread was 16 instructions per store; a
        // bulk group belongs to the thread that committed it, so the same lanes wait for theirs below)
        if (warp == 0) {
          for (int o = lane * BCG_EGS_ZERO_BYTES; o < body; o += 32 * BCG_EGS_ZERO_BYTES) {
            if (e >= evict_from) bulk_store_evict_first(dst + head + o, zero_u32, (uint32_t)min(body - o, BCG_EGS_ZERO_BYTES));
            else bulk_store(dst + head + o, zero_u32, (uint32_t)min(body - o, BCG_EGS_ZERO_BYTES));
          }
          bulk_commit();
        }
        if (warp == NT / 32 - 1) {
          if (lane < head) dst[lane] = 0;
          if (lane >= 16 && lane - 16 < tail) dst[head + body + lane - 16] = 0;
        }
      }
      // ---- fixed-point tables of the crop (as the dense kernel) --------------------------------------------------
      // (a i) 1024 == (1024 a) i and (a t + b) 1024 == (1024 a) t + 1024 b bit for bit (a power of two commutes with
      // every rounding), so the scale is folded into the coefficients: one multiplication less per table value
      {
        const EgoAffine A = r->aff;
        const double a11 = A.a11 * 1024, a21 = A.a21 * 1024, a12 = A.a12 * 1024, a22 = A.a22 * 1024;
        const double b1 = A.b1 * 1024, b2 = A.b2 * 1024;
        const int ox = 512 - (X0 << 10), oy = 512 - (Y0 << 10);
        const int2 never = make_int2(0x40000000, 0x40000000);      // a + b - (r << 10) stays far above 1023 (mod 2^32)
        for (int i = tid; i < ego_w + ego_h + 4; i += NT) {
          if (i < ego_w + 2) {
            const int u = i - 1;
            egs_tab[i] = (u < 0 || u >= ego_w) ? never : make_int2(__double2int_rn(a11 * u), __double2int_rn(a21 * u));
          } else {
            const int t = i - (ego_w + 2) - 1;
            egs_tab[i] = (t < 0 || t >= ego_h) ? never
                                               : make_int2(__double2int_rn(a12 * t + b1) + ox, __double2int_rn(a22 * t + b2) + oy);
          }
        }
      }
      // ---- 2. occupied cells of the window: four lanes per 32 x 16 bit tile (a 16-byte load = 4 rows each).  All loads
      // of a thread are issued before the first is used (one DRAM round trip per env instead of one per round).
      // Walls are thin: only a few of a warp's 32 pieces hold a cell, so expanding them where they were loaded would
      // keep most lanes idle.  Each warp queues its non-empty pieces (16 bytes + band / column / row-group tag) in a
      // shared ring and expands them 32 at a time, one piece per lane. ------------------------------------------------
      const int tiles_x = (int)(r->tiles_xy & 0xffffu);
      const uint4* occ = reinterpret_cast<const uint4*>(b.occ_tile_arena + ((int64_t)r->tile_off16 << 4));
      const int g = lane & 3;                                                     // rows 4 g .. 4 g + 3 of the tile
      constexpr int TPR = NT / 4;                                                // tiles per round
      const uint32_t span_u32 = sbase + (uint32_t)offsetof(EgsShared, span) + (uint32_t)par * (uint32_t)sizeof(S.span[0]);
      auto expand = [&](const uint32_t qhead, const int nitems) {
        uint4 wd = make_uint4(0u, 0u, 0u, 0u);
        uint32_t tag = 0u;
        if (lane < nitems) {
          const uint32_t at = (qhead + (uint32_t)lane) & (BCG_EGS_QCAP - 1);
          wd = lds_v4(qword_u32 + 16u * at);
          tag = lds_u32(qtag_u32 + 4u * at);
        }
        __syncwarp();                                                            // ring slots are free again
        const int band = (int)(tag >> 8), jw = (int)((tag >> 2) & 63u), gq = (int)(tag & 3u);
        const int tx = wx0 + jw;
        const int yr0 = (((by0 + band) << 4) + 4 * gq) - Y0;                      // window row of word .x; 4 | yr0
        uint32_t bits[4] = {wd.x, wd.y, wd.z, wd.w};
        uint32_t keep = 0u;
        if (yr0 >= 0 && yr0 < 8 * nty) {                                          // clip to the tile span of these rows
          const uint32_t sp = lds_u16(span_u32 + 2 * (yr0 >> 3));
          const int lo = max(X0 + 16 * (int)(sp & 0xff) - (tx << 5), 0);
          const int hi = min(X0 + 16 * (int)(sp >> 8) + 15 - (tx << 5), 31);
          if (lo <= hi) keep = (0xffffffffu >> (31 - hi)) & (0xffffffffu << lo);
        }
        int cnt = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          bits[k] &= keep;
          cnt += __popc(bits[k]);
        }
        // list slots: one shared-memory atomic per lane that holds a cell (the kernel is bound by issue slots: a warp
        // scan of the counts was ~25 instructions per call, the atomic is one; the order of the list is irrelevant)
        if (cnt == 0) return;
        const uint32_t base = atomicAdd(&T.count[par], (uint32_t)cnt);
        if (base + (uint32_t)cnt > BCG_EGS_LIST) return;                          // overflow: the env goes to the dense kernel
        uint32_t at = list_u32 + 4u * base;
        const int key = (yr0 << 16) + ((tx << 5) - X0);          // x_rel of bit 0 may be negative, of a kept bit never
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          uint32_t w = bits[k];
          while (w) {
            const int bit = 31 - __clz(w);                       // order within the list is irrelevant
            w ^= 1u << bit;
            sts_u32(at, (uint32_t)(key + (k << 16) + bit));
            at += 4u;
          }
        }
      };
      const uint32_t lt_mask = (1u << lane) - 1u;
      uint32_t qhead = 0u, qtail = 0u;
      auto push = [&](const uint4& w, const uint32_t tag) {
        const bool nz = (w.x | w.y | w.z | w.w) != 0u;
        const uint32_t bal = __ballot_sync(BCG_FULL, nz);
        if (bal == 0u) return;                                                    // free space
        if (nz) {
          const uint32_t at = (qtail + (uint32_t)__popc(bal & lt_mask)) & (BCG_EGS_QCAP - 1);
          sts_v4(qword_u32 + 16u * at, w);
          sts_u32(qtag_u32 + 4u * at, tag);
        }
        qtail += (uint32_t)__popc(bal);
        if (qtail - qhead >= 32u) {
          __syncwarp();
          expand(qhead, 32);
          qhead += 32u;
        }
      };
      if (cix) {
        // cell index: nothing to list, the scatter below reads the window's cells from the index
      } else {
        uint32_t slo = cur_lo, shi = cur_hi;
        if (has_index) summary_words(r, slo, shi, false);                       // the prefetched words were prefix counts
        // (a) which tiles of the window hold a cell at all: lane <-> band of 16 rows, one or two words of the map's tile
        // summary each, loaded one env ahead (`summary_words`; every warp holds the same words: no barrier)
        const uint32_t tmask = (uint32_t)((((uint64_t)shi << 32) | slo) >> (wx0 & 31)) & ((1u << nwx) - 1u);
        // (b) the list of those tiles (band << 6 | column), in band order: inclusive warp scan of the per-band counts
        int tincl = __popc(tmask);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int v = __shfl_up_sync(BCG_FULL, tincl, d);
          if (lane >= d) tincl += v;
        }
        const int ntl = __shfl_sync(BCG_FULL, tincl, 31);                         // <= ntile <= BCG_EGS_MAX_TILES
        {
          uint32_t at = tlist_u32 + 2u * (uint32_t)(tincl - __popc(tmask));
          uint32_t m2 = tmask;
          while (m2) {
            const int jw = __ffs((int)m2) - 1;
            m2 &= m2 - 1u;
            sts_u16(at, (uint32_t)((lane << 6) | jw));
            at += 2u;
          }
        }
        __syncwarp();
        // (c) their pieces, BCG_EGS_SUM_ROUNDS x 16 tiles per pass (one pass unless the window is crowded)
        constexpr int RS = BCG_EGS_SUM_ROUNDS;
        for (int base = 0; base < ntl; base += RS * TPR) {
          uint4 word[RS];
          uint32_t tag[RS];
#pragma unroll
          for (int rd = 0; rd < RS; ++rd) {
            const int i = base + (tid >> 2) + rd * TPR;
            word[rd] = make_uint4(0u, 0u, 0u, 0u);
            tag[rd] = 0u;
            if (i < ntl) {
              const uint32_t code = lds_u16(tlist_u32 + 2u * (uint32_t)i);
              const int band = (int)(code >> 6), jw = (int)(code & 63u);
              tag[rd] = (code << 2) | (uint32_t)g;
              word[rd] = __ldg(occ + ((((by0 + band) * tiles_x + wx0 + jw) << 2) + g));
            }
          }
#pragma unroll
          for (int rd = 0; rd < RS; ++rd) push(word[rd], tag[rd]);
        }
      }
      if (qtail != qhead) {
        __syncwarp();
        expand(qhead, (int)(qtail - qhead));
      }
      if (warp == 0) bulk_wait_all();         // the zeros have landed (they had the whole scan to do so)
    }
    cp_async_wait_group_1();                  // the record needed next iteration has landed
    __syncthreads();                          // zeros (incl. head / tail bytes), tables, list and count are complete
    const uint32_t count = T.count[par];
    const bool sparse = try_sparse && (cix || count <= BCG_EGS_LIST);
    if (sparse) {
      // ---- 3. scatter the listed cells ----------------------------------------------------------------------------
      const bool only_lethal = (r->dense_map & 2) != 0;
      const uint8_t* src = nullptr;
      int pitch = 0;
      if (!only_lethal) {                               // other cost values: they are read from the map's uint8 rows
        const BcgMapDesc* md = b.maps + r->map_id;
        src = b.map_arena + md->data_off;
        pitch = md->pitch;
      }
      const int m0 = r->fwd[0], m1 = r->fwd[1], m2 = r->fwd[2], m3 = r->fwd[3], m4 = r->fwd[4], m5 = r->fwd[5];
      // the loop is instantiated per kind of map: with every occupied cell lethal the value is a constant and the address
      // arithmetic of the cost-byte load (predicated off, but issued) is gone
      // (the table bases and the constant go through an empty asm: the compiler otherwise re-derives the shared-memory
      // addresses from the CTA's window and re-materialises 254 once per store, inside the loop)
      uint32_t abase = adxy_u32, bbase = bxy_u32, lethal_value = 254u + ((uint32_t)hit_cap >> 31);   // hit_cap >= 0
      asm volatile("" : "+r"(abase), "+r"(bbase), "+r"(lethal_value));
      auto scatter = [&](auto lethal_tag) {
      constexpr bool LETHAL = decltype(lethal_tag)::value;
      auto resolve = [&](const int xr, const int yr) {
        // candidates only, in 16.16 integers (no conversions: they run on the quarter-rate unit); the fixed-point test
        // below decides
        const int fu = (m0 * xr + m1 * yr + m2) >> 16;
        const int fv = (m3 * xr + m4 * yr + m5) >> 16;
        if (fu < -1 || fu >= ego_w || fv < -1 || fv >= ego_h) return;       // every candidate is outside the crop
        uint32_t val = lethal_value;
        if (!LETHAL) val = __ldg(src + (int64_t)(Y0 + yr) * pitch + (X0 + xr));
        // candidates (fu | fu + 1, fv | fv + 1); fu in [-1, ego_w - 1], fv in [-1, ego_h - 1]: the outer ones are sentinels
        const uint32_t ta = abase + 8u * (uint32_t)fu, tb = bbase + 8u * (uint32_t)fv;
        const uint2 a0 = lds_v2(ta), a1 = lds_v2(ta + 8u);
        const uint2 b0 = lds_v2(tb), b1 = lds_v2(tb + 8u);
        // (a + b) >> 10 == r  <=>  0 <= a + b - (r << 10) < 1024   (unsigned arithmetic: the sentinels may wrap)
        const uint32_t xs = (uint32_t)xr << 10, ys = (uint32_t)yr << 10;
        const uint32_t ax0 = a0.x - xs, ax1 = a1.x - xs, ay0 = a0.y - ys, ay1 = a1.y - ys;
        const bool h00 = (ax0 + b0.x) < 1024u && (ay0 + b0.y) < 1024u;
        const bool h10 = (ax1 + b0.x) < 1024u && (ay1 + b0.y) < 1024u;
        const bool h01 = (ax0 + b1.x) < 1024u && (ay0 + b1.y) < 1024u;
        const bool h11 = (ax1 + b1.x) < 1024u && (ay1 + b1.y) < 1024u;
        const int o00 = fv * ego_w + fu;                                      // may lie outside the crop; only hits are stored
        uint8_t* const p0 = dst + o00, * const p1 = p0 + ego_w;
        if (h00) p0[0] = (uint8_t)val;
        if (h10) p0[1] = (uint8_t)val;
        if (h01) p1[0] = (uint8_t)val;
        if (h11) p1[1] = (uint8_t)val;
        if (HITS && !final_crop) {
          // compact observation (BcgStepOut.ego_hits): pixel offset | value << 16 of every non-zero crop pixel.  A crop
          // pixel samples exactly one cell and the four candidates of a cell are distinct pixels: no duplicates.
          const int nh = (int)h00 + (int)h10 + (int)h01 + (int)h11;
          if (nh) {
            uint32_t at = atomicAdd(&T.hits[par], (uint32_t)nh);
            uint32_t* const out = hit_list + (int64_t)e * hit_cap;
            const uint32_t tagged = (val & 0xffu) << 16;
            if (h00) { if (at < (uint32_t)hit_cap) out[at] = tagged | (uint32_t)o00; ++at; }
            if (h10) { if (at < (uint32_t)hit_cap) out[at] = tagged | (uint32_t)(o00 + 1); ++at; }
            if (h01) { if (at < (uint32_t)hit_cap) out[at] = tagged | (uint32_t)(o00 + ego_w); ++at; }
            if (h11) { if (at < (uint32_t)hit_cap) out[at] = tagged | (uint32_t)(o00 + ego_w + 1); ++at; }
          }
        }
      };
      if (cix) {
        // BCG_EGS_CELL_ROUNDS cells per thread are loaded before the first is resolved; a cell's band is found by a
        // binary search over the band scan (lanes >= the window's bands hold `total`)
        constexpr int CR = BCG_EGS_CELL_ROUNDS;
        for (int base = warp * 32; base < total; base += CR * NT) {
          uint32_t cell[CR];
#pragma unroll
          for (int rd = 0; rd < CR; ++rd) {
            const int j = base + rd * NT + lane;
            cell[rd] = 0u;
            if (base + rd * NT < total) {                                      // warp-uniform
              int bnd = 0;                                                     // bands whose cells all precede j
#pragma unroll
              for (int s = 16; s > 0; s >>= 1)
                if (__shfl_sync(BCG_FULL, bincl, bnd + s - 1) <= j) bnd += s;
              const int off = __shfl_sync(BCG_FULL, boff, bnd);
              if (j < total) cell[rd] = __ldg(cells + j + off);
            }
          }
#pragma unroll
          for (int rd = 0; rd < CR; ++rd)
            if (base + rd * NT + lane < total) resolve((int)(cell[rd] & 0xffffu) - X0, (int)(cell[rd] >> 16) - Y0);
        }
      } else {
        for (uint32_t i = tid; i < count; i += NT) {
          const uint32_t key = lds_u32(list_u32 + 4u * i);
          resolve((int)(key & 0xffffu), (int)(key >> 16));
        }
      }
      };
      if (only_lethal) scatter(std::true_type{});
      else scatter(std::false_type{});
    } else if (b.flags & BCG_BATCH_SPARSE_EGO_ONLY) {
      // No dense pass follows this kernel (the host knows that no map of the batch is dense): the rare window that
      // overflows the cell list, or lies outside any sane range, is rendered here by the bounds-checked per-pixel gather.
      ego_gather_crop(b, r->aff, r->map_id, ego_w, ego_h, dst, egs_tab, tid, NT);
    } else if (final_crop) {
      if (tid == 0) ends.final_list[atomicAdd(ends.count + 1, 1)] = e - n;
    } else if (tid == 0) {
      const int at = atomicAdd(b.ego_list + n, 1);
      b.ego_list[at] = e;
    }
    if (tid == 0) T.count[par ^ 1] = 0;         // nobody reads the other counter before the next barrier
    if (HITS) {                                 // (the hit counter of this env is complete after the barrier below)
      if (!sparse && tid == 0 && !final_crop) hit_count[e] = -1;       // rendered densely: the consumer reads the image itself
      __syncthreads();
      if (sparse && tid == 0 && !final_crop) hit_count[e] = (int32_t)T.hits[par];      // > hit_cap: the list overflowed, read the image
      if (tid == 0) T.hits[par ^ 1] = 0;
    }
    if (tid == 0) ids_s[(it + RD + 1) & 7] = drawn;
    __syncthreads();                            // list, tables and record `it` are free
  }
}

// Auto-reset into a new world (BcgParams.auto_reset == BCG_AUTO_RESET_NEW_WORLD), launched behind reward_kernel: a fixed
// grid (a captured graph replays it unchanged) whose CTAs take the envs reward_kernel listed in BcgWorldGen.list through the
// item counter.  For each listed env:
//   1. with episode ends, the egocentric image and a final slot: the final crop, gathered from the OLD world before its
//      walls are erased (the egocentric kernels behind this one render the step's crops only);
//   2. the new world, built by the body bcg_generate_aisles / bcg_generate_minis run for a masked env, drawn with
//      (seed; env id, BCG_NEW_WORLD_DRAW | the step's index);
//   3. the initial observation, written like the in-kernel reset writes it.  When the world failed (slot overflow, sampler
//      out of tries; counted in the status words) the env restarts its current world, as auto_reset 1 does.
// The last CTA to finish zeroes the list counters, so that every step's reward_kernel finds them zero.
// ROWS: the aisle initial states use each env's own goal tolerances (as bcg_generate_aisles with rows).
#define BCG_REGEN_THREADS 128
#define BCG_REGEN_CTAS 4          // CTAs per SM of the fixed grid
template <bool ROWS>
__global__ void __launch_bounds__(BCG_REGEN_THREADS) regenerate_kernel(const BcgParams p, const BcgBatch b, const BcgStateLayout L,
                                                                       const BcgEnvRows rows, const BcgStepOut out, const int ego_cap,
                                                                       const BcgEpisodeEnds ends, const uint64_t step_index_arg) {
  __shared__ int item_s;
  __shared__ int2 tab_s[2 * BCG_EGO_MAX];
  pdl_wait();                                            // reward_kernel's list, final records and step counter
  const BcgWorldGen* const wg = b.world_gen;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int64_t N = b.n_envs;
  // (reward_kernel has advanced the device-side step counter already: this step's index is one less)
  const uint64_t step_index = b.step_counter ? *reinterpret_cast<const volatile uint64_t*>(b.step_counter) - 1ull : step_index_arg;
  const uint64_t draw = BCG_NEW_WORLD_DRAW | step_index;
  const int listed = *reinterpret_cast<const volatile int32_t*>(wg->count);
  const int kind = wg->kind;
  const BcgAisleSlots slots = wg->slots;
  const bool finals = out.ego_image && ends.final_ego_image;
  for (;;) {
    if (tid == 0) item_s = atomicAdd(wg->count + 1, 1);
    __syncthreads();
    const int item = item_s;
    __syncthreads();                                     // item_s is written again at the next item
    if (item >= listed) break;
    const int e = wg->list[item];
    const int slot = finals ? ends.final_slot[e] : -1;
    if (slot >= 0) {
      const EgoTileWork* const rec =
          reinterpret_cast<const EgoTileWork*>(reinterpret_cast<const uint8_t*>(ends.final_ego_work) + (int64_t)slot * BCG_EGO_WORK_BYTES);
      ego_gather_crop(b, rec->aff, rec->map_id, p.ego_w, p.ego_h, ends.final_ego_image + (int64_t)slot * p.ego_w * p.ego_h, tab_s,
                      tid, nthr);
      __syncthreads();                                   // the old walls are read before they are erased
    }
    bool made;
    if (kind == BCG_WORLD_MINI)
      made = mini_world(p, b, L, slots, wg->mini, nullptr, reinterpret_cast<BcgMiniParams*>(slots.params_out), e, draw,
                        wg->path_delta) == 1;
    else
      made = aisle_world<ROWS>(p, b, L, slots, rows, e, draw_turn_params(p.seed, p.env_id_base + (uint64_t)e, draw), wg->path_delta);
    if (!made) {                                         // the current world's initial state
      for (int r = tid; r < b.n_frows; r += nthr) b.state_f[(int64_t)r * N + e] = b.init_f[(int64_t)r * N + e];
      for (int r = tid; r < b.n_irows; r += nthr) b.state_i[(int64_t)r * N + e] = b.init_i[(int64_t)r * N + e];
    }
    __syncthreads();                                     // the initial rows, path and map descriptor are complete
    if (tid == 0) write_initial_observation(p, b, out, e, ego_cap);
  }
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(wg->count + 2, 1) == (int)gridDim.x - 1) wg->count[0] = wg->count[1] = wg->count[2] = 0;
  }
}

// egocentric records and / or goal_n_state from the current state (stand-alone bcg_observe_ego): one thread per env
__global__ void __launch_bounds__(128) ego_prep_kernel(const BcgParams p, const BcgBatch b, const int want_image,
                                                       float* __restrict__ goal_n_state, const int ego_cap) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= b.n_envs) return;
  const int64_t N = b.n_envs;
  const double* sf = b.state_f + e;
  const int prow = p.ego_variant == 1 ? BCG_F_ROBOT : BCG_F_DPOSE;
  const double px = sf[(prow + 0) * N], py = sf[(prow + 1) * N], pth = sf[(prow + 2) * N];
  if (want_image) {
    const int map_id = b.map_id[e];
    write_ego_tile_record(p, b, e, map_id, b.maps[map_id], px, py, pth, ego_cap);
  }
  if (e == 0 && b.ego_list) b.ego_list[N] = b.ego_list[N + 1] = 0;       // hand-over count, env counter of the sparse kernel
  if (goal_n_state) {
    double drobot[7];
#pragma unroll
    for (int r = 0; r < 7; ++r) drobot[r] = sf[(BCG_F_DROBOT + r) * N];
    write_goal_n_state(p, b, e, b.paths[b.path_id[e]], px, py, pth, b.state_i[BCG_I_TARGET * N + e], drobot, goal_n_state);
  }
}

__global__ void __launch_bounds__(256) gather_kernel(const BcgBatch b, const int64_t* __restrict__ idx, const int k,
                                                     double* __restrict__ out_f, int32_t* __restrict__ out_i) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= k) return;
  const int64_t e = idx[j], N = b.n_envs;
  if (e < 0 || e >= N) return;
  for (int r = 0; r < b.n_frows; ++r) out_f[(int64_t)r * k + j] = b.state_f[(int64_t)r * N + e];
  for (int r = 0; r < b.n_irows; ++r) out_i[(int64_t)r * k + j] = b.state_i[(int64_t)r * N + e];
}

__global__ void __launch_bounds__(256) scatter_kernel(const BcgBatch b, const int64_t* __restrict__ idx, const int k,
                                                      const double* __restrict__ in_f, const int32_t* __restrict__ in_i,
                                                      const int load_delayed_robot) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= k) return;
  const int64_t e = idx[j], N = b.n_envs;
  if (e < 0 || e >= N) return;
  for (int r = 0; r < b.n_frows; ++r) {
    int src = r;
    if (load_delayed_robot && r >= BCG_F_ROBOT && r < BCG_F_ROBOT + 7) src = r - BCG_F_ROBOT + BCG_F_DROBOT;  // env.py:284
    b.state_f[(int64_t)r * N + e] = in_f[(int64_t)src * k + j];
  }
  for (int r = 0; r < b.n_irows; ++r) b.state_i[(int64_t)r * N + e] = in_i[(int64_t)r * k + j];
}

// ego_hits lists of all envs, fixed stride -> one contiguous array (offsets: exclusive prefix sum of the clamped counts);
// eight lanes per env.  OFFSETS_ONLY: 16-bit pixel offsets without the cost values (batches whose maps hold no cost value
// but 254: the value is implied)
template <bool OFFSETS_ONLY>
__global__ void __launch_bounds__(256) pack_hits_kernel(const uint32_t* __restrict__ hits, const int32_t* __restrict__ counts,
                                                        const int cap, const int n, const int64_t* __restrict__ offsets,
                                                        void* __restrict__ packed) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, gl = threadIdx.x & 7;
  if (e >= n) return;
  const int c = counts[e];
  if (c <= 0 || c > cap) return;                 // rendered densely / list overflowed: the consumer reads the image
  const uint32_t* src = hits + (int64_t)e * cap;
  if (OFFSETS_ONLY) {
    uint16_t* dst = reinterpret_cast<uint16_t*>(packed) + offsets[e];
    for (int i = gl; i < c; i += 8) dst[i] = (uint16_t)(src[i] & 0xffffu);
  } else {
    uint32_t* dst = reinterpret_cast<uint32_t*>(packed) + offsets[e];
    for (int i = gl; i < c; i += 8) dst[i] = src[i];
  }
}

// is_footprint_colliding_impl: any(values[mask] == value) over flattened arrays
__global__ void __launch_bounds__(256) masked_any_equal_kernel(const uint8_t* __restrict__ values, const uint8_t* __restrict__ mask,
                                                               const int64_t n, const uint8_t value, int32_t* __restrict__ flag) {
  bool hit = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    hit |= (mask[i] != 0) && (values[i] == value);
  if (__any_sync(BCG_FULL, hit) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

// inverse_transform (utilities/coordinate_transformations.py:57-84) of n transforms [n][3]
__global__ void __launch_bounds__(256) inverse_transform_kernel(const double* __restrict__ in, const int64_t n, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = in[3 * i], y = in[3 * i + 1], th = in[3 * i + 2];
  double sn, cs;
  sincos(th, &sn, &cs);
  out[3 * i] = -x * cs - y * sn;
  out[3 * i + 1] = x * sn - y * cs;
  out[3 * i + 2] = wrap_angle(-th);
}

// project_poses (utilities/coordinate_transformations.py:289-328): rotate by the transform's angle, translate, wrap the angle
__global__ void __launch_bounds__(256) project_poses_kernel(const double tx, const double ty, const double tt,
                                                            const double* __restrict__ poses, const int64_t n, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double sn, cs;
  sincos(tt, &sn, &cs);
  const double x = poses[3 * i], y = poses[3 * i + 1];
  out[3 * i] = cs * x - sn * y + tx;
  out[3 * i + 1] = sn * x + cs * y + ty;
  out[3 * i + 2] = wrap_angle(poses[3 * i + 2] + tt);
}

// Observation.path (envs/base/env.py:421-433: path[target_idx:]) of every env as a device tensor, in the robot frame
// (from_global_to_egocentric, utilities/coordinate_transformations.py:341-362): out [n][max_points][3], zero padded;
// len_out[e] = number of remaining way points (may exceed max_points).  One warp per env, lanes <-> points.
__global__ void __launch_bounds__(256) ego_path_kernel(const BcgParams p, const BcgBatch b, const int max_points,
                                                       double* __restrict__ out, int32_t* __restrict__ len_out) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned lane = threadIdx.x & 31;
  if (e >= b.n_envs) return;
  const int64_t N = b.n_envs;
  const BcgPathDesc pd = b.paths[b.path_id[e]];
  const double* P = b.path_arena + pd.off;
  const int target = b.state_i[BCG_I_TARGET * N + e];
  const bool pursuit = p.reward_kind == BCG_REWARD_PURE_PURSUIT;      // reward.py:120-124: path[:target_idx + 1]
  const int first = pursuit ? 0 : min(max(target, 0), pd.n);
  const int count = pursuit ? min(target + 1, pd.n) : pd.n - first;
  const int prow = p.ego_variant == 1 ? BCG_F_ROBOT : BCG_F_DPOSE;
  double ct, st, tx, ty, tt;
  inverse_transform(b.state_f[(prow + 0) * N + e], b.state_f[(prow + 1) * N + e], b.state_f[(prow + 2) * N + e], ct, st, tx, ty, tt);
  double* o = out + (int64_t)e * max_points * 3;
  for (int j = lane; j < max_points; j += 32) {
    double ex = 0.0, ey = 0.0, ea = 0.0;
    if (j < count) {
      const double gx = P[first + j], gy = P[pd.pitch + first + j], gt = P[2 * pd.pitch + first + j];
      ex = ct * gx - st * gy + tx;
      ey = st * gx + ct * gy + ty;
      ea = wrap_angle(gt + tt);
    }
    o[3 * j] = ex;
    o[3 * j + 1] = ey;
    o[3 * j + 2] = ea;
  }
  if (lane == 0 && len_out) len_out[e] = count;
}

__global__ void w2p_kernel(const double* __restrict__ xy, const int64_t n, const double ox, const double oy,
                           const double inv_res, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[2 * i] = world_to_pixel_1d(xy[2 * i], ox, inv_res);
  out[2 * i + 1] = world_to_pixel_1d(xy[2 * i + 1], oy, inv_res);
}

__global__ void wrap_kernel(const double* __restrict__ in, const int64_t n, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = wrap_angle(in[i]);
}

inline int blocks_for(int64_t work, int per_block) { return (int)((work + per_block - 1) / per_block); }

}  // namespace

// ---- C-ABI -------------------------------------------------------------------------------------------
extern "C" {

int bcg_abi_version(void) { return BCG_ABI_VERSION; }

size_t bcg_last_error(char* buf, size_t cap) {
  if (buf && cap) {
    const size_t n = g_last_error.size() < cap - 1 ? g_last_error.size() : cap - 1;
    memcpy(buf, g_last_error.data(), n);
    buf[n] = 0;
  }
  return g_last_error.size();
}

int64_t bcg_sizeof(int32_t which) {
  switch (which) {
    case 0: return sizeof(BcgParams);
    case 1: return sizeof(BcgMapDesc);
    case 2: return sizeof(BcgPathDesc);
    case 3: return sizeof(BcgFootprintLut);
    case 4: return sizeof(BcgBatch);
    case 5: return sizeof(BcgStateLayout);
    case 6: return sizeof(BcgStepOut);
    case 7: return sizeof(BcgTurnParams);
    case 8: return sizeof(BcgAisleSlots);
    case 9: return sizeof(BcgMiniGenParams);
    case 10: return sizeof(BcgMiniParams);
    case 11: return sizeof(BcgEnvRows);
    case 12: return sizeof(BcgEpisodeEnds);
    case 13: return sizeof(BcgWorldGen);
    default: return -1;
  }
}

int bcg_device_count(void) {
  int n = 0;
  const cudaError_t err = cudaGetDeviceCount(&n);
  if (err != cudaSuccess) {
    cudaGetLastError();
    return fail(BCG_ERR_NO_DEVICE, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(err));
  }
  return n;
}

int bcg_state_layout(const BcgParams* p, BcgStateLayout* out) {
  BCG_REQUIRE(p && out, "null argument");
  BCG_REQUIRE(p->delay_control >= 0 && p->delay_pose >= 0 && p->delay_state >= 0, "negative delay");
  *out = make_layout(*p);
  return BCG_OK;
}

int bcg_build_lethal_tiles(const BcgBatch* b, int32_t first, int32_t count, void* stream) {
  BCG_REQUIRE(b && b->maps && b->map_arena && b->tile_arena, "null map arena");
  BCG_REQUIRE(b->occ_tile_arena, "null occupancy plane (BcgBatch.occ_tile_arena)");
  BCG_REQUIRE(b->occ_sum_arena, "null tile summary (BcgBatch.occ_sum_arena)");
  BCG_REQUIRE(first >= 0 && count >= 0 && first + count <= b->n_maps, "map range out of bounds");
  cudaStream_t s = (cudaStream_t)stream;
  if (count > 0) zero_occupied_kernel<<<blocks_for(count, 256), 256, 0, s>>>(*b, first, count);
  for (int32_t done = 0; done < count; done += 32768) {
    const int32_t chunk = (count - done) < 32768 ? (count - done) : 32768;
    tiles_kernel<<<dim3(8, chunk), 256, 0, s>>>(*b, first + done);
    BCG_CHECK_CUDA(cudaGetLastError());
  }
  if ((b->flags & BCG_BATCH_CELL_INDEX) && count > 0) {
    cell_index_kernel<<<count, BCG_CIX_THREADS, 0, s>>>(*b, first);
    BCG_CHECK_CUDA(cudaGetLastError());
  }
  return BCG_OK;
}

int bcg_build_cell_tiles(const BcgBatch* b, int32_t first, int32_t count, void* stream) {
  BCG_REQUIRE(b && b->maps && b->map_arena && b->cell_tile_arena, "null map / cell-tile arena");
  BCG_REQUIRE(first >= 0 && count >= 0 && first + count <= b->n_maps, "map range out of bounds");
  cudaStream_t s = (cudaStream_t)stream;
  for (int32_t done = 0; done < count; done += 32768) {
    const int32_t chunk = (count - done) < 32768 ? (count - done) : 32768;
    cell_tiles_kernel<<<dim3(8, chunk), 256, 0, s>>>(*b, first + done);
    BCG_CHECK_CUDA(cudaGetLastError());
  }
  return BCG_OK;
}

int bcg_alloc_image_memory(int64_t bytes, int32_t want_compression, void** dptr, int64_t* mapped_bytes, int32_t* compressed) {
  BCG_REQUIRE(bytes > 0 && dptr && mapped_bytes && compressed, "bad argument");
  decltype(&cuMemGetAllocationGranularity) get_gran = nullptr;
  decltype(&cuMemCreate) create = nullptr;
  decltype(&cuMemGetAllocationPropertiesFromHandle) get_prop = nullptr;
  decltype(&cuMemAddressReserve) reserve = nullptr;
  decltype(&cuMemMap) map = nullptr;
  decltype(&cuMemSetAccess) set_access = nullptr;
  decltype(&cuMemRelease) release = nullptr;
  decltype(&cuMemAddressFree) address_free = nullptr;
  decltype(&cuDeviceGetAttribute) get_attr = nullptr;
  if (int rc = driver_fn("cuMemGetAllocationGranularity", &get_gran)) return rc;
  if (int rc = driver_fn("cuMemCreate", &create)) return rc;
  if (int rc = driver_fn("cuMemGetAllocationPropertiesFromHandle", &get_prop)) return rc;
  if (int rc = driver_fn("cuMemAddressReserve", &reserve)) return rc;
  if (int rc = driver_fn("cuMemMap", &map)) return rc;
  if (int rc = driver_fn("cuMemSetAccess", &set_access)) return rc;
  if (int rc = driver_fn("cuMemRelease", &release)) return rc;
  if (int rc = driver_fn("cuMemAddressFree", &address_free)) return rc;
  if (int rc = driver_fn("cuDeviceGetAttribute", &get_attr)) return rc;
  int dev = 0;
  BCG_CHECK_CUDA(cudaGetDevice(&dev));
  BCG_CHECK_CUDA(cudaFree(nullptr));                        // the primary context exists
  int supported = 0;
  BCG_CHECK_CU(get_attr(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev));
  CUmemAllocationProp prop = {};
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = dev;
  if (want_compression && supported) prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
  size_t gran = 0;
  BCG_CHECK_CU(get_gran(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
  BCG_REQUIRE(gran > 0, "zero allocation granularity");
  const size_t size = ((size_t)bytes + gran - 1) / gran * gran;
  CUmemGenericAllocationHandle h;
  BCG_CHECK_CU(create(&h, size, &prop, 0));
  CUmemAllocationProp got = {};
  if (get_prop(&got, h) != CUDA_SUCCESS) got = prop;
  CUdeviceptr p = 0;
  if (reserve(&p, size, 0, 0, 0) != CUDA_SUCCESS) {
    release(h);
    return fail(BCG_ERR_CUDA, "cuMemAddressReserve failed");
  }
  if (map(p, size, 0, h, 0) != CUDA_SUCCESS) {
    address_free(p, size);
    release(h);
    return fail(BCG_ERR_CUDA, "cuMemMap failed");
  }
  release(h);                                                // the mapping keeps the memory until it is unmapped
  CUmemAccessDesc acc = {};
  acc.location = prop.location;
  acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  if (set_access(p, size, &acc, 1) != CUDA_SUCCESS) {
    bcg_free_image_memory(reinterpret_cast<void*>(p), (int64_t)size);
    return fail(BCG_ERR_CUDA, "cuMemSetAccess failed");
  }
  *dptr = reinterpret_cast<void*>(p);
  *mapped_bytes = (int64_t)size;
  *compressed = got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC ? 1 : 0;
  return BCG_OK;
}

int bcg_free_image_memory(void* dptr, int64_t mapped_bytes) {
  BCG_REQUIRE(dptr && mapped_bytes > 0, "bad argument");
  decltype(&cuMemUnmap) unmap = nullptr;
  decltype(&cuMemAddressFree) address_free = nullptr;
  if (int rc = driver_fn("cuMemUnmap", &unmap)) return rc;
  if (int rc = driver_fn("cuMemAddressFree", &address_free)) return rc;
  BCG_CHECK_CU(unmap(reinterpret_cast<CUdeviceptr>(dptr), (size_t)mapped_bytes));
  BCG_CHECK_CU(address_free(reinterpret_cast<CUdeviceptr>(dptr), (size_t)mapped_bytes));
  return BCG_OK;
}

int bcg_init_state(const BcgParams* p, const BcgBatch* b, const BcgEnvRows* rows, void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  if (int rc = check_rows(rows)) return rc;
  const int64_t grid = blocks_for((int64_t)b->n_envs * 32, 256);
  if (rows)
    init_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(*p, *b, make_layout(*p), *rows);
  else
    init_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(*p, *b, make_layout(*p), BcgEnvRows{nullptr, nullptr});
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_generate_aisles(const BcgParams* p, const BcgBatch* b, const BcgEnvRows* rows, const BcgAisleSlots* slots,
                        const uint8_t* mask, const BcgTurnParams* turn_params, uint64_t draw_index, double path_delta,
                        void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  if (int rc = check_rows(rows)) return rc;
  if (int rc = check_slots(p, b, slots, path_delta, "bcg_generate_aisles")) return rc;
  if (rows)
    generate_aisles_kernel<true><<<b->n_envs, 256, 0, (cudaStream_t)stream>>>(*p, *b, make_layout(*p), *slots, mask, turn_params,
                                                                           draw_index, path_delta, *rows);
  else
    generate_aisles_kernel<false><<<b->n_envs, 256, 0, (cudaStream_t)stream>>>(*p, *b, make_layout(*p), *slots, mask, turn_params,
                                                                            draw_index, path_delta, BcgEnvRows{nullptr, nullptr});
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_generate_minis(const BcgParams* p, const BcgBatch* b, const BcgAisleSlots* slots, const uint8_t* mask,
                       const BcgMiniGenParams* gen, const BcgMiniParams* mini_params, BcgMiniParams* params_out,
                       uint64_t draw_index, double path_delta, void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  if (int rc = check_slots(p, b, slots, path_delta, "bcg_generate_minis")) return rc;
  BCG_REQUIRE(gen || mini_params, "need the sampling space (gen) or explicit MiniEnvParams");
  BcgMiniGenParams g;
  memset(&g, 0, sizeof(g));
  if (gen) g = *gen;
  generate_minis_kernel<<<b->n_envs, 128, 0, (cudaStream_t)stream>>>(*p, *b, make_layout(*p), *slots, mask, g, mini_params,
                                                                    params_out, draw_index, path_delta);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_reset_where(const BcgBatch* b, const uint8_t* mask, void* stream) {
  BCG_REQUIRE(b && b->state_f && b->init_f && b->state_i && b->init_i && b->n_envs > 0, "bad batch");
  reset_kernel<<<blocks_for(b->n_envs, 256), 256, 0, (cudaStream_t)stream>>>(*b, mask);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

static int check_ego(const BcgParams* p, const BcgBatch* b, const uint8_t* ego_image) {
  BCG_REQUIRE(p->ego_w > 0 && p->ego_h > 0 && p->ego_w <= BCG_EGO_MAX && p->ego_h <= BCG_EGO_MAX,
              "egocentric crop must be 1..256 pixels per side");
  if (ego_image) {
    BCG_REQUIRE(b->ego_work, "BcgBatch.ego_work is needed for the egocentric image");
    BCG_REQUIRE(b->cell_tile_arena, "the egocentric image needs the cell-tile planes (BcgBatch.cell_tile_arena)");
  }
  return BCG_OK;
}

}  // extern "C"

// window capacity handed to the record writers.  Crops wider than the dense kernel's column table get 0: every record is
// then in direct mode, and the crop is rendered by the bounds-checked global gather
static int ego_capacity(const BcgParams& p) {
  return p.ego_w <= BCG_EGT_MAX_W ? ego_window_capacity(p) : 0;
}

static int sm_count_of_current_device(int* out) {
  static int cached[64] = {0};
  int dev = 0;
  BCG_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || cached[dev] == 0) {
    int n = 0;
    BCG_CHECK_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    if (dev >= 0 && dev < 64) cached[dev] = n;
    *out = n;
    return BCG_OK;
  }
  *out = cached[dev];
  return BCG_OK;
}

template <int NG, bool ENDS>
static int launch_ego_tiles(const BcgParams* p, const BcgBatch* b, uint8_t* ego_image, const int* env_list, const BcgEpisodeEnds& ends,
                            cudaStream_t s) {
  const int win = ego_window_capacity(*p);
  const int smem = win + (int)sizeof(EgoTab) + BCG_EGT_REC_SLOTS * BCG_EGO_WORK_BYTES;
  static int configured[64] = {0};    // per template instance and device: the attribute is per function and context
  int dev = 0;
  BCG_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || configured[dev] < smem) {
    BCG_CHECK_CUDA(cudaFuncSetAttribute(ego_tiles_kernel<NG, ENDS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (dev >= 0 && dev < 64) configured[dev] = smem;
  }
  int sms = 0;
  if (int rc = sm_count_of_current_device(&sms)) return rc;
  const int grid = b->n_envs < BCG_EGT_CTAS * sms ? b->n_envs : BCG_EGT_CTAS * sms;
  ego_tiles_kernel<NG, ENDS><<<grid, BCG_EGT_THREADS, smem, s>>>(*p, *b, ego_image, win, env_list, ends);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

template <bool ENDS>
static int launch_ego_dense(const BcgParams* p, const BcgBatch* b, uint8_t* ego_image, const int* env_list, const BcgEpisodeEnds& ends,
                            cudaStream_t s) {
  switch ((p->ego_w + 31) / 32) {
    case 1: return launch_ego_tiles<1, ENDS>(p, b, ego_image, env_list, ends, s);
    case 2: return launch_ego_tiles<2, ENDS>(p, b, ego_image, env_list, ends, s);
    case 3: return launch_ego_tiles<3, ENDS>(p, b, ego_image, env_list, ends, s);
    case 4: return launch_ego_tiles<4, ENDS>(p, b, ego_image, env_list, ends, s);
    default: return launch_ego_tiles<5, ENDS>(p, b, ego_image, env_list, ends, s);
  }
}

// the dense kernel, with the final crops of `ends` (may be NULL) behind the envs
static int launch_ego_dense(const BcgParams* p, const BcgBatch* b, uint8_t* ego_image, const int* env_list, const BcgEpisodeEnds* ends,
                            cudaStream_t s) {
  if (ends) return launch_ego_dense<true>(p, b, ego_image, env_list, *ends, s);
  return launch_ego_dense<false>(p, b, ego_image, env_list, BcgEpisodeEnds{}, s);
}

// sparse scatter kernel for every env, then the dense kernel for the envs it handed over (usually none)
struct EgoHits {       // BcgStepOut.ego_hits / ego_hit_count / ego_hit_cap (all zero: no compact output)
  uint32_t* list;
  int32_t* count;
  int cap;
  bool pdl;            // launch the sparse kernel as a programmatic dependent of the kernel before it (the step path)
};

static int launch_ego_sparse(const BcgParams* p, const BcgBatch* b, uint8_t* ego_image, const EgoHits& hits, const BcgEpisodeEnds* ends,
                             cudaStream_t s) {
  int sms = 0;
  if (int rc = sm_count_of_current_device(&sms)) return rc;
  // (the hand-over count and the env counter in ego_list[n_envs ..] were zeroed by the state / prep kernel)
  // persistent CTAs, as many per SM as fit with this crop's tables (18 for the 117 x 133 crop)
  const int tab_bytes = (p->ego_w + p->ego_h + 4) * (int)sizeof(int2);     // + a sentinel before and after each table
  using SparseKernel = decltype(&ego_sparse_kernel<false, false>);
  static const SparseKernel kernels[2][2] = {         // [HITS][ENDS]
      {ego_sparse_kernel<false, false>, ego_sparse_kernel<false, true>},
      {ego_sparse_kernel<true, false>, ego_sparse_kernel<true, true>}};
  static int per_sm_cache[64] = {0}, tab_cache[64] = {0};
  int dev = 0;
  BCG_CHECK_CUDA(cudaGetDevice(&dev));
  int per_sm = 0;
  if (dev >= 0 && dev < 64 && per_sm_cache[dev] > 0 && tab_cache[dev] == tab_bytes) {
    per_sm = per_sm_cache[dev];
  } else {
    BCG_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernels[0][0], BCG_EGS_THREADS, tab_bytes));
    BCG_REQUIRE(per_sm > 0, "the sparse egocentric kernel does not fit an SM with this crop size");
    if (dev >= 0 && dev < 64) {
      per_sm_cache[dev] = per_sm;
      tab_cache[dev] = tab_bytes;
    }
  }
  const int grid = b->n_envs < per_sm * sms ? b->n_envs : per_sm * sms;
  // (the variant that also records the compact hit lists has the same shared-memory footprint and register budget)
  // When the batch's crops are about as large as L2 they linger there as dirty lines, and the next step's first kernels
  // start against their write-back: zero-filled with an L2 evict-first policy they leave early (8 192 envs: move_kernel
  // 0.029 -> 0.025 ms, reward_kernel 0.018 -> 0.017; profiles/r2ze_evict_first_by_batch.txt).  Larger batches stream
  // through L2 anyway; there the policy only makes the hit bytes miss the lines just written (65 536 envs: 0.209 ->
  // 0.225 ms), also when it is applied to the last crops alone (r2zf): off above the threshold.
  static const long long evict_bytes = [] {
    const char* v = getenv("BCG_EGO_EVICT_FIRST_BYTES");
    return v ? atoll(v) : 160ll << 20;
  }();
  const int evict = (long long)b->n_envs * p->ego_w * p->ego_h <= evict_bytes ? 0 : b->n_envs;   // evict_from: envs >= it use the policy
  const bool with_hits = hits.list != nullptr;
  // (the final crops of episode ends, when asked for, are the items behind the envs)
  const BcgEpisodeEnds en = ends ? *ends : BcgEpisodeEnds{};
  BCG_CHECK_CUDA(launch_step_kernel(kernels[with_hits][ends != nullptr], grid, BCG_EGS_THREADS, tab_bytes, s, hits.pdl, *p, *b,
                                    ego_image, hits.list, with_hits ? hits.count : nullptr, with_hits ? hits.cap : 0, evict, en));
  BCG_CHECK_CUDA(cudaGetLastError());
  if (b->flags & BCG_BATCH_SPARSE_EGO_ONLY) return BCG_OK;     // the sparse kernel rendered every env itself
  return launch_ego_dense(p, b, ego_image, b->ego_list, ends, s);
}

// BCG_EGO_KERNEL=dense forces the dense cell-tile kernel for every env (A/B timing of the sparse path)
static bool ego_dense_kernel_requested() {
  static const bool dense = [] {
    const char* v = getenv("BCG_EGO_KERNEL");
    return v && strcmp(v, "dense") == 0;
  }();
  return dense;
}

// the image kernel(s); the per-env records must already be in b->ego_work (and those of the final crops of `ends`, which
// may be NULL, in ends->final_ego_work)
static int launch_ego_image(const BcgParams* p, const BcgBatch* b, uint8_t* ego_image, const EgoHits& hits, const BcgEpisodeEnds* ends,
                            cudaStream_t s) {
  if (b->ego_list && !ego_dense_kernel_requested()) return launch_ego_sparse(p, b, ego_image, hits, ends, s);
  BCG_REQUIRE(!hits.list, "the compact egocentric output (BcgStepOut.ego_hits) comes from the sparse kernel: ego_list is needed");
  return launch_ego_dense(p, b, ego_image, nullptr, ends, s);
}

extern "C" {

int bcg_observe_ego(const BcgParams* p, const BcgBatch* b, uint8_t* ego_image, float* goal_n_state, void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  BCG_REQUIRE(ego_image || goal_n_state, "nothing to compute");
  if (int rc = check_ego(p, b, ego_image)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  ego_prep_kernel<<<blocks_for(b->n_envs, 128), 128, 0, s>>>(*p, *b, ego_image ? 1 : 0, goal_n_state,
                                                            ego_capacity(*p));
  BCG_CHECK_CUDA(cudaGetLastError());
  if (ego_image) return launch_ego_image(p, b, ego_image, EgoHits{nullptr, nullptr, 0, false}, nullptr, s);
  return BCG_OK;
}

}  // extern "C"

static int check_ends(const BcgStepOut* out, const BcgEpisodeEnds* ends) {
  if (!ends) return BCG_OK;
  BCG_REQUIRE(ends->capacity >= 1, "BcgEpisodeEnds.capacity must be at least 1");
  BCG_REQUIRE(ends->reason && ends->final_slot && ends->final_obs_vec && ends->final_return && ends->final_length && ends->count,
              "BcgEpisodeEnds: reason, final_slot, final_obs_vec, final_return, final_length and count are needed");
  if (out->goal_n_state) BCG_REQUIRE(ends->final_goal_n_state, "BcgEpisodeEnds.final_goal_n_state is needed with goal_n_state");
  if (out->ego_image)
    BCG_REQUIRE(ends->final_ego_work && ends->final_ego_image && ends->final_list,
                "BcgEpisodeEnds: final_ego_work, final_ego_image and final_list are needed with ego_image");
  return BCG_OK;
}

extern "C" {

int bcg_step(const BcgParams* p, const BcgBatch* b, const BcgEnvRows* rows, const void* actions, int32_t action_is_f64,
             uint64_t step_index, const BcgStepOut* out, const BcgEpisodeEnds* ends, void* const* events, void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  if (int rc = check_rows(rows)) return rc;
  BCG_REQUIRE(actions && out, "null actions/out");
  if (int rc = check_ends(out, ends)) return rc;
  const bool ego = out->ego_image || out->goal_n_state;
  if (ego) {
    if (int rc = check_ego(p, b, out->ego_image)) return rc;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const BcgStateLayout L = make_layout(*p);
  const bool new_world = p->auto_reset == BCG_AUTO_RESET_NEW_WORLD;
  if (events && events[0]) BCG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)events[0], s));
  {
    if (events && events[1]) BCG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)events[1], s));
    const int cap = ego ? ego_capacity(*p) : 0;
    // (event records between the kernels are stream operations of their own: the timed form runs without the overlap)
    const bool pdl = !(events && (events[0] || events[1]));          // an event right before a kernel: no overlap for it
    const bool pdl_reward = !(events && events[2]);
    const BcgEnvRows r = rows ? *rows : BcgEnvRows{nullptr, nullptr};
    const BcgEpisodeEnds en = ends ? *ends : BcgEpisodeEnds{};
    // move_kernel at the register tier the batch size picks
    using MoveKernel = decltype(&move_kernel<BCG_MOVE_MIN_BLOCKS, false, false>);
    static const MoveKernel moves[3][2][2] = {      // [tier][ROWS][ENDS]
        {{move_kernel<BCG_MOVE_FEWER_BLOCKS, false, false>, move_kernel<BCG_MOVE_FEWER_BLOCKS, false, true>},
         {move_kernel<BCG_MOVE_FEWER_BLOCKS, true, false>, move_kernel<BCG_MOVE_FEWER_BLOCKS, true, true>}},
        {{move_kernel<BCG_MOVE_FEW_BLOCKS, false, false>, move_kernel<BCG_MOVE_FEW_BLOCKS, false, true>},
         {move_kernel<BCG_MOVE_FEW_BLOCKS, true, false>, move_kernel<BCG_MOVE_FEW_BLOCKS, true, true>}},
        {{move_kernel<BCG_MOVE_MIN_BLOCKS, false, false>, move_kernel<BCG_MOVE_MIN_BLOCKS, false, true>},
         {move_kernel<BCG_MOVE_MIN_BLOCKS, true, false>, move_kernel<BCG_MOVE_MIN_BLOCKS, true, true>}}};
    int sms = 0;
    if (int rc = sm_count_of_current_device(&sms)) return rc;
    const int move_blocks = (int)blocks_for(b->n_envs, BCG_MOVE_THREADS);
    const int tier = move_blocks <= sms * BCG_MOVE_FEWER_BLOCKS ? 0 : move_blocks <= sms * BCG_MOVE_FEW_BLOCKS ? 1 : 2;
    BCG_CHECK_CUDA(launch_step_kernel(moves[tier][rows != nullptr][ends != nullptr], move_blocks, BCG_MOVE_THREADS, 0, s, pdl,
                                      *p, *b, L, actions, (int)action_is_f64, step_index, *out, cap, r, en.count));
    if (events && events[2]) BCG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)events[2], s));
    // reward_kernel with the lane group the batch size picks
    using RewardKernel = decltype(&reward_kernel<8, false, false>);
    static const RewardKernel rewards[3][2][2] = {  // [group 8, 16, 32][ROWS][ENDS]
        {{reward_kernel<8, false, false>, reward_kernel<8, false, true>}, {reward_kernel<8, true, false>, reward_kernel<8, true, true>}},
        {{reward_kernel<16, false, false>, reward_kernel<16, false, true>}, {reward_kernel<16, true, false>, reward_kernel<16, true, true>}},
        {{reward_kernel<32, false, false>, reward_kernel<32, false, true>}, {reward_kernel<32, true, false>, reward_kernel<32, true, true>}}};
    const int64_t ns = b->n_envs;
    const int group = ns > 16384 ? 0 : ns > 2048 ? 1 : 2;
    BCG_CHECK_CUDA(launch_step_kernel(rewards[group][rows != nullptr][ends != nullptr], blocks_for(ns * (8 << group), BCG_REWARD_THREADS),
                                      BCG_REWARD_THREADS, 0, s, pdl_reward, *p, *b, *out, cap, en));
    BCG_CHECK_CUDA(cudaGetLastError());
    if (new_world) {
      const int grid = b->n_envs < BCG_REGEN_CTAS * sms ? b->n_envs : BCG_REGEN_CTAS * sms;
      BCG_CHECK_CUDA(launch_step_kernel(rows ? regenerate_kernel<true> : regenerate_kernel<false>, grid, BCG_REGEN_THREADS, 0, s, true,
                                        *p, *b, L, r, *out, cap, en, step_index));
    }
  }
  if (events && events[3]) BCG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)events[3], s));
  if (out->ego_image) {
    BCG_REQUIRE((out->ego_hits != nullptr) == (out->ego_hit_count != nullptr) && (!out->ego_hits || out->ego_hit_cap > 0),
                "ego_hits, ego_hit_count and ego_hit_cap go together");
    // (a new-world batch's final crops were rendered by regenerate_kernel)
    if (int rc = launch_ego_image(p, b, out->ego_image, EgoHits{out->ego_hits, out->ego_hit_count, out->ego_hit_cap, !(events && events[3])},
                                  new_world ? nullptr : ends, s))
      return rc;
  }
  if (events && events[4]) BCG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)events[4], s));
  return BCG_OK;
}

int bcg_rollout(const BcgParams* p, const BcgBatch* b, const BcgEnvRows* rows, const float* plan, int32_t horizon,
                uint64_t step_index, const BcgStepOut* out, const BcgEpisodeEnds* ends, void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  BCG_REQUIRE(plan && horizon >= 0, "null plan / negative horizon");
  for (int32_t h = 0; h < horizon; ++h)
    if (int rc = bcg_step(p, b, rows, plan + (int64_t)h * b->n_envs * 2, 0, step_index + (uint64_t)h, out, ends, nullptr, stream))
      return rc;
  return BCG_OK;
}

static int launch_collision_kernel(const BcgBatch* b, uint8_t* flags_out, int32_t* pixels_out, int use_u8, cudaStream_t s) {
  const int grid = blocks_for((int64_t)b->n_envs * 32, 256);
  if (use_u8) collision_kernel<2><<<grid, 256, 0, s>>>(*b, flags_out, nullptr);
  else if (pixels_out) collision_kernel<1><<<grid, 256, 0, s>>>(*b, flags_out, pixels_out);
  else collision_thread_kernel<<<blocks_for(b->n_envs, 64), 64, 0, s>>>(*b, flags_out);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

static int launch_collision(const BcgParams* p, const BcgBatch* b, const double* poses, uint8_t* flags_out,
                            int32_t* pixels_out, int use_u8, cudaStream_t s) {
  // NULL: the poses the last step proposed (rows 0..2 of b->cand have the [3][n] layout of `poses`)
  pose_prep_kernel<<<blocks_for(b->n_envs, 128), 128, 0, s>>>(*p, *b, poses ? poses : b->cand);
  BCG_CHECK_CUDA(cudaGetLastError());
  return launch_collision_kernel(b, flags_out, pixels_out, use_u8, s);
}

int bcg_collision(const BcgParams* p, const BcgBatch* b, const double* poses, uint8_t* flags_out, int32_t* pixels_out,
                  void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  BCG_REQUIRE(flags_out, "null flags");
  return launch_collision(p, b, poses, flags_out, pixels_out, 0, (cudaStream_t)stream);
}

int bcg_collision_u8(const BcgParams* p, const BcgBatch* b, const double* poses, uint8_t* flags_out, void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  BCG_REQUIRE(flags_out, "null flags");
  return launch_collision(p, b, poses, flags_out, nullptr, 1, (cudaStream_t)stream);
}

int bcg_collision_recheck(const BcgParams* p, const BcgBatch* b, uint8_t* flags_out, int32_t use_u8, void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  BCG_REQUIRE(flags_out, "null flags");
  return launch_collision_kernel(b, flags_out, nullptr, use_u8, (cudaStream_t)stream);
}

int bcg_gather_state(const BcgBatch* b, const int64_t* idx, int32_t k, double* out_f, int32_t* out_i, void* stream) {
  BCG_REQUIRE(b && idx && out_f && out_i && k >= 0, "bad gather arguments");
  if (k == 0) return BCG_OK;
  gather_kernel<<<blocks_for(k, 256), 256, 0, (cudaStream_t)stream>>>(*b, idx, k, out_f, out_i);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_scatter_state(const BcgBatch* b, const int64_t* idx, int32_t k, const double* in_f, const int32_t* in_i,
                      int32_t load_delayed_robot, void* stream) {
  BCG_REQUIRE(b && idx && in_f && in_i && k >= 0, "bad scatter arguments");
  if (k == 0) return BCG_OK;
  scatter_kernel<<<blocks_for(k, 256), 256, 0, (cudaStream_t)stream>>>(*b, idx, k, in_f, in_i, load_delayed_robot);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_pack_ego_hits(const uint32_t* hits, const int32_t* counts, int32_t cap, int32_t n, const int64_t* offsets,
                      void* packed, int32_t offsets_only, void* stream) {
  BCG_REQUIRE(hits && counts && offsets && packed && cap > 0 && n >= 0, "bad pack arguments");
  if (n == 0) return BCG_OK;
  if (offsets_only) pack_hits_kernel<true><<<blocks_for((int64_t)n * 8, 256), 256, 0, (cudaStream_t)stream>>>(hits, counts, cap, n, offsets, packed);
  else pack_hits_kernel<false><<<blocks_for((int64_t)n * 8, 256), 256, 0, (cudaStream_t)stream>>>(hits, counts, cap, n, offsets, packed);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_masked_any_equal(const uint8_t* values, const uint8_t* mask, int64_t n, int32_t value, int32_t* flag_out, void* stream) {
  BCG_REQUIRE(values && mask && flag_out && n >= 0 && value >= 0 && value <= 255, "bad masked_any_equal arguments");
  cudaStream_t s = (cudaStream_t)stream;
  BCG_CHECK_CUDA(cudaMemsetAsync(flag_out, 0, sizeof(int32_t), s));
  if (n == 0) return BCG_OK;
  const int grid = (int)(n < 256 * 1024 ? blocks_for(n, 256) : 1024);
  masked_any_equal_kernel<<<grid, 256, 0, s>>>(values, mask, n, (uint8_t)value, flag_out);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_inverse_transform(const double* transforms, int64_t n, double* out, void* stream) {
  BCG_REQUIRE(transforms && out && n >= 0, "bad inverse_transform arguments");
  if (n == 0) return BCG_OK;
  inverse_transform_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(transforms, n, out);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_project_poses(const double* transform_host, const double* poses, int64_t n, double* out, void* stream) {
  BCG_REQUIRE(transform_host && poses && out && n >= 0, "bad project_poses arguments");
  if (n == 0) return BCG_OK;
  project_poses_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(transform_host[0], transform_host[1], transform_host[2],
                                                                           poses, n, out);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_observe_ego_path(const BcgParams* p, const BcgBatch* b, int32_t max_points, double* out, int32_t* len_out, void* stream) {
  if (int rc = check_batch(p, b)) return rc;
  BCG_REQUIRE(out && max_points > 0, "bad ego path arguments");
  ego_path_kernel<<<blocks_for((int64_t)b->n_envs * 32, 256), 256, 0, (cudaStream_t)stream>>>(*p, *b, max_points, out, len_out);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_world_to_pixel(const double* xy, int64_t n, double origin_x, double origin_y, double resolution, int32_t* out,
                       void* stream) {
  BCG_REQUIRE(xy && out && n >= 0 && resolution > 0, "bad world_to_pixel arguments");
  if (n == 0) return BCG_OK;
  w2p_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(xy, n, origin_x, origin_y, 1. / resolution, out);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

int bcg_normalize_angle(const double* in, int64_t n, double* out, void* stream) {
  BCG_REQUIRE(in && out && n >= 0, "bad normalize_angle arguments");
  if (n == 0) return BCG_OK;
  wrap_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(in, n, out);
  BCG_CHECK_CUDA(cudaGetLastError());
  return BCG_OK;
}

}  // extern "C"
