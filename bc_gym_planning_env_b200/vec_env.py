"""VecPlanEnv: N independent `PlanEnv`s stepped as one batch on a B200.

State lives in HBM as structure-of-arrays (fp64 rows x N, int32 rows x N; row map in
include/bcg_b200.h), costmaps and refined paths in arenas with per-map / per-path descriptors.
`step` is one call into the C-ABI (`bcg_step`): kinematics -> collision -> reward -> done
(-> egocentric observation), i.e. reference envs/base/env.py:334-361 for every env at once.
PyTorch is used for device memory, streams and (elsewhere) torch.distributed only.
"""
import ctypes as C
import os

import numpy as np
import torch

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200 import env_params as envp
from bc_gym_planning_env_b200.envs.base.params import CONTINUOUS_REWARD, CONTINUOUS_REWARD_PURE_PURSUIT, EnvParams
from bc_gym_planning_env_b200.footprint_lut import FootprintLut
from bc_gym_planning_env_b200.robot_models.robot_dimensions import TRICYCLE, get_dimensions_example
from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
from bc_gym_planning_env_b200.utilities.path_tools import refine_path

# PlanEnv's hard-wired odometry noise (reference envs/base/env.py:226-232)
DEFAULT_NOISE = dict(alpha1=0.0, alpha2=0.0, alpha3=1.e-2, alpha4=1.e-2, alpha5=1.e-3, alpha6=1.e-3)

EGO_X_BOUNDS = (-0.5, 3.)   # reference envs/egocentric.py:113-114
EGO_Y_BOUNDS = (-2., 2.)

_LUT_CACHE = {}


def _round_up(v, m):
    return (v + m - 1) // m * m


def footprint_lut_for(robot_name, resolution, footprint_scale=1.0, footprint=None):
    """Angle-bin table of a standard robot (cached) or of an explicit footprint polygon (n, 2)."""
    if footprint is not None:
        footprint = np.asarray(footprint, dtype=np.float64)
        key = ('custom', footprint.tobytes(), float(resolution), float(footprint_scale))
    else:
        key = (robot_name, float(resolution), float(footprint_scale))
    if key not in _LUT_CACHE:
        if footprint is None:
            footprint = get_dimensions_example(robot_name).footprint()
        _LUT_CACHE[key] = FootprintLut(footprint * footprint_scale, resolution)
    return _LUT_CACHE[key]


def _device_world_types():
    """batch classes whose maps are rewritten on the device (their descriptors' flags can change after a reset)"""
    from bc_gym_planning_env_b200 import vec_aisle_env
    return (vec_aisle_env._VecSlotEnv,)


class VecObservation(object):
    """Batched Observation (reference envs/base/obs.py:14-23): views into the live state tensors --
    like the reference's Observation they alias env state and change on the next step."""

    def __init__(self, env):
        self._env = env
        sf, si = env.state_f, env.state_i
        self.pose = sf[nat.F_DPOSE:nat.F_DPOSE + 3].t()            # [N, 3] delayed pose
        self.robot_state = sf[nat.F_DROBOT:nat.F_DROBOT + 7].t()   # [N, 7] delayed robot state
        self.time = sf[nat.F_TIME]
        self.target_idx = si[nat.I_TARGET]
        self.dt = env.params.dt

    def path(self, e):
        """Observation.path of env e (reference envs/base/env.py:421-433): `path[target_idx:]`, or
        `path[:target_idx + 1]` with the pure-pursuit reward provider (reward.py:120-124)."""
        t = int(self.target_idx[e])
        full = self._env.full_path(e)
        return full[:t + 1] if self._env.params.reward_provider_name == CONTINUOUS_REWARD_PURE_PURSUIT else full[t:]

    def costmap(self, e):
        return self._env.costmap(e)


class FinalObservation(object):
    """What the episodes that ended at the last step looked like at their end, before the auto-reset (device tensors,
    reused buffers that the next step overwrites; nothing here synchronises).  Rows are indexed by env and valid where
    `ended` is true:
      ended           bool [N]          the episode of env e ended at the last step
      obs_vec         float32 [N, 12]   the compact observation (delayed pose, delayed robot state, time, target index)
      goal_n_state    float32 [N, 9, 1] with the egocentric observation, else None
      episode_return  float64 [N]       the episode's return, this step's reward included
      episode_length  int32 [N]         its iterations
      slot            int32 [N]         env e's row of ego_image, -1 when it did not end or found no free slot
      ego_image       uint8 [capacity, H, W, 1] final crops by slot (with the egocentric observation, else None)
      count           int32 scalar      episodes that ended at the last step; more than `capacity` means that some ended
                                        envs (which ones is unspecified) have no crop: see VecPlanEnv.final_ego"""

    def __init__(self, **fields):
        self.__dict__.update(fields)


class VecState(object):
    """Snapshot of k env columns (reference `State`, envs/base/env.py:52-68): fp64 rows [F, k] and
    int32 rows [I, k].  Costmaps and paths are immutable per env, so a snapshot holds no copy of them."""

    def __init__(self, f, i):
        self.f, self.i = f, i

    def clone(self):
        return VecState(self.f.clone(), self.i.clone())


class VecPlanEnv(object):
    def __init__(self, costmaps, paths, params=None, n_envs=None, map_ids=None, path_ids=None,
                 noise_parameters=DEFAULT_NOISE, seed=0, auto_reset=False, device=None, env_id_base=0,
                 private_map_copies=False, with_ego=False, footprint_scale=1.0, footprint=None,
                 ego_staging='tiles', ego_sparse=True, compact_ego=False, params_ids=None, episode_ends=False,
                 episode_end_capacity=None):
        """
        :param costmaps: pool of CostMap2D (uint8), one resolution
        :param paths: pool of oriented paths, array(n, 3); refined here when params.refine_path
        :param params: one EnvParams shared by the batch, or a sequence of them (a pool: env e uses
            params[params_ids[e]]).  Delays, iteration_timeout, the goal tolerances and the progress multiplier may
            differ between the sets of a pool; dt, robot, resolution, reward provider, refine_path and path_delta may not
        :param map_ids, path_ids: [n_envs] indices into the pools (default: env e uses entry e % len)
        :param noise_parameters: dict alpha1..alpha6 or None (noise off); PlanEnv's default is on.  With a pool also a
            sequence of such settings, one per set
        :param params_ids: [n_envs] indices into the params pool (default e % len(pool)); only with a pool
        :param private_map_copies: give every env its own copy of its costmap in HBM (pool replicated
            on device) instead of sharing pool entries
        :param with_ego: assemble the egocentric observation inside every step
        :param footprint: explicit footprint polygon array(n, 2) in metres (default: the robot's own)
        :param ego_staging: how the egocentric kernels stage the source window; 'tiles' is the only value: a derived
            copy of every costmap in 128-byte cell tiles, of which only the tiles the rotated window touches are read
        :param compact_ego: also keep, per env, the list of non-zero crop pixels (BcgStepOut.ego_hits): what
            `step_host(images='compact')` sends to the host instead of whole crops (needs with_ego and the sparse kernel)
        :param ego_sparse: render crops with the sparse scatter kernel (occupancy plane; the dense
            cell-tile kernel only takes the envs it hands over).  False: the dense kernel renders every env
        :param episode_ends: report every step why envs are done (`terminated`, `truncated`, `episode_reason`) and keep
            the final observation of every episode that ends (`final_observation()`), also when `auto_reset` has already
            replaced it.  Computed in the step's own kernels (no extra launch)
        :param episode_end_capacity: final crops kept per step (default n_envs, which never overflows; 1 .. n_envs)
        """
        costmaps = list(costmaps)
        paths = list(paths)
        if not costmaps or not paths:
            raise ValueError("need at least one costmap and one path")
        n = int(n_envs if n_envs is not None else max(len(costmaps), len(paths)))
        # the sparse kernel pays off on maps that are mostly free space; when every map of the pool is above the
        # library's dense threshold (1 cell in 20 occupied) it would only hand every env over: leave it out
        self._ego_sparse = bool(ego_sparse) and not all(
            np.count_nonzero(c.get_data()) * 20 > c.get_data().size for c in costmaps)
        self._compact_ego = bool(compact_ego)
        self._configure(params, n, float(costmaps[0].get_resolution()), noise_parameters, seed, auto_reset, device,
                        env_id_base, with_ego, ego_staging, params_ids, episode_ends, episode_end_capacity)
        self._map_pool = costmaps
        self._map_ids_host = (np.arange(n) % len(costmaps)) if map_ids is None else np.asarray(map_ids, dtype=np.int64)
        self._path_ids_host = (np.arange(n) % len(paths)) if path_ids is None else np.asarray(path_ids, dtype=np.int64)
        assert self._map_ids_host.shape == (n,) and self._path_ids_host.shape == (n,)
        self._upload_maps(costmaps, private_map_copies)
        self._upload_paths(paths)
        self._upload_lut(footprint_lut_for(self.params.robot_name, self.resolution, footprint_scale, footprint))
        self._alloc_state()
        self._make_batch()
        s = self._stream()
        nat.check(nat.lib().bcg_build_lethal_tiles(C.byref(self._batch), 0, self._batch.n_maps, s))
        nat.check(nat.lib().bcg_build_cell_tiles(C.byref(self._batch), 0, self._batch.n_maps, s))
        nat.check(nat.lib().bcg_init_state(C.byref(self._c_params), C.byref(self._batch), self._rows, s))
        self.check_status()
        if self._ego_list is not None:
            # bcg_build_lethal_tiles counted the occupied cells of every map: when none is above the library's dense
            # threshold (1 cell in 20) no env is ever handed to the dense egocentric kernel, so it is not launched
            d = np.frombuffer(self.map_descs.cpu().numpy().tobytes(), dtype=np.dtype(nat.BcgMapDesc))
            dense = d['occupied'].astype(np.int64) * 20 > d['width'].astype(np.int64) * d['height'].astype(np.int64)
            if not dense.any():
                self._batch.flags |= nat.BATCH_SPARSE_EGO_ONLY

    def _configure(self, params, n_envs, resolution, noise_parameters, seed, auto_reset, device, env_id_base, with_ego,
                   ego_staging, params_ids=None, episode_ends=False, episode_end_capacity=None):
        """Everything that does not depend on where the maps and paths come from."""
        if isinstance(auto_reset, str):
            if auto_reset != 'new_world':
                raise ValueError("auto_reset must be True, False or 'new_world', got %r" % (auto_reset,))
            if not isinstance(self, _device_world_types()):
                raise ValueError("auto_reset='new_world' needs worlds drawn on the device (VecRandomAisleTurnEnv, "
                                 "VecRandomMiniEnv): the maps of this batch were uploaded by the host and have no slots")
        self.new_world_reset = auto_reset == 'new_world'      # (the batch of device-drawn worlds sets it up)
        self.episode_ends = bool(episode_ends)
        self.episode_end_capacity = None
        if self.episode_ends:
            cap = int(n_envs) if episode_end_capacity is None else int(episode_end_capacity)
            if not 1 <= cap <= int(n_envs):
                raise ValueError("episode_end_capacity must be in [1, n_envs=%d], got %d" % (int(n_envs), cap))
            self.episode_end_capacity = cap
        elif episode_end_capacity is not None:
            raise ValueError("episode_end_capacity needs episode_ends=True")
        nat.require_cuda()
        self._pool = self._noise_pool = self._env_rows = None
        if envp.is_pool(params):
            # a pool: per-env rows (BcgEnvRows); self.params is set 0, whose batch-wide fields every set shares
            self._pool = envp.check_pool(params)
            self._noise_pool = envp.normalize_noise(len(self._pool), noise_parameters)
            self._env_rows = envp.build_env_rows(self._pool, self._noise_pool, params_ids, n_envs)
            self._params_ids_host = (np.arange(int(n_envs)) % len(self._pool) if params_ids is None
                                     else np.asarray(params_ids, dtype=np.int64).copy())
            params, noise_parameters = self._pool[0], self._noise_pool[0]
        elif params_ids is not None:
            raise ValueError("params_ids needs a pool of EnvParams (a sequence) as params")
        self.params = params if params is not None else EnvParams()
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        if self.device.type != 'cuda':
            raise nat.BcgError("VecPlanEnv runs on a CUDA device only (no CPU path)")
        self.n_envs = int(n_envs)
        self.resolution = float(resolution)
        self.dims = get_dimensions_example(self.params.robot_name)
        self.robot_kind = nat.ROBOT_TRICYCLE if self.dims.drive_type == TRICYCLE else nat.ROBOT_DIFFDRIVE
        self.auto_reset = bool(auto_reset)
        self.with_ego = bool(with_ego)
        if ego_staging != 'tiles':
            raise ValueError("ego_staging must be 'tiles' (the TMA and span staging were removed), got %r" % (ego_staging,))
        self.ego_staging = ego_staging
        self._step_index = 0
        self._graph = None
        self._plan_graph = None
        self._c_params = self._make_params(noise_parameters, seed, env_id_base)
        self._rows = None                                  # BcgEnvRows* of the library calls (None: batch-wide params)
        if self._env_rows is not None:
            cp = self._c_params
            cp.delay_control, cp.delay_pose, cp.delay_state = self._env_rows.capacities     # ring capacities
            self.env_rows_f = self._to_device(self._env_rows.f)
            self.env_rows_i = self._to_device(self._env_rows.i)
            self._c_rows = nat.BcgEnvRows(self.env_rows_f.data_ptr(), self.env_rows_i.data_ptr())
            self._rows = C.byref(self._c_rows)
        self.layout = nat.state_layout(self._c_params)

    # ---- setup -------------------------------------------------------------------------------
    def _make_params(self, noise, seed, env_id_base):
        p, rp, d = self.params, self.params.reward_provider_params, self.dims
        cp = nat.BcgParams()
        cp.dt, cp.resolution, cp.inv_resolution = p.dt, self.resolution, 1. / self.resolution
        cp.spatial_precision, cp.angular_precision = rp.spatial_precision, rp.angular_precision
        cp.progress_multiplier = rp.spatial_progress_multiplier
        cp.wheel_base, cp.max_wheel_angle = d.front_wheel_from_axis, d.max_front_wheel_angle
        cp.max_wheel_delta = d.max_front_wheel_speed * p.dt
        cp.p_gain, cp.max_lin_acc, cp.max_ang_acc = d.front_column_model_p_gain, d.max_linear_acceleration, d.max_angular_acceleration
        if noise is not None:
            for k in range(6):
                cp.alpha[k] = float(noise['alpha%d' % (k + 1)])
        cp.noise_on = 0 if noise is None else 1
        # egocentric crop geometry (reference envs/egocentric.py:113-119, utilities/costmap_utils.py:46-49)
        size = np.array([EGO_X_BOUNDS[1] - EGO_X_BOUNDS[0], EGO_Y_BOUNDS[1] - EGO_Y_BOUNDS[0]])
        wh = np.round(size * (1. / self.resolution)).astype(int)
        cp.ego_w, cp.ego_h = int(wh[0]), int(wh[1])
        cp.ego_x0, cp.ego_y0 = EGO_X_BOUNDS[0], EGO_Y_BOUNDS[0]
        cp.ego_world_w = (cp.ego_x0 + self.resolution * cp.ego_w) - cp.ego_x0   # CostMap2D.world_size()
        cp.ego_world_h = (cp.ego_y0 + self.resolution * cp.ego_h) - cp.ego_y0
        cp.seed, cp.env_id_base = int(seed) & (2 ** 64 - 1), int(env_id_base)
        cp.robot_kind = self.robot_kind
        cp.delay_control, cp.delay_pose, cp.delay_state = p.control_delay, p.pose_delay, p.state_delay
        cp.iteration_timeout = p.iteration_timeout
        kinds = {CONTINUOUS_REWARD: nat.REWARD_CONTINUOUS, CONTINUOUS_REWARD_PURE_PURSUIT: nat.REWARD_PURE_PURSUIT}
        if p.reward_provider_name not in kinds:          # reward_provider_examples_factory.py:44-47
            raise AssertionError("Unknown reward provider: {}. Should be one of {}".format(p.reward_provider_name, list(kinds)))
        cp.reward_kind = kinds[p.reward_provider_name]
        cp.auto_reset = nat.AUTO_RESET_NEW_WORLD if self.new_world_reset else 1 if self.auto_reset else 0
        return cp

    def _to_device(self, arr):
        t = torch.from_numpy(np.ascontiguousarray(arr))
        return t.to(self.device, non_blocking=False)

    def _upload_maps(self, costmaps, private_copies):
        descs = (nat.BcgMapDesc * len(costmaps))()
        data_off, tile_off, ctile_off, sum_off = 0, 0, 0, 0
        capacity_at, capacities = [], []
        for k, cm in enumerate(costmaps):
            data = cm.get_data()
            if data.dtype != np.uint8 or data.ndim != 2:
                raise TypeError("costmap data must be a 2-d uint8 array")
            if float(cm.get_resolution()) != self.resolution:
                raise ValueError("all costmaps of a batch must share one resolution")
            h, w = data.shape
            d = descs[k]
            if h >= 32768 or w >= 32768:
                raise ValueError("costmaps are limited to 32767 cells per side")
            d.height, d.width, d.pitch = h, w, _round_up(w, 32)
            d.tiles_x, d.tiles_y = d.pitch // 32, (h + 15) // 16
            d.flags = nat.MAP_ONLY_LETHAL                   # cleared on device when a cell is neither 0 nor 254
            d.origin_x, d.origin_y = float(cm.get_origin()[0]), float(cm.get_origin()[1])
            d.ctiles_x, d.ctiles_y = d.pitch // 16, (h + 7) // 8
            d.data_off, d.tile_off, d.cell_tile_off, d.sum_off = data_off, tile_off, ctile_off, sum_off
            sum_off += d.tiles_y * ((d.tiles_x + 31) // 32)
            # the map's cell index (BCG_BATCH_CELL_INDEX trailer, filled by bcg_build_lethal_tiles): dense maps get none
            nnz = int(np.count_nonzero(data))
            if nnz * 20 <= h * w:
                capacity_at.append(sum_off)
                capacities.append(nnz)
                sum_off += 3 + d.tiles_x * d.tiles_y + nnz
            data_off += _round_up(h * d.pitch, 128)
            tile_off += d.tiles_x * d.tiles_y * 16
            ctile_off += d.ctiles_x * d.ctiles_y * 128
        arena = np.zeros(data_off, dtype=np.uint8)
        for k, cm in enumerate(costmaps):
            d = descs[k]
            view = arena[d.data_off:d.data_off + d.height * d.pitch].reshape(d.height, d.pitch)
            view[:, :d.width] = cm.get_data()
        pool_bytes, pool_words, pool_ctile_bytes, pool_sum_words = data_off, tile_off, ctile_off, sum_off
        sum_init = np.zeros(max(pool_sum_words, 1), dtype=np.int32)     # tile summaries zero, trailer capacities set
        sum_init[np.asarray(capacity_at, dtype=np.int64)] = capacities
        map_arena = self._to_device(arena)
        ids = self._map_ids_host
        if private_copies:
            # copy index = how many earlier envs use the same pool entry
            order = np.argsort(ids, kind='stable')
            copy_idx = np.empty(self.n_envs, dtype=np.int64)
            sorted_ids = ids[order]
            starts = np.r_[0, np.flatnonzero(np.diff(sorted_ids)) + 1]
            run_start = np.repeat(starts, np.diff(np.r_[starts, len(ids)]))
            copy_idx[order] = np.arange(len(ids)) - run_start
            copies = int(copy_idx.max()) + 1
            map_arena = map_arena.repeat(copies)
            # one descriptor per env: its pool entry's, with the offsets moved into the env's own copy of the pool
            pool = np.frombuffer(bytes(descs), dtype=np.dtype(nat.BcgMapDesc))
            rows = pool[ids].copy()
            rows['data_off'] += copy_idx * pool_bytes
            rows['tile_off'] += copy_idx * pool_words
            rows['cell_tile_off'] += copy_idx * pool_ctile_bytes
            if int((rows['sum_off'] + copy_idx * pool_sum_words).max()) >= 2 ** 31:
                raise ValueError("tile summaries of this batch exceed the 32-bit offsets of BcgMapDesc.sum_off")
            rows['sum_off'] += (copy_idx * pool_sum_words).astype(np.int32)
            table = (nat.BcgMapDesc * self.n_envs).from_buffer_copy(rows.tobytes())
            descs = table
            ids = np.arange(self.n_envs)
            pool_words *= copies
            pool_ctile_bytes *= copies
            pool_sum_words *= copies
            sum_init = np.tile(sum_init, copies)                     # every copy owns its trailers
        self._map_descs_host = descs
        self.map_arena = map_arena
        self.tile_arena = torch.zeros(max(pool_words, 1), dtype=torch.int32, device=self.device)
        self.cell_tile_arena = torch.empty(max(pool_ctile_bytes, 128), dtype=torch.uint8, device=self.device)
        # occupancy plane (cell != 0; same layout as the lethal plane) and its tile summary (one bit per 32 x 16 tile):
        # the sparse egocentric kernel scans them, and the collision check uses the summary to skip empty tiles
        self.occ_tile_arena = torch.zeros(max(pool_words, 1), dtype=torch.int32, device=self.device)
        if pool_sum_words >= 2 ** 31:
            raise ValueError("tile summaries of this batch exceed the 32-bit offsets of BcgMapDesc.sum_off")
        self.occ_sum_arena = self._to_device(sum_init)
        self._cell_index_trailers = True
        self.map_descs = self._to_device(np.frombuffer(bytes(descs), dtype=np.uint8).copy())
        self.map_id = self._to_device(ids.astype(np.int32))
        self._n_maps = len(descs)

    def _upload_paths(self, paths):
        p = self.params
        refined, descs = [], (nat.BcgPathDesc * len(paths))()
        off = 0
        for k, path in enumerate(paths):
            path = np.asarray(path, dtype=np.float64)
            if p.refine_path:
                path = refine_path(path, p.path_delta)
            assert path.ndim == 2 and path.shape[1] == 3
            refined.append(np.ascontiguousarray(path))
            d = descs[k]
            d.n, d.pitch = len(path), _round_up(len(path), 4)
            d.n_chunks = (d.n + 31) // 32
            d.chunk_pitch = _round_up(d.n_chunks, 4)
            d.off = off
            d.chunk_off = off + 5 * d.pitch
            off = d.chunk_off + 3 * d.chunk_pitch
        arena = np.zeros(off, dtype=np.float64)
        for k, path in enumerate(refined):
            d = descs[k]
            rows = arena[d.off:d.off + 5 * d.pitch].reshape(5, d.pitch)
            rows[0, :d.n], rows[1, :d.n], rows[2, :d.n] = path[:, 0], path[:, 1], path[:, 2]
            rows[3, :d.n], rows[4, :d.n] = np.cos(path[:, 2]), np.sin(path[:, 2])   # as path_tools.py:405 evaluates them
            ch = arena[d.chunk_off:d.chunk_off + 3 * d.chunk_pitch].reshape(3, d.chunk_pitch)
            for c in range(d.n_chunks):
                pts = path[32 * c:32 * c + 32, :2]
                ctr = 0.5 * (pts.min(axis=0) + pts.max(axis=0))
                rad = np.hypot(pts[:, 0] - ctr[0], pts[:, 1] - ctr[1]).max()
                ch[0, c], ch[1, c], ch[2, c] = ctr[0], ctr[1], rad * (1 + 1e-12) + 1e-9   # conservative bound
        self._paths_host = refined
        self._n_paths = len(refined)
        self._path_descs_host = descs
        self.path_arena = self._to_device(arena)
        self.path_descs = self._to_device(np.frombuffer(bytes(descs), dtype=np.uint8).copy())
        self.path_id = self._to_device(self._path_ids_host.astype(np.int32))

    def _upload_lut(self, lut):
        self.lut = lut
        a = lut.arrays()
        self._lut_dev = {k: self._to_device(v.view(np.int64) if v.dtype == np.uint64 else v) for k, v in a.items()}

    def _alloc_state(self):
        n, L = self.n_envs, self.layout
        dev = self.device
        self.state_f = torch.zeros((L.n_frows, n), dtype=torch.float64, device=dev)
        self.state_i = torch.zeros((L.n_irows, n), dtype=torch.int32, device=dev)
        self.init_f = torch.zeros_like(self.state_f)
        self.init_i = torch.zeros_like(self.state_i)
        self._cand = torch.zeros((3, n), dtype=torch.float64, device=dev)
        self._cand_i = torch.zeros((2, n), dtype=torch.int32, device=dev)
        self._work = torch.zeros((n, 192), dtype=torch.uint8, device=dev)
        self._ego_work = torch.zeros((n, 128), dtype=torch.uint8, device=dev)
        self._step_counter = torch.zeros(2, dtype=torch.int64, device=dev)
        self._status = torch.zeros(nat.STATUS_WORDS, dtype=torch.int32, device=dev)
        self._stats = torch.zeros(nat.STATS_WORDS, dtype=torch.float64, device=dev)
        self.reward = torch.zeros(n, dtype=torch.float64, device=dev)
        self._done_u8 = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._hit_u8 = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.obs_vec = torch.zeros((n, 12), dtype=torch.float32, device=dev)
        cp = self._c_params
        if self.episode_ends:
            cap = self.episode_end_capacity
            self._end_reason = torch.zeros(n, dtype=torch.uint8, device=dev)
            self._final_slot = torch.full((n,), -1, dtype=torch.int32, device=dev)
            self._final_obs_vec = torch.zeros((n, 12), dtype=torch.float32, device=dev)
            self._final_return = torch.zeros(n, dtype=torch.float64, device=dev)
            self._final_length = torch.zeros(n, dtype=torch.int32, device=dev)
            self._ends_count = torch.zeros(2, dtype=torch.int32, device=dev)
            self._end_flags = torch.zeros((3, n), dtype=torch.bool, device=dev)      # ended, terminated, truncated
            self._end_scratch = torch.zeros(n, dtype=torch.uint8, device=dev)
            self._final_goal_n_state = self._final_ego_work = self.final_ego_image = self._final_list = None
            if self.with_ego:
                self._final_goal_n_state = torch.zeros((n, 9, 1), dtype=torch.float32, device=dev)
                self._final_ego_work = torch.zeros((cap, 128), dtype=torch.uint8, device=dev)
                self._final_list = torch.zeros(cap, dtype=torch.int32, device=dev)
                # (before the step's crops: _new_image_tensor records whether the step's crops got compressed memory)
                self.final_ego_image = self._new_image_tensor((cap, cp.ego_h, cp.ego_w, 1))
        if self.with_ego:
            self.ego_image = self._new_image_tensor((n, cp.ego_h, cp.ego_w, 1))
            self.goal_n_state = torch.zeros((n, 9, 1), dtype=torch.float32, device=dev)
        else:
            self.ego_image = self.goal_n_state = None

    def _new_image_tensor(self, shape):
        """uint8 zeros for the egocentric crops, in an allocation with compute-data compression when the device grants
        one (bcg_alloc_image_memory: crops are mostly zeros -- the scatter kernel writes them 2 % faster, a GPU-resident
        consumer reads them 1.6 x faster; profiles/r2y_image_memory.txt).  BCG_IMAGE_MEMORY=plain: a torch tensor;
        =vmm: the same virtual-memory allocation without compression (the probe's control)."""
        mode = os.environ.get("BCG_IMAGE_MEMORY", "compressed")
        if mode not in ("plain", "compressed", "vmm"):
            raise ValueError("BCG_IMAGE_MEMORY must be plain, compressed or vmm")
        self.image_memory_compressed = False
        if mode != "plain" and int(np.prod(shape)) >= (1 << 20):      # small batches: not worth a 2 MB mapping of their own
            with torch.cuda.device(self.device):
                try:
                    block = nat.ImageMemory(int(np.prod(shape)), want_compression=(mode == "compressed"))
                except nat.BcgError:
                    if mode == "vmm":
                        raise
                    block = None                           # no virtual-memory API on this device / driver: torch's pool
                if block is not None and (block.compressed or mode == "vmm"):
                    self.image_memory_compressed = block.compressed
                    return block.tensor(shape)
                del block                                  # no compression on this device: nothing gained over torch's pool
        return torch.zeros(shape, dtype=torch.uint8, device=self.device)

    def _make_batch(self):
        b = nat.BcgBatch()
        b.n_envs, b.n_frows, b.n_irows = self.n_envs, self.layout.n_frows, self.layout.n_irows
        b.n_maps, b.n_paths = self._n_maps, self._n_paths
        b.state_f, b.state_i = self.state_f.data_ptr(), self.state_i.data_ptr()
        b.init_f, b.init_i = self.init_f.data_ptr(), self.init_i.data_ptr()
        b.cand, b.cand_i, b.work = self._cand.data_ptr(), self._cand_i.data_ptr(), self._work.data_ptr()
        b.ego_work = self._ego_work.data_ptr()
        b.map_id, b.path_id = self.map_id.data_ptr(), self.path_id.data_ptr()
        b.maps, b.paths = self.map_descs.data_ptr(), self.path_descs.data_ptr()
        b.map_arena, b.tile_arena, b.path_arena = self.map_arena.data_ptr(), self.tile_arena.data_ptr(), self.path_arena.data_ptr()
        d = self._lut_dev
        b.lut.edges, b.lut.verts, b.lut.header = d['edges'].data_ptr(), d['verts'].data_ptr(), d['header'].data_ptr()
        b.lut.rows, b.lut.fp_pix = d['rows'].data_ptr(), d['fp_pix'].data_ptr()
        b.lut.bucket_first, b.lut.n_buckets = d['bucket_first'].data_ptr(), self.lut.n_buckets
        b.lut.bins, b.lut.bin_stride = d['bins'].data_ptr(), int(d['bins'].shape[1])
        b.lut.bucket_scale = self.lut.bucket_scale
        b.lut.n_bins, b.lut.n_verts, b.lut.max_rows, b.lut.wpr = self.lut.n_bins, self.lut.n_verts, self.lut.max_rows, self.lut.wpr
        b.status, b.stats = self._status.data_ptr(), self._stats.data_ptr()
        b.cell_tile_arena = self.cell_tile_arena.data_ptr()
        b.occ_tile_arena, b.occ_sum_arena = self.occ_tile_arena.data_ptr(), self.occ_sum_arena.data_ptr()
        if getattr(self, '_cell_index_trailers', False):
            b.flags |= nat.BATCH_CELL_INDEX
        self._ego_list = None
        if getattr(self, '_ego_sparse', True):
            self._ego_list = torch.zeros(self.n_envs + 4, dtype=torch.int32, device=self.device)
            b.ego_list = self._ego_list.data_ptr()
        self._batch = b
        out = nat.BcgStepOut()
        out.reward, out.done, out.hit = self.reward.data_ptr(), self._done_u8.data_ptr(), self._hit_u8.data_ptr()
        out.obs_vec = self.obs_vec.data_ptr()
        if self.with_ego:
            out.ego_image, out.goal_n_state = self.ego_image.data_ptr(), self.goal_n_state.data_ptr()
        self._ego_hits = self._ego_hit_count = None
        if getattr(self, '_compact_ego', False):
            if not self.with_ego or self._ego_list is None:
                raise ValueError("compact_ego needs with_ego=True and the sparse egocentric kernel (ego_sparse, sparse maps)")
            self.EGO_HIT_CAP = 1024
            self._ego_hits = torch.zeros((self.n_envs, self.EGO_HIT_CAP), dtype=torch.int32, device=self.device)
            self._ego_hit_count = torch.zeros(self.n_envs, dtype=torch.int32, device=self.device)
            # (BcgStepOut.ego_hits is only set for the steps whose lists are wanted: step_host(images='compact'))
        self._out = out
        self._ends = None                                  # BcgEpisodeEnds* of the step calls (None: episode_ends off)
        if getattr(self, 'episode_ends', False):
            en = nat.BcgEpisodeEnds()
            en.reason, en.final_slot = self._end_reason.data_ptr(), self._final_slot.data_ptr()
            en.final_obs_vec, en.final_return = self._final_obs_vec.data_ptr(), self._final_return.data_ptr()
            en.final_length, en.count = self._final_length.data_ptr(), self._ends_count.data_ptr()
            if self.with_ego:
                en.final_goal_n_state, en.final_ego_work = self._final_goal_n_state.data_ptr(), self._final_ego_work.data_ptr()
                en.final_ego_image, en.final_list = self.final_ego_image.data_ptr(), self._final_list.data_ptr()
            en.capacity = self.episode_end_capacity
            self._c_ends = en
            self._ends = C.byref(self._c_ends)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- the env API ---------------------------------------------------------------------------
    @property
    def done(self):
        return self._done_u8.view(torch.bool)

    @property
    def hit(self):
        return self._hit_u8.view(torch.bool)

    def _ends_on(self):
        if not self.episode_ends:
            raise ValueError("this batch was built without episode_ends=True")

    @property
    def episode_reason(self):
        """uint8 [N] of the last step (needs episode_ends): nat.END_GOAL | END_COLLIDED | END_TIMEOUT, the causes of `done`,
        set while the env is done; nat.END_NOW, the episode ended at this step"""
        self._ends_on()
        return self._end_reason

    @property
    def terminated(self):
        """bool [N] (needs episode_ends): done by reaching the goal or by a collision -- no bootstrap from the final
        observation.  A reused buffer, like `done`."""
        self._ends_on()
        torch.bitwise_and(self._end_reason, nat.END_GOAL | nat.END_COLLIDED, out=self._end_scratch)
        return torch.ne(self._end_scratch, 0, out=self._end_flags[1])

    @property
    def truncated(self):
        """bool [N] (needs episode_ends): done by the iteration timeout alone (a goal or a collision on the same step
        terminates) -- bootstrap from the final observation.  A reused buffer, like `done`."""
        self._ends_on()
        torch.bitwise_and(self._end_reason, nat.END_GOAL | nat.END_COLLIDED | nat.END_TIMEOUT, out=self._end_scratch)
        return torch.eq(self._end_scratch, nat.END_TIMEOUT, out=self._end_flags[2])

    def action_bounds(self):
        """low, high of the action Box (reference envs/base/env.py:237-240), float32."""
        s = self.dims.max_front_wheel_speed
        return (np.array([s / 10, -np.pi / 2]).astype(np.float32), np.array([s / 2, np.pi / 2]).astype(np.float32))

    def _as_actions(self, actions):
        if isinstance(actions, np.ndarray):
            if actions.dtype not in (np.float32, np.float64):
                actions = actions.astype(np.float64)
            actions = torch.from_numpy(np.ascontiguousarray(actions)).to(self.device)
        if actions.dtype not in (torch.float32, torch.float64):
            actions = actions.to(torch.float64)
        if actions.device != self.device:
            actions = actions.to(self.device)
        if tuple(actions.shape) != (self.n_envs, 2):
            raise ValueError("actions must have shape (%d, 2), got %s" % (self.n_envs, tuple(actions.shape)))
        return actions.contiguous()

    def step(self, actions):
        """One env step for every env.  actions: [N, 2] float32/float64 (tensor or ndarray).
        Returns (VecObservation, reward fp64 [N], done bool [N], {}) -- tensors are reused buffers."""
        self._bcg_step(self._as_actions(actions), self._step_index, self._stream())
        self._step_index += 1
        return self.observation(), self.reward, self.done, {}

    def _bcg_step(self, actions, step_index, stream, events=None):
        """One bcg_step call on this batch: actions a float32 / float64 [N, 2] device tensor, stream a c_void_p,
        events None or the five cudaEvent_t handles."""
        nat.check(nat.lib().bcg_step(C.byref(self._c_params), C.byref(self._batch), self._rows, nat.ptr(actions),
                                     1 if actions.dtype == torch.float64 else 0, step_index, C.byref(self._out), self._ends,
                                     events, stream))

    def step_graph(self, actions=None):
        """`step` as ONE CUDA-graph launch: the first call captures the step's kernels (reading `self.actions`, a
        persistent float32 [N, 2] device buffer, and the device-side step counter) and every call replays them --
        one driver call per step instead of one per kernel plus the argument marshalling, which is what a small
        batch spends its time on.  `actions` (optional) is copied into `self.actions` first; a GPU-resident policy
        writes into `self.actions` itself and calls step_graph().  From the first call on the step index lives on the
        device (BcgBatch.step_counter); `step` keeps working and uses it too."""
        if self._graph is None:
            self.actions = torch.zeros((self.n_envs, 2), dtype=torch.float32, device=self.device)
            if actions is not None:
                self.actions.copy_(self._as_actions(actions))
            self._step_counter[0] = self._step_index
            self._step_counter[1] = 0
            self._batch.step_counter = self._step_counter.data_ptr()
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                with torch.cuda.graph(g, stream=side):
                    self._bcg_step(self.actions, 0, C.c_void_p(side.cuda_stream))
            torch.cuda.current_stream(self.device).wait_stream(side)
            self._graph = g
        elif actions is not None:
            self.actions.copy_(self._as_actions(actions), non_blocking=True)
        self._graph.replay()
        self._step_index += 1
        return self.observation(), self.reward, self.done, {}

    def rollout(self, plan):
        """H steps of a fixed action plan from ONE library call (bcg_rollout): the 2-3 kernels of every step are launched
        back to back, each a programmatic dependent of the one before -- no Python between the steps.  plan: float
        [H, N, 2] on the device.  Read `state_f` / `reward` (last step) / `done` afterwards; the episode return
        accumulates in row F_EP_RETURN."""
        plan = plan.to(self.device)
        if plan.dim() != 3 or tuple(plan.shape[1:]) != (self.n_envs, 2):
            raise ValueError("plan must have shape [H, %d, 2]" % self.n_envs)
        plan = plan.to(torch.float32).contiguous()
        horizon = int(plan.shape[0])
        nat.check(nat.lib().bcg_rollout(C.byref(self._c_params), C.byref(self._batch), self._rows, nat.ptr(plan), horizon,
                                        self._step_index, C.byref(self._out), self._ends, self._stream()))
        self._step_index += horizon

    def rollout_graph(self, plan):
        """H steps of a fixed action plan as ONE CUDA-graph launch (Monte-Carlo fan-outs: README.md:45-61 of the
        reference steps a copied env through a candidate plan).  plan: float [H, N, 2]; it is copied into a persistent
        device buffer whose H slices the captured steps read, the Philox step index comes from the device-side counter.
        The graph is captured on the first call for a given H and replayed afterwards.  Returns nothing: read
        `state_f` / `reward` (last step) / `done` afterwards; the episode return accumulates in row F_EP_RETURN."""
        plan = plan.to(self.device)
        if plan.dim() != 3 or tuple(plan.shape[1:]) != (self.n_envs, 2):
            raise ValueError("plan must have shape [H, %d, 2]" % self.n_envs)
        horizon = int(plan.shape[0])
        if self._plan_graph is None or self._plan_graph[0] != horizon:
            buf = torch.zeros((horizon, self.n_envs, 2), dtype=torch.float32, device=self.device)
            buf.copy_(plan)
            if self._batch.step_counter == 0 or self._batch.step_counter is None:
                self._step_counter[0] = self._step_index
                self._step_counter[1] = 0
                self._batch.step_counter = self._step_counter.data_ptr()
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                with torch.cuda.graph(g, stream=side):
                    for h in range(horizon):
                        self._bcg_step(buf[h], 0, C.c_void_p(side.cuda_stream))
            torch.cuda.current_stream(self.device).wait_stream(side)
            self._plan_graph = (horizon, g, buf)
        else:
            self._plan_graph[2].copy_(plan, non_blocking=True)
        self._plan_graph[1].replay()
        self._step_index += horizon

    def launches_per_step(self):
        """Kernels one `step` launches: move_kernel + reward_kernel (+ regenerate_kernel with auto_reset='new_world'), then
        the egocentric kernel(s)."""
        n = 3 if self.new_world_reset else 2
        if not self.with_ego:
            return n
        if self._ego_list is None or os.environ.get("BCG_EGO_KERNEL") == "dense":
            return n + 1                                   # one dense kernel
        return n + (1 if self._batch.flags & nat.BATCH_SPARSE_EGO_ONLY else 2)

    def step_timed(self, actions, events):
        """`step` with five torch.cuda.Event (enable_timing=True, already recorded once so that their
        handles exist; entries may be None) recorded around the kernels; see the `events` of bcg_step."""
        handles = (C.c_void_p * 5)(*[C.c_void_p(ev.cuda_event if ev is not None else None) for ev in events])
        self._bcg_step(self._as_actions(actions), self._step_index, self._stream(), handles)
        self._step_index += 1
        return self.observation(), self.reward, self.done, {}

    def step_host(self, actions_host, images=False):
        """One env step driven from the host: `actions_host` float32 [N, 2] in pinned memory goes to the device, and
        reward (fp64 [N]), done (uint8 [N]) and the compact observation (float32 [N, 12]: delayed pose, delayed
        robot state, time, target index) come back in pinned host buffers -- what a CPU-side policy or logger needs
        every step.  The device->host copies wait only for reward_kernel and run on a side stream while the
        egocentric kernel is still working; the images stay in HBM (`ego_image`) for a GPU-resident consumer.
        With `images` the egocentric crops (uint8 [N, H, W]) and goal_n_state (float32 [N, 9]) are copied to pinned
        host memory as well, after the egocentric kernel (N x 15.6 KB per step: the PCIe link then sets the pace).
        Returns (reward, done, obs_vec) host tensors -- plus (ego_image, goal_n_state) with `images` --, valid when
        this call returns.  It waits for exactly what it returns: without `images` that is the copies of reward / done /
        obs, not the egocentric kernel, which finishes in stream order behind them.  With episode_ends the episode ends
        and final observations are computed but stay on the device (`final_observation()`); copying them to the host
        here is not implemented yet."""
        if getattr(self, '_host_io', None) is None:
            n = self.n_envs
            self._host_io = dict(
                actions=torch.empty((n, 2), dtype=torch.float32, device=self.device),
                reward=torch.empty(n, dtype=torch.float64).pin_memory(),
                done=torch.empty(n, dtype=torch.uint8).pin_memory(),
                obs=torch.empty((n, 12), dtype=torch.float32).pin_memory(),
                stream=torch.cuda.Stream(device=self.device),
                upload=torch.cuda.Stream(device=self.device), uploaded=torch.cuda.Event(enable_timing=False),
                events=[torch.cuda.Event(enable_timing=False) for _ in range(5)])
            for ev in self._host_io['events']:
                ev.record()                                   # creates the handles bcg_step records into
        io = self._host_io
        if tuple(actions_host.shape) != (self.n_envs, 2) or actions_host.dtype != torch.float32:
            raise ValueError("actions_host must be a float32 tensor of shape (%d, 2)" % self.n_envs)
        main = torch.cuda.current_stream(self.device)
        # the actions go up on a stream of their own: the previous step's egocentric kernel may still be running on the
        # main stream (see below), and its move_kernel -- the reader of this buffer -- finished before that step returned
        with torch.cuda.stream(io['upload']):
            io['actions'].copy_(actions_host, non_blocking=True)
            io['uploaded'].record()
        main.wait_event(io['uploaded'])
        if images == 'compact':
            if self._ego_hits is None:
                raise ValueError("this batch was built without compact_ego=True")
            self._out.ego_hits, self._out.ego_hit_count = self._ego_hits.data_ptr(), self._ego_hit_count.data_ptr()
            self._out.ego_hit_cap = self.EGO_HIT_CAP
        try:
            # (only the event after reward_kernel: the kernels before it stay programmatic dependents of one another)
            self.step_timed(io['actions'], [None, None, None, io['events'][3], None])
        finally:
            self._out.ego_hits = self._out.ego_hit_count = None
            self._out.ego_hit_cap = 0
        side = io['stream']
        side.wait_event(io['events'][3])                      # recorded right after reward_kernel
        with torch.cuda.stream(side):
            io['reward'].copy_(self.reward, non_blocking=True)
            io['done'].copy_(self._done_u8, non_blocking=True)
            io['obs'].copy_(self.obs_vec, non_blocking=True)
        compact = None
        if images == 'compact':
            compact = self._compact_to_host(io, side)
            images = False
        if images:
            if self.ego_image is None:
                raise ValueError("this batch was built without the egocentric observation (with_ego=False)")
            if 'ego_image' not in io:
                io['ego_image'] = torch.empty(tuple(self.ego_image.shape), dtype=torch.uint8).pin_memory()
                io['goal_n_state'] = torch.empty(tuple(self.goal_n_state.shape), dtype=torch.float32).pin_memory()
            io['ego_image'].copy_(self.ego_image, non_blocking=True)
            io['goal_n_state'].copy_(self.goal_n_state, non_blocking=True)
        side.synchronize()
        if compact is not None or images:
            main.synchronize()                                # the crops were asked for: wait for the egocentric kernel too
        # (without `images` the call returns when reward / done / obs are on the host.  The egocentric kernel may still be
        # running: `ego_image` is valid for whatever is enqueued on the current stream next, and the next step_host call
        # queues behind it -- the host prepares the next actions meanwhile instead of leaving the GPU idle)
        if compact is not None:
            return io['reward'], io['done'], io['obs'], compact, io['goal_n_state']
        if images:
            return io['reward'], io['done'], io['obs'], io['ego_image'], io['goal_n_state']
        return io['reward'], io['done'], io['obs']

    def _compact_to_host(self, io, side):
        """The egocentric observation of the step just launched as per-env lists of non-zero pixels, packed on the
        device and copied to pinned host memory: dict(counts int32 [N] (-1 / > cap: see dense_envs), offsets int64 [N],
        packed (uint32 [total]: pixel offset | value << 16 -- or, when every map of the batch holds no cost value but 254,
        uint16 [total]: the pixel offsets alone, `value` = 254), dense_envs int64 [k], dense_images uint8 [k, H, W],
        bytes = bytes that crossed the link for the images).  Expand with `expand_compact`."""
        if self._ego_hits is None:
            raise ValueError("this batch was built without compact_ego=True")
        n, cap = self.n_envs, self.EGO_HIT_CAP
        if getattr(self, '_only_lethal', None) is None:          # (read once: do all maps hold nothing but 0 and 254?)
            d = np.frombuffer(self.map_descs.cpu().numpy().tobytes(), dtype=np.dtype(nat.BcgMapDesc))
            self._only_lethal = bool(np.all(d['flags'] & nat.MAP_ONLY_LETHAL)) and not isinstance(self, _device_world_types())
        short = self._only_lethal
        counts = self._ego_hit_count
        listed = (counts > 0) & (counts <= cap)
        c = torch.where(listed, counts, torch.zeros_like(counts)).to(torch.int64)
        ends = torch.cumsum(c, 0)
        offsets = (ends - c).contiguous()
        dense = torch.nonzero((counts < 0) | (counts > cap)).reshape(-1)
        total = int(ends[-1])                                    # (synchronises: the size of the copy is data)
        if 'packed_dev' not in io or io['packed_dev'].numel() < total:
            size = max(total * 5 // 4, n * 64)
            dt = torch.int16 if short else torch.int32
            io['packed_dev'] = torch.empty(size, dtype=dt, device=self.device)
            io['packed'] = torch.empty(size, dtype=dt).pin_memory()
            io['counts'] = torch.empty(n, dtype=torch.int32).pin_memory()
            io['offsets'] = torch.empty(n, dtype=torch.int64).pin_memory()
            io['goal_n_state'] = torch.empty(tuple(self.goal_n_state.shape), dtype=torch.float32).pin_memory()
        nat.check(nat.lib().bcg_pack_ego_hits(nat.ptr(self._ego_hits), nat.ptr(counts), cap, n, nat.ptr(offsets),
                                              nat.ptr(io['packed_dev']), 1 if short else 0, self._stream()))
        io['packed'][:total].copy_(io['packed_dev'][:total], non_blocking=True)
        io['counts'].copy_(counts, non_blocking=True)
        io['offsets'].copy_(offsets, non_blocking=True)
        io['goal_n_state'].copy_(self.goal_n_state, non_blocking=True)
        dense_images = None
        if dense.numel():
            dense_images = self.ego_image[dense].reshape(dense.numel(), self.ego_image.shape[1], self.ego_image.shape[2]).cpu()
        return dict(counts=io['counts'], offsets=io['offsets'], packed=io['packed'][:total], dense_envs=dense.cpu(),
                    dense_images=dense_images, cap=cap, value=254 if short else None,
                    bytes=total * (2 if short else 4) + n * 12 + (0 if dense_images is None else dense_images.numel()))

    @staticmethod
    def expand_compact(compact, height, width):
        """Host-side expander of `step_host(images='compact')`: uint8 [N, H, W] equal to `ego_image` byte for byte."""
        counts = compact['counts'].numpy()
        n = len(counts)
        out = np.zeros((n, height * width), dtype=np.uint8)
        listed = (counts > 0) & (counts <= compact['cap'])
        c = np.where(listed, counts, 0).astype(np.int64)
        env = np.repeat(np.arange(n), c)
        if compact['value'] is not None:                         # 16-bit offsets, one implied cost value
            out[env, compact['packed'].numpy().view(np.uint16)] = compact['value']
        else:
            words = compact['packed'].numpy().view(np.uint32)
            out[env, words & 0xffff] = (words >> 16).astype(np.uint8)
        out = out.reshape(n, height, width)
        if compact['dense_images'] is not None:
            out[compact['dense_envs'].numpy()] = compact['dense_images'].numpy()
        return out

    def reset(self, mask=None):
        """PlanEnv.reset for all envs (mask None) or those with mask[e] true."""
        m = self._mask(mask)
        nat.check(nat.lib().bcg_reset_where(C.byref(self._batch), nat.ptr(m), self._stream()))
        return self.observation()

    def _mask(self, mask):
        """uint8 [N] device tensor of a per-env mask (None stays None); the kernels index it by env id unchecked"""
        if mask is None:
            return None
        m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        if tuple(m.shape) != (self.n_envs,):
            raise ValueError("mask must have shape (%d,)" % self.n_envs)
        return m

    def observation(self):
        return VecObservation(self)

    def observe_colored_ego(self):
        """ColoredEgoCostmapRandomAisleTurnEnv._extract_egocentric_observation (reference
        envs/synth_turn_env.py:396-420) for every env: ('environment' uint8 [N,133,133,1] cropped about the TRUE
        robot pose over x in [-0.5, 3.5], y in [-2, 2]; 'goal' float32 [N,5,1] = unit vector towards the last
        path point in crop units, then v, w, wheel angle)."""
        import copy
        cp = copy.copy(self._c_params)
        x_bounds, y_bounds = (-0.5, 3.5), (-2., 2.)
        size = np.array([x_bounds[1] - x_bounds[0], y_bounds[1] - y_bounds[0]])
        wh = np.round(size * (1. / self.resolution)).astype(int)
        cp.ego_w, cp.ego_h = int(wh[0]), int(wh[1])
        cp.ego_x0, cp.ego_y0 = x_bounds[0], y_bounds[0]
        cp.ego_world_w = (cp.ego_x0 + self.resolution * cp.ego_w) - cp.ego_x0
        cp.ego_world_h = (cp.ego_y0 + self.resolution * cp.ego_h) - cp.ego_y0
        cp.ego_variant = 1
        if getattr(self, '_colored_image', None) is None:
            self._colored_image = torch.zeros((self.n_envs, cp.ego_h, cp.ego_w, 1), dtype=torch.uint8, device=self.device)
            self._colored_goal = torch.zeros((self.n_envs, 9), dtype=torch.float32, device=self.device)
        nat.check(nat.lib().bcg_observe_ego(C.byref(cp), C.byref(self._batch), nat.ptr(self._colored_image),
                                            nat.ptr(self._colored_goal), self._stream()))
        return self._colored_image, self._colored_goal[:, :5].unsqueeze(-1)

    def observe_ego(self):
        """EgocentricCostmap.observation of the current state -> ('env' uint8 [N,H,W,1],
        'goal_n_state' float32 [N,9,1])."""
        if not self.with_ego:
            cp = self._c_params
            self.ego_image = torch.zeros((self.n_envs, cp.ego_h, cp.ego_w, 1), dtype=torch.uint8, device=self.device)
            self.goal_n_state = torch.zeros((self.n_envs, 9, 1), dtype=torch.float32, device=self.device)
        nat.check(nat.lib().bcg_observe_ego(C.byref(self._c_params), C.byref(self._batch), nat.ptr(self.ego_image),
                                            nat.ptr(self.goal_n_state), self._stream()))
        return self.ego_image, self.goal_n_state

    def observe_ego_path(self, max_points=64):
        """Observation.path of every env as device tensors (reference envs/base/env.py:421-433: `path[target_idx:]`, with
        the pure-pursuit provider `path[:target_idx + 1]`), in the robot frame like the egocentric wrapper sees it
        (from_global_to_egocentric, utilities/coordinate_transformations.py:341-362): (fp64 [N, max_points, 3] zero
        padded, int32 [N] way points left) -- what a GPU-resident policy consumes instead of the ragged per-env slices
        of `VecObservation.path`."""
        out = torch.empty((self.n_envs, int(max_points), 3), dtype=torch.float64, device=self.device)
        left = torch.empty(self.n_envs, dtype=torch.int32, device=self.device)
        nat.check(nat.lib().bcg_observe_ego_path(C.byref(self._c_params), C.byref(self._batch), int(max_points), nat.ptr(out),
                                                 nat.ptr(left), self._stream()))
        return out, left

    def get_state(self, indices=None):
        idx = self._indices(indices)
        k = idx.numel()
        f = torch.empty((self.layout.n_frows, k), dtype=torch.float64, device=self.device)
        i = torch.empty((self.layout.n_irows, k), dtype=torch.int32, device=self.device)
        nat.check(nat.lib().bcg_gather_state(C.byref(self._batch), nat.ptr(idx), k, nat.ptr(f), nat.ptr(i), self._stream()))
        return VecState(f, i)

    def set_state(self, state, indices=None, load_delayed_robot=True):
        """Restore columns.  Like the reference (envs/base/env.py:282-285) the live robot is loaded
        from the *delayed* robot state of the snapshot unless load_delayed_robot is False."""
        idx = self._indices(indices)
        k = idx.numel()
        if tuple(state.f.shape) != (self.layout.n_frows, k) or tuple(state.i.shape) != (self.layout.n_irows, k):
            raise ValueError("snapshot shape does not match the env layout / index count")
        f, i = state.f.to(self.device).contiguous(), state.i.to(self.device).contiguous()
        if self._env_rows is not None and k:
            # a column must fit the target env's own rings: queue length <= its delay, head inside it (empty when 0)
            d = self.env_rows_i[nat.EP_I_DELAY_CONTROL:nat.EP_I_DELAY_STATE + 1][:, idx]
            q = i[nat.I_QC:nat.I_QS + 1]
            head, length = q & 0xffff, q >> 16
            bad = (length > d) | ((head >= d) & (q != 0))
            if bool(bad.any()):
                col = int(torch.nonzero(bad.any(dim=0))[0, 0])
                raise ValueError("set_state: snapshot column %d holds queues (head | len << 16 = %s) that do not fit the "
                                 "delays %s of env %d" % (col, q[:, col].tolist(), d[:, col].tolist(), int(idx[col])))
        nat.check(nat.lib().bcg_scatter_state(C.byref(self._batch), nat.ptr(idx), k, nat.ptr(f), nat.ptr(i),
                                              1 if load_delayed_robot else 0, self._stream()))

    def _indices(self, indices):
        if indices is None:
            return torch.arange(self.n_envs, dtype=torch.int64, device=self.device)
        idx = torch.as_tensor(indices, dtype=torch.int64, device=self.device).reshape(-1).contiguous()
        if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= self.n_envs):
            raise IndexError("env index out of range")
        return idx

    # ---- pieces of the path, individually addressable ---------------------------------------------
    def _poses_rows(self, poses):
        p = torch.as_tensor(poses, dtype=torch.float64, device=self.device)
        if tuple(p.shape) != (self.n_envs, 3):
            raise ValueError("poses must have shape (%d, 3)" % self.n_envs)
        return p.t().contiguous()

    def pose_collides(self, poses, count_pixels=False, use_u8=False):
        """Batched `pose_collides` (reference envs/base/env.py:464-489): pose e against env e's costmap."""
        rows = self._poses_rows(poses)
        flags = torch.empty(self.n_envs, dtype=torch.uint8, device=self.device)
        if use_u8:
            nat.check(nat.lib().bcg_collision_u8(C.byref(self._c_params), C.byref(self._batch), nat.ptr(rows),
                                                 nat.ptr(flags), self._stream()))
            return flags.view(torch.bool)
        pixels = torch.empty(self.n_envs, dtype=torch.int32, device=self.device) if count_pixels else None
        nat.check(nat.lib().bcg_collision(C.byref(self._c_params), C.byref(self._batch), nat.ptr(rows), nat.ptr(flags),
                                          nat.ptr(pixels), self._stream()))
        return (flags.view(torch.bool), pixels) if count_pixels else flags.view(torch.bool)

    # ---- bookkeeping ---------------------------------------------------------------------------
    def check_status(self):
        """Poll the device anomaly counters (synchronises).  Raises like the reference would."""
        st = self._status.cpu().numpy().astype(np.int64)
        if st[nat.STATUS_PATH_EXHAUSTED]:
            self._status.zero_()
            raise ValueError("Goal pose too close to initial pose")   # reference envs/base/reward.py:275-277
        if st[nat.STATUS_LUT_MISS]:
            self._status.zero_()
            raise nat.BcgError("%d footprint lookups fell outside the angle-bin table" % st[nat.STATUS_LUT_MISS])
        if st[nat.STATUS_SLOT_OVERFLOW]:
            self._status.zero_()
            raise nat.BcgError("%d generated worlds did not fit their map / path slots (envs left unchanged)"
                               % st[nat.STATUS_SLOT_OVERFLOW])

    def final_observation(self):
        """The final observation of every episode that ended at the last step (needs episode_ends), as it was before
        the auto-reset replaced it: a FinalObservation of device tensors.  Does not synchronise; `ended` and the rows
        combine with the step's outputs by torch.where."""
        self._ends_on()
        torch.bitwise_and(self._end_reason, nat.END_NOW, out=self._end_scratch)
        ended = torch.ne(self._end_scratch, 0, out=self._end_flags[0])
        return FinalObservation(ended=ended, obs_vec=self._final_obs_vec, goal_n_state=self._final_goal_n_state,
                                episode_return=self._final_return, episode_length=self._final_length, slot=self._final_slot,
                                ego_image=self.final_ego_image, count=self._ends_count[0])

    def final_ego(self, env_ids):
        """Final crops (uint8 [k, H, W, 1]) of envs `env_ids` whose episodes ended at the last step.  Synchronises; raises
        when the step had more episode ends than episode_end_capacity (some crops were not kept) or when an env did not
        end at the last step."""
        self._ends_on()
        if not self.with_ego:
            raise ValueError("this batch was built without the egocentric observation (with_ego=False)")
        count, cap = int(self._ends_count[0]), self.episode_end_capacity
        if count > cap:
            raise nat.BcgError("%d episodes ended at the last step but episode_end_capacity is %d: the final crops of %d "
                               "of them were not kept" % (count, cap, count - cap))
        idx = self._indices(env_ids)
        slots = self._final_slot[idx]
        if bool((slots < 0).any()):
            raise ValueError("env %d did not end at the last step" % int(idx[torch.nonzero(slots < 0)[0, 0]]))
        return self.final_ego_image[slots.to(torch.int64)]

    def episode_stats(self, reset=False):
        """Device-accumulated episode statistics as a fp64 tensor [STATS_WORDS] (see STAT_NAMES)."""
        out = self._stats.clone()
        if reset:
            self._stats.zero_()
        return out

    def path_lengths(self):
        """Refined path length of every env, int64 [N] on the device -- read from the path descriptors where they live
        (device-generated worlds rewrite them), no host round trip."""
        n_of_path = self.path_descs.view(torch.int32).view(-1, C.sizeof(nat.BcgPathDesc) // 4)[:, nat.BcgPathDesc.n.offset // 4]
        return n_of_path[self.path_id.to(torch.int64)].to(torch.int64)

    def goal_reached(self):
        """bool [N]: has env e finished its path?  ContinuousRewardProvider: target_idx past the last way point
        (reference envs/base/reward.py:66-69); pure pursuit: observed pose within 1 m of the last point (:139-149)."""
        n = self.path_lengths()
        if self.params.reward_provider_name != CONTINUOUS_REWARD_PURE_PURSUIT:
            return self.state_i[nat.I_TARGET].to(torch.int64) > n - 1
        d = self.path_descs.view(torch.int64).view(-1, C.sizeof(nat.BcgPathDesc) // 8)
        pid = self.path_id.to(torch.int64)
        off = d[:, nat.BcgPathDesc.off.offset // 8][pid]
        pitch = self.path_descs.view(torch.int32).view(-1, C.sizeof(nat.BcgPathDesc) // 4)[:, nat.BcgPathDesc.pitch.offset // 4][pid].to(torch.int64)
        gx, gy = self.path_arena[off + n - 1], self.path_arena[off + pitch + n - 1]
        return torch.hypot(gx - self.state_f[nat.F_DPOSE], gy - self.state_f[nat.F_DPOSE + 1]) < 1.0

    def full_path(self, e):
        return self._paths_host[int(self._path_ids_host[e])]

    def costmap(self, e):
        return self._map_pool[int(self._map_ids_host[e])]

    def queue_rows(self, which, e=None):
        """(first fp64 row, slots, components, int row) of a delay ring: 'control' | 'pose' | 'state'.  `slots` is the
        ring's capacity, or with `e` the delay of env e: the slots its queue uses (the modulus of its head)."""
        L, p = self.layout, self.params
        if e is not None:
            p = self.params_of(e)
        elif self._pool is not None:
            cp = self._c_params
            return {'control': (L.ring_control, cp.delay_control, 2, nat.I_QC),
                    'pose': (L.ring_pose, cp.delay_pose, 3, nat.I_QP),
                    'state': (L.ring_state, cp.delay_state, 7, nat.I_QS)}[which]
        return {'control': (L.ring_control, p.control_delay, 2, nat.I_QC),
                'pose': (L.ring_pose, p.pose_delay, 3, nat.I_QP),
                'state': (L.ring_state, p.state_delay, 7, nat.I_QS)}[which]

    # ---- per-env parameters ----------------------------------------------------------------------
    def params_of(self, e):
        """The EnvParams env e steps with."""
        return self.params if self._pool is None else self._pool[int(self._params_ids_host[int(e)])]

    def noise_of(self, e):
        """The odometry noise setting (dict alpha1..alpha6, or None for off) env e steps with."""
        if self._pool is None:
            cp = self._c_params
            return dict(('alpha%d' % (k + 1), cp.alpha[k]) for k in range(6)) if cp.noise_on else None
        return self._noise_pool[int(self._params_ids_host[int(e)])]

    @property
    def params_ids(self):
        """int64 [N] host array: the pool entry of every env (None without a pool)"""
        return None if self._pool is None else self._params_ids_host.copy()

    @property
    def delays(self):
        """int32 [N, 3] device tensor: the control, pose and state delay of every env"""
        if self._pool is not None:
            return self.env_rows_i[nat.EP_I_DELAY_CONTROL:nat.EP_I_DELAY_STATE + 1].t()
        p = self.params
        return torch.tensor([[p.control_delay, p.pose_delay, p.state_delay]], dtype=torch.int32,
                            device=self.device).expand(self.n_envs, 3)
