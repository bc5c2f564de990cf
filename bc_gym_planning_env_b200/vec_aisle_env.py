"""VecRandomAisleTurnEnv / VecRandomMiniEnv: batches whose worlds are drawn and rasterised on the GPU.

The reference rebuilds a random aisle turn on the host at every `reset` (envs/synth_turn_env.py:278-291:
draw TurnParams :317-332, path_and_costmap_from_config :110-192, cv2.line walls, refine_path, initial reward
state) at about 1 k worlds/s per core.  Here `bcg_generate_aisles` does the same for any subset of the batch
in one launch: every env owns a fixed-size slot of the map / tile / path arenas and its world is rewritten in
place, so a 65 536-env reset storm is a single kernel instead of a minute of host work.
Draws come from Philox4x32-10 keyed (seed; env id, draw index) instead of the reference's MT19937; explicit
TurnParams can be supplied instead (that is how the parity tests replay the reference's own worlds).
`VecRandomMiniEnv` does the same for `RandomMiniEnv` (envs/mini_env.py:269-389: rejection sampler, two clipped
walls, two-point path) through `bcg_generate_minis`.
"""
import ctypes as C

import numpy as np
import torch

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200 import env_params as envp
from bc_gym_planning_env_b200.envs.synth_turn_env import TurnParams
from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE, VecPlanEnv, _round_up, footprint_lut_for

TURN_DTYPE = np.dtype([("main_corridor_length", "<f8"), ("turn_corridor_length", "<f8"), ("turn_corridor_angle", "<f8"),
                       ("main_corridor_width", "<f8"), ("turn_corridor_width", "<f8"), ("margin", "<f8"),
                       ("rot_theta", "<f8"), ("flip_arnd_oy", "<i4"), ("flip_arnd_ox", "<i4")])
assert TURN_DTYPE.itemsize == C.sizeof(nat.BcgTurnParams)


def turn_params_array(turns):
    """list of TurnParams (or dicts with its fields) -> structured array in the layout of BcgTurnParams"""
    out = np.zeros(len(turns), dtype=TURN_DTYPE)
    for k, t in enumerate(turns):
        get = (lambda f: t[f]) if isinstance(t, dict) else (lambda f: getattr(t, f))
        for f in TURN_DTYPE.names:
            out[f][k] = get(f)
    return out


def worst_case_world(resolution, path_delta):
    """Upper bounds (map cells incl. row padding, refined path points) over the RandomAisleTurnEnv distribution
    (envs/synth_turn_env.py:317-332).  The extents grow with every length and width, so only the two angles are
    searched (dense grid); 6 % head-room covers the grid spacing and the 32-cell row padding."""
    al, rt = np.meshgrid(np.linspace(-3. / 8. * np.pi, 3. / 8. * np.pi, 201), np.linspace(0, 2 * np.pi, 721))
    h, far, d, z = 8.0, 6.0, 1.5, 1.5
    ta, ca = np.tan(al), np.cos(al)
    lower, upper = -z / ca, z / ca
    o = np.ones_like(al)
    cx = np.stack([-d * o, 0 * o, d * o, d * o, far * o, far * o, d * o, far * o, -d * o, d * o])
    cy = np.stack([-h * o, -h * o, -h * o, d * ta + lower, far * ta + lower, far * ta, d * ta + upper, far * ta + upper,
                   h * o, h * o])
    c, s = np.cos(rt), np.sin(rt)
    X, Y = c * cx - s * cy, s * cx + c * cy
    w = (X.max(0) - X.min(0) + 2.0) / resolution + 33
    hh = (Y.max(0) - Y.min(0) + 2.0) / resolution + 9
    cells = int(np.ceil((w * hh).max() * 1.06))
    ca_min = np.cos(3. / 8. * np.pi)
    length = (h + d * np.tan(3. / 8. * np.pi) + z / ca_min) + np.hypot(d, z / ca_min) + (far + d / ca_min)
    return cells, int(np.ceil(length / path_delta)) + 8


class _VecSlotEnv(VecPlanEnv):
    """Common part of the batch envs whose worlds are generated on the device: one fixed-size slot per env in the map,
    cell-tile, tile-plane and path arenas, and host accessors that read a world back."""

    def _setup_slots(self, params, n_envs, resolution, noise_parameters, seed, auto_reset, device, env_id_base, with_ego,
                     footprint_scale, footprint, map_cells, path_points, record_bytes, world_kind, params_ids=None,
                     episode_ends=False, episode_end_capacity=None):
        if auto_reset == 'new_world' and not self._draw_new_turn_on_reset:
            raise ValueError("auto_reset='new_world' draws a new world at every episode end: it needs draw_new_turn_on_reset=True")
        self._configure(params, n_envs, resolution, noise_parameters, seed, auto_reset, device, env_id_base, with_ego, 'tiles',
                        params_ids, episode_ends, episode_end_capacity)
        if not self.params.refine_path:
            raise ValueError("device-side generation always refines the path (EnvParams.refine_path)")
        if max(1, int(0.05 / self.resolution)) != 1:
            raise ValueError("device-side walls are one pixel thick: resolution must be above 0.025 m")
        self._slot_bytes = _round_up(int(map_cells), 128)
        self._path_pitch = _round_up(int(path_points), 4)
        self._chunk_pitch = _round_up((self._path_pitch + 31) // 32, 4)
        self._tile_slot_words = _round_up(self._slot_bytes // 32 + 16 * 64, 16)   # 1 bit per cell + partial-tile slack
        self._draw_index = 0
        self._alloc_slots(record_bytes)
        self._upload_lut(footprint_lut_for(self.params.robot_name, self.resolution, footprint_scale, footprint))
        self._alloc_state()
        self._make_batch()
        # generated worlds are thin walls (BcgMapDesc.occupied stays 0): no env ever needs the dense egocentric kernel
        self._batch.flags |= nat.BATCH_SPARSE_EGO_ONLY
        if self.new_world_reset:
            self._setup_world_gen(world_kind)

    def _setup_world_gen(self, kind):
        """auto_reset='new_world': the BcgWorldGen the step's regeneration kernel reads (in device memory), its list of the
        envs to regenerate and its counters"""
        self._regen_list = torch.zeros(self.n_envs, dtype=torch.int32, device=self.device)
        self._regen_count = torch.zeros(4, dtype=torch.int32, device=self.device)
        wg = nat.BcgWorldGen()
        wg.kind = kind
        C.memmove(C.addressof(wg.slots), C.addressof(self._slots), C.sizeof(nat.BcgAisleSlots))
        wg.slots.params_out = self._records.data_ptr()
        if kind == nat.WORLD_MINI:
            wg.mini = self._gen
        wg.path_delta = float(self.params.path_delta)
        wg.list, wg.count = self._regen_list.data_ptr(), self._regen_count.data_ptr()
        self._world_gen = self._to_device(np.frombuffer(bytes(wg), dtype=np.uint8).copy())
        self._batch.world_gen = self._world_gen.data_ptr()

    def _alloc_slots(self, record_bytes):
        n, dev = self.n_envs, self.device
        path_slot = 5 * self._path_pitch + 3 * self._chunk_pitch
        # tile summary of a slot: at most one word per tile row and 32 tile columns, i.e. never more words than tiles
        sum_slot_words = self._tile_slot_words // 16
        if n * sum_slot_words >= 2 ** 31:
            raise ValueError("tile summaries of this batch exceed the 32-bit offsets of BcgMapDesc.sum_off")
        ids = np.arange(n, dtype=np.int64)
        md = np.zeros(n, dtype=np.dtype(nat.BcgMapDesc))
        md['data_off'] = md['cell_tile_off'] = ids * self._slot_bytes
        md['tile_off'] = ids * self._tile_slot_words
        md['sum_off'] = ids * sum_slot_words
        pdd = np.zeros(n, dtype=np.dtype(nat.BcgPathDesc))
        pdd['off'] = ids * path_slot
        pdd['chunk_off'] = ids * path_slot + 5 * self._path_pitch
        pdd['pitch'], pdd['chunk_pitch'] = self._path_pitch, self._chunk_pitch
        descs, pdescs = md.tobytes(), pdd.tobytes()
        self.map_arena = torch.zeros(n * self._slot_bytes, dtype=torch.uint8, device=dev)
        self.cell_tile_arena = torch.zeros(n * self._slot_bytes, dtype=torch.uint8, device=dev)
        self.tile_arena = torch.zeros(n * self._tile_slot_words, dtype=torch.int32, device=dev)
        self.occ_tile_arena = torch.zeros(n * self._tile_slot_words, dtype=torch.int32, device=dev)
        self.occ_sum_arena = torch.zeros(n * sum_slot_words, dtype=torch.int32, device=dev)
        self.path_arena = torch.zeros(n * path_slot, dtype=torch.float64, device=dev)
        self.map_descs = self._to_device(np.frombuffer(bytes(descs), dtype=np.uint8).copy())
        self.path_descs = self._to_device(np.frombuffer(bytes(pdescs), dtype=np.uint8).copy())
        self.map_id = torch.arange(n, dtype=torch.int32, device=dev)
        self.path_id = torch.arange(n, dtype=torch.int32, device=dev)
        self._n_maps = self._n_paths = n
        self._gen_state = torch.zeros((n, 128), dtype=torch.uint8, device=dev)
        self._records = torch.zeros((n, record_bytes), dtype=torch.uint8, device=dev)     # the parameters each world has
        slots = nat.BcgAisleSlots()
        slots.map_slot_bytes, slots.tile_slot_words = self._slot_bytes, self._tile_slot_words
        slots.path_pitch, slots.chunk_pitch = self._path_pitch, self._chunk_pitch
        slots.gen_state = self._gen_state.data_ptr()
        self._slots = slots

    # ---- accessors: the worlds live on the device ----------------------------------------------------
    def _map_desc(self, e):
        sz = C.sizeof(nat.BcgMapDesc)
        raw = self.map_descs[int(e) * sz:(int(e) + 1) * sz].cpu().numpy().tobytes()
        return nat.BcgMapDesc.from_buffer_copy(raw)

    def _path_desc(self, e):
        sz = C.sizeof(nat.BcgPathDesc)
        raw = self.path_descs[int(e) * sz:(int(e) + 1) * sz].cpu().numpy().tobytes()
        return nat.BcgPathDesc.from_buffer_copy(raw)

    def costmap(self, e):
        d = self._map_desc(e)
        rows = self.map_arena[d.data_off:d.data_off + d.height * d.pitch].view(d.height, d.pitch)[:, :d.width]
        return CostMap2D(rows.cpu().numpy().copy(), self.resolution, np.array([d.origin_x, d.origin_y], dtype=np.float64))

    def full_path(self, e):
        d = self._path_desc(e)
        rows = self.path_arena[d.off:d.off + 3 * d.pitch].view(3, d.pitch)[:, :d.n]
        return np.ascontiguousarray(rows.t().cpu().numpy())

    def check_status(self):
        st = self._status.cpu().numpy().astype(np.int64)
        if st[nat.STATUS_SAMPLER_EMPTY]:
            self._status.zero_()
            raise ValueError("Something went wrong, the sampling space looks empty.")     # mini_env.py:138,361
        super(_VecSlotEnv, self).check_status()


class VecRandomAisleTurnEnv(_VecSlotEnv):
    def __init__(self, n_envs, params=None, draw_new_turn_on_reset=True, seed=0, turn_params=None,
                 noise_parameters=DEFAULT_NOISE, auto_reset=False, device=None, env_id_base=0, with_ego=False,
                 footprint_scale=1.0, footprint=None, resolution=0.03, max_map_cells=None, max_path_points=None,
                 params_ids=None, episode_ends=False, episode_end_capacity=None, compact_ego=False):
        """
        :param n_envs: batch size; env e draws from the Philox stream (seed; env_id_base + e, draw index)
        :param params, noise_parameters, params_ids: one EnvParams and noise setting for the batch, or a pool of them
            and the set of every env (see VecPlanEnv); `reset(mask, params_ids=...)` moves envs to other sets
        :param draw_new_turn_on_reset: `reset` draws a new turn for the envs it resets (reference default)
        :param auto_reset: the step's own reset of the envs whose episodes end (no host round trip).
            'new_world': the reference's behaviour -- a new turn for every episode (synth_turn_env.py:278-291) -- inside
            the step: its regeneration kernel draws the finished envs' new turns (Philox (seed; env id, 2^63 | step
            index)), builds them and writes their initial observations; works with step_graph, rollout(_graph) and
            step_host.  Needs draw_new_turn_on_reset.  A turn that overflows its slot restarts the env's current
            world and `check_status()` raises.
            True: restores the initial state of the env's CURRENT world and does NOT draw a new turn, whatever
            draw_new_turn_on_reset says: an episode that ends is replayed on the same aisle.
            False: no reset; `env.reset(done)` after the step gives the finished envs new turns (one generation launch
            plus a full egocentric pass).
        :param turn_params: optional list of n_envs TurnParams for the first worlds (default: drawn on device)
        :param max_map_cells, max_path_points: slot capacities per env (default: worst case of the distribution)
        :param episode_ends, episode_end_capacity: see VecPlanEnv.  The final observations (`final_observation()`) of
            envs that got a new turn, in the step ('new_world') or by `reset(done)` after it, are those of the old one
        :param compact_ego: see VecPlanEnv (`step_host(images='compact')`)
        """
        from bc_gym_planning_env_b200.envs.base.params import EnvParams
        first = params[0] if envp.is_pool(params) and len(params) else params
        pd = (first if first is not None else EnvParams()).path_delta
        cells, points = worst_case_world(float(resolution), pd)
        self._draw_new_turn_on_reset = bool(draw_new_turn_on_reset)
        self._compact_ego = bool(compact_ego)
        self._setup_slots(params, n_envs, resolution, noise_parameters, seed, auto_reset, device, env_id_base, with_ego,
                          footprint_scale, footprint, max_map_cells if max_map_cells is not None else cells,
                          max_path_points if max_path_points is not None else points, TURN_DTYPE.itemsize, nat.WORLD_AISLE,
                          params_ids, episode_ends, episode_end_capacity)
        self._turns = self._records
        self._slots.params_out = self._turns.data_ptr()
        self.generate(turn_params=turn_params)
        self.check_status()

    # ---- generation ------------------------------------------------------------------------------
    def generate(self, mask=None, turn_params=None):
        """Give the envs with mask[e] true (None: all) a new world and its initial state.
        turn_params: list of n_envs TurnParams / structured array (TURN_DTYPE) to use instead of drawing;
        entries of unmasked envs are ignored."""
        m = self._mask(mask)
        tp = None
        if turn_params is not None:
            arr = turn_params if isinstance(turn_params, np.ndarray) else turn_params_array(turn_params)
            if arr.dtype != TURN_DTYPE or arr.shape != (self.n_envs,):
                raise ValueError("turn_params must hold one TurnParams per env")
            tp = self._to_device(arr.view(np.uint8).reshape(self.n_envs, TURN_DTYPE.itemsize))
        nat.check(nat.lib().bcg_generate_aisles(C.byref(self._c_params), C.byref(self._batch), self._rows,
                                                C.byref(self._slots), nat.ptr(m), nat.ptr(tp), self._draw_index,
                                                float(self.params.path_delta), self._stream()))
        self._draw_index += 1
        if tp is not None:
            torch.cuda.current_stream(self.device).synchronize()     # tp is released when this returns

    def reset(self, mask=None, params_ids=None):
        """RandomAisleTurnEnv.reset (envs/synth_turn_env.py:278-291) for all envs (mask None) or those with
        mask[e] true: a new turn when draw_new_turn_on_reset, the initial state either way.
        params_ids (batches built with a pool only): [n_envs] pool indices; the envs being reset move to their entry
        before their world and initial state are built (the entries of the other envs are ignored) -- domain
        randomisation at episode boundaries in the same single generation launch.  Without draw_new_turn_on_reset an env
        whose set changes gets its current world rebuilt from its recorded TurnParams, so that its initial state follows
        the new goal tolerances."""
        changed = None
        if params_ids is not None:
            changed = self._assign_params(mask, params_ids)
        if not self._draw_new_turn_on_reset:
            if changed is not None and changed.any():
                draw_index = self._draw_index
                self.generate(torch.from_numpy(changed), turn_params=self.turn_params())
                self._draw_index = draw_index              # (no draw was made)
            return super(VecRandomAisleTurnEnv, self).reset(mask)
        self.generate(mask)
        if self.with_ego:
            self.observe_ego()
        return self.observation()

    def _assign_params(self, mask, params_ids):
        """Move the masked envs to pool entries params_ids[e] (rows rebuilt and validated on the host, then uploaded);
        returns the bool [n_envs] host mask of the envs whose set changed."""
        if self._pool is None:
            raise ValueError("params_ids needs a batch built with a pool of EnvParams")
        new = np.asarray(params_ids.cpu() if isinstance(params_ids, torch.Tensor) else params_ids)
        if new.shape != (self.n_envs,) or not np.issubdtype(new.dtype, np.integer):
            raise ValueError("params_ids must be %d integers" % self.n_envs)
        m = np.ones(self.n_envs, dtype=bool) if mask is None else np.asarray(
            mask.cpu() if isinstance(mask, torch.Tensor) else mask).astype(bool).reshape(-1)
        ids = np.where(m, new, self._params_ids_host).astype(np.int64)
        rows = envp.build_env_rows(self._pool, self._noise_pool, ids, self.n_envs)
        changed = ids != self._params_ids_host
        self._params_ids_host = ids
        self.env_rows_f.copy_(torch.from_numpy(rows.f))
        self.env_rows_i.copy_(torch.from_numpy(rows.i))
        return changed

    # ---- accessors: the worlds live on the device ----------------------------------------------------
    def turn_params(self, e=None):
        """TurnParams of env e, or the structured array (TURN_DTYPE) of the whole batch."""
        arr = self._turns.cpu().numpy().reshape(-1).view(TURN_DTYPE)
        if e is None:
            return arr
        r = arr[int(e)]
        kw = {f: float(r[f]) for f in TURN_DTYPE.names}
        kw["flip_arnd_oy"], kw["flip_arnd_ox"] = bool(r["flip_arnd_oy"]), bool(r["flip_arnd_ox"])
        return TurnParams(**kw)


MINI_DTYPE = np.dtype([("h", "<f8"), ("w", "<f8"), ("start", "<f8", 3), ("end", "<f8", 3), ("a", "<f8", 2), ("o", "<f8", 2),
                       ("b", "<f8", 2)])
assert MINI_DTYPE.itemsize == C.sizeof(nat.BcgMiniParams)


def mini_params_array(configs):
    """list of MiniEnvParams (envs/mini_env.py) -> structured array in the layout of BcgMiniParams"""
    out = np.zeros(len(configs), dtype=MINI_DTYPE)
    for k, c in enumerate(configs):
        out["h"][k], out["w"][k] = c.h, c.w
        out["start"][k], out["end"][k] = c.start_pos.as_np(), c.end_pos.as_np()
        out["a"][k], out["o"][k], out["b"][k] = c.obstacle_a.as_np(), c.obstacle_o.as_np(), c.obstacle_b.as_np()
    return out


class VecRandomMiniEnv(_VecSlotEnv):
    """N `RandomMiniEnv`s (reference envs/mini_env.py:408-494) whose worlds are sampled, rasterised and checked on the
    GPU (`bcg_generate_minis`): the reference builds a new env at every reset on the host, about 100 per second."""

    def __init__(self, n_envs, params=None, draw_new_turn_on_reset=True, seed=0, mini_params=None,
                 noise_parameters=DEFAULT_NOISE, auto_reset=False, device=None, env_id_base=0, with_ego=False,
                 footprint_scale=1.0, footprint=None, episode_ends=False, episode_end_capacity=None):
        """
        :param params RandomMiniEnvParams: the sampling space and its EnvParams (default: RandomMiniEnv's own,
            goal tolerances 0.2 m / pi/8)
        :param mini_params: optional list of n_envs MiniEnvParams for the first worlds (built as they are, like
            MiniEnv(config)); default: sampled on the device
        :param auto_reset: 'new_world': the reference's new env per episode (mini_env.py:447-470) inside the step,
            sampled with (seed; env id, 2^63 | step index); a sampler that runs out of tries restarts the env's current
            world and `check_status()` raises.  True: in-kernel reset to the initial state of the env's CURRENT world,
            never a new one (see VecRandomAisleTurnEnv).  False: no reset; `env.reset(done)` samples new worlds.
        :param episode_ends, episode_end_capacity: see VecPlanEnv
        """
        from bc_gym_planning_env_b200.envs.base.params import EnvParams
        from bc_gym_planning_env_b200.envs.mini_env import RandomMiniEnvParams
        if envp.is_pool(params):
            # the device sampler's final check uses batch-wide goal tolerances (BcgMiniGenParams)
            raise ValueError("VecRandomMiniEnv takes one RandomMiniEnvParams; per-env parameter pools are not supported")
        if params is None:
            params = RandomMiniEnvParams(env_params=EnvParams(goal_ang_dist=np.pi / 8., goal_spat_dist=0.2))
        self.gen_params = params
        ep = params.env_params
        g = nat.BcgMiniGenParams()
        for f in ("inner_h", "inner_w", "mid_margin", "out_margin", "min_obstacle_angle", "max_obstacle_angle", "lim_euc_dist",
                  "lim_ang_dist", "angular_pose_noise_scale"):
            setattr(g, f, float(getattr(params, f)))
        g.goal_spat_dist, g.goal_ang_dist = float(ep.goal_spat_dist), float(ep.goal_ang_dist)
        self._gen = g
        self._draw_new_turn_on_reset = bool(draw_new_turn_on_reset)
        h = params.inner_h + 2 * params.mid_margin + 2 * params.out_margin
        w = params.inner_w + 2 * params.mid_margin + 2 * params.out_margin
        side_x, side_y = int(round(h / ep.resolution)) + 33, int(round(w / ep.resolution)) + 9
        diag = np.hypot(params.inner_w + 2 * params.mid_margin, params.inner_h + 2 * params.mid_margin)
        self._setup_slots(ep, n_envs, ep.resolution, noise_parameters, seed, auto_reset, device, env_id_base, with_ego,
                          footprint_scale, footprint, side_x * side_y, int(np.ceil(diag / ep.path_delta)) + 8, MINI_DTYPE.itemsize,
                          nat.WORLD_MINI, episode_ends=episode_ends, episode_end_capacity=episode_end_capacity)
        self.generate(mini_params=mini_params)
        self.check_status()

    def generate(self, mask=None, mini_params=None):
        """Give the envs with mask[e] true (None: all) a new world and its initial state; `mini_params` (list of
        MiniEnvParams or structured array MINI_DTYPE, one per env) builds those worlds instead of sampling."""
        m = self._mask(mask)
        mp = None
        if mini_params is not None:
            arr = mini_params if isinstance(mini_params, np.ndarray) else mini_params_array(mini_params)
            if arr.dtype != MINI_DTYPE or arr.shape != (self.n_envs,):
                raise ValueError("mini_params must hold one MiniEnvParams per env")
            mp = self._to_device(arr.view(np.uint8).reshape(self.n_envs, MINI_DTYPE.itemsize))
        nat.check(nat.lib().bcg_generate_minis(C.byref(self._c_params), C.byref(self._batch), C.byref(self._slots), nat.ptr(m),
                                               C.byref(self._gen), nat.ptr(mp), nat.ptr(self._records), self._draw_index,
                                               float(self.params.path_delta), self._stream()))
        self._draw_index += 1
        if mp is not None:
            torch.cuda.current_stream(self.device).synchronize()     # mp is released when this returns

    def reset(self, mask=None):
        """RandomMiniEnv.reset (envs/mini_env.py:465-477): a new world when draw_new_turn_on_reset, the initial state
        either way."""
        if not self._draw_new_turn_on_reset:
            return super(VecRandomMiniEnv, self).reset(mask)
        self.generate(mask)
        if self.with_ego:
            self.observe_ego()
        return self.observation()

    def mini_params(self, e=None):
        """The accepted MiniEnvParams as a structured array (MINI_DTYPE), or the row of env e."""
        arr = self._records.cpu().numpy().reshape(-1).view(MINI_DTYPE)
        return arr if e is None else arr[int(e)]
