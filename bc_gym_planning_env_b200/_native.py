"""ctypes binding of libbcg_b200.so (include/bcg_b200.h).

This is the only route from the Python host into the hot path.  There is no CPU fallback: if the
library is missing it is (re)built with nvcc, and if no CUDA device is present every compute entry
point raises.
"""
import ctypes as C
import os

from .csrc import build as _build

c_f64p = C.c_void_p  # device pointers travel as integers (tensor.data_ptr())


class BcgParams(C.Structure):
    _fields_ = [
        ("dt", C.c_double), ("resolution", C.c_double), ("inv_resolution", C.c_double),
        ("spatial_precision", C.c_double), ("angular_precision", C.c_double), ("progress_multiplier", C.c_double),
        ("wheel_base", C.c_double), ("max_wheel_angle", C.c_double), ("max_wheel_delta", C.c_double),
        ("p_gain", C.c_double), ("max_lin_acc", C.c_double), ("max_ang_acc", C.c_double),
        ("alpha", C.c_double * 6),
        ("ego_x0", C.c_double), ("ego_y0", C.c_double), ("ego_world_w", C.c_double), ("ego_world_h", C.c_double),
        ("seed", C.c_uint64), ("env_id_base", C.c_uint64),
        ("robot_kind", C.c_int32), ("noise_on", C.c_int32),
        ("delay_control", C.c_int32), ("delay_pose", C.c_int32), ("delay_state", C.c_int32),
        ("iteration_timeout", C.c_int32), ("ego_w", C.c_int32), ("ego_h", C.c_int32),
        ("reward_kind", C.c_int32), ("reserved", C.c_int32),
        ("auto_reset", C.c_int32), ("ego_variant", C.c_int32),
    ]


class BcgMapDesc(C.Structure):
    _fields_ = [
        ("data_off", C.c_int64), ("tile_off", C.c_int64), ("origin_x", C.c_double), ("origin_y", C.c_double),
        ("height", C.c_int32), ("width", C.c_int32), ("pitch", C.c_int32),
        ("tiles_x", C.c_int32), ("tiles_y", C.c_int32), ("flags", C.c_int32),
        ("cell_tile_off", C.c_int64), ("ctiles_x", C.c_int32), ("ctiles_y", C.c_int32),
        ("occupied", C.c_int32), ("sum_off", C.c_int32),
    ]


class BcgPathDesc(C.Structure):
    _fields_ = [
        ("off", C.c_int64), ("chunk_off", C.c_int64),
        ("n", C.c_int32), ("pitch", C.c_int32), ("n_chunks", C.c_int32), ("chunk_pitch", C.c_int32),
    ]


class BcgFootprintLut(C.Structure):
    _fields_ = [
        ("edges", C.c_void_p), ("verts", C.c_void_p), ("header", C.c_void_p), ("rows", C.c_void_p),
        ("fp_pix", C.c_void_p), ("bucket_first", C.c_void_p), ("bucket_scale", C.c_double),
        ("n_bins", C.c_int32), ("n_verts", C.c_int32), ("max_rows", C.c_int32), ("wpr", C.c_int32),
        ("n_buckets", C.c_int32), ("bin_stride", C.c_int32), ("bins", C.c_void_p),
    ]


class BcgBatch(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32), ("n_frows", C.c_int32), ("n_irows", C.c_int32),
        ("n_maps", C.c_int32), ("n_paths", C.c_int32), ("flags", C.c_int32),
        ("state_f", C.c_void_p), ("state_i", C.c_void_p), ("init_f", C.c_void_p), ("init_i", C.c_void_p),
        ("cand", C.c_void_p), ("cand_i", C.c_void_p), ("ego_work", C.c_void_p), ("work", C.c_void_p), ("map_id", C.c_void_p), ("path_id", C.c_void_p),
        ("maps", C.c_void_p), ("paths", C.c_void_p),
        ("map_arena", C.c_void_p), ("tile_arena", C.c_void_p), ("path_arena", C.c_void_p),
        ("lut", BcgFootprintLut),
        ("cell_tile_arena", C.c_void_p), ("occ_tile_arena", C.c_void_p), ("ego_list", C.c_void_p),
        ("occ_sum_arena", C.c_void_p), ("status", C.c_void_p), ("stats", C.c_void_p), ("step_counter", C.c_void_p),
        ("world_gen", C.c_void_p),
    ]


class BcgTurnParams(C.Structure):
    _fields_ = [
        ("main_corridor_length", C.c_double), ("turn_corridor_length", C.c_double), ("turn_corridor_angle", C.c_double),
        ("main_corridor_width", C.c_double), ("turn_corridor_width", C.c_double), ("margin", C.c_double),
        ("rot_theta", C.c_double), ("flip_arnd_oy", C.c_int32), ("flip_arnd_ox", C.c_int32),
    ]


class BcgAisleSlots(C.Structure):
    _fields_ = [
        ("map_slot_bytes", C.c_int64), ("tile_slot_words", C.c_int64),
        ("path_pitch", C.c_int32), ("chunk_pitch", C.c_int32),
        ("gen_state", C.c_void_p), ("params_out", C.c_void_p),
    ]


class BcgMiniGenParams(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("inner_h", "inner_w", "mid_margin", "out_margin", "min_obstacle_angle",
                                          "max_obstacle_angle", "lim_euc_dist", "lim_ang_dist", "angular_pose_noise_scale",
                                          "goal_spat_dist", "goal_ang_dist")]


class BcgMiniParams(C.Structure):
    _fields_ = [("h", C.c_double), ("w", C.c_double), ("start", C.c_double * 3), ("end", C.c_double * 3),
                ("a", C.c_double * 2), ("o", C.c_double * 2), ("b", C.c_double * 2)]


class BcgWorldGen(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("reserved", C.c_int32), ("slots", BcgAisleSlots), ("mini", BcgMiniGenParams),
        ("path_delta", C.c_double), ("list", C.c_void_p), ("count", C.c_void_p),
    ]


class BcgStateLayout(C.Structure):
    _fields_ = [
        ("n_frows", C.c_int32), ("n_irows", C.c_int32),
        ("ring_control", C.c_int32), ("ring_pose", C.c_int32), ("ring_state", C.c_int32),
    ]


class BcgStepOut(C.Structure):
    _fields_ = [
        ("reward", C.c_void_p), ("done", C.c_void_p), ("hit", C.c_void_p),
        ("ego_image", C.c_void_p), ("goal_n_state", C.c_void_p), ("obs_vec", C.c_void_p),
        ("ego_hits", C.c_void_p), ("ego_hit_count", C.c_void_p), ("ego_hit_cap", C.c_int32), ("reserved", C.c_int32),
    ]


class BcgEnvRows(C.Structure):
    _fields_ = [("f", C.c_void_p), ("i", C.c_void_p)]


class BcgEpisodeEnds(C.Structure):
    _fields_ = [
        ("reason", C.c_void_p), ("final_slot", C.c_void_p), ("final_obs_vec", C.c_void_p), ("final_goal_n_state", C.c_void_p),
        ("final_return", C.c_void_p), ("final_length", C.c_void_p), ("final_ego_work", C.c_void_p),
        ("final_ego_image", C.c_void_p), ("final_list", C.c_void_p), ("count", C.c_void_p),
        ("capacity", C.c_int32), ("reserved", C.c_int32),
    ]


_STRUCTS = [BcgParams, BcgMapDesc, BcgPathDesc, BcgFootprintLut, BcgBatch, BcgStateLayout, BcgStepOut, BcgTurnParams,
            BcgAisleSlots, BcgMiniGenParams, BcgMiniParams, BcgEnvRows, BcgEpisodeEnds, BcgWorldGen]

# fixed rows / words of include/bcg_b200.h
F_ROBOT, F_DROBOT, F_DPOSE, F_TIME, F_MIN_DIST, F_EP_RETURN, F_FIXED = 0, 7, 14, 17, 18, 19, 20
I_ITER, I_TARGET, I_COLLIDED, I_QC, I_QP, I_QS, I_FIXED = 0, 1, 2, 3, 4, 5, 6
STATUS_LUT_MISS, STATUS_PATH_EXHAUSTED, STATUS_SLOT_OVERFLOW, STATUS_SAMPLER_EMPTY, STATUS_WORDS = 0, 1, 2, 3, 8
STAT_NAMES = ("episodes", "return", "length", "collided", "goal", "timeout")
STATS_WORDS = 8
ROBOT_TRICYCLE, ROBOT_DIFFDRIVE = 0, 1
MAP_ONLY_LETHAL, MAP_CELL_INDEX = 1, 4
BATCH_SPARSE_EGO_ONLY, BATCH_CELL_INDEX = 1, 2
REWARD_CONTINUOUS, REWARD_PURE_PURSUIT = 0, 1
# per-env parameter rows (BcgEnvRows)
EP_F_SP, EP_F_AP, EP_F_PM, EP_F_ALPHA, EP_F_ROWS = 0, 1, 2, 3, 9
EP_I_DELAY_CONTROL, EP_I_DELAY_POSE, EP_I_DELAY_STATE, EP_I_TIMEOUT, EP_I_NOISE_ON, EP_I_ROWS = 0, 1, 2, 3, 4, 5
# BcgParams.auto_reset, BcgWorldGen.kind, the draw-index domain of the worlds a step draws
AUTO_RESET_NEW_WORLD = 2
WORLD_AISLE, WORLD_MINI = 0, 1
NEW_WORLD_DRAW = 1 << 63
# episode-end reason bits (BcgEpisodeEnds.reason)
END_GOAL, END_COLLIDED, END_TIMEOUT, END_NOW = 1, 2, 4, 8

# every symbol include/bcg_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "bcg_abi_version": (C.c_int, []),
    "bcg_last_error": (C.c_size_t, [C.c_char_p, C.c_size_t]),
    "bcg_sizeof": (C.c_int64, [C.c_int32]),
    "bcg_device_count": (C.c_int, []),
    "bcg_state_layout": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgStateLayout)]),
    "bcg_build_lethal_tiles": (C.c_int, [C.POINTER(BcgBatch), C.c_int32, C.c_int32, _P]),
    "bcg_build_cell_tiles": (C.c_int, [C.POINTER(BcgBatch), C.c_int32, C.c_int32, _P]),
    "bcg_init_state": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), C.POINTER(BcgEnvRows), _P]),
    "bcg_generate_aisles": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), C.POINTER(BcgEnvRows),
                                      C.POINTER(BcgAisleSlots), _P, _P, C.c_uint64, C.c_double, _P]),
    "bcg_generate_minis": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), C.POINTER(BcgAisleSlots), _P,
                                     C.POINTER(BcgMiniGenParams), _P, _P, C.c_uint64, C.c_double, _P]),
    "bcg_reset_where": (C.c_int, [C.POINTER(BcgBatch), _P, _P]),
    "bcg_step": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), C.POINTER(BcgEnvRows), _P, C.c_int32, C.c_uint64,
                           C.POINTER(BcgStepOut), C.POINTER(BcgEpisodeEnds), C.POINTER(C.c_void_p), _P]),
    "bcg_collision": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), _P, _P, _P, _P]),
    "bcg_collision_u8": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), _P, _P, _P]),
    "bcg_collision_recheck": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), _P, C.c_int32, _P]),
    "bcg_observe_ego": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), _P, _P, _P]),
    "bcg_gather_state": (C.c_int, [C.POINTER(BcgBatch), _P, C.c_int32, _P, _P, _P]),
    "bcg_scatter_state": (C.c_int, [C.POINTER(BcgBatch), _P, C.c_int32, _P, _P, C.c_int32, _P]),
    "bcg_pack_ego_hits": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P, C.c_int32, _P]),
    "bcg_world_to_pixel": (C.c_int, [_P, C.c_int64, C.c_double, C.c_double, C.c_double, _P, _P]),
    "bcg_normalize_angle": (C.c_int, [_P, C.c_int64, _P, _P]),
    "bcg_masked_any_equal": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, _P]),
    "bcg_inverse_transform": (C.c_int, [_P, C.c_int64, _P, _P]),
    "bcg_project_poses": (C.c_int, [C.POINTER(C.c_double), _P, C.c_int64, _P, _P]),
    "bcg_observe_ego_path": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), C.c_int32, _P, _P, _P]),
    "bcg_rollout": (C.c_int, [C.POINTER(BcgParams), C.POINTER(BcgBatch), C.POINTER(BcgEnvRows), _P, C.c_int32, C.c_uint64,
                              C.POINTER(BcgStepOut), C.POINTER(BcgEpisodeEnds), _P]),
    "bcg_alloc_image_memory": (C.c_int, [C.c_int64, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "bcg_free_image_memory": (C.c_int, [_P, C.c_int64]),
}


class BcgError(RuntimeError):
    """A C-ABI call returned a negative status."""


_lib = None


def library_path():
    return _build.TARGET


def lib():
    """Load (building first if the sources are newer) libbcg_b200.so and verify the struct mirrors."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("BCG_B200_LIB") or _build.build()    # BCG_B200_LIB: a tuning variant (csrc/build.py build_variant)
    handle = C.CDLL(path)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(handle, name)  # AttributeError here = header and library disagree
        fn.restype = restype
        fn.argtypes = argtypes
    for which, struct in enumerate(_STRUCTS):
        if handle.bcg_sizeof(which) != C.sizeof(struct):
            raise BcgError("ABI mismatch: sizeof(%s) is %d in the library, %d in the binding"
                           % (struct.__name__, handle.bcg_sizeof(which), C.sizeof(struct)))
    _lib = handle
    return _lib


def last_error():
    buf = C.create_string_buffer(1024)
    lib().bcg_last_error(buf, len(buf))
    return buf.value.decode("utf-8", "replace")


def check(status):
    if status < 0:
        raise BcgError("libbcg_b200: %s (status %d)" % (last_error(), status))
    return status


def require_cuda():
    """The product has no CPU path: fail loudly when the CUDA device or the extension is missing."""
    n = lib().bcg_device_count()
    if n <= 0:
        raise BcgError("bc_gym_planning_env_b200 needs a CUDA device (B200, sm_100a); none is visible: %s"
                       % last_error())
    return n


def state_layout(params):
    out = BcgStateLayout()
    check(lib().bcg_state_layout(C.byref(params), C.byref(out)))
    return out


class ImageMemory(object):
    """A device block from bcg_alloc_image_memory (compute-data compression when the device has it), exposed through
    the CUDA array interface so that torch can view it; unmapped when the last view is gone."""

    def __init__(self, nbytes, want_compression=True):
        dptr, mapped, compressed = C.c_void_p(), C.c_int64(), C.c_int32()
        check(lib().bcg_alloc_image_memory(int(nbytes), 1 if want_compression else 0, C.byref(dptr), C.byref(mapped),
                                           C.byref(compressed)))
        self.ptr, self.mapped_bytes, self.compressed, self.nbytes = int(dptr.value), int(mapped.value), bool(compressed.value), int(nbytes)
        self.__cuda_array_interface__ = {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 3,
                                         "strides": None}

    def tensor(self, shape):
        """uint8 torch tensor of `shape` on this block, zero filled; it keeps the block alive"""
        import torch
        t = torch.as_tensor(self, device="cuda").view(shape)
        t.zero_()
        return t

    def __del__(self):
        ptr_, self.ptr = getattr(self, "ptr", 0), 0
        if ptr_ and _lib is not None:
            try:
                import torch
                torch.cuda.synchronize()
            except Exception:
                pass
            _lib.bcg_free_image_memory(C.c_void_p(ptr_), self.mapped_bytes)


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())
