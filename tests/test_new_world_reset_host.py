"""auto_reset='new_world' without a GPU: the struct mirror, the library's refusal of a batch without the world generator,
and the Python argument errors."""
import ctypes as C

import numpy as np
import pytest

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
from bc_gym_planning_env_b200.vec_aisle_env import VecRandomAisleTurnEnv, VecRandomMiniEnv
from bc_gym_planning_env_b200.vec_env import VecPlanEnv

BCG_ERR_INVALID = -1


def test_world_gen_struct_mirror():
    assert nat._STRUCTS[13] is nat.BcgWorldGen
    assert nat.lib().bcg_sizeof(13) == C.sizeof(nat.BcgWorldGen)


def _batch_with_dummy_pointers():
    # every field check_batch requires, as non-null pointers that no kernel ever reads (the calls below launch nothing)
    p, b = nat.BcgParams(), nat.BcgBatch()
    L = nat.state_layout(p)
    b.n_envs, b.n_frows, b.n_irows = 1, L.n_frows, L.n_irows
    dummy = 0x1000
    for name in ("state_f", "state_i", "init_f", "init_i", "cand", "cand_i", "work", "map_id", "path_id", "maps", "paths",
                 "map_arena", "tile_arena", "path_arena", "occ_tile_arena", "occ_sum_arena", "status", "stats"):
        setattr(b, name, dummy)
    for name in ("edges", "verts", "header", "rows", "fp_pix", "bucket_first"):
        setattr(b.lut, name, dummy)
    b.lut.n_buckets, b.lut.bucket_scale, b.lut.n_verts = 1, 1.0, 4
    b.lut.n_bins, b.lut.wpr, b.lut.max_rows = 1, 1, 1
    return p, b


def test_new_world_batch_needs_the_world_generator_and_slots():
    lib = nat.lib()
    p, b = _batch_with_dummy_pointers()
    plan = C.c_void_p(0x1000)
    p.auto_reset = nat.AUTO_RESET_NEW_WORLD
    acts, out = C.c_void_p(0x1000), nat.BcgStepOut()
    assert lib.bcg_step(C.byref(p), C.byref(b), None, acts, 0, 0, C.byref(out), None, None, None) == BCG_ERR_INVALID
    assert "world_gen" in nat.last_error()
    b.world_gen = 0x1000
    assert lib.bcg_rollout(C.byref(p), C.byref(b), None, plan, 0, 0, None, None, None) == BCG_ERR_INVALID
    assert "world_gen" in nat.last_error() and "slots" in nat.last_error()
    b.n_maps = b.n_paths = 1
    b.cell_tile_arena = 0x1000
    assert lib.bcg_rollout(C.byref(p), C.byref(b), None, plan, 0, 0, None, None, None) == 0
    p.auto_reset = 1
    b.world_gen = None
    assert lib.bcg_rollout(C.byref(p), C.byref(b), None, plan, 0, 0, None, None, None) == 0


def test_new_world_argument_errors():
    # raised before anything needs a device
    with pytest.raises(ValueError, match="draw_new_turn_on_reset"):
        VecRandomAisleTurnEnv(4, auto_reset='new_world', draw_new_turn_on_reset=False)
    with pytest.raises(ValueError, match="draw_new_turn_on_reset"):
        VecRandomMiniEnv(4, auto_reset='new_world', draw_new_turn_on_reset=False)
    cm = CostMap2D(np.zeros((40, 40), dtype=np.uint8), 0.05, np.zeros(2))
    path = np.array([[0.2, 0.2, 0.0], [1.5, 0.2, 0.0]])
    with pytest.raises(ValueError, match="slots"):
        VecPlanEnv([cm], [path], auto_reset='new_world')
    for bad in ("new-world", "same_world", "True"):
        with pytest.raises(ValueError, match="new_world"):
            VecRandomAisleTurnEnv(4, auto_reset=bad)
        with pytest.raises(ValueError, match="new_world"):
            VecPlanEnv([cm], [path], auto_reset=bad)
