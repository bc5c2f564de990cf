"""CPU: the C-ABI shared library builds, loads, exports every symbol include/bcg_b200.h declares and
agrees with the ctypes mirrors.  No compute call needs a GPU here; the ones that do must fail loudly."""
import ctypes as C
import os
import re

import pytest

from bc_gym_planning_env_b200 import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BCG_ERR_INVALID = -1                                   # include/bcg_b200.h


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "bcg_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(bcg_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_the_declared_abi_version_14():
    lib = nat.lib()
    declared = _declared_symbols()
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), "libbcg_b200.so does not export %s" % name
    assert sorted(nat.SYMBOLS) == declared, "ctypes binding and header disagree"
    assert lib.bcg_abi_version() == 14


def test_one_entry_point_per_operation():
    # bcg_step, bcg_rollout, bcg_init_state and bcg_generate_aisles take NULL rows / ends / events themselves: no
    # suffixed variant of them is exported, no stand-alone kinematics step and no tensor-map encoder (the egocentric
    # kernels stage their windows from the cell tiles only)
    lib = nat.lib()
    for name in ("bcg_init_state_rows", "bcg_generate_aisles_rows", "bcg_step_events", "bcg_step_rows", "bcg_step_ends",
                 "bcg_rollout_rows", "bcg_rollout_ends", "bcg_kinematic_step", "bcg_encode_map_tensor_maps"):
        assert not hasattr(lib, name), "libbcg_b200.so still exports %s" % name
        assert name not in nat.SYMBOLS


def test_struct_mirrors_match_library():
    lib = nat.lib()
    for which, struct in enumerate(nat._STRUCTS):
        assert lib.bcg_sizeof(which) == C.sizeof(struct), struct.__name__
    assert lib.bcg_sizeof(99) == -1


def test_state_layout_follows_delays():
    L0 = nat.state_layout(nat.BcgParams())
    assert (L0.n_frows, L0.n_irows) == (nat.F_FIXED, nat.I_FIXED)
    L = nat.state_layout(nat.BcgParams(delay_control=2, delay_pose=1, delay_state=3))
    assert L.ring_control == nat.F_FIXED and L.ring_pose == L.ring_control + 4
    assert L.ring_state == L.ring_pose + 3 and L.n_frows == L.ring_state + 21
    with pytest.raises(nat.BcgError):
        nat.state_layout(nat.BcgParams(delay_pose=-1))


def test_bad_arguments_return_error_codes():
    lib = nat.lib()
    assert lib.bcg_step(None, None, None, None, 0, 0, None, None, None, None) < 0
    assert "null" in nat.last_error()
    assert lib.bcg_world_to_pixel(None, 4, 0.0, 0.0, 0.05, None, None) < 0
    p, b = nat.BcgParams(), nat.BcgBatch()
    assert lib.bcg_step(C.byref(p), C.byref(b), None, None, 0, 0, None, None, None, None) < 0
    assert "n_envs" in nat.last_error()


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


@pytest.mark.parametrize("field", ["occ_tile_arena", "occ_sum_arena"])
def test_batch_without_occupancy_plane_or_summary_is_refused(field):
    # the collision check, the egocentric kernels and the world generators read the occupancy plane and its tile
    # summary unconditionally: a batch without either is refused before anything is launched
    lib = nat.lib()
    p, b = _batch_with_dummy_pointers()
    plan = C.c_void_p(0x1000)
    assert lib.bcg_rollout(C.byref(p), C.byref(b), None, plan, 0, 0, None, None, None) == 0
    assert lib.bcg_build_lethal_tiles(C.byref(b), 0, 0, None) == 0
    setattr(b, field, None)
    assert lib.bcg_rollout(C.byref(p), C.byref(b), None, plan, 0, 0, None, None, None) == BCG_ERR_INVALID
    assert field in nat.last_error()
    assert lib.bcg_build_lethal_tiles(C.byref(b), 0, 0, None) == BCG_ERR_INVALID
    assert field in nat.last_error()


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(nat.BcgError):
        nat.require_cuda()
    from bc_gym_planning_env_b200.envs.base.params import EnvParams
    from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
    from bc_gym_planning_env_b200.vec_env import VecPlanEnv
    costmaps, paths = random_aisle_pool(1, 0)
    with pytest.raises(nat.BcgError):
        VecPlanEnv(costmaps, paths, EnvParams())


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "bc_gym_planning_env_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), os.path.join(dirpath, f)
