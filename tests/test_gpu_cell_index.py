"""GPU: the per-map cell index (BCG_BATCH_CELL_INDEX) equals the occupancy plane, and the sparse egocentric kernel that
reads it renders the same crops and compact hit lists as the oracle and as the listing from the occupancy plane."""
import ctypes as C

import numpy as np
import pytest
import torch

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200.envs.base.params import EnvParams
from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
from bc_gym_planning_env_b200.vec_env import VecPlanEnv
from oracle import plan_env_oracle as O
from tests.test_cell_index_host import cell_index_reference

pytestmark = pytest.mark.gpu


def _device_descs(env):
    return np.frombuffer(env.map_descs.cpu().numpy().tobytes(), dtype=np.dtype(nat.BcgMapDesc))


def _trailer_at(d):
    return int(d['sum_off']) + int(d['tiles_y']) * ((int(d['tiles_x']) + 31) // 32)


def _trailer(env, d):
    arena = env.occ_sum_arena.cpu().numpy().view(np.uint32)
    at, ntiles = _trailer_at(d), int(d['tiles_x']) * int(d['tiles_y'])
    cap, total = int(arena[at]), int(arena[at + 1])
    return cap, total, arena[at + 2:at + 3 + ntiles], arena[at + 3 + ntiles:at + 3 + ntiles + min(cap, total)]


def _pool(n_maps, seed):
    ep = EnvParams()
    costmaps, paths = random_aisle_pool(n_maps, seed, ep)
    return ep, costmaps, paths


@pytest.mark.parametrize("private", [False, True])
def test_index_equals_numpy_recomputation(private):
    ep, costmaps, paths = _pool(5, 31)
    env = VecPlanEnv(costmaps, paths, ep, n_envs=13, noise_parameters=None, with_ego=True, private_map_copies=private)
    assert env._batch.flags & nat.BATCH_CELL_INDEX
    descs = _device_descs(env)
    assert len(descs) == (13 if private else 5)
    for k, d in enumerate(descs):
        data = costmaps[int(env._map_ids_host[k]) if private else k].get_data()
        prefix_want, cells_want = cell_index_reference(data)
        cap, total, prefix, cells = _trailer(env, d)
        assert d['flags'] & nat.MAP_CELL_INDEX, k
        assert cap == total == len(cells_want)
        assert np.array_equal(prefix, prefix_want) and np.array_equal(cells, cells_want), k
    assert len({int(d['sum_off']) for d in descs}) == len(descs)       # every private copy owns its index


def _crops_at_random_poses(env, costmaps, rng, n_trials=6):
    n, res = env.n_envs, env.resolution
    for _ in range(n_trials):
        poses = np.zeros((n, 3))
        for e in range(n):
            c = costmaps[int(env._map_ids_host[e])]
            size = np.array([c.get_data().shape[1], c.get_data().shape[0]]) * res
            poses[e, :2] = c.get_origin() + rng.uniform(-0.1, 1.1, 2) * size
            poses[e, 2] = rng.uniform(-np.pi, np.pi)
        env.state_f[nat.F_DPOSE:nat.F_DPOSE + 3] = torch.from_numpy(poses.T.copy()).cuda()
        img, _ = env.observe_ego()
        yield poses, img.cpu().numpy()[..., 0], int(env._ego_list[n])


def _assert_crops_match_oracle(env, costmaps, seed):
    for poses, img, handed_over in _crops_at_random_poses(env, costmaps, np.random.RandomState(seed)):
        assert handed_over == 0
        for e in range(env.n_envs):
            c = costmaps[int(env._map_ids_host[e])]
            assert np.array_equal(img[e], O.ego_costmap(c.get_data(), poses[e], c.get_origin(), env.resolution)), e


def test_crops_from_the_index_match_the_oracle():
    ep, costmaps, paths = _pool(6, 5)
    env = VecPlanEnv(costmaps, paths, ep, n_envs=96, noise_parameters=None, with_ego=True, private_map_copies=True)
    _assert_crops_match_oracle(env, costmaps, 8)
    env.check_status()


def test_map_past_its_capacity_loses_its_bit_and_still_renders_exactly():
    ep, costmaps, paths = _pool(4, 9)
    env = VecPlanEnv(costmaps, paths, ep, n_envs=32, noise_parameters=None, with_ego=True, private_map_copies=True)
    d3 = _device_descs(env)[3]
    cap, _, _, _ = _trailer(env, d3)
    at = _trailer_at(d3)
    env.occ_sum_arena[at] = cap - 1                   # one cell short: nothing may be written past the capacity
    guard_at = at + 3 + int(d3['tiles_x']) * int(d3['tiles_y']) + cap - 1
    env.occ_sum_arena[guard_at] = 0x5eed
    nat.check(nat.lib().bcg_build_lethal_tiles(C.byref(env._batch), 0, env._batch.n_maps, env._stream()))
    torch.cuda.synchronize()
    descs = _device_descs(env)
    assert not descs[3]['flags'] & nat.MAP_CELL_INDEX
    assert all(descs[k]['flags'] & nat.MAP_CELL_INDEX for k in range(len(descs)) if k != 3)
    assert env.occ_sum_arena[guard_at].item() == 0x5eed
    _assert_crops_match_oracle(env, costmaps, 4)
    env.check_status()


def _hit_sets(compact):
    counts = compact['counts'].numpy()
    words = compact['packed'].numpy().view(np.uint16 if compact['value'] is not None else np.uint32)
    starts = np.r_[0, np.cumsum(np.where((counts > 0) & (counts <= compact['cap']), counts, 0))]
    return [frozenset(words[starts[e]:starts[e + 1]].tolist()) if counts[e] > 0 else int(counts[e]) for e in range(len(counts))]


def test_compact_hits_and_crops_equal_those_of_the_occupancy_listing():
    """Per env, the compact hit list (as a set) and the crop are the same with the index and without it (batch bit
    cleared: the sparse kernel lists the window's cells from the occupancy plane), and the list expands to the crop."""
    ep, costmaps, paths = _pool(8, 17)
    runs = []
    for use_index in (True, False):
        env = VecPlanEnv(costmaps, paths, ep, n_envs=512, seed=3, with_ego=True, private_map_copies=True, compact_ego=True)
        if not use_index:
            env._batch.flags &= ~nat.BATCH_CELL_INDEX
        lo, hi = env.action_bounds()
        rng = np.random.RandomState(1)
        h, w = env.ego_image.shape[1], env.ego_image.shape[2]
        steps = []
        for t in range(12):
            acts = torch.from_numpy((lo + (hi - lo) * rng.random_sample((env.n_envs, 2))).astype(np.float32))
            res = env.step_host(acts.pin_memory(), images="compact")
            img = env.ego_image.cpu().numpy()[..., 0]
            assert np.array_equal(VecPlanEnv.expand_compact(res[3], h, w), img), (use_index, t)
            steps.append((img, _hit_sets(res[3])))
        assert int(env._ego_list[env.n_envs]) == 0
        env.check_status()
        runs.append(steps)
    for (img_a, hits_a), (img_b, hits_b) in zip(*runs):
        assert np.array_equal(img_a, img_b)
        assert hits_a == hits_b
