"""-m gpu: edge cases of the batched step against the oracle -- robots that leave their (tiny) map, maps smaller than the
footprint, two-point paths, batch sizes that do not fill a warp or a block, a finished path stepped on, and the error
codes of the C entry points for malformed calls (reference behaviour: envs/base/env.py:464-489 skips out-of-map
footprint pixels, utilities/costmap_utils.py:72 pads the egocentric crop with zeros, envs/base/reward.py:223-224 pays
nothing once the path is finished)."""
import ctypes as C

import numpy as np
import pytest
import torch

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200.envs.base.params import EnvParams
from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
from bc_gym_planning_env_b200.vec_env import VecPlanEnv
from oracle import plan_env_oracle as O
from tests import common

pytestmark = pytest.mark.gpu


_tiny_worlds = common.tiny_worlds


def _build(worlds, n_envs=None, **kw):
    costmaps = [CostMap2D(m, 0.03, o.astype(np.float64)) for m, o, _ in worlds]
    paths = [p for _, _, p in worlds]
    ep = EnvParams(control_delay=1, pose_delay=1, state_delay=2)
    env = VecPlanEnv(costmaps, paths, ep, n_envs=n_envs, noise_parameters=None, with_ego=True, **kw)
    n = env.n_envs
    oracles = [O.OraclePlanEnv(worlds[e % len(worlds)][0], worlds[e % len(worlds)][1], 0.03, worlds[e % len(worlds)][2],
                               delays=(1, 1, 2)) for e in range(n)]
    return env, oracles


def _compare_step(env, oracles, actions, t, check_images):
    obs, r, done, _ = env.step(actions)
    pose, rew, dn = obs.pose.cpu().numpy(), r.cpu().numpy(), done.cpu().numpy()
    tgt, hit = obs.target_idx.cpu().numpy(), env.hit.cpu().numpy()
    img = env.ego_image.cpu().numpy()[..., 0] if check_images else None
    goal = env.goal_n_state.cpu().numpy() if check_images else None
    for e, o in enumerate(oracles):
        oo, r2, d2, h2 = o.step(actions[e])
        np.testing.assert_allclose(pose[e], oo["pose"], rtol=0, atol=1e-9, err_msg="step %d env %d" % (t, e))
        assert rew[e] == pytest.approx(r2, abs=1e-9) and bool(dn[e]) == d2 and bool(hit[e]) == bool(h2), (t, e)
        assert int(tgt[e]) == o.target_idx, (t, e)
        if check_images:
            assert np.array_equal(img[e], O.ego_costmap(o.costmap, o.pose, o.origin, o.resolution)), (t, e)
            want = O.goal_n_state(oo["path"], oo["pose"], oo["robot_state"], o.resolution)
            np.testing.assert_allclose(goal[e, :, 0], want, rtol=0, atol=2e-6)
    return hit


def test_robots_leaving_tiny_maps_match_the_oracle():
    worlds = _tiny_worlds()
    env, oracles = _build(worlds)
    rng = np.random.RandomState(7)
    low, high = env.action_bounds()
    hits = 0
    for t in range(260):
        a = rng.uniform(low, high, size=(env.n_envs, 2)).astype(np.float32)
        a[:, 1] = rng.uniform(-0.15, 0.15, size=env.n_envs)   # nearly straight: the robots do leave their maps
        hits += int(_compare_step(env, oracles, a, t, check_images=(t % 13 == 0 or t > 250)).sum())
    # every robot ended up outside its map (the last crops are compared above: all zeros where no map is)
    for e, o in enumerate(oracles):
        h, w = o.costmap.shape
        px = (o.pose[:2] - o.origin) / o.resolution
        assert not (0 <= px[0] < w and 0 <= px[1] < h), e
    assert hits > 0                                      # the all-lethal map was driven into
    env.check_status()


@pytest.mark.parametrize("n_envs", [1, 31, 33, 67, 130])
def test_batch_sizes_that_do_not_fill_a_warp_or_block(n_envs):
    """Env e of a batch of any size computes what env e % 4 computes alone (same world, same actions)."""
    worlds = _tiny_worlds()
    env, _ = _build(worlds, n_envs=n_envs)
    ref, _ = _build(worlds)
    rng = np.random.RandomState(3)
    low, high = env.action_bounds()
    for t in range(60):
        a4 = rng.uniform(low, high, size=(4, 2)).astype(np.float32)
        a = a4[np.arange(n_envs) % 4]
        env.step(a)
        ref.step(a4)
    idx = torch.arange(n_envs, device="cuda") % 4
    assert torch.equal(env.state_f, ref.state_f[:, idx]) and torch.equal(env.state_i, ref.state_i[:, idx])
    assert torch.equal(env.ego_image, ref.ego_image[idx]) and torch.equal(env.goal_n_state, ref.goal_n_state[idx])
    assert torch.equal(env.reward, ref.reward[idx]) and torch.equal(env.done, ref.done[idx])
    env.check_status()


def test_two_point_path_and_stepping_after_the_goal():
    """A path that is not refined (two points 2.5 m apart): once the robot is within the goal tolerance of the second
    point the reference keeps stepping with reward 0, done True and an empty remaining path (goal_n_state all zeros)."""
    m = np.zeros((120, 120), dtype=np.uint8)
    path = np.array([[0., 0., 0.], [2.5, 0., 0.]])
    ep = EnvParams(refine_path=False)
    env = VecPlanEnv([CostMap2D(m, 0.03, np.array([-1.8, -1.8]))], [path], ep, noise_parameters=None, with_ego=True)
    o = O.OraclePlanEnv(m, np.array([-1.8, -1.8]), 0.03, path, refine=False)
    a = np.array([[0.5, 0.0]], dtype=np.float32)
    seen_done = 0
    for t in range(140):
        obs, r, done, _ = env.step(a)
        oo, r2, d2, _ = o.step(a[0])
        np.testing.assert_allclose(obs.pose.cpu().numpy()[0], oo["pose"], rtol=0, atol=1e-9)
        assert float(r[0]) == r2 and bool(done[0]) == d2 and int(obs.target_idx[0]) == o.target_idx, t
        want = O.goal_n_state(oo["path"], oo["pose"], oo["robot_state"], 0.03)
        np.testing.assert_allclose(env.goal_n_state.cpu().numpy().reshape(-1), want, rtol=0, atol=2e-6)
        seen_done += int(d2)
    assert seen_done > 20 and o.target_idx == len(path)          # finished early, kept stepping
    assert float(env.goal_n_state.abs().sum()) == 0.0
    env.check_status()


def test_malformed_step_calls_return_error_codes():
    """The C entry points report bad arguments through their return code and bcg_last_error -- nothing is thrown,
    nothing is launched."""
    env, _ = _build(_tiny_worlds())
    lib = nat.lib()
    s = env._stream()
    a = torch.zeros((env.n_envs, 2), dtype=torch.float32, device="cuda")
    before = env.state_f.clone()
    assert lib.bcg_step(C.byref(env._c_params), C.byref(env._batch), None, None, 0, 0, C.byref(env._out), None, None, s) < 0
    assert lib.bcg_step(C.byref(env._c_params), C.byref(env._batch), None, nat.ptr(a), 0, 0, None, None, None, s) < 0
    assert "null" in nat.last_error()
    assert lib.bcg_observe_ego(C.byref(env._c_params), C.byref(env._batch), None, None, s) < 0
    torch.cuda.synchronize()
    assert torch.equal(env.state_f, before)
    with pytest.raises(ValueError):
        env.step(np.zeros((env.n_envs + 1, 2), dtype=np.float32))
    with pytest.raises(ValueError):
        VecPlanEnv([], [], EnvParams())


def _summary_is_exact(env, desc):
    """Tile summary bit (tx, ty) == tile (tx, ty) of the occupancy plane holds a cell."""
    tx, ty = desc.tiles_x, desc.tiles_y
    occ = env.occ_tile_arena[desc.tile_off:desc.tile_off + tx * ty * 16].view(ty, tx, 16)
    want = (occ != 0).any(dim=2).cpu().numpy()
    sw = (tx + 31) // 32
    words = env.occ_sum_arena[desc.sum_off:desc.sum_off + ty * sw].view(ty, sw).cpu().numpy().astype(np.uint32)
    got = ((words[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1).reshape(ty, sw * 32)
    assert not got[:, tx:].any()
    return np.array_equal(got[:, :tx].astype(bool), want)


def test_tile_summary_follows_the_occupancy_plane():
    """The one-bit-per-tile summary the sparse egocentric kernel trusts: exact for uploaded maps (shared and private
    copies) and for device-generated worlds after repeated regeneration in place."""
    from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
    from bc_gym_planning_env_b200.vec_aisle_env import VecRandomAisleTurnEnv, VecRandomMiniEnv
    ep = EnvParams()
    costmaps, paths = random_aisle_pool(6, 77, ep)
    costmaps = list(costmaps) + [CostMap2D(m, 0.03, o.astype(np.float64)) for m, o, _ in _tiny_worlds()]
    paths = list(paths) + [p for _, _, p in _tiny_worlds()]
    for private in (False, True):
        env = VecPlanEnv(costmaps, paths, ep, n_envs=23, noise_parameters=None, with_ego=True, private_map_copies=private)
        assert env.occ_sum_arena is not None
        for d in env._map_descs_host:
            assert _summary_is_exact(env, d)
    for cls in (VecRandomAisleTurnEnv, VecRandomMiniEnv):
        genv = cls(48, seed=11, with_ego=True) if cls is VecRandomMiniEnv else cls(48, ep, seed=11, with_ego=True)
        for rep in range(4):
            genv.generate()
            mask = torch.zeros(48, dtype=torch.bool, device="cuda")
            mask[rep::3] = True
            genv.generate(mask)
            for e in range(48):
                assert _summary_is_exact(genv, genv._map_desc(e)), (cls.__name__, rep, e)
        genv.check_status()
