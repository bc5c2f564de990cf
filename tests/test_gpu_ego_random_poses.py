"""-m gpu: egocentric crops at arbitrary poses -- deep inside, straddling every map edge and far
outside the map -- against the oracle's closed form of cv2.warpAffine (itself pinned against cv2 in the
CPU suite)."""
import numpy as np
import pytest
import torch

from bc_gym_planning_env_b200 import _native as nat
from oracle import plan_env_oracle as O
from tests import common

pytestmark = pytest.mark.gpu


def _random_poses(maps, res, rng, trial):
    """One pose per (costmap, origin, path): anywhere inside, hugging an edge, on the path or well outside the map."""
    poses = np.zeros((len(maps), 3))
    for e, (cm, origin, path) in enumerate(maps):
        size = np.array([cm.shape[1], cm.shape[0]]) * res
        kind = trial % 4
        if kind == 0:      # anywhere inside
            poses[e, :2] = origin + rng.uniform(0, 1, 2) * size
        elif kind == 1:    # hugging an edge
            poses[e, :2] = origin + rng.choice([0.0, 1.0], 2) * size + rng.uniform(-1.5, 1.5, 2)
        elif kind == 2:    # on the path
            poses[e, :2] = path[rng.randint(len(path)), :2]
        else:              # well outside
            poses[e, :2] = origin + size / 2 + rng.choice([-1, 1], 2) * (size / 2 + rng.uniform(0, 6, 2))
        poses[e, 2] = rng.uniform(-np.pi, np.pi) if trial % 5 else rng.choice([0, np.pi / 2, -np.pi / 2, -np.pi])
    return poses


def _wide_crop_env(dense_map):
    """Random aisle turns at resolution 0.02 m, where the crop (175 x 200 px) is wider than the dense kernel's 160-entry
    column table; with `dense_map` one map gets a filled region of every cost class (more than 1 cell in 20 occupied)."""
    from bc_gym_planning_env_b200.envs.base.params import EnvParams
    from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
    from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
    from bc_gym_planning_env_b200.vec_env import VecPlanEnv
    res = 0.02
    params = EnvParams(resolution=res)
    costmaps, paths = random_aisle_pool(6, 41, params)
    if dense_map:
        rng = np.random.RandomState(5)
        data = costmaps[0].get_data().copy()
        h, w = data.shape
        data[h // 4:3 * h // 4, w // 4:3 * w // 4] = rng.choice([1, 100, 253, 254, 255], size=(3 * h // 4 - h // 4, 3 * w // 4 - w // 4))
        costmaps[0] = CostMap2D(data, res, np.array(costmaps[0].get_origin(), dtype=np.float64))
    env = VecPlanEnv(costmaps, paths, params, noise_parameters=None, with_ego=True)
    assert (env._c_params.ego_w, env._c_params.ego_h) == (175, 200)
    assert bool(env._batch.flags & nat.BATCH_SPARSE_EGO_ONLY) != dense_map
    maps = [(c.get_data(), np.array(c.get_origin()), np.asarray(p)) for c, p in zip(costmaps, paths)]
    return env, maps, res


@pytest.mark.parametrize("world", ["aisle_collision", "res002_sparse", "res002_dense"])
def test_ego_crops_at_random_poses(world):
    """`aisle_collision`: the fixture's maps at 0.03 m.  `res002_*`: crops wider than the dense kernel's column table, which
    every env gets from a bounds-checked direct gather -- the sparse kernel's own when every map is sparse, the dense
    kernel's when a dense map in the batch makes the sparse kernel hand its envs over."""
    if world == "aisle_collision":
        d = common.load(world)
        env = common.make_vec_env(d, with_ego=True)
        maps, res, trials = common.fixture_envs(d), float(d["resolution"]), 40
    else:
        env, maps, res = _wide_crop_env(world == "res002_dense")
        trials = 20
    rng = np.random.RandomState(3)
    nonzero = 0
    for trial in range(trials):
        poses = _random_poses(maps, res, rng, trial)
        env.state_f[nat.F_DPOSE:nat.F_DPOSE + 3] = torch.from_numpy(poses.T.copy()).cuda()
        img, _ = env.observe_ego()
        img = img.cpu().numpy()[..., 0]
        for e, (cm, origin, _) in enumerate(maps):
            want = O.ego_costmap(cm, poses[e], origin, res)
            assert np.array_equal(img[e], want), (trial, e, poses[e])
            nonzero += int((want != 0).sum())
    assert nonzero > 1000
    # the step's own record writers give the same crops
    env.step(torch.zeros((env.n_envs, 2), dtype=torch.float32, device="cuda"))
    img_step = env.ego_image.clone()
    img, _ = env.observe_ego()
    assert torch.equal(img, img_step)
    env.check_status()


def _painted_maps(d, rng, fill):
    """The fixture's aisle maps with extra cost values: a sprinkle of cells of every cost class (sparse: the
    scatter kernel must fetch the values) or a filled inscribed region (dense: handed to the dense kernel)."""
    from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
    res = float(d["resolution"])
    out = []
    for cm, origin, path in common.fixture_envs(d):
        cm = cm.copy()
        h, w = cm.shape
        if fill:
            cm[h // 4:3 * h // 4, w // 4:3 * w // 4] = rng.choice([253, 255, 100, 1], size=(3 * h // 4 - h // 4, 3 * w // 4 - w // 4))
        else:
            ys, xs = rng.randint(0, h, 600), rng.randint(0, w, 600)
            cm[ys, xs] = rng.choice([1, 100, 253, 254, 255], size=600)
            cm[0, :] = 255                      # map border rows / columns are sampled by crops that straddle an edge
            cm[:, w - 1] = 7
        out.append((CostMap2D(cm, res, np.array(origin, dtype=np.float64)), path))
    return out


@pytest.mark.parametrize("fill", [False, True])
def test_sparse_and_dense_paths_carry_every_cost_value(fill):
    from bc_gym_planning_env_b200.vec_env import VecPlanEnv
    d = common.load("aisle_collision")
    rng = np.random.RandomState(11)
    worlds = _painted_maps(d, rng, fill)
    env = VecPlanEnv([c for c, _ in worlds], [p for _, p in worlds], common.env_params(d["params"]) if "params" in d else None,
                     noise_parameters=None, with_ego=True)
    n, res = env.n_envs, float(d["resolution"])
    seen = set()
    for trial in range(24):
        poses = np.zeros((n, 3))
        for e, (c, path) in enumerate(worlds):
            size = np.array([c.get_data().shape[1], c.get_data().shape[0]]) * res
            poses[e, :2] = c.get_origin() + rng.uniform(-0.1, 1.1, 2) * size
            poses[e, 2] = rng.uniform(-np.pi, np.pi) if trial % 4 else rng.choice([0, np.pi / 2, np.pi, -np.pi / 2])
        env.state_f[nat.F_DPOSE:nat.F_DPOSE + 3] = torch.from_numpy(poses.T.copy()).cuda()
        img, _ = env.observe_ego()
        img = img.cpu().numpy()[..., 0]
        # (a pool in which every map is dense is built without the sparse kernel: all envs go through the dense one)
        handed_over = int(env._ego_list[n]) if env._ego_list is not None else n
        seen.add(handed_over > 0)
        for e, (c, _) in enumerate(worlds):
            want = O.ego_costmap(c.get_data(), poses[e], c.get_origin(), res)
            assert np.array_equal(img[e], want), (fill, trial, e, poses[e])
    assert (True in seen) == fill        # filled maps overflow the cell list at least once; sprinkled ones never do
    env.check_status()
