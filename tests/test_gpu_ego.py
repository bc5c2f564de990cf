"""-m gpu: egocentric observation (crop image + goal_n_state) against the reference's
EgocentricCostmap wrapper (fixture aisle_ego) -- images bit-exact, vector to one fp32 ulp."""
import numpy as np
import pytest
import torch

from tests import common

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kernel,name", [("tiles", "aisle_ego"), ("dense", "aisle_ego"), ("tiles", "edge_worlds"),
                                         ("dense", "edge_worlds"), ("tiles", "aisle_goal_reached"), ("dense", "aisle_goal_reached")])
def test_ego_observation_matches_reference(kernel, name):
    """Both egocentric kernels against cv2: `tiles` is the default (the sparse scatter kernel, the dense cell-tile kernel
    for the envs it hands over), `dense` the dense cell-tile kernel for every env (ego_sparse=False); `edge_worlds`: crops
    that lie partly or wholly outside tiny maps (the reference pads with zeros)."""
    d = common.load(name)
    env = common.make_vec_env(d, with_ego=True, ego_sparse=(kernel == "tiles"))
    actions = torch.from_numpy(d["actions"]).cuda()
    every = int(d["every"])
    k = 0
    for t in range(actions.shape[1]):
        env.step(actions[:, t].contiguous())
        if "ref_goal_n_state_all" in d:              # the goal vector at every step, across the goal-reached transition
            vec = env.goal_n_state.cpu().numpy()[..., 0]
            ref = d["ref_goal_n_state_all"][:, t]
            assert np.all(np.abs(vec - ref) <= np.spacing(np.abs(ref).astype(np.float32)) + 1e-12), t
            assert np.array_equal((vec == 0).all(axis=1), (ref == 0).all(axis=1)), t    # all zeros once the path is finished
        if t % every == every - 1:
            img = env.ego_image.cpu().numpy()[..., 0]
            vec = env.goal_n_state.cpu().numpy()[..., 0]
            assert np.array_equal(img, d["ref_ego_image"][:, k]), "ego image differs at step %d" % t
            ref = d["ref_goal_n_state"][:, k]
            assert np.all(np.abs(vec - ref) <= np.spacing(np.abs(ref).astype(np.float32)) + 1e-12), t
            k += 1
    assert k == d["ref_ego_image"].shape[1]
    assert (d["ref_ego_image"] != 0).any()
    env.check_status()


def test_observe_ego_standalone_equals_step_output():
    d = common.load("aisle_ego")
    env = common.make_vec_env(d, with_ego=True)
    actions = torch.from_numpy(d["actions"]).cuda()
    for t in range(10):
        env.step(actions[:, t].contiguous())
    img_step = env.ego_image.clone()
    vec_step = env.goal_n_state.clone()
    img, vec = env.observe_ego()
    assert torch.equal(img, img_step) and torch.equal(vec, vec_step)


def test_colored_ego_variant_matches_reference():
    """ColoredEgoCostmapRandomAisleTurnEnv (reference envs/synth_turn_env.py:380-451): 133x133 crop about the
    TRUE robot pose, goal = unit vector to the last path point + (v, w, wheel)."""
    d = common.load("aisle_colored_ego")
    env = common.make_vec_env(d)                       # EnvParams(): no delays, like the reference class
    actions = torch.from_numpy(d["actions"]).cuda()
    every = int(d["every"])
    k = 0
    for t in range(actions.shape[1]):
        env.step(actions[:, t].contiguous())
        if t % every == every - 1:
            image, goal = env.observe_colored_ego()
            assert tuple(image.shape[1:]) == (133, 133, 1) and tuple(goal.shape[1:]) == (5, 1)
            assert np.array_equal(image.cpu().numpy()[..., 0], d["ref_environment"][:, k]), t
            np.testing.assert_allclose(goal.cpu().numpy()[..., 0], d["ref_goal"][:, k], rtol=2e-7, atol=1e-7)
            k += 1
    assert (d["ref_environment"] != 0).any()
    # the wrapper-style observation is unaffected by the variant call
    img9, vec9 = env.observe_ego()
    assert tuple(img9.shape[1:]) == (133, 117, 1) and tuple(vec9.shape[1:]) == (9, 1)
