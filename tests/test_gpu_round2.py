"""-m gpu: what round 2 added around the step -- the CUDA-graph step with its device-side step counter, the compact
egocentric observation and its host expander, the sparse kernel's in-kernel fallback for windows that overflow its cell
list, the device-side goal flags of the Monte-Carlo fan-out, and the unmodified reference stepped live beside the CUDA
batch when its package is importable on this box (oracle/_ref, installed by oracle/make_ref.py)."""
import numpy as np
import pytest
import torch

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200.envs.base.params import EnvParams
from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE, VecPlanEnv
from oracle import plan_env_oracle as O
from tests import common

pytestmark = pytest.mark.gpu


def _actions(env, steps, seed):
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    low, high = env.action_bounds()
    lo, hi = torch.from_numpy(low).cuda(), torch.from_numpy(high).cuda()
    return [(lo + (hi - lo) * torch.rand((env.n_envs, 2), generator=gen, device="cuda")).contiguous() for _ in range(steps)]


def test_graph_step_equals_plain_step_with_noise_and_auto_reset():
    """step_graph replays one captured graph per step and takes the Philox step index from the device-side counter: 150
    steps with noise and auto-reset give the same bits as 150 plain steps, and the two ways of stepping can be mixed."""
    params = EnvParams(control_delay=2, pose_delay=1, state_delay=1)
    costmaps, paths = random_aisle_pool(24, 77, params)
    kw = dict(n_envs=600, seed=5, auto_reset=True, with_ego=True, noise_parameters=DEFAULT_NOISE)
    a, b = VecPlanEnv(costmaps, paths, params, **kw), VecPlanEnv(costmaps, paths, params, **kw)
    acts = _actions(a, 150, 3)
    for t, act in enumerate(acts):
        a.step(act)
        if 60 <= t < 80:
            b.step(act)                                  # plain steps in between: they use the device counter too
        else:
            b.step_graph(act)
        if t % 25 == 24:
            assert torch.equal(a.state_f, b.state_f) and torch.equal(a.state_i, b.state_i), t
            assert torch.equal(a.ego_image, b.ego_image) and torch.equal(a.goal_n_state, b.goal_n_state), t
            assert torch.equal(a.reward, b.reward) and torch.equal(a.done, b.done) and torch.equal(a.obs_vec, b.obs_vec), t
    assert float(a.episode_stats()[0]) > 0 and torch.equal(a.episode_stats(), b.episode_stats())
    assert int(b._step_counter[0]) == 150 and int(b._step_counter[1]) == 0
    a.check_status()
    b.check_status()


def test_compact_observation_expands_to_the_image():
    d = common.load("aisle_ego")
    env = common.make_vec_env(d, with_ego=True, compact_ego=True)
    actions = torch.from_numpy(d["actions"])
    h, w = env.ego_image.shape[1], env.ego_image.shape[2]
    for t in range(actions.shape[1]):
        res = env.step_host(actions[:, t].contiguous().pin_memory(), images="compact")
        compact, goal = res[3], res[4]
        got = VecPlanEnv.expand_compact(compact, h, w)
        assert np.array_equal(got, env.ego_image.cpu().numpy()[..., 0]), t
        assert torch.equal(goal, env.goal_n_state.cpu())
        counts = compact["counts"].numpy()
        assert np.array_equal(np.where(counts > 0, counts, 0), (got != 0).reshape(len(got), -1).sum(axis=1))
        if t % 6 == 5:
            assert np.array_equal(got, d["ref_ego_image"][:, t // 6])      # ... which is the reference's crop
    assert compact["bytes"] < 0.2 * env.ego_image.numel()
    env.check_status()


def _blob_world():
    """a map far below the dense threshold (1 cell in 20) with one filled block next to the path: its windows hold more
    occupied cells than the sparse kernel's list"""
    m = np.zeros((500, 500), dtype=np.uint8)
    m[230:290, 300:360] = 254
    m[100, 50:450] = 253
    return CostMap2D(m, 0.03, np.array([0., 0.])), np.array([[7.4, 7.8, 0.0], [14.0, 7.8, 0.0]])     # starts 1.6 m before the block


def test_sparse_kernel_renders_overflowing_windows_itself():
    cm, path = _blob_world()
    assert np.count_nonzero(cm.get_data()) * 20 < cm.get_data().size
    env = VecPlanEnv([cm], [path], EnvParams(), n_envs=64, noise_parameters=None, with_ego=True, compact_ego=True)
    assert env._batch.flags & nat.BATCH_SPARSE_EGO_ONLY and env.launches_per_step() == 3
    rng = np.random.RandomState(0)
    poses = np.stack([rng.uniform(5.0, 12.0, 64), rng.uniform(5.5, 9.5, 64), rng.uniform(-np.pi, np.pi, 64)], axis=1)
    env.state_f[nat.F_DPOSE:nat.F_DPOSE + 3] = torch.from_numpy(poses.T.copy()).cuda()
    img, _ = env.observe_ego()
    img = img.cpu().numpy()[..., 0]
    overflowed = 0
    for e in range(64):
        want = O.ego_costmap(cm.get_data(), poses[e], cm.get_origin(), 0.03)
        assert np.array_equal(img[e], want), e
        overflowed += int((want != 0).sum() > 1200)
    assert overflowed >= 5                               # the block fills many of the crops
    # through a step: the compact lists flag those envs (-1) and the host gets their crops densely
    acts = torch.zeros((64, 2), dtype=torch.float32).pin_memory()
    res = env.step_host(acts, images="compact")
    got = VecPlanEnv.expand_compact(res[3], img.shape[1], img.shape[2])
    assert np.array_equal(got, env.ego_image.cpu().numpy()[..., 0])
    assert (res[3]["counts"].numpy() < 0).sum() == len(res[3]["dense_envs"]) >= 1
    assert int(env._ego_list[64]) == 0                   # nothing was handed to the dense kernel
    env.check_status()


def test_goal_flags_and_path_lengths_on_device():
    d = common.load("aisle_goal_reached")
    env = common.make_vec_env(d)
    assert [int(v) for v in env.path_lengths()] == [len(d["path_%d" % e]) for e in range(int(d["n_envs"]))]
    actions = torch.from_numpy(d["actions"]).cuda()
    for t in range(actions.shape[1]):
        env.step(actions[:, t].contiguous())
        assert np.array_equal(env.goal_reached().cpu().numpy(), d["ref_path_len"][:, t] == 0), t
    assert bool(env.goal_reached().all())
    with pytest.raises(ValueError):
        env.reset(mask=np.ones(3, dtype=bool))          # a mask of the wrong length never reaches the kernel


def _stored_reference_beside_the_cuda_batch():
    """Where the reference package is not importable: the same comparison against its outputs recorded in tests/golden,
    the CUDA batch stepped with the egocentric observation on.  aisle_delays_211 (12 envs x 300 steps, delays (2, 1, 1),
    noise off, iteration_timeout 220: collisions and timeouts) and aisle_goal_reached (6 envs x 240 steps, delays
    (2, 1, 1), paths driven to their end; goal_n_state of every step, crops of every 3rd) -- flags exact, floats to
    1e-9, goal_n_state to one fp32 spacing, crops exact."""
    seen_done = seen_hit = crops = 0
    for name in ("aisle_delays_211", "aisle_goal_reached"):
        d = common.load(name)
        env = common.make_vec_env(d, with_ego=True)
        actions = torch.from_numpy(d["actions"]).cuda()
        every = int(d["every"]) if "every" in d else 0
        for t in range(actions.shape[1]):
            obs, r, done, _ = env.step(actions[:, t].contiguous())
            np.testing.assert_allclose(obs.pose.cpu().numpy(), d["ref_pose"][:, t], rtol=0, atol=1e-9)
            np.testing.assert_allclose(obs.robot_state.cpu().numpy(), d["ref_robot_state"][:, t], rtol=0, atol=1e-9)
            assert np.array_equal(r.cpu().numpy(), d["ref_reward"][:, t]) and np.array_equal(done.cpu().numpy(), d["ref_done"][:, t]), t
            assert np.array_equal(obs.target_idx.cpu().numpy(), d["ref_target_idx"][:, t]), t
            assert np.array_equal(env.state_i[nat.I_COLLIDED].cpu().numpy().astype(bool), d["ref_collided"][:, t]), t
            if "ref_goal_n_state_all" in d:
                vec, ref = env.goal_n_state.cpu().numpy()[..., 0], d["ref_goal_n_state_all"][:, t]
                assert np.all(np.abs(vec - ref) <= np.spacing(np.abs(ref).astype(np.float32)) + 1e-12), t
            if every and t % every == every - 1:
                assert np.array_equal(env.ego_image.cpu().numpy()[..., 0], d["ref_ego_image"][:, t // every]), t
                crops += 1
        seen_done += int(d["ref_done"].sum())
        seen_hit += int(d["ref_collided"].sum())
        env.check_status()
    assert seen_done > 0 and seen_hit > 0 and crops == 80


def test_live_reference_beside_the_cuda_batch():
    """No fixtures in between: 16 envs of the UNMODIFIED reference stepped beside the CUDA batch for 300 steps, delays
    (2, 1, 1), noise off -- flags exact, floats to 1e-9, crops exact.  Without the reference package: its recorded
    outputs instead (_stored_reference_beside_the_cuda_batch)."""
    from oracle.ref_loader import load_reference, reference_available
    if not reference_available():
        _stored_reference_beside_the_cuda_batch()
        return
    load_reference()
    from bc_gym_planning_env.envs.base.action import Action
    from bc_gym_planning_env.envs.base.params import EnvParams as RefParams
    from bc_gym_planning_env.envs.egocentric import EgocentricCostmap
    from bc_gym_planning_env.envs.synth_turn_env import RandomAisleTurnEnv
    n, steps = 16, 300
    refs = []
    for s in range(n):
        base = RandomAisleTurnEnv(params=RefParams(control_delay=2, pose_delay=1, state_delay=1, iteration_timeout=250), seed=4000 + s)
        base._env._robot.set_noise_parameters(None)
        refs.append((base, EgocentricCostmap(base)))
    costmaps = [CostMap2D(b._env._state.costmap.get_data().copy(), 0.03, np.array(b._env._state.costmap.get_origin())) for b, _ in refs]
    paths = [np.array(b._env._state.original_path) for b, _ in refs]
    params = EnvParams(control_delay=2, pose_delay=1, state_delay=1, iteration_timeout=250, refine_path=False)
    env = VecPlanEnv(costmaps, paths, params, noise_parameters=None, with_ego=True)
    rng = np.random.RandomState(12)
    low, high = env.action_bounds()
    seen_done = seen_hit = 0
    for t in range(steps):
        a = rng.uniform(low, high, size=(n, 2)).astype(np.float32)
        obs, r, done, _ = env.step(a)
        pose, rs = obs.pose.cpu().numpy(), obs.robot_state.cpu().numpy()
        rew, dn, tgt = r.cpu().numpy(), done.cpu().numpy(), obs.target_idx.cpu().numpy()
        img = env.ego_image.cpu().numpy()[..., 0] if t % 10 == 9 else None
        vec = env.goal_n_state.cpu().numpy()[..., 0]
        for e, (base, wrapped) in enumerate(refs):
            o2, r2, d2, _ = wrapped.step(Action(command=a[e]))
            plain = base._env._extract_obs()
            st = plain.robot_state
            np.testing.assert_allclose(pose[e], plain.pose, rtol=0, atol=1e-9)
            np.testing.assert_allclose(rs[e], [st.x, st.y, st.angle, st.v, st.w, st.steering_motor_command, st.wheel_angle], rtol=0, atol=1e-9)
            assert rew[e] == r2 and bool(dn[e]) == d2, (t, e)
            assert tgt[e] == base._env._state.reward_provider_state.target_idx, (t, e)
            assert bool(env.state_i[nat.I_COLLIDED][e]) == base._env._state.robot_collided
            ref_vec = o2["goal_n_state"][:, 0]
            assert np.all(np.abs(vec[e] - ref_vec) <= np.spacing(np.abs(ref_vec).astype(np.float32)) + 1e-12), (t, e)
            if img is not None:
                assert np.array_equal(img[e], o2["env"][..., 0]), (t, e)
            seen_done += int(d2)
            seen_hit += int(base._env._state.robot_collided)
    assert seen_done > 0 and seen_hit > 0
    env.check_status()


def test_move_kernel_register_tiers_give_the_same_bits():
    """move_kernel is built three times (230 / 168 / 128 registers) and bcg_step picks one by its block count (64 threads
    per block) on S SMs: tier 0 up to 4 S blocks, tier 1 up to 6 S, tier 2 above.  The same envs stepped as the head of
    a 4 096-env batch (tier 0), of a 320 S + 13 one (the middle of tier 1: 47 373 envs on a 148-SM B200) and of a
    448 S + 29 one (tier 2: 66 333) agree bit for bit: state, rewards, done flags, compact observation, egocentric crops
    and goal vectors, with noise, delays and auto-reset on."""
    from tests.test_gpu_step_matrix import move_tier
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    params = EnvParams(control_delay=2, pose_delay=1, state_delay=1)
    costmaps, paths = random_aisle_pool(16, 31, params)
    head = 4096
    sizes = (head, 320 * sms + 13, 448 * sms + 29)
    assert [move_tier(n, sms) for n in sizes] == [0, 1, 2], (sms, sizes)
    envs = [VecPlanEnv(costmaps, paths, params, n_envs=n, seed=9, auto_reset=True, with_ego=True, noise_parameters=DEFAULT_NOISE)
            for n in sizes]
    acts = _actions(envs[0], 120, 11)
    for t, act in enumerate(acts):
        for env in envs:
            full = act if env.n_envs == head else act.repeat((env.n_envs + head - 1) // head, 1)[:env.n_envs].contiguous()
            env.step(full)
        if t % 20 == 19:
            ref = envs[0]
            for env in envs[1:]:
                assert torch.equal(ref.state_f, env.state_f[:, :head]) and torch.equal(ref.state_i, env.state_i[:, :head]), (t, env.n_envs)
                assert torch.equal(ref.reward, env.reward[:head]) and torch.equal(ref.done, env.done[:head]), (t, env.n_envs)
                assert torch.equal(ref.obs_vec, env.obs_vec[:head]), (t, env.n_envs)
                assert torch.equal(ref.ego_image, env.ego_image[:head]), (t, env.n_envs)
                assert torch.equal(ref.goal_n_state, env.goal_n_state[:head]), (t, env.n_envs)
    assert float(envs[0].episode_stats()[0]) > 0
    for env in envs:
        env.check_status()


def test_rollout_and_rollout_graph_equal_plain_steps():
    """rollout (one library call launching the H steps back to back) and rollout_graph (the H steps as one captured
    graph, device-side step counter): state, last rewards and accumulated returns equal H plain steps, also on a second
    plan."""
    params = EnvParams(control_delay=2, pose_delay=1, state_delay=1)
    costmaps, paths = random_aisle_pool(12, 5, params)
    kw = dict(n_envs=300, seed=21, auto_reset=False, with_ego=False, noise_parameters=DEFAULT_NOISE)
    a, b, c = (VecPlanEnv(costmaps, paths, params, **kw) for _ in range(3))
    H = 40
    for rep in range(2):
        plan = torch.stack(_actions(a, H, 100 + rep))
        for h in range(H):
            a.step(plan[h])
        b.rollout_graph(plan)
        c.rollout(plan)
        for other in (b, c):
            assert torch.equal(a.state_f, other.state_f) and torch.equal(a.state_i, other.state_i), rep
            assert torch.equal(a.reward, other.reward) and torch.equal(a.done, other.done), rep
    with pytest.raises(ValueError):
        b.rollout_graph(plan[:, :10])
    with pytest.raises(ValueError):
        c.rollout(plan[:, :10])
    for env in (a, b, c):
        env.check_status()
