"""-m gpu: the collision check for footprint tables of every shape, against the CPU oracle.

The thread-per-env check (collide_warp_balanced, which move_kernel and collision_thread_kernel inline) takes boxes of one
shape on its fast path: one-word mask rows (masks at most 64 px wide) in aligned pairs, at most 4 tile columns and 6
bands.  Every other box goes to collide_thread's plain loop, which reads each row with mask_bits32.  The tricycle at
0.03 m has 60-row masks of one word at footprint_scale 1.0 (the fast path); at 1.5 (88 rows) and 2.0 (118 rows, up to 9
bands: two batches of 6) its rows take two words and every check runs that loop, as do the multi-word arms of the
warp-per-env tile and uint8 kernels.

Poses are points of random aisle paths jittered by +-0.8 m and +-3 rad, poses that straddle the map's border and poses
wholly outside it, in batches of 4 096, 37 and 5 envs (partly filled warps), each with hits and misses, and in one batch
whose warps each share one map and one pose (collide_warp_balanced's equal-list branch: no dealing).  The three stand-alone kernels must agree flag
for flag, and a sample matches the oracle's verdicts and in-map pixel counts.  Then the step with that loop inside
move_kernel: 16 envs at footprint_scale 1.5 beside OraclePlanEnv, and a batch large enough for the 128-register move_kernel
build (the one with the most register pressure), sampled.
"""
import numpy as np
import pytest
import torch

from oracle import plan_env_oracle as O
from tests.test_gpu_step_matrix import MOVE_THREADS, action_stream, move_tier, sample_envs

pytestmark = pytest.mark.gpu

ROBOT = "industrial_tricycle_v1"
SCALES = (1.0, 1.5, 2.0)
WPR = {1.0: 1, 1.5: 2, 2.0: 2}         # words per mask row of the tricycle's table at 0.03 m
POOL = 32
SAMPLE = 320                           # oracle-checked envs per batch (all of a smaller batch)


def _pool():
    from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
    return random_aisle_pool(POOL, 5)


def _poses(env, seed):
    """[n, 3]: per env a jittered point of its path; every tenth env straddles its map's border (a pose within 0.6 m of an
    edge, half of them also of a corner), every tenth lies 6 m outside the map"""
    rng = np.random.RandomState(seed)
    poses = np.empty((env.n_envs, 3))
    for e in range(env.n_envs):
        cm = env.costmap(e)
        h, w = cm.get_data().shape
        (ox, oy), res = cm.get_origin(), cm.get_resolution()
        lo, hi = np.array([ox, oy]), np.array([ox + w * res, oy + h * res])
        th = rng.uniform(-np.pi, np.pi)
        kind = e % 10
        if kind == 8:
            xy = rng.uniform(lo, hi)
            axes = [rng.randint(2)] if rng.rand() < 0.5 else [0, 1]
            for a in axes:
                xy[a] = (lo[a] if rng.rand() < 0.5 else hi[a]) + rng.uniform(-0.6, 0.6)
        elif kind == 9:
            xy = rng.uniform(lo, hi)
            a = rng.randint(2)
            xy[a] = lo[a] - 6.0 if rng.rand() < 0.5 else hi[a] + 6.0
        else:
            p = env.full_path(e)
            q = p[rng.randint(len(p))]
            xy = q[:2] + rng.uniform(-0.8, 0.8, 2)
            th = q[2] + rng.uniform(-3.0, 3.0)
        poses[e] = (xy[0], xy[1], th)
    return poses


def _check_batch(env, poses, scale, seed):
    """the three kernels against one another, and a sample against the oracle; returns the flags"""
    pt = torch.from_numpy(poses).cuda()
    thread = env.pose_collides(pt).cpu().numpy()
    u8 = env.pose_collides(pt, use_u8=True).cpu().numpy()
    flags, pixels = env.pose_collides(pt, count_pixels=True)
    flags, pixels = flags.cpu().numpy(), pixels.cpu().numpy()
    what = (scale, env.n_envs)
    assert np.array_equal(thread, u8), (what, np.flatnonzero(thread != u8)[:20])
    assert np.array_equal(thread, flags), (what, np.flatnonzero(thread != flags)[:20])
    n = env.n_envs
    sample = np.arange(n) if n <= SAMPLE else np.random.RandomState(seed).choice(n, SAMPLE, replace=False)
    footprint = np.asarray(O.ROBOTS[ROBOT]["footprint"]) * scale
    for e in sample:
        cm = env.costmap(int(e))
        data, origin, res = cm.get_data(), cm.get_origin(), cm.get_resolution()
        x, y, th = poses[e]
        assert bool(thread[e]) == O.pose_collides(x, y, th, footprint, data, origin, res), what + (int(e), poses[e])
        assert pixels[e] == O.footprint_pixels_in_map(x, y, th, footprint, data.shape, origin, res), what + (int(e), poses[e])
    env.check_status()
    return thread


@pytest.mark.parametrize("scale", SCALES)
def test_three_collision_kernels_match_the_oracle(scale):
    from bc_gym_planning_env_b200.envs.base.params import EnvParams
    from bc_gym_planning_env_b200.vec_env import VecPlanEnv, footprint_lut_for
    ep = EnvParams()
    assert ep.resolution == 0.03 and footprint_lut_for(ROBOT, ep.resolution, scale).wpr == WPR[scale]
    costmaps, paths = _pool()
    env = VecPlanEnv(costmaps, paths, ep, n_envs=4096, seed=1, footprint_scale=scale)
    poses = _poses(env, seed=4096)
    hits = _check_batch(env, poses, scale, seed=4096)
    assert hits.any() and not hits.all(), (scale, int(hits.sum()))
    assert not hits[9::10].any(), scale                                     # (a pose outside the map never collides)
    # partly filled warps: env e takes a pose of the large batch on its own map (e % POOL), a hit for even e and a miss
    # for odd e where that map has one
    for n in (37, 5):
        pick = []
        for e in range(n):
            same = np.arange(e % POOL, len(hits), POOL)
            want = same[hits[same] == (e % 2 == 0)]
            pick.append(want[e // POOL % len(want)] if len(want) else same[0])
        small = VecPlanEnv(costmaps, paths, ep, n_envs=n, seed=1, footprint_scale=scale)
        h = _check_batch(small, poses[pick], scale, seed=n)
        assert h.any() and not h.all(), (scale, n, int(h.sum()))
    # every warp on one map and one pose: the lanes' tile lists are equal, collide_warp_balanced does not deal
    n = 4096
    ids = (np.arange(n) // 32) % POOL
    env = VecPlanEnv(costmaps, paths, ep, n_envs=n, map_ids=ids, path_ids=ids, seed=1, footprint_scale=scale)
    poses = np.repeat(_poses(env, seed=7)[::32], 32, axis=0)
    hits = _check_batch(env, poses, scale, seed=7)
    assert hits.any() and not hits.all(), (scale, int(hits.sum()))
    assert (hits.reshape(-1, 32) == hits[::32, None]).all()


def _oracle(costmap, path, ep, scale):
    return O.OraclePlanEnv(costmap.get_data(), costmap.get_origin(), costmap.get_resolution(), path,
                           delays=(ep.control_delay, ep.pose_delay, ep.state_delay), timeout=ep.iteration_timeout,
                           footprint_scale=scale)


def _step_beside_oracles(n, sample, steps=150, scale=1.5):
    """n envs at footprint_scale `scale`, noise off, stepped `steps` times; envs `sample` beside their oracles (pose to
    1e-9, reward and done exact).  Returns how many of the sampled envs collided."""
    from bc_gym_planning_env_b200.envs.base.params import EnvParams
    from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
    from bc_gym_planning_env_b200.vec_env import VecPlanEnv
    ep = EnvParams(control_delay=1, pose_delay=1, state_delay=0)
    costmaps, paths = random_aisle_pool(16, 41, ep)
    env = VecPlanEnv(costmaps, paths, ep, n_envs=n, noise_parameters=None, seed=3, footprint_scale=scale)
    oracles = [_oracle(costmaps[e % 16], paths[e % 16], ep, scale) for e in sample]
    idx = torch.from_numpy(np.asarray(sample, dtype=np.int64)).cuda()
    for t, a in enumerate(action_stream(steps=steps, n=n)):
        obs, r, d, _ = env.step(torch.from_numpy(a).cuda())
        pose, rew, done = obs.pose[idx].cpu().numpy(), r[idx].cpu().numpy(), d[idx].cpu().numpy()
        for k, (e, o) in enumerate(zip(sample, oracles)):
            oo, r2, d2, _ = o.step(a[e])
            assert np.all(np.abs(pose[k] - oo["pose"]) <= 1e-9), (n, int(e), t, pose[k], oo["pose"])
            assert rew[k] == r2 and bool(done[k]) == d2, (n, int(e), t)
    env.check_status()
    return sum(o.collided for o in oracles)


def test_wide_footprint_step_matches_the_oracle():
    """16 envs: collide_thread inside move_kernel's lowest tier, and the rollback of a pose it finds in collision"""
    assert _step_beside_oracles(16, np.arange(16)) > 0


def test_wide_footprint_step_at_the_128_register_build():
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 7 * sms * MOVE_THREADS + 13        # in the middle of tier 2 (more than 6 blocks per SM), not a multiple of 32
    assert move_tier(n, sms) == 2
    assert _step_beside_oracles(n, sample_envs(n, sms, [])) > 0
