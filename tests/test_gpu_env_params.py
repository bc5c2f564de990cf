"""GPU: per-env parameters in one batch (BcgEnvRows).  A batch built from a pool computes, column by column, exactly what a
batch of one setting computes: bit for bit, state rows, rings and outputs."""
import numpy as np
import pytest
import torch

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200.envs.base.params import EnvParams, RewardParams
from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
from bc_gym_planning_env_b200.vec_aisle_env import VecRandomAisleTurnEnv
from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE, VecPlanEnv

pytestmark = pytest.mark.gpu

N = 4096
RINGS = ('control', 'pose', 'state')


def _actions(env, steps, seed):
    lo, hi = env.action_bounds()
    rng = np.random.RandomState(seed)
    a = rng.uniform(lo, hi, size=(steps, env.n_envs, 2)).astype(np.float32)
    return torch.from_numpy(a).to(env.device)


def _pool4():
    """four sets that differ in every per-env field"""
    sets = [
        EnvParams(control_delay=0, pose_delay=0, state_delay=0),
        EnvParams(control_delay=2, pose_delay=1, state_delay=1, goal_spat_dist=0.2, goal_ang_dist=np.pi / 8, iteration_timeout=150),
        EnvParams(control_delay=1, pose_delay=2, state_delay=0,
                  reward_provider_params=RewardParams(spatial_precision=1.0, angular_precision=np.pi / 2,
                                                      spatial_progress_multiplier=0.5)),
        EnvParams(control_delay=3, pose_delay=0, state_delay=2, goal_spat_dist=0.2, goal_ang_dist=np.pi / 8, iteration_timeout=150,
                  reward_provider_params=RewardParams(spatial_precision=0.2, angular_precision=np.pi / 8,
                                                      spatial_progress_multiplier=0.5)),
    ]
    noise = [DEFAULT_NOISE, None, {k: 4 * v for k, v in DEFAULT_NOISE.items()},
             dict(alpha1=1e-3, alpha2=2e-3, alpha3=0.0, alpha4=5e-3, alpha5=0.0, alpha6=1e-2)]
    return sets, noise


def _columns_equal(mixed, single, envs, outputs=True):
    """fixed rows, the env's own ring slots (same slot positions: its queue heads run modulo its own delay) and outputs"""
    idx = torch.as_tensor(envs, dtype=torch.int64, device=mixed.device)
    assert torch.equal(mixed.state_f[:nat.F_FIXED][:, idx], single.state_f[:nat.F_FIXED][:, idx])
    assert torch.equal(mixed.state_i[:, idx], single.state_i[:, idx])
    for which in RINGS:
        row0, _, ncomp, _ = mixed.queue_rows(which)
        srow0, d, _, _ = single.queue_rows(which)
        assert torch.equal(mixed.state_f[row0:row0 + d * ncomp][:, idx], single.state_f[srow0:srow0 + d * ncomp][:, idx]), which
    if not outputs:
        return
    assert torch.equal(mixed.reward[idx], single.reward[idx])
    assert torch.equal(mixed.done[idx], single.done[idx])
    assert torch.equal(mixed.hit[idx], single.hit[idx])
    assert torch.equal(mixed.obs_vec[idx], single.obs_vec[idx])
    if mixed.with_ego:
        assert torch.equal(mixed.ego_image[idx], single.ego_image[idx])
        assert torch.equal(mixed.goal_n_state[idx], single.goal_n_state[idx])


def _assert_same(a, b):
    for name in ('state_f', 'state_i', 'reward', '_done_u8', '_hit_u8', 'obs_vec', 'ego_image', 'goal_n_state'):
        assert torch.equal(getattr(a, name), getattr(b, name)), name


@pytest.fixture(scope="module")
def worlds():
    return random_aisle_pool(64, 0)


def test_rows_of_one_set_equal_no_rows(worlds):
    costmaps, paths = worlds
    ep = EnvParams(control_delay=2, pose_delay=1, state_delay=1)
    kw = dict(n_envs=N, noise_parameters=DEFAULT_NOISE, auto_reset=True, with_ego=True, compact_ego=True, seed=3)
    plain = VecPlanEnv(costmaps, paths, ep, **kw)
    rows = VecPlanEnv(costmaps, paths, [ep], **kw)
    assert plain._rows is None and rows._rows is not None
    _assert_same(plain, rows)
    acts = _actions(plain, 300, 1)
    for t in range(300):
        plain.step(acts[t])
        rows.step(acts[t])
        if t % 25 == 0 or t == 299:
            _assert_same(plain, rows)
    assert torch.equal(plain.episode_stats(), rows.episode_stats())
    assert plain.episode_stats()[0] > 0                     # episodes ended (and auto-reset) along the way
    for t in range(20):
        plain.step_graph(acts[t])
        rows.step_graph(acts[t])
    _assert_same(plain, rows)
    plain.rollout(acts[:20])
    rows.rollout(acts[:20])
    _assert_same(plain, rows)
    for t in range(3):
        host = acts[t].cpu().pin_memory()
        ra = plain.step_host(host, images='compact')
        ca = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in ra[3].items()}
        rb = rows.step_host(host, images='compact')
        for k in ('counts', 'offsets'):
            assert torch.equal(ca[k], rb[3][k]), k
        h, w = plain.ego_image.shape[1:3]                     # (a crop's hit list comes in no particular order)
        assert np.array_equal(VecPlanEnv.expand_compact(ca, h, w), VecPlanEnv.expand_compact(rb[3], h, w))
        torch.cuda.synchronize()
        _assert_same(plain, rows)
    assert torch.equal(plain.episode_stats(), rows.episode_stats())


@pytest.mark.parametrize("assign", ["interleaved", "random"])
def test_columns_equal_single_setting_batches(worlds, assign):
    costmaps, paths = worlds
    sets, noise = _pool4()
    ids = np.arange(N) % 4 if assign == "interleaved" else np.random.RandomState(7).randint(0, 4, N)
    kw = dict(n_envs=N, auto_reset=True, with_ego=True, seed=11)
    mixed = VecPlanEnv(costmaps, paths, sets, noise_parameters=noise, params_ids=ids, **kw)
    singles = [VecPlanEnv(costmaps, paths, sets[k], noise_parameters=noise[k], **kw) for k in range(4)]
    assert mixed.queue_rows('control')[1] == 3 and mixed.queue_rows('state', e=int(np.flatnonzero(ids == 1)[0]))[1] == 1
    assert torch.equal(mixed.delays.cpu(), torch.tensor([[sets[k].control_delay, sets[k].pose_delay, sets[k].state_delay]
                                                         for k in ids], dtype=torch.int32))
    for e in (0, 1, 2, 3):
        assert mixed.params_of(e) is sets[ids[e]] and mixed.noise_of(e) is noise[ids[e]]
    members = [np.flatnonzero(ids == k) for k in range(4)]
    for k in range(4):
        _columns_equal(mixed, singles[k], members[k])
    acts = _actions(mixed, 400, 2)
    for t in range(400):
        mixed.step(acts[t])
        for s in singles:
            s.step(acts[t])
        if t % 40 == 0 or t == 399:
            for k in range(4):
                _columns_equal(mixed, singles[k], members[k])


def test_contiguous_blocks_equal_sub_batches(worlds):
    costmaps, paths = worlds
    sets, noise = _pool4()
    block = N // 4
    ids = np.repeat(np.arange(4), block)
    env_map = np.arange(N) % len(costmaps)
    kw = dict(auto_reset=True, with_ego=True, seed=5)
    mixed = VecPlanEnv(costmaps, paths, sets, n_envs=N, noise_parameters=noise, params_ids=ids, map_ids=env_map,
                       path_ids=env_map, **kw)
    subs = [VecPlanEnv(costmaps, paths, sets[k], n_envs=block, noise_parameters=noise[k], env_id_base=k * block,
                       map_ids=env_map[k * block:(k + 1) * block], path_ids=env_map[k * block:(k + 1) * block], **kw)
            for k in range(4)]
    acts = _actions(mixed, 400, 3)
    for t in range(400):
        mixed.step(acts[t])
        for k, s in enumerate(subs):
            s.step(acts[t, k * block:(k + 1) * block])
    for k, s in enumerate(subs):
        sl = slice(k * block, (k + 1) * block)
        assert torch.equal(mixed.state_f[:nat.F_FIXED, sl], s.state_f[:nat.F_FIXED])
        assert torch.equal(mixed.state_i[:, sl], s.state_i)
        assert torch.equal(mixed.reward[sl], s.reward) and torch.equal(mixed.done[sl], s.done)
        assert torch.equal(mixed.ego_image[sl], s.ego_image) and torch.equal(mixed.goal_n_state[sl], s.goal_n_state)
    st = mixed.episode_stats().cpu().numpy()
    parts = np.sum([s.episode_stats().cpu().numpy() for s in subs], axis=0)
    counters = [nat.STAT_NAMES.index(n) for n in ("episodes", "length", "collided", "goal", "timeout")]
    assert np.array_equal(st[counters], parts[counters])
    assert st[0] > 0
    assert abs(st[1] - parts[1]) <= 1e-9 * max(1.0, abs(parts[1]))


@pytest.mark.parametrize("draw_new_turn", [True, False])
def test_randomisation_at_reset(draw_new_turn):
    sets, noise = _pool4()
    n = 1024
    kw = dict(seed=9, with_ego=True, draw_new_turn_on_reset=draw_new_turn)
    ids0 = np.arange(n) % 4
    mixed = VecRandomAisleTurnEnv(n, params=sets, noise_parameters=noise, params_ids=ids0, **kw)
    singles = [VecRandomAisleTurnEnv(n, params=sets[k], noise_parameters=noise[k], **kw) for k in range(4)]
    acts = _actions(mixed, 120, 4)
    for t in range(60):
        mixed.step(acts[t])
        for s in singles:
            s.step(acts[t])
    rng = np.random.RandomState(12)
    mask = rng.rand(n) < 0.5
    new = rng.randint(0, 4, n)
    mixed.reset(torch.from_numpy(mask), params_ids=new)
    for s in singles:
        s.reset(torch.from_numpy(mask))
    ids = np.where(mask, new, ids0)
    assert np.array_equal(mixed.params_ids, ids)
    members = [np.flatnonzero(ids == k) for k in range(4)]
    moved = np.flatnonzero(mask & (new != ids0))
    assert len(moved) > 0
    for k in range(4):                                        # (the outputs are still those of the last step)
        _columns_equal(mixed, singles[k], np.intersect1d(members[k], moved), outputs=False)
    for t in range(60, 120):
        mixed.step(acts[t])
        for s in singles:
            s.step(acts[t])
    for k in range(4):
        _columns_equal(mixed, singles[k], members[k])
    # reset without params_ids keeps every env's set
    mixed.reset(torch.from_numpy(mask))
    assert np.array_equal(mixed.params_ids, ids)


def test_snapshots_between_envs(worlds):
    costmaps, paths = worlds
    pool = [EnvParams(control_delay=2, pose_delay=1, state_delay=1), EnvParams()]
    env = VecPlanEnv(costmaps[:1], paths[:1], pool, n_envs=3, noise_parameters=None, params_ids=[0, 1, 0])
    acts = _actions(env, 40, 5)
    for t in range(20):
        env.step(acts[t])
    env.set_state(env.get_state([0]), [2], load_delayed_robot=False)
    same = acts.clone()
    same[:, 2] = same[:, 0]
    for t in range(20, 40):
        env.step(same[t])
        assert torch.equal(env.state_f[:, 0], env.state_f[:, 2])
        assert torch.equal(env.state_i[:, 0], env.state_i[:, 2])
    with pytest.raises(ValueError, match="do not fit"):
        env.set_state(env.get_state([0]), [1])


def test_reference_fixtures_in_one_batch():
    """Four recorded reference fixtures (delays 1/2/0, 2/1/1 with timeout 220, the mini env's tolerances without delays,
    2/1/1 to the goal) as ONE batch of 36 envs, each with its own EnvParams: every env matches its fixture's recorded
    reference trajectory like test_gpu_rollouts.py::test_step_matches_reference, the goal-reached envs also its crops."""
    from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
    from tests import common
    names = ["aisle_delays_120", "aisle_delays_211", "mini_noise_off", "aisle_goal_reached"]
    fx = [common.load(n) for n in names]
    costmaps, paths, pool, ids, spans = [], [], [], [], []
    for k, d in enumerate(fx):
        res = float(d["resolution"])
        for cm, origin, path in common.fixture_envs(d):
            costmaps.append(CostMap2D(cm, res, np.array(origin, dtype=np.float64)))
            paths.append(path)
            ids.append(k)
        pool.append(common.env_params(d["params"]))
        spans.append((len(ids) - int(d["n_envs"]), len(ids)))
    n = len(ids)
    assert n == 36
    T = max(d["actions"].shape[1] for d in fx)
    acts = np.zeros((n, T, 2), dtype=np.float32)
    for (a, b), d in zip(spans, fx):
        acts[a:b, :d["actions"].shape[1]] = d["actions"]
    env = VecPlanEnv(costmaps, paths, pool, n_envs=n, noise_parameters=None, params_ids=ids, with_ego=True)
    assert env.queue_rows('control')[1] == 2 and env.queue_rows('pose')[1] == 2 and env.queue_rows('state')[1] == 1
    actions = torch.from_numpy(acts).cuda()
    rec = {k: [] for k in ("pose", "robot_state", "true_pose", "reward", "done", "collided", "target_idx", "min_dist", "time")}
    crops, k_goal = [], names.index("aisle_goal_reached")
    every = int(fx[k_goal]["every"])
    for t in range(T):
        obs, r, done, _ = env.step(actions[:, t].contiguous())
        rec["pose"].append(obs.pose.cpu().numpy().copy())
        rec["robot_state"].append(obs.robot_state.cpu().numpy().copy())
        rec["true_pose"].append(env.state_f[nat.F_ROBOT:nat.F_ROBOT + 3].t().cpu().numpy().copy())
        rec["reward"].append(r.cpu().numpy().copy())
        rec["done"].append(done.cpu().numpy().copy())
        rec["collided"].append(env.state_i[nat.I_COLLIDED].cpu().numpy().astype(bool))
        rec["target_idx"].append(obs.target_idx.cpu().numpy().copy())
        rec["min_dist"].append(env.state_f[nat.F_MIN_DIST].cpu().numpy().copy())
        rec["time"].append(obs.time.cpu().numpy().copy())
        if t % every == every - 1 and t < fx[k_goal]["actions"].shape[1]:
            a, b = spans[k_goal]
            crops.append(env.ego_image[a:b, ..., 0].cpu().numpy())
    env.check_status()
    got = {k: np.swapaxes(np.array(v), 0, 1) for k, v in rec.items()}
    for (a, b), d, name in zip(spans, fx, names):
        steps = d["actions"].shape[1]
        for k in ("done", "collided", "target_idx"):
            assert np.array_equal(got[k][a:b, :steps], d["ref_" + k]), (name, k)
        for k in ("pose", "robot_state", "true_pose", "reward", "min_dist", "time"):
            np.testing.assert_allclose(got[k][a:b, :steps], d["ref_" + k], rtol=0, atol=common.TIGHT_ATOL, err_msg="%s %s" % (name, k))
    assert np.array_equal(np.stack(crops, axis=1), fx[k_goal]["ref_ego_image"])
