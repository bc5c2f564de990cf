"""Episode ends of auto-reset batches (episode_ends=True): reason bits, terminated / truncated and the final observation
of every episode that ends, checked against a twin batch that steps the same envs without auto-reset -- whose step
outputs ARE the final observations -- and is reset by the host afterwards."""
import numpy as np
import pytest
import torch

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200.envs.base.params import CONTINUOUS_REWARD_PURE_PURSUIT, EnvParams
from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE, VecPlanEnv
from tests import common

pytestmark = pytest.mark.gpu

CAUSES = nat.END_GOAL | nat.END_COLLIDED | nat.END_TIMEOUT


# ---- worlds and batches ----------------------------------------------------------------------------------------------
def _goal_fixture():
    return common.load("aisle_goal_reached")


def _cost_block(cm, origin, path, res, side, value=50):
    """a square of a non-lethal cost around the start pose: its windows hold more cells than the sparse kernel's list"""
    m = cm.copy()
    px, py = int((path[0, 0] - origin[0]) / res), int((path[0, 1] - origin[1]) / res)
    h = side // 2
    blk = m[max(py - h, 0):py + h + 1, max(px - h, 0):px + h + 1]
    blk[blk == 0] = value
    return m


def _speckled(cm, density=0.08, value=30, seed=3):
    """non-lethal costs on a fraction of the free cells: a dense map (more than 1 cell in 20 occupied)"""
    m = cm.copy()
    rng = np.random.RandomState(seed)
    m[(rng.rand(*m.shape) < density) & (m == 0)] = value
    return m


def _worlds(d, extra=()):
    """the six goal-fixture worlds, plus variants: 'dense' (world 1 speckled), 'overflow' (world 2 with a cost block)"""
    res = float(d["resolution"])
    worlds = [(cm, np.array(o, dtype=np.float64), p) for cm, o, p in common.fixture_envs(d)]
    out = list(worlds)
    for kind in extra:
        if kind == "dense":
            cm, o, p = worlds[1]
            m = _speckled(cm)
            assert np.count_nonzero(m) * 20 > m.size
            out.append((m, o, p))
        elif kind == "overflow":
            cm, o, p = worlds[2]
            m = _cost_block(cm, o, p, res, 45)
            assert np.count_nonzero(m) * 20 <= m.size and np.count_nonzero(m) - np.count_nonzero(cm) > 896
            out.append((m, o, p))
    return [CostMap2D(cm, res, o) for cm, o, _ in out], [p for _, _, p in out]


def _pool(d, provider=None):
    """the fixture's own set (the recorded goal actions reach their goals with it) and three sets with short timeouts"""
    over = {} if provider is None else dict(reward_provider_name=provider)
    p = d["params"]
    sets = [common.env_params(p, **over),
            common.env_params(p, iteration_timeout=25, **over),
            common.env_params(p, iteration_timeout=40, control_delay=0, pose_delay=0, state_delay=0, **over),
            common.env_params(p, iteration_timeout=60, control_delay=1, pose_delay=2, state_delay=0, **over)]
    return sets, [None, DEFAULT_NOISE, None, DEFAULT_NOISE]


def _twins(d, n=48, provider=None, extra=(), capacity=None, **kw):
    costmaps, paths = _worlds(d, extra)
    k = len(costmaps)
    ids = np.arange(n) % k
    pset = np.where(np.arange(n) < 6, 0, 1 + np.arange(n) % 3)
    sets, noise = _pool(d, provider)
    common_kw = dict(n_envs=n, map_ids=ids, path_ids=ids, params_ids=pset, noise_parameters=noise, seed=7, with_ego=True)
    common_kw.update(kw)
    a = VecPlanEnv(costmaps, paths, sets, auto_reset=True, episode_ends=True, episode_end_capacity=capacity, **common_kw)
    b = VecPlanEnv(costmaps, paths, sets, auto_reset=False, episode_ends=True, **common_kw)
    return a, b


def _actions(env, d, steps, seed=11):
    """uniform random actions; envs 0..5 replay the fixture's recorded goal-reaching actions first"""
    low, high = env.action_bounds()
    acts = np.random.RandomState(seed).uniform(low, high, size=(steps, env.n_envs, 2)).astype(np.float32)
    rec = np.swapaxes(d["actions"], 0, 1)
    t = min(steps, rec.shape[0])
    acts[:t, :rec.shape[1]] = rec[:t]
    return torch.from_numpy(acts).cuda()


# ---- checks -------------------------------------------------------------------------------------------------------------
def _bits(t):
    t = t.contiguous()
    return (t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int64) if t.element_size() == 8 else t).cpu().numpy()


def _timeouts(env):
    return np.array([env.params_of(e).iteration_timeout for e in range(env.n_envs)])


def _causes_from_state(env, timeouts):
    """the reason bits a done env must report, from its state after the step (env.py:407-419)"""
    goal = env.goal_reached().cpu().numpy()
    coll = env.state_i[nat.I_COLLIDED].cpu().numpy() != 0
    tmo = env.state_i[nat.I_ITER].cpu().numpy() >= timeouts
    causes = goal * nat.END_GOAL | coll * nat.END_COLLIDED | tmo * nat.END_TIMEOUT
    return np.where(env.done.cpu().numpy(), causes, 0)


def _check_finals(fo, b, idx, images=None):
    """final rows of the envs `idx` (which ended) equal what twin `b`, not reset, observes after the same step; the final
    crops (in `images`, default fo.ego_image) of those that have a slot equal its crops"""
    it = torch.from_numpy(idx).cuda()
    assert np.array_equal(_bits(fo.obs_vec[it]), _bits(b.obs_vec[it]))
    assert np.array_equal(_bits(fo.episode_return[it]), _bits(b.state_f[nat.F_EP_RETURN][it]))
    assert np.array_equal(fo.episode_length[it].cpu().numpy(), b.state_i[nat.I_ITER][it].cpu().numpy())
    if b.with_ego:
        assert np.array_equal(_bits(fo.goal_n_state[it]), _bits(b.goal_n_state[it]))
        slot = fo.slot.cpu().numpy()[idx]
        have = slot >= 0
        got = (fo.ego_image if images is None else images)[torch.from_numpy(slot[have]).cuda().long()]
        assert np.array_equal(got.cpu().numpy(), b.ego_image[it[torch.from_numpy(have).cuda()]].cpu().numpy())


def _check_step(a, b, timeouts):
    """a (auto-reset) and b (its twin without) have just made the same step; b has not been reset since its last step's
    done envs were.  Returns the ended envs."""
    assert torch.equal(a.done, b.done) and np.array_equal(_bits(a.reward), _bits(b.reward))
    causes = _causes_from_state(b, timeouts)
    reason = a.episode_reason.cpu().numpy().astype(np.int64)
    assert np.array_equal(reason & CAUSES, causes)
    now = (reason & nat.END_NOW) != 0
    assert np.array_equal(now, b.done.cpu().numpy())              # b enters every step with no env done
    assert np.array_equal(b.episode_reason.cpu().numpy(), reason)  # the same bits without auto-reset
    term = (causes & (nat.END_GOAL | nat.END_COLLIDED)) != 0
    assert np.array_equal(a.terminated.cpu().numpy(), term)
    assert np.array_equal(a.truncated.cpu().numpy(), ((causes & nat.END_TIMEOUT) != 0) & ~term)
    fo = a.final_observation()
    assert np.array_equal(fo.ended.cpu().numpy(), now)
    count = int(fo.count)
    assert count == int(now.sum())
    slot = fo.slot.cpu().numpy()
    assert (slot[~now] == -1).all()
    cap = a.episode_end_capacity
    assert sorted(slot[now][slot[now] >= 0].tolist()) == list(range(min(count, cap)))
    idx = np.flatnonzero(now)
    if len(idx):
        _check_finals(fo, b, idx)
        _check_finals(b.final_observation(), b, idx)              # without auto-reset the finals are the step's outputs
        if count <= cap:
            assert torch.equal(a.final_ego(idx), b.ego_image[torch.from_numpy(idx).cuda()])
    return now


def _reset_and_compare(a, b, now):
    """b.reset(b.done) must leave b where a's in-kernel reset left a: rows, crops and goal vectors"""
    img_b, goal_b = b.ego_image.clone(), b.goal_n_state.clone()
    b.reset(b.done)
    sa, sb = a.get_state(), b.get_state()
    assert np.array_equal(_bits(sa.f), _bits(sb.f)) and torch.equal(sa.i, sb.i)
    b.observe_ego()
    keep = torch.from_numpy(~now).cuda()
    done = torch.from_numpy(now).cuda()
    assert torch.equal(a.ego_image[keep], img_b[keep]) and torch.equal(a.ego_image[done], b.ego_image[done])
    assert np.array_equal(_bits(a.goal_n_state[keep]), _bits(goal_b[keep]))
    assert np.array_equal(_bits(a.goal_n_state[done]), _bits(b.goal_n_state[done]))


def _run_twins(a, b, acts, on_step=None):
    timeouts = _timeouts(b)
    seen, ends = 0, 0
    for t in range(acts.shape[0]):
        a.step(acts[t])
        b.step(acts[t])
        now = _check_step(a, b, timeouts)
        seen |= int(np.bitwise_or.reduce(a.episode_reason.cpu().numpy().astype(np.int64)))
        ends += int(now.sum())
        if on_step is not None:
            on_step(a, b, t)
        _reset_and_compare(a, b, now)
    assert a.episode_stats()[0].item() == ends == b.episode_stats()[0].item()
    a.check_status()
    b.check_status()
    return seen, ends


# ---- 1. twin-batch equivalence ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("provider", [None, CONTINUOUS_REWARD_PURE_PURSUIT])
def test_finals_equal_the_twin_without_auto_reset(provider):
    d = _goal_fixture()
    a, b = _twins(d, provider=provider)
    assert a._rows is not None                                    # the per-env parameter path (ROWS kernels)
    seen, ends = _run_twins(a, b, _actions(a, d, 300))
    assert seen & CAUSES == CAUSES and seen & nat.END_NOW, seen   # goal, collision and timeout all occurred
    assert ends > 50


# ---- 2. final crops through the sparse kernel's own gather and through the dense kernel -------------------------------
@pytest.mark.parametrize("case", ["handover", "sparse_only", "dense_kernel"])
def test_finals_of_dense_and_overflowing_windows(case):
    d = _goal_fixture()
    extra = {"handover": ("dense", "overflow"), "sparse_only": ("overflow",), "dense_kernel": ("overflow",)}[case]
    a, b = _twins(d, n=40, extra=extra, ego_sparse=(case != "dense_kernel"))
    if case == "handover":
        assert not a._batch.flags & nat.BATCH_SPARSE_EGO_ONLY
    elif case == "sparse_only":
        assert a._batch.flags & nat.BATCH_SPARSE_EGO_ONLY
    else:
        assert a._ego_list is None
    handed = []

    def on_step(a, b, t):
        handed.append(int(a._ends_count[1]))
    seen, ends = _run_twins(a, b, _actions(a, d, 160), on_step)
    assert ends > 20
    if case == "handover":
        assert max(handed) > 0                                    # finals went to the dense kernel


# ---- 3. device worlds ---------------------------------------------------------------------------------------------------
def test_device_worlds_twins():
    from bc_gym_planning_env_b200.vec_aisle_env import VecRandomAisleTurnEnv
    pool = [EnvParams(iteration_timeout=30), EnvParams(iteration_timeout=50, control_delay=1, pose_delay=0, state_delay=1)]
    kw = dict(params=pool, draw_new_turn_on_reset=True, seed=5, with_ego=True)
    a = VecRandomAisleTurnEnv(64, auto_reset=True, episode_ends=True, **kw)
    b = VecRandomAisleTurnEnv(64, auto_reset=False, episode_ends=True, **kw)
    timeouts = _timeouts(b)
    acts = _actions(a, {"actions": np.zeros((0, 0, 2), np.float32)}, 120, seed=3)
    ends = 0
    for t in range(acts.shape[0]):
        a.step(acts[t])
        b.step(acts[t])
        now = _check_step(a, b, timeouts)
        ends += int(now.sum())
        a.reset(a.done)                                           # a new turn for the finished envs of both
        b.reset(b.done)
        sa, sb = a.get_state(), b.get_state()
        assert np.array_equal(_bits(sa.f), _bits(sb.f)) and torch.equal(sa.i, sb.i)
        assert torch.equal(a.ego_image, b.ego_image) and np.array_equal(_bits(a.goal_n_state), _bits(b.goal_n_state))
    assert ends > 64 and a.episode_stats()[0].item() == ends
    assert np.array_equal(a.turn_params(), b.turn_params())


# ---- 4. off means off ---------------------------------------------------------------------------------------------------
def test_episode_ends_change_no_step_output():
    d = _goal_fixture()
    costmaps, paths = _worlds(d, ("overflow",))
    sets, noise = _pool(d)
    n = 42
    ids = np.arange(n) % len(costmaps)
    kw = dict(n_envs=n, map_ids=ids, path_ids=ids, params_ids=1 + np.arange(n) % 3, noise_parameters=noise, seed=9,
              with_ego=True, auto_reset=True, compact_ego=True)
    off = VecPlanEnv(costmaps, paths, sets, **kw)
    on = VecPlanEnv(costmaps, paths, sets, episode_ends=True, **kw)
    acts = _actions(off, d, 120)
    H, W = off.ego_image.shape[1:3]
    for t in range(acts.shape[0]):
        if t % 3 == 2:
            host = acts[t].cpu().pin_memory()
            ro = off.step_host(host, images='compact')
            rn = on.step_host(host, images='compact')
            for x, y in zip(ro[:3], rn[:3]):
                assert torch.equal(x, y)
            assert torch.equal(ro[3]['counts'], rn[3]['counts'])
            assert np.array_equal(VecPlanEnv.expand_compact(ro[3], H, W), VecPlanEnv.expand_compact(rn[3], H, W))
        else:
            off.step(acts[t])
            on.step(acts[t])
        assert np.array_equal(_bits(off.reward), _bits(on.reward)) and torch.equal(off.done, on.done)
        assert np.array_equal(_bits(off.obs_vec), _bits(on.obs_vec))
        assert np.array_equal(_bits(off.goal_n_state), _bits(on.goal_n_state))
        assert torch.equal(off.ego_image, on.ego_image)
        so, sn = off.get_state(), on.get_state()
        assert np.array_equal(_bits(so.f), _bits(sn.f)) and torch.equal(so.i, sn.i)
    assert torch.equal(off.episode_stats(), on.episode_stats())
    assert off.launches_per_step() == on.launches_per_step()


# ---- 5. capacity overflow -----------------------------------------------------------------------------------------------
def test_capacity_overflow():
    d = _goal_fixture()
    costmaps, paths = _worlds(d)
    ep = common.env_params(d["params"], iteration_timeout=12)
    n, cap, guard = 64, 4, 2
    ids = np.arange(n) % len(costmaps)
    kw = dict(n_envs=n, map_ids=ids, path_ids=ids, noise_parameters=None, seed=3, with_ego=True)
    a = VecPlanEnv(costmaps, paths, ep, auto_reset=True, episode_ends=True, episode_end_capacity=cap, **kw)
    b = VecPlanEnv(costmaps, paths, ep, auto_reset=False, episode_ends=True, **kw)
    H, W = a.ego_image.shape[1:3]
    # the final crops and records go to buffers with a guard region behind the capacity
    images = torch.full((cap + guard, H, W, 1), 0xA5, dtype=torch.uint8, device="cuda")
    records = torch.full((cap + guard, 128), 0x5A, dtype=torch.uint8, device="cuda")
    a._c_ends.final_ego_image, a._c_ends.final_ego_work = images.data_ptr(), records.data_ptr()
    low, high = a.action_bounds()
    acts = torch.from_numpy(np.tile(((low + high) / 4).astype(np.float32), (n, 1))).cuda()   # slow: no collisions
    timeouts = _timeouts(b)
    overflowed = False
    for t in range(30):
        a.step(acts)
        b.step(acts)
        causes = _causes_from_state(b, timeouts)
        reason = a.episode_reason.cpu().numpy().astype(np.int64)
        assert np.array_equal(reason & CAUSES, causes)
        now = (reason & nat.END_NOW) != 0
        fo = a.final_observation()
        count = int(fo.count)
        assert count == now.sum()
        slot = fo.slot.cpu().numpy()
        assert (slot >= 0).sum() == min(count, cap) and (slot[~now] == -1).all()
        assert sorted(slot[slot >= 0].tolist()) == list(range(min(count, cap)))
        idx = np.flatnonzero(now)
        if len(idx):
            _check_finals(fo, b, idx, images)
        assert (images[cap:] == 0xA5).all() and (records[cap:] == 0x5A).all()
        if count > cap:
            overflowed = True
            with pytest.raises(nat.BcgError, match="episode_end_capacity"):
                a.final_ego(idx)
        b.reset(b.done)
    assert overflowed


# ---- 6. graphs and rollouts ---------------------------------------------------------------------------------------------
def _ends_of(env):
    """the episode ends of the last step, with the final crops in env order (slots are handed out in no order)"""
    fo = env.final_observation()
    now = fo.ended.cpu().numpy()
    idx = np.flatnonzero(now)
    crops = env.final_ego(idx).cpu().numpy() if len(idx) else None
    return dict(reason=env.episode_reason.cpu().numpy(), count=int(fo.count), obs=_bits(fo.obs_vec)[now],
                goal=_bits(fo.goal_n_state)[now], ret=_bits(fo.episode_return)[now], length=fo.episode_length.cpu().numpy()[now],
                crops=crops)


def _same_ends(x, y):
    assert x.keys() == y.keys()
    for k in x:
        if x[k] is None or y[k] is None:
            assert x[k] is None and y[k] is None, k
        else:
            assert np.array_equal(x[k], y[k]), k


def test_step_graph_and_rollouts_leave_the_same_ends():
    d = _goal_fixture()
    costmaps, paths = _worlds(d)
    n = 48
    ids = np.arange(n) % len(costmaps)
    ep = common.env_params(d["params"], iteration_timeout=25)
    kw = dict(n_envs=n, map_ids=ids, path_ids=ids, noise_parameters=DEFAULT_NOISE, seed=4, with_ego=True, auto_reset=True,
              episode_ends=True)
    plain, graph = VecPlanEnv(costmaps, paths, ep, **kw), VecPlanEnv(costmaps, paths, ep, **kw)
    acts = _actions(plain, d, 80)
    for t in range(acts.shape[0]):
        plain.step(acts[t])
        graph.step_graph(acts[t])
        _same_ends(_ends_of(plain), _ends_of(graph))
    assert plain.episode_stats()[0].item() >= n
    # H steps from one rollout call / one graph launch leave the ends of their last step (the timeout falls on it)
    H = 25
    plan = _actions(plain, d, H, seed=12)
    envs = [VecPlanEnv(costmaps, paths, ep, **kw) for _ in range(3)]
    for h in range(H):
        envs[0].step(plan[h])
    envs[1].rollout(plan)
    envs[2].rollout_graph(plan)
    ref = _ends_of(envs[0])
    assert ref["count"] > 0
    for e in envs[1:]:
        _same_ends(ref, _ends_of(e))


# ---- 7. validation and the semantics without auto-reset ------------------------------------------------------------------
def test_validation():
    d = _goal_fixture()
    costmaps, paths = _worlds(d)
    for cap in (0, 7):
        with pytest.raises(ValueError, match="episode_end_capacity"):
            VecPlanEnv(costmaps, paths, n_envs=6, with_ego=True, episode_ends=True, episode_end_capacity=cap)
    for with_ego in (True, False):                      # 'tiles' is the only staging of the egocentric window
        for staging in ("tma", "spans"):
            with pytest.raises(ValueError, match="ego_staging"):
                VecPlanEnv(costmaps, paths, n_envs=6, with_ego=with_ego, episode_ends=True, ego_staging=staging)
    env = VecPlanEnv(costmaps, paths, n_envs=6)
    with pytest.raises(ValueError, match="episode_ends"):
        env.final_observation()


def test_reasons_stay_set_without_auto_reset():
    d = _goal_fixture()
    costmaps, paths = _worlds(d)
    ep = common.env_params(d["params"], iteration_timeout=10)
    env = VecPlanEnv(costmaps, paths, ep, noise_parameters=None, episode_ends=True)       # no egocentric observation
    acts = torch.zeros((6, 2), dtype=torch.float32, device="cuda")
    for t in range(14):
        env.step(acts)
        r = env.episode_reason.cpu().numpy()
        if t < 9:
            assert (r == 0).all()
        else:
            assert ((r & CAUSES) == nat.END_TIMEOUT).all() and env.truncated.all() and not env.terminated.any()
            assert ((r & nat.END_NOW) != 0).all() == (t == 9)
            assert int(env.final_observation().count) == (6 if t == 9 else 0)
    assert env.final_observation().ego_image is None
    assert env.episode_stats()[0].item() == 6
