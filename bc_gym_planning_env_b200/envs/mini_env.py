"""Mini "parallel parking" environments: one corner obstacle, start and goal poses a few metres apart.

Mirrors the reference's envs/mini_env.py API (RandomMiniEnvParams :30-46, MiniEnvParams :80-92,
prepare_map_and_path :364-389, MiniEnv :392-405, RandomMiniEnv :408-494).  The rejection sampler
(_sample_mini_env_params :323-361) consumes the RandomState in the reference's order; its two
collision checks per candidate run through the batched CUDA collision kernel (there is no CPU
collision path in this package), candidates being drawn speculatively in small batches.
"""
import copy

import attr
import numpy as np

from bc_gym_planning_env_b200.envs.base.env import PlanEnv
from bc_gym_planning_env_b200.envs.base.maps import Wall
from bc_gym_planning_env_b200.envs.base.params import EnvParams
from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D


class SpaceSeemsEmptyError(Exception):
    """Rejection sampling ran out of tries."""


def _wrap(z):
    return (np.array(z) + np.pi) % (2 * np.pi) - np.pi


@attr.s
class RandomMiniEnvParams(object):
    inner_h = attr.ib(default=3, type=float)
    inner_w = attr.ib(default=3, type=float)
    mid_margin = attr.ib(default=0.25, type=float)
    out_margin = attr.ib(default=1, type=float)
    min_obstacle_angle = attr.ib(default=np.pi / 8., type=float)
    max_obstacle_angle = attr.ib(default=np.pi, type=float)
    lim_euc_dist = attr.ib(default=1000, type=float)
    lim_ang_dist = attr.ib(default=np.pi, type=float)
    angular_pose_noise_scale = attr.ib(default=np.pi / 2.0, type=float)
    env_params = attr.ib(factory=EnvParams)


@attr.s
class OrientedPoint(object):
    x = attr.ib(type=float)
    y = attr.ib(type=float)
    theta = attr.ib(type=float, converter=_wrap)

    def as_np(self):
        return np.array([self.x, self.y, self.theta], dtype=float)


@attr.s
class Point(object):
    x = attr.ib(type=float)
    y = attr.ib(type=float)

    def as_np(self):
        return np.array([self.x, self.y], dtype=float)


@attr.s
class MiniEnvParams(object):
    h = attr.ib(type=float)
    w = attr.ib(type=float)
    start_pos = attr.ib(type=OrientedPoint)
    end_pos = attr.ib(type=OrientedPoint)
    obstacle_a = attr.ib(type=Point)
    obstacle_o = attr.ib(type=Point)
    obstacle_b = attr.ib(type=Point)
    env_params = attr.ib(factory=EnvParams)


def _polar_point(r, phi, tx, ty):
    return Point(x=r * np.cos(phi) + tx, y=r * np.sin(phi) + ty)


def _outside_obstacle_wedge(pt, corner, start_angle, opening):
    """True when pt is not inside the wedge [start_angle, start_angle + opening] seen from the corner
    (reference :215-225: the polar angle is tested as is and shifted by 2 pi)."""
    phi = float(_wrap(np.arctan2(pt.y - corner.y, pt.x - corner.x)))
    for shifted in (phi, phi + 2 * np.pi):
        if start_angle <= shifted <= start_angle + opening:
            return False
    return True


def _sample_pose(rng, params, constraints):
    for _ in range(1000):
        pt = OrientedPoint(
            x=rng.uniform(-params.inner_w / 2 - params.mid_margin, params.inner_w / 2 + params.mid_margin),
            y=rng.uniform(-params.inner_h / 2 - params.mid_margin, params.inner_h / 2 + params.mid_margin),
            theta=rng.uniform(0, 2 * np.pi))
        if all(c(pt) for c in constraints):
            return pt
    raise ValueError("Something went wrong, the sampling space looks empty.")


def _pick_on_circle(rng, params, outside):
    """Start and goal diametrically opposite on a circle, both heading from start to goal (:145-185)."""
    for _ in range(1000):
        r = min((params.inner_w + params.inner_h) / 4. + params.mid_margin, params.lim_euc_dist)
        phi = rng.uniform(0, 2 * np.pi)
        x, y = r * np.cos(phi), r * np.sin(phi)
        rng.uniform(0, 2 * np.pi)      # the reference draws a heading here and then overrides it
        heading = np.arctan2(-y - y, -x - x)
        start, end = OrientedPoint(x, y, heading), OrientedPoint(-x, -y, heading)
        if outside(start) and outside(end):
            return start, end
    raise SpaceSeemsEmptyError("Something went wrong, the sampling space looks empty.")


def _pick_in_square(rng, params, outside):
    """Start anywhere legal, goal anywhere legal within the distance limits, both heading start->goal (:188-240)."""
    start = _sample_pose(rng, params, [outside])

    def near_angle(pt):
        return np.mod(start.theta - pt.theta, 2 * np.pi) < params.lim_ang_dist

    def near_euclid(pt):
        return np.linalg.norm(np.array([start.x - pt.x, start.y - pt.y])) < params.lim_euc_dist

    end = _sample_pose(rng, params, [outside, near_angle, near_euclid])
    heading = np.arctan2(end.y - start.y, end.x - start.x)
    return OrientedPoint(start.x, start.y, heading), OrientedPoint(end.x, end.y, heading)


def sample_candidate(params, rng):
    """One draw of _sample_mini_env_params_no_final_check (:269-320), same RandomState consumption."""
    corner = Point(x=rng.uniform(-params.inner_w / 2, params.inner_w / 2),
                   y=rng.uniform(-params.inner_h / 2, params.inner_h / 2))
    start_angle = rng.uniform(0, 2 * np.pi)
    opening = rng.uniform(params.min_obstacle_angle, params.max_obstacle_angle)
    r = 3 * (params.inner_h + params.inner_w + params.mid_margin + params.out_margin)
    obstacle_a = _polar_point(r, start_angle, corner.x, corner.y)
    obstacle_b = _polar_point(r, start_angle + opening, corner.x, corner.y)
    h = params.inner_h + 2 * params.mid_margin + 2 * params.out_margin
    w = params.inner_w + 2 * params.mid_margin + 2 * params.out_margin

    def outside(pt):
        return _outside_obstacle_wedge(pt, corner, start_angle, opening)

    if rng.rand() < 0.7:
        start, end = _pick_on_circle(rng, params, outside)
    else:
        start, end = _pick_in_square(rng, params, outside)
    noise = rng.uniform(-params.angular_pose_noise_scale / 2.0, params.angular_pose_noise_scale / 2.0)
    start = OrientedPoint(start.x, start.y, start.theta + noise)
    noise = rng.uniform(-params.angular_pose_noise_scale / 2.0, params.angular_pose_noise_scale / 2.0)
    end = OrientedPoint(end.x, end.y, end.theta + noise)
    return MiniEnvParams(h, w, start, end, obstacle_a, corner, obstacle_b, params.env_params)


def prepare_map_and_path(params):
    """(costmap, coarse 2-point path) of a MiniEnvParams (:364-389)."""
    costmap = CostMap2D.create_empty(world_size=(params.h, params.w), resolution=params.env_params.resolution,
                                     world_origin=(-params.h / 2., -params.w / 2.))
    for far in (params.obstacle_a, params.obstacle_b):
        Wall(from_pt=params.obstacle_o.as_np(), to_pt=far.as_np()).render(costmap)
    return costmap, np.array([params.start_pos.as_np(), params.end_pos.as_np()])


def _poses_collide(costmaps, poses, env_params):
    """pose_collides (reference envs/base/env.py:464-489) of pose k on costmap k, on the GPU."""
    from bc_gym_planning_env_b200.vec_env import VecPlanEnv
    # a far-apart dummy path keeps the initial-state kernel happy; only the collision kernel is used
    dummy = [np.array([[0., 0., 0.], [100., 0., 0.]]) for _ in costmaps]
    checker = VecPlanEnv(costmaps, dummy, attr.evolve(env_params, refine_path=False), noise_parameters=None)
    return checker.pose_collides(np.asarray(poses, dtype=np.float64)).cpu().numpy()


def sample_mini_env_params(gen_params, rng, batch=8):
    """_sample_mini_env_params (:323-361): first candidate whose start and goal poses are collision free
    and not already within the goal tolerances.  Candidates are drawn `batch` at a time (collision
    verdicts do not feed back into the draws), both poses of each are checked in one kernel call, and
    the RandomState is rewound to just after the accepted candidate -- exactly where the reference's
    sequential loop would have left it."""
    ep = gen_params.env_params
    tries = 0
    while tries < 1000:
        cands, states = [], []
        while len(cands) < batch and tries < 1000:
            tries += 1
            try:
                cand = sample_candidate(gen_params, rng)
            except SpaceSeemsEmptyError:
                continue
            cands.append(cand)
            states.append(copy.deepcopy(rng.get_state()))
        if not cands:
            break
        built = [prepare_map_and_path(c) for c in cands]
        costmaps = [cm for cm, _ in built for _ in range(2)]
        poses = [path[k] for _, path in built for k in range(2)]
        hits = _poses_collide(costmaps, poses, ep).reshape(-1, 2)
        for k, (cand, (_, path)) in enumerate(zip(cands, built)):
            d = float(np.hypot(path[0, 0] - path[1, 0], path[0, 1] - path[1, 1]))
            a = float(np.abs(_wrap(path[0, 2] - path[1, 2])))
            too_close = d < ep.goal_spat_dist and a < ep.goal_ang_dist
            if not hits[k].any() and not too_close:
                rng.set_state(states[k])
                return cand
    raise ValueError("Something went wrong, the sampling space looks empty.")


def random_mini_pool(n, seed, gen_params=None, max_rounds=1000):
    """n mini envs for a batch: ([CostMap2D], [coarse path]) where entry i is what RandomMiniEnv(seed=seed + i)
    draws first.  All pending candidates of a round are collision-checked in one kernel call."""
    if gen_params is None:
        gen_params = RandomMiniEnvParams(env_params=EnvParams(goal_ang_dist=np.pi / 8., goal_spat_dist=0.2))
    ep = gen_params.env_params
    rngs = [np.random.RandomState(seed + i) for i in range(n)]
    result = [None] * n
    pending = list(range(n))
    for _ in range(max_rounds):
        if not pending:
            break
        built = []
        for i in pending:
            try:
                built.append((i, prepare_map_and_path(sample_candidate(gen_params, rngs[i]))))
            except SpaceSeemsEmptyError:
                pass
        if built:
            costmaps = [cm for _, (cm, _) in built for _ in range(2)]
            poses = [path[k] for _, (_, path) in built for k in range(2)]
            hits = _poses_collide(costmaps, poses, ep).reshape(-1, 2)
            for (i, (cm, path)), hit in zip(built, hits):
                d = float(np.hypot(path[0, 0] - path[1, 0], path[0, 1] - path[1, 1]))
                a = float(np.abs(_wrap(path[0, 2] - path[1, 2])))
                if not hit.any() and not (d < ep.goal_spat_dist and a < ep.goal_ang_dist):
                    result[i] = (cm, path)
        pending = [i for i in pending if result[i] is None]
    if pending:
        raise ValueError("Something went wrong, the sampling space looks empty.")
    return [r[0] for r in result], [r[1] for r in result]


class MiniEnv(PlanEnv):
    def __init__(self, config, **kw):
        self._config = config
        costmap, path = prepare_map_and_path(config)
        super(MiniEnv, self).__init__(costmap, path, config.env_params, **kw)


class RandomMiniEnv(object):
    """MiniEnv with the geometry drawn at random on construction and (by default) on every reset."""

    def __init__(self, params=None, draw_new_turn_on_reset=True, seed=None, rng=None, **kw):
        self._params = params if params is not None else RandomMiniEnvParams(
            env_params=EnvParams(goal_ang_dist=np.pi / 8., goal_spat_dist=0.2))
        self._rng = np.random.RandomState(seed=0) if rng is None else rng
        self.seed(seed)
        self._draw_new_turn_on_reset = draw_new_turn_on_reset
        self._kw = kw
        self._env = MiniEnv(sample_mini_env_params(self._params, self._rng), **kw)
        self.action_space = self._env.action_space

    def seed(self, seed=None):
        if seed is not None:
            self._rng.seed(seed)

    def step(self, action):
        return self._env.step(action)

    def reset(self):
        if self._draw_new_turn_on_reset:
            self._env = MiniEnv(sample_mini_env_params(self._params, self._rng), **self._kw)
        return self._env.reset()

    def render(self, mode='human'):
        return self._env.render(mode)

    def close(self):
        self._env.close()
