"""The step at the batch sizes that select each kernel instantiation, against the CPU oracle (-m gpu; the rule table
test runs without a device).

bcg_step (bc_gym_planning_env_b200/csrc/bcg_kernels.cu: bcg_step, launch_ego_sparse) picks its kernels by the batch size
n on a device with S SMs:

  move_kernel<MIN_BLOCKS, ROWS, ENDS>  64 threads per block.  Tier 0 (4 blocks per SM, 230 registers) while the blocks
                                       fit 4 S, tier 1 (6 per SM, 168 registers) while they fit 6 S, tier 2 (8 per SM,
                                       128 registers, with spills) above.
  reward_kernel<G, ROWS, ENDS>         lane group G = 32 for n <= 2048, 16 for n <= 16384, 8 above.
  ego_sparse_kernel<HITS, ENDS>        persistent CTAs, grid = min(n, 18 S).  CTA c renders c + k grid for k <= RD = 3,
                                       then items drawn from the global counter ego_list[n + 1]: every env >= 4 grid, and
                                       with episode ends the final crops (items n + s) beyond the first four rounds.

  size (S = 148)      move tier   reward G   egocentric CTAs
  1 000               0           32         one env each
  6 007               0           16         ring, no counter draws
  16 001              0           16         counter draws
  30 000              0           8          counter draws
  320 S + 13 = 47 373 1           8          counter draws
  65 536              2           8          counter draws (the benchmark's size)

Four configurations cover the (ROWS, ENDS) builds and both reward providers with and without episode ends; each runs
the six sizes in lockstep on the same actions.  About 48 sampled envs per batch are stepped beside an OraclePlanEnv of
their own (pose and robot state to 1e-9, flags exact, crops bit-exact); the first 1 000 envs, which have the same ids,
seed and actions at every size, must be bit-identical across the sizes.  A batch of device-generated worlds above
4 grid closes the module.
"""
import functools
import os
import re

import numpy as np
import pytest
import torch

from bc_gym_planning_env_b200 import _native as nat
from oracle import plan_env_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
KERNELS_CU = os.path.join(HERE, os.pardir, "bc_gym_planning_env_b200", "csrc", "bcg_kernels.cu")

# ---- the selection rules of bcg_step and launch_ego_sparse, restated -------------------------------------------------
MOVE_THREADS = 64
MOVE_BLOCKS_PER_SM = (4, 6, 8)         # BCG_MOVE_FEWER_BLOCKS, BCG_MOVE_FEW_BLOCKS, BCG_MOVE_MIN_BLOCKS: tiers 0, 1, 2
REWARD_GROUPS = ((16384, 8), (2048, 16), (-1, 32))       # (n above, G), first match
EGS_CTAS = 18                          # ego_sparse_kernel CTAs per SM (BCG_EGS_CTAS) for the 117 x 133 crop
EGS_RD = 3                             # its record prefetch distance: the first RD + 1 envs of a CTA are fixed
HEAD = 1000                            # envs that are the same at every size
ONE, RING, COUNTER = "one env per CTA", "ring, no counter draws", "counter draws"
# (move tier, reward G, egocentric regime) of each size of batch_sizes, in order
EXPECTED = ((0, 32, ONE), (0, 16, RING), (0, 16, COUNTER), (0, 8, COUNTER), (1, 8, COUNTER), (2, 8, COUNTER))


def move_tier(n, sms):
    blocks = -(-n // MOVE_THREADS)
    return 0 if blocks <= sms * MOVE_BLOCKS_PER_SM[0] else 1 if blocks <= sms * MOVE_BLOCKS_PER_SM[1] else 2


def reward_group(n):
    return next(g for above, g in REWARD_GROUPS if n > above)


def ego_grid(n, sms):
    return min(n, EGS_CTAS * sms)


def ego_regime(n, sms):
    grid = ego_grid(n, sms)
    return ONE if n <= grid else RING if n <= (EGS_RD + 1) * grid else COUNTER


def regime(n, sms):
    return move_tier(n, sms), reward_group(n), ego_regime(n, sms)


def batch_sizes(sms):
    """the six sizes of the table; the tier-1 size (a midpoint of that tier, not a multiple of 32) follows the SM count"""
    return (HEAD, 6007, 16001, 30000, 320 * sms + 13, 65536)


def _kernel_source():
    with open(KERNELS_CU) as f:
        return f.read()


def _define(src, name):
    m = re.search(r"#define\s+%s\s+(\d+)" % name, src)
    assert m, name
    return int(m.group(1))


def test_rule_table_matches_the_kernel_source():
    """The constants and selection expressions restated above are the ones bcg_kernels.cu launches with, and the sizes
    of the table land in the regimes it names on a 148-SM B200: a retune cannot quietly move a regime out of coverage."""
    src = _kernel_source()
    flat = " ".join(src.split())
    assert _define(src, "BCG_MOVE_THREADS") == MOVE_THREADS
    assert tuple(_define(src, k) for k in ("BCG_MOVE_FEWER_BLOCKS", "BCG_MOVE_FEW_BLOCKS", "BCG_MOVE_MIN_BLOCKS")) == MOVE_BLOCKS_PER_SM
    assert ("const int tier = move_blocks <= sms * BCG_MOVE_FEWER_BLOCKS ? 0 : move_blocks <= sms * BCG_MOVE_FEW_BLOCKS ? 1 : 2;"
            in flat)
    assert "const int move_blocks = (int)blocks_for(b->n_envs, BCG_MOVE_THREADS);" in flat
    moves = re.search(r"static const MoveKernel moves\[3\]\[2\]\[2\] = \{(.*?)\};", flat).group(1)
    assert re.findall(r"move_kernel<(\w+),", moves) == ["BCG_MOVE_FEWER_BLOCKS"] * 4 + ["BCG_MOVE_FEW_BLOCKS"] * 4 + ["BCG_MOVE_MIN_BLOCKS"] * 4
    m = re.search(r"const int group = ns > (\d+) \? 0 : ns > (\d+) \? 1 : 2;", flat)
    assert m and (int(m.group(1)), int(m.group(2))) == (REWARD_GROUPS[0][0], REWARD_GROUPS[1][0])
    rewards = re.search(r"static const RewardKernel rewards\[3\]\[2\]\[2\] = \{(.*?)\};", flat).group(1)
    assert [int(g) for g in re.findall(r"reward_kernel<(\d+),", rewards)] == [8] * 4 + [16] * 4 + [32] * 4
    assert _define(src, "BCG_EGS_CTAS") == EGS_CTAS
    assert "const int grid = b->n_envs < per_sm * sms ? b->n_envs : per_sm * sms;" in flat
    body = flat[flat.index("ego_sparse_kernel(const BcgParams p"):]
    body = body[:body.index("ego_prep_kernel")]
    assert int(re.search(r"constexpr int RD = (\d+);", body).group(1)) == EGS_RD
    assert "if (tid <= RD) ids_s[tid] = e0 + tid * G;" in body
    assert "drawn = (RD + 1) * G + atomicAdd(b.ego_list + n + 1, 1);" in body
    # the sizes of the table on a 148-SM B200
    sizes = batch_sizes(148)
    assert sizes[4] == 47373 and sizes[4] % 32 and sizes[0] % 32 and sizes[0] % reward_group(sizes[0])
    assert sizes[4] % reward_group(sizes[4])
    assert tuple(regime(n, 148) for n in sizes) == EXPECTED
    assert ego_grid(65536, 148) == 2664
    # the launch asks the occupancy calculator for its CTAs per SM (EGS_CTAS is its upper bound, the launch bound): every
    # size keeps its egocentric regime for any occupancy from 12 to 18 CTAs per SM
    for per_sm in range(12, EGS_CTAS + 1):
        grid = [min(n, per_sm * 148) for n in sizes]
        assert [ONE if n <= g else RING if n <= (EGS_RD + 1) * g else COUNTER for n, g in zip(sizes, grid)] == \
            [r[2] for r in EXPECTED], per_sm


# ---- worlds, parameters, actions (host only) ----------------------------------------------------------------------------
POOL = 24
# paths cut to their first metres (goals within the 150 steps); every sixth map keeps its whole path (about 10 m, 200+
# refined points): reward_kernel's chunk scans then cover many 32-point chunks at every lane group
LENGTHS = (1.25, 1.5, 1.9, 2.4, 1.5, None)
DENSE_BASE = 5                         # the map the filled variant is made from
STEPS = 150
SEED = 17


@functools.lru_cache(maxsize=None)
def worlds():
    """(costmaps, coarse paths, the filled map): a random aisle pool whose paths are cut to the first LENGTHS metres of
    their main corridor (None: the whole path), and a copy of one map with its central region filled with non-lethal costs (more than 1 cell
    in 20 occupied: no cell index, every env on it is handed to the dense kernel)"""
    from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
    from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
    costmaps, coarse = random_aisle_pool(POOL, 900)
    paths = []
    for k, p in enumerate(coarse):
        p = np.asarray(p, dtype=np.float64)
        if LENGTHS[k % len(LENGTHS)] is None:
            paths.append(p)
            continue
        length = min(LENGTHS[k % len(LENGTHS)], float(np.hypot(*(p[1, :2] - p[0, :2]))))
        th = p[0, 2]
        paths.append(np.array([p[0], [p[0, 0] + length * np.cos(th), p[0, 1] + length * np.sin(th), th]]))
    base = costmaps[DENSE_BASE]
    data = base.get_data().copy()
    h, w = data.shape
    data[h // 4:3 * h // 4, w // 4:3 * w // 4] = np.random.RandomState(5).choice([253, 255, 100, 1], size=(3 * h // 4 - h // 4, 3 * w // 4 - w // 4))
    dense = CostMap2D(data, base.get_resolution(), np.array(base.get_origin(), dtype=np.float64))
    assert np.count_nonzero(data) * 20 > data.size
    return costmaps, paths, dense


def env_ids(n, with_dense):
    """map, path and parameter-set ids of envs 0..n-1: functions of the env id alone (the head is the same at every
    size).  With `with_dense` some envs past the head drive on the filled map (pool entry POOL)."""
    e = np.arange(n)
    maps = e % POOL
    paths = maps.copy()
    if with_dense:
        on = (e >= HEAD) & (e % 53 == 11)
        maps = np.where(on, POOL, maps)
        paths = np.where(on, DENSE_BASE, paths)
    sets = np.random.RandomState(4).randint(0, 4, 65536)[:n]
    return maps, paths, sets


def noise_sets():
    from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE
    return [None, DEFAULT_NOISE, {k: 4 * v for k, v in DEFAULT_NOISE.items()},
            dict(alpha1=2e-3, alpha2=1e-3, alpha3=5e-3, alpha4=0.0, alpha5=2e-3, alpha6=4e-3)]


def param_pool(provider):
    """four sets: no delays and a short timeout; the ring maxima (3, 2, 2); others in between.  Goal tolerances,
    progress multipliers, timeouts and noise differ"""
    from bc_gym_planning_env_b200.envs.base.params import EnvParams, RewardParams
    kw = dict(reward_provider_name=provider)
    return [EnvParams(control_delay=0, pose_delay=0, state_delay=0, iteration_timeout=45, **kw),
            EnvParams(control_delay=3, pose_delay=2, state_delay=2, iteration_timeout=130, **kw,
                      reward_provider_params=RewardParams(spatial_precision=0.6, angular_precision=np.pi / 3,
                                                          spatial_progress_multiplier=0.5)),
            EnvParams(control_delay=1, pose_delay=0, state_delay=2, iteration_timeout=30, **kw,
                      reward_provider_params=RewardParams(spatial_precision=0.9, angular_precision=np.pi / 2,
                                                          spatial_progress_multiplier=1.0)),
            EnvParams(control_delay=2, pose_delay=1, state_delay=0, iteration_timeout=90, **kw,
                      reward_provider_params=RewardParams(spatial_precision=0.8, angular_precision=np.pi / 4,
                                                          spatial_progress_multiplier=0.25))]


CONTINUOUS, PURSUIT = "continuous_reward", "continuous_reward_pure_pursuit"
# name: (reward provider, per-env pool, episode ends, compact lists, auto-reset)
CONFIGS = {"c0": (CONTINUOUS, False, False, False, False),
           "c1": (PURSUIT, True, False, True, True),
           "c2": (PURSUIT, False, True, False, True),
           "c3": (CONTINUOUS, True, True, True, True)}


def batch_params(config):
    """(params, noise) of a configuration: the pool, or one batch-wide set with delays, noise and a timeout"""
    from bc_gym_planning_env_b200.envs.base.params import EnvParams
    from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE
    provider, pool = CONFIGS[config][:2]
    if pool:
        return param_pool(provider), noise_sets()
    timeout = 80 if provider == CONTINUOUS else 45            # (pure pursuit is done 1 m before the end of the path)
    return EnvParams(control_delay=2, pose_delay=1, state_delay=1, iteration_timeout=timeout, reward_provider_name=provider), DEFAULT_NOISE


def action_stream(steps=STEPS, n=65536, seed=SEED):
    """float32 [n, 2] per step, forward-biased: speed in the upper fifth of its range; the wheel angle of an env follows
    one of four styles (straight, wavering, hard left, hard right) so that goals, collisions and timeouts all occur"""
    lo_v, hi_v = 0.1 * np.pi / 3, 0.5 * np.pi / 3                          # action_bounds of the tricycle
    style = np.random.RandomState(3).randint(0, 4, n)
    sigma = np.array([0.15, 0.6, 0.3, 0.3])[style]
    bias = np.array([0.0, 0.0, 0.9, -0.9])[style]
    rng = np.random.RandomState(seed)
    for _ in range(steps):
        v = rng.uniform(0.8, 1.0, n) * hi_v
        phi = np.clip(bias + sigma * rng.standard_normal(n), -np.pi / 2, np.pi / 2)
        a = np.stack([np.maximum(v, lo_v), phi], axis=1).astype(np.float32)
        yield a


def make_oracle(params, noise, costmap, path, env_id, clock, seed=SEED, refine=None):
    """env `env_id`'s oracle (`path` coarse, refined here unless refine=False); its noise is keyed by the batch's step
    index clock[0]: the oracle's own `iter` restarts at an auto-reset, the device's step index does not"""
    rp = params.reward_provider_params
    alphas = None if noise is None else tuple(float(noise["alpha%d" % (k + 1)]) for k in range(6))
    src = None if noise is None else (lambda it: O.philox_normal_source(seed, env_id, clock[0]))
    return O.OraclePlanEnv(costmap.get_data(), costmap.get_origin(), costmap.get_resolution(), path,
                           dt=params.dt, sp=rp.spatial_precision, ap=rp.angular_precision,
                           multiplier=rp.spatial_progress_multiplier, timeout=params.iteration_timeout,
                           delays=(params.control_delay, params.pose_delay, params.state_delay), alphas=alphas,
                           normal_source=src, refine=params.refine_path if refine is None else refine, path_delta=params.path_delta,
                           reward_provider=params.reward_provider_name)


def oracle_causes(o):
    """the END_* bits of a done oracle: goal, sticky collision, timeout"""
    goal = O.pure_pursuit_done(o.pose, o.path) if o.pure_pursuit else o.target_idx > len(o.path) - 1
    return (nat.END_GOAL if goal else 0) | (nat.END_COLLIDED if o.collided else 0) | (nat.END_TIMEOUT if o.iter >= o.timeout else 0)


def sample_envs(n, sms, dense_envs, k=48, seed=0):
    """~k envs of an n-env batch: the ends, the last warp, both sides of the reward-group, warp, block and egocentric
    grid boundaries, envs rendered from counter draws, envs >= 32 768, envs on the filled map, and a seeded random rest"""
    grid = ego_grid(n, sms)
    g = reward_group(n)
    last_warp = (n - 1) // 32 * 32
    want = {0, n - 1, last_warp, min(last_warp + 31, n - 1), g - 1, g, 31, 32, 63, 64}
    mid = n // 2 // 64 * 64
    want |= {mid - 1, mid}
    rng = np.random.RandomState(seed + n)
    if n > grid:
        want |= {grid - 1, grid}
    if n > 4 * grid:
        want |= {4 * grid - 1, 4 * grid}
        want |= set(rng.randint(4 * grid, n, 4).tolist())
    if n > 32768:
        want |= set(rng.randint(32768, n, 4).tolist())
    if len(dense_envs):
        want |= set(rng.choice(dense_envs, min(4, len(dense_envs)), replace=False).tolist())
    want = {e for e in want if 0 <= e < n}
    while len(want) < k:
        want.add(int(rng.randint(0, n)))
    return np.array(sorted(want), dtype=np.int64)


# ---- per-env comparison -------------------------------------------------------------------------------------------------
def _near(got, want, atol, what):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert np.all(np.abs(got - want) <= atol), (what, got, want)


def _fp32_near(got, want, what):
    """fp32 outputs of fp64 values that agree to 1e-9: equal up to one fp32 spacing"""
    want32 = np.asarray(want, dtype=np.float64).astype(np.float32)
    got = np.asarray(got, dtype=np.float32)
    assert np.all(np.abs(got.astype(np.float64) - want32) <= np.spacing(np.abs(want32)).astype(np.float64) + 1e-12), (what, got, want32)


def _obs_of(o):
    """obs_vec of an oracle: delayed pose, delayed robot state, time, target index"""
    return np.r_[o.pose, o.delayed_robot_state, o.time, o.target_idx]


def _goal_of(o):
    return O.goal_n_state(o.observation()["path"], o.pose, o.delayed_robot_state, o.resolution)


def _crop_of(o):
    return O.ego_costmap(o.costmap, o.pose, o.origin, o.resolution)


def check_env(o, f, i, obs, goal, img, what):
    """device column (fp64 rows f, int rows i; obs_vec, goal_n_state, crop: each may be None) against oracle o"""
    _near(f[nat.F_DPOSE:nat.F_DPOSE + 3], o.pose, 1e-9, ("pose",) + what)
    _near(f[nat.F_ROBOT:nat.F_ROBOT + 7], o.robot_state, 1e-9, ("robot state",) + what)
    _near(f[nat.F_DROBOT:nat.F_DROBOT + 7], o.delayed_robot_state, 1e-9, ("delayed robot state",) + what)
    _near(f[nat.F_TIME], o.time, 1e-9, ("time",) + what)
    _near(f[nat.F_MIN_DIST], o.min_dist, 1e-9, ("min_dist",) + what)
    assert (i[nat.I_ITER], i[nat.I_TARGET], bool(i[nat.I_COLLIDED])) == (o.iter, o.target_idx, o.collided), what
    if obs is not None:
        rows = np.r_[f[nat.F_DPOSE:nat.F_DPOSE + 3], f[nat.F_DROBOT:nat.F_DROBOT + 7], f[nat.F_TIME], i[nat.I_TARGET]]
        assert np.array_equal(obs, rows.astype(np.float32)), ("obs_vec of the rows",) + what
        _fp32_near(obs, _obs_of(o), ("obs_vec",) + what)
    if goal is not None:
        _fp32_near(goal, _goal_of(o), ("goal_n_state",) + what)
    if img is not None:
        want = _crop_of(o)
        assert np.array_equal(img, want), ("crop",) + what
        return want
    return None


class _Run(object):
    """One batch stepped beside the oracles of its sampled envs, with the per-step checks and what they covered."""

    def __init__(self, env, sample, oracle_of, sms, compact=False):
        self.env, self.sample, self.oracle_of = env, np.asarray(sample), oracle_of
        self.n = env.n_envs
        self.grid = ego_grid(self.n, sms)
        self.ends, self.auto, self.compact = env.episode_ends, env.auto_reset, compact
        self.clock = [0]
        self.oracles = [oracle_of(int(e), self.clock) for e in self.sample]
        self.ret = np.zeros(len(self.sample))
        self.idx = torch.from_numpy(self.sample).to(env.device)
        self.host = torch.empty((self.n, 2), dtype=torch.float32).pin_memory() if compact else None
        self.compact_out = None
        self.dense_map = np.zeros(self.n, dtype=bool)
        self.seen = dict(goal=0, collided=0, timeout=0, finals=0, dense=0, counter=0, counter_finals=0, batch_finals=0)

    def step(self, acts, acts_dev):
        if self.compact:
            self.host.copy_(torch.from_numpy(acts[:self.n]))
            self.compact_out = self.env.step_host(self.host, images="compact")[3]
        else:
            self.env.step(acts_dev[:self.n])

    def _gather(self):
        env, idx = self.env, self.idx
        g = dict(f=env.state_f[:nat.F_FIXED][:, idx], i=env.state_i[:nat.I_FIXED][:, idx], r=env.reward[idx], d=env.done[idx],
                 obs=env.obs_vec[idx], goal=env.goal_n_state[idx, :, 0], img=env.ego_image[idx, ..., 0])
        if self.ends:
            fo = env.final_observation()
            g.update(reason=env.episode_reason[idx], term=env.terminated[idx], trunc=env.truncated[idx],
                     fobs=fo.obs_vec[idx], fgoal=fo.goal_n_state[idx, :, 0], fret=fo.episode_return[idx],
                     flen=fo.episode_length[idx], fslot=fo.slot[idx])
        if self.compact:
            g.update(count=env._ego_hit_count[idx], hits=env._ego_hits[idx])
        return {k: v.cpu().numpy() for k, v in g.items()}

    def check(self, t, acts):
        """the sampled envs after step t (actions `acts`) against their oracles"""
        g = self._gather()
        self.clock[0] = t
        ended = []
        for k, e in enumerate(self.sample):
            o = self.oracles[k]
            what = (self.n, int(e), t)
            was_done = o.done()
            _, r2, d2, _ = o.step(acts[e])
            self.ret[k] += r2
            _near(g["r"][k], r2, 1e-9, ("reward",) + what)
            assert bool(g["d"][k]) == d2, ("done",) + what
            now = d2 and not was_done
            causes = oracle_causes(o) if d2 else 0
            if now:
                self.seen["goal"] += bool(causes & nat.END_GOAL)
                self.seen["collided"] += bool(causes & nat.END_COLLIDED)
                self.seen["timeout"] += bool(causes & nat.END_TIMEOUT)
            if self.ends:
                assert int(g["reason"][k]) == causes | (nat.END_NOW if now else 0), ("reason",) + what
                term = bool(causes & (nat.END_GOAL | nat.END_COLLIDED))
                assert (bool(g["term"][k]), bool(g["trunc"][k])) == (term, bool(causes & nat.END_TIMEOUT) and not term), what
                if now:                                   # the final observation: the oracle before its reset
                    _fp32_near(g["fobs"][k], _obs_of(o), ("final obs_vec",) + what)
                    assert g["fobs"][k][11] == o.target_idx, what
                    _fp32_near(g["fgoal"][k], _goal_of(o), ("final goal_n_state",) + what)
                    _near(g["fret"][k], self.ret[k], 1e-9, ("final return",) + what)
                    assert g["flen"][k] == o.iter and g["fslot"][k] >= 0, what
                    ended.append((k, _crop_of(o)))
                else:
                    assert g["fslot"][k] == -1, what
            if d2 and self.auto:
                o.reset()
                self.ret[k] = 0.0
            _near(g["f"][nat.F_EP_RETURN, k], self.ret[k], 1e-9, ("return",) + what)
            crop = check_env(o, g["f"][:, k], g["i"][:, k], g["obs"][k], g["goal"][k], g["img"][k], what)
            if self.compact:
                c = int(g["count"][k])
                flat = crop.reshape(-1)
                nz = np.flatnonzero(flat)
                if c != -1:                                # -1: rendered by the dense kernel, the consumer reads the image
                    assert c == len(nz), ("hit count",) + what
                    if c <= self.env.EGO_HIT_CAP:
                        words = g["hits"][k, :c].astype(np.int64)
                        assert np.array_equal(np.sort(words), np.sort(nz | (flat[nz].astype(np.int64) << 16))), ("hits",) + what
            self.seen["dense"] += bool(self.dense_map[e])
            self.seen["counter"] += bool(e >= 4 * self.grid)
        if ended:
            ks = [k for k, _ in ended]
            got = self.env.final_ego(self.sample[ks]).cpu().numpy()[..., 0]
            for j, (k, want) in enumerate(ended):
                assert np.array_equal(got[j], want), ("final crop", self.n, int(self.sample[k]), t)
            self.seen["finals"] += len(ended)
            if self.n >= 4 * self.grid:                    # items n + s: all of them drawn from the counter
                self.seen["counter_finals"] += len(ended)

    def check_batch(self, t):
        """whole-batch invariants of step t, without the oracle"""
        env = self.env
        if self.ends:
            fo = env.final_observation()
            count = int(fo.count)
            assert int(fo.ended.sum()) == count and int(((env.episode_reason & nat.END_NOW) != 0).sum()) == count, t
            assert int((fo.slot >= 0).sum()) == min(count, env.episode_end_capacity), t
            self.seen["batch_finals"] += count
        if env._ego_list is not None:
            # one counter stream hands out every item: the n envs, then the final crops kept (items n + s)
            items = self.n + (min(count, env.episode_end_capacity) if self.ends else 0)
            assert int(env._ego_list[self.n + 1]) == items, t
        if self.compact:
            _check_hit_lists(env)
            if t % 50 == 49:
                h, w = env.ego_image.shape[1:3]
                assert np.array_equal(type(env).expand_compact(self.compact_out, h, w), env.ego_image.cpu().numpy()[..., 0]), t

    def report(self):
        return "n=%d %s" % (self.n, " ".join("%s=%d" % kv for kv in sorted(self.seen.items())))


def _check_hit_lists(env):
    """every env's compact list holds each non-zero pixel of its crop once (count -1: rendered densely; a count above
    the capacity: the list overflowed, the consumer reads the image)"""
    cnt, hits, cap = env._ego_hit_count, env._ego_hits, env.EGO_HIT_CAP
    n, h, w = env.ego_image.shape[:3]
    img = env.ego_image.view(n, h * w)
    listed = cnt >= 0
    assert bool((listed | (cnt == -1)).all())
    assert torch.equal((img != 0).sum(1, dtype=torch.int32)[listed], cnt[listed])
    full = listed & (cnt <= cap)
    keep = torch.arange(cap, device=cnt.device)[None, :] < torch.where(full, cnt, 0)[:, None]
    words = hits[keep]
    rebuilt = torch.zeros_like(img)
    rebuilt[keep.nonzero()[:, 0], (words & 0xffff).long()] = ((words >> 16) & 0xff).to(torch.uint8)
    assert torch.equal(rebuilt[full], img[full])


def _sorted_lists(hits, cnt, cap):
    keep = torch.arange(cap, device=cnt.device)[None, :] < torch.where(cnt <= cap, cnt, 0)[:, None]
    return torch.sort(torch.where(keep, hits, torch.full_like(hits, 0x7fffffff)), dim=1)[0]


def _same_head(ref, run):
    """the first HEAD envs of `run` are bit-identical to those of `ref` (a HEAD-env batch)"""
    a, b, h = ref.env, run.env, HEAD
    assert torch.equal(a.state_f, b.state_f[:, :h]) and torch.equal(a.state_i, b.state_i[:, :h]), run.n
    for name in ("reward", "_done_u8", "obs_vec", "goal_n_state", "ego_image"):
        assert torch.equal(getattr(a, name), getattr(b, name)[:h]), (name, run.n)
    if ref.ends:
        assert torch.equal(a.episode_reason, b.episode_reason[:h]), run.n
        now = (a.episode_reason & nat.END_NOW) != 0
        for name in ("_final_obs_vec", "_final_goal_n_state", "_final_return", "_final_length"):
            assert torch.equal(getattr(a, name)[now], getattr(b, name)[:h][now]), (name, run.n)
        ids = now.nonzero()[:, 0]
        if ids.numel():                                   # (slots are handed out in no order: by env id)
            assert torch.equal(a.final_ego(ids), b.final_ego(ids)), run.n
    if ref.compact:
        ca, cb = a._ego_hit_count, b._ego_hit_count[:h]
        assert torch.equal(ca, cb), run.n
        cap = a.EGO_HIT_CAP
        assert torch.equal(_sorted_lists(a._ego_hits, ca, cap), _sorted_lists(b._ego_hits[:h], cb, cap)), run.n


def _matrix_run(config, n, sms, with_dense):
    from bc_gym_planning_env_b200.vec_env import VecPlanEnv
    provider, pool, ends, compact, auto = CONFIGS[config]
    costmaps, paths, dense = worlds()
    maps, pids, sets = env_ids(n, with_dense)
    params, noise = batch_params(config)
    env = VecPlanEnv(costmaps + [dense] if with_dense else costmaps, paths, params, n_envs=n, map_ids=maps, path_ids=pids,
                     noise_parameters=noise, seed=SEED, auto_reset=auto, with_ego=True, compact_ego=compact,
                     episode_ends=ends, params_ids=sets if pool else None)
    assert (env._rows is not None) == pool and bool(env._batch.flags & nat.BATCH_SPARSE_EGO_ONLY) != with_dense

    # (the oracles take their set, noise and world from the test's own lists, not from the batch's bookkeeping)
    def oracle_of(e, clock):
        k = sets[e] if pool else None
        return make_oracle(params[k] if pool else params, noise[k] if pool else noise,
                           dense if maps[e] == POOL else costmaps[maps[e]], paths[pids[e]], e, clock)
    run = _Run(env, sample_envs(n, sms, np.flatnonzero(maps == POOL)), oracle_of, sms, compact=compact)
    run.dense_map = maps == POOL
    return run


@pytest.mark.gpu
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_every_instantiation_matches_the_oracle(config):
    """c0: batch-wide parameters, continuous reward, noise, no auto-reset.  c1: the parameter pool, pure pursuit,
    compact lists, auto-reset.  c2: batch-wide parameters, episode ends, pure pursuit, auto-reset.  c3: the pool, episode
    ends, compact lists, continuous reward, auto-reset.  The six sizes step in lockstep."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sizes = batch_sizes(sms)
    assert tuple(regime(n, sms) for n in sizes) == EXPECTED, (sms, sizes)
    runs = [_matrix_run(config, n, sms, with_dense=n in (16001, 65536)) for n in sizes]
    for t, acts in enumerate(action_stream()):
        acts_dev = torch.from_numpy(acts).cuda()
        for run in runs:
            run.step(acts, acts_dev)
        for run in runs:
            run.check(t, acts)
            run.check_batch(t)
        for run in runs[1:]:
            _same_head(runs[0], run)
    for run, n in zip(runs, sizes):
        run.env.check_status()
        print("step matrix %s %s tier=%d G=%d ego=%s" % ((config, run.report()) + regime(n, sms)))
        s = run.seen
        assert s["goal"] and s["collided"] and s["timeout"], (config, run.report())
        if run.ends:
            assert s["finals"] and s["batch_finals"], (config, run.report())
        if n > 4 * run.grid:
            assert s["counter"] and (s["counter_finals"] or not run.ends), (config, run.report())
        if n in (16001, 65536):
            assert s["dense"], (config, run.report())


@pytest.mark.gpu
def test_device_worlds_above_the_counter_threshold():
    """12 000 device-generated worlds (no cell index: crops from the occupancy listing), pure pursuit, episode ends and
    auto-reset, and two reset(done) storms that give the finished envs new worlds: a sample against oracles built from
    each env's turn parameters by the host restatement of the generator.  The first worlds of the even envs have their
    corridors cut to 15 % (paths of 1.5 - 3 m: goals), those of the odd envs are drawn as they come (about 10 m:
    timeouts); the storms draw new ones on the device."""
    from bc_gym_planning_env_b200.envs.base.params import EnvParams
    from bc_gym_planning_env_b200.vec_aisle_env import VecRandomAisleTurnEnv
    from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE
    from oracle import aisle_oracle as A
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 12000
    assert ego_regime(n, sms) == COUNTER and move_tier(n, sms) == 0 and reward_group(n) == 16
    ep = EnvParams(control_delay=1, pose_delay=1, state_delay=1, iteration_timeout=60, reward_provider_name=PURSUIT)
    rng = np.random.RandomState(SEED)
    first = [A.draw_turn_params(rng) for _ in range(n)]
    for tp in first[::2]:
        tp["main_corridor_length"] *= 0.15
        tp["turn_corridor_length"] *= 0.15
    env = VecRandomAisleTurnEnv(n, ep, seed=SEED, turn_params=first, noise_parameters=DEFAULT_NOISE, with_ego=True,
                                auto_reset=True, episode_ends=True)

    def oracle_of(e, clock):
        r = env.turn_params()[e]
        tp = {f: (bool(r[f]) if f.startswith("flip") else float(r[f])) for f in A.TURN_FIELDS}
        coarse, costmap, origin = A.aisle_world(tp, ep.resolution)
        from bc_gym_planning_env_b200.utilities.costmap_2d import CostMap2D
        return make_oracle(ep, DEFAULT_NOISE, CostMap2D(costmap, ep.resolution, origin), coarse, e, clock)
    run = _Run(env, sample_envs(n, sms, []), oracle_of, sms)
    storms = 0
    for t, acts in enumerate(action_stream(n=n, seed=SEED + 1)):
        run.step(acts, torch.from_numpy(acts).cuda())
        run.check(t, acts)
        run.check_batch(t)
        if t in (60, 110):
            mask = env.done.clone()
            env.reset(mask)                                # new worlds for the envs that finished this step
            m = mask.cpu().numpy()
            storms += int(m.sum())
            for k, e in enumerate(run.sample):
                if m[e]:
                    run.oracles[k] = oracle_of(int(e), run.clock)
                    run.ret[k] = 0.0
            g = run._gather()
            for k, e in enumerate(run.sample):
                # (obs_vec is a step output: reset leaves it alone)
                check_env(run.oracles[k], g["f"][:, k], g["i"][:, k], None, g["goal"][k], g["img"][k], (n, int(e), t, "storm"))
    env.check_status()
    print("step matrix device worlds %s storms=%d" % (run.report(), storms))
    s = run.seen
    assert storms > 0 and s["counter"] and s["goal"] and s["collided"] and s["timeout"] and s["counter_finals"], run.report()


@pytest.mark.gpu
def test_pure_pursuit_goal_vector_points_at_the_first_path_point():
    """With pure pursuit Observation.path is path[:target + 1] (reward.py:120-124), and goal_n_state points at its first
    point (envs/egocentric.py:141-160), not at the way point at the target index.  All three writers of the vector --
    the step's, the final observation's and the auto-reset's -- and observe_ego, against the oracle for every env."""
    from bc_gym_planning_env_b200.envs.base.params import EnvParams
    from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE, VecPlanEnv
    costmaps, paths, _ = worlds()
    ep = EnvParams(control_delay=1, pose_delay=1, state_delay=0, iteration_timeout=40, reward_provider_name=PURSUIT)
    n = 48
    env = VecPlanEnv(costmaps, paths, ep, n_envs=n, noise_parameters=DEFAULT_NOISE, seed=SEED, auto_reset=True,
                     with_ego=True, episode_ends=True)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    run = _Run(env, np.arange(n), lambda e, clock: make_oracle(ep, DEFAULT_NOISE, costmaps[e % POOL], paths[e % POOL], e, clock), sms)
    moved = 0
    for t, acts in enumerate(action_stream(steps=60, n=n)):
        run.step(acts, torch.from_numpy(acts).cuda())
        run.check(t, acts)
        moved += sum(o.target_idx > 1 for o in run.oracles)       # the target index has left the first point behind
    assert moved > 0 and run.seen["finals"] and run.seen["goal"], run.report()
    _, goal = env.observe_ego()
    goal = goal[..., 0].cpu().numpy()
    for k, o in enumerate(run.oracles):
        _fp32_near(goal[k], _goal_of(o), ("observe_ego goal_n_state", k))
    env.check_status()
