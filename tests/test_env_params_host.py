"""CPU: per-env parameter rows (BcgEnvRows) are built and validated on the host."""
import numpy as np
import pytest

from bc_gym_planning_env_b200 import _native as nat
from bc_gym_planning_env_b200.env_params import build_env_rows, is_pool
from bc_gym_planning_env_b200.envs.base.params import CONTINUOUS_REWARD_PURE_PURSUIT, EnvParams, RewardParams
from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE

NOISE_B = dict(alpha1=0.1, alpha2=0.2, alpha3=0.3, alpha4=0.4, alpha5=0.5, alpha6=0.6)


def _pool():
    return [EnvParams(control_delay=2, pose_delay=1, state_delay=1),
            EnvParams(goal_spat_dist=0.2, goal_ang_dist=np.pi / 8, iteration_timeout=150),
            EnvParams(control_delay=3, pose_delay=0, state_delay=2,
                      reward_provider_params=RewardParams(spatial_precision=0.5, angular_precision=0.3,
                                                          spatial_progress_multiplier=0.5))]


def test_rows_hold_each_envs_values_and_capacities_are_maxima():
    pool = _pool()
    ids = np.array([2, 0, 1, 1, 0, 2, 0])
    rows = build_env_rows(pool, [DEFAULT_NOISE, None, NOISE_B], ids, len(ids))
    assert rows.f.shape == (nat.EP_F_ROWS, 7) and rows.f.dtype == np.float64
    assert rows.i.shape == (nat.EP_I_ROWS, 7) and rows.i.dtype == np.int32
    assert rows.capacities == (3, 1, 2)
    for e, k in enumerate(ids):
        p = pool[k]
        rp = p.reward_provider_params
        assert rows.f[nat.EP_F_SP, e] == rp.spatial_precision
        assert rows.f[nat.EP_F_AP, e] == rp.angular_precision
        assert rows.f[nat.EP_F_PM, e] == rp.spatial_progress_multiplier
        assert tuple(rows.i[nat.EP_I_DELAY_CONTROL:nat.EP_I_DELAY_STATE + 1, e]) == (p.control_delay, p.pose_delay, p.state_delay)
        assert tuple(rows.delays[e]) == (p.control_delay, p.pose_delay, p.state_delay)
        assert rows.i[nat.EP_I_TIMEOUT, e] == p.iteration_timeout
        noise = [DEFAULT_NOISE, None, NOISE_B][k]
        assert rows.i[nat.EP_I_NOISE_ON, e] == (0 if noise is None else 1)
        want = [0.0] * 6 if noise is None else [noise['alpha%d' % (j + 1)] for j in range(6)]
        assert list(rows.f[nat.EP_F_ALPHA:nat.EP_F_ALPHA + 6, e]) == want


def test_default_ids_and_shared_noise():
    pool = _pool()
    rows = build_env_rows(pool, DEFAULT_NOISE, None, 7)
    assert list(rows.i[nat.EP_I_TIMEOUT]) == [pool[e % 3].iteration_timeout for e in range(7)]
    assert list(rows.i[nat.EP_I_NOISE_ON]) == [1] * 7
    # capacities cover the whole pool, also sets no env uses yet (a reset may move envs there)
    assert build_env_rows(pool, None, np.zeros(4, dtype=np.int64), 4).capacities == (3, 1, 2)


def test_pool_selection():
    assert is_pool([EnvParams()]) and is_pool((EnvParams(),))
    assert not is_pool(EnvParams()) and not is_pool(None)


@pytest.mark.parametrize("field,value", [("dt", 0.1), ("robot_name", "standard_logistic_tricycle_v1"), ("resolution", 0.05),
                                         ("reward_provider_name", CONTINUOUS_REWARD_PURE_PURSUIT), ("refine_path", False),
                                         ("path_delta", 0.1)])
def test_batch_wide_fields_must_agree(field, value):
    import attr
    pool = [EnvParams(), attr.evolve(EnvParams(), **{field: value})]
    with pytest.raises(ValueError, match=field):
        build_env_rows(pool, None, None, 4)


@pytest.mark.parametrize("field,value", [("control_delay", -1), ("pose_delay", 4096), ("state_delay", -3),
                                         ("control_delay", 1.5), ("iteration_timeout", 0), ("iteration_timeout", -5)])
def test_delays_and_timeout_are_checked(field, value):
    with pytest.raises(ValueError, match=field):
        build_env_rows([EnvParams(), EnvParams(**{field: value})], None, None, 2)


def test_largest_delay_is_accepted():
    rows = build_env_rows([EnvParams(pose_delay=4095)], None, None, 1)
    assert rows.capacities == (0, 4095, 0)


@pytest.mark.parametrize("ids", [[0, 1, 2], [0, -1, 1, 0], [0, 1, 3, 0], [0.0, 1.0, 0.0, 1.0], [[0, 1, 0, 1]]])
def test_bad_ids(ids):
    with pytest.raises(ValueError, match="params_ids"):
        build_env_rows(_pool(), None, np.asarray(ids), 4)


def test_noise_list_length_and_alphas():
    with pytest.raises(ValueError, match="noise_parameters"):
        build_env_rows(_pool(), [None, DEFAULT_NOISE], None, 3)
    bad = dict(DEFAULT_NOISE, alpha4=-1e-3)
    with pytest.raises(ValueError, match="alphas"):
        build_env_rows(_pool(), [None, bad, None], None, 3)
    with pytest.raises(ValueError, match="alphas"):
        build_env_rows(_pool(), dict(DEFAULT_NOISE, alpha1=float('nan')), None, 3)


def test_empty_pool():
    with pytest.raises(ValueError, match="empty"):
        build_env_rows([], None, None, 1)
