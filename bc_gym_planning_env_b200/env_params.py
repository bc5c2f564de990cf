"""Per-env parameters of one batch: a pool of `EnvParams` (and noise settings) and the index of the set each env uses.

The reference gives every `PlanEnv` its own `EnvParams` and its own odometry noise (envs/base/env.py:218-232,
`set_noise_parameters`).  A batch here carries, per env, the fields the step reads that may differ between such envs --
delays, timeout, goal tolerances, progress multiplier, noise on/off and alphas -- as the rows of `BcgEnvRows`
(include/bcg_b200.h).  Everything else must agree across the pool.  This module builds and validates those rows on the
host; it needs no GPU.
"""
import numpy as np

from bc_gym_planning_env_b200 import _native as nat

# fields that stay batch-wide: a pool that disagrees on one of them is refused
BATCH_WIDE_FIELDS = ("dt", "robot_name", "resolution", "reward_provider_name", "refine_path", "path_delta")
MAX_DELAY = 4096          # exclusive bound of every delay (queue words hold 16-bit heads and lengths)


class EnvRows(object):
    """The per-env rows of a batch: `f` fp64 [EP_F_ROWS, n], `i` int32 [EP_I_ROWS, n], and the ring capacities
    (control, pose, state) = the per-field maxima of the delays over the pool."""

    def __init__(self, f, i, capacities):
        self.f, self.i, self.capacities = f, i, capacities

    @property
    def delays(self):
        """int32 [n, 3]: control, pose and state delay of every env"""
        return self.i[nat.EP_I_DELAY_CONTROL:nat.EP_I_DELAY_STATE + 1].T


def is_pool(params):
    """A list / tuple of EnvParams (even of length one) selects the per-env path; one EnvParams or None does not."""
    return isinstance(params, (list, tuple))


def normalize_noise(pool_len, noise_parameters):
    """One noise dict / None shared by every set, or a sequence of them with one entry per set -> list of pool_len"""
    if noise_parameters is None or isinstance(noise_parameters, dict):
        return [noise_parameters] * pool_len
    noise = list(noise_parameters)
    if len(noise) != pool_len:
        raise ValueError("noise_parameters must be one dict / None or a sequence of %d (one per parameter set), got %d"
                         % (pool_len, len(noise)))
    for nz in noise:
        if nz is not None and not isinstance(nz, dict):
            raise ValueError("every noise setting must be a dict alpha1..alpha6 or None")
    return noise


def check_pool(pool):
    """The fields that stay batch-wide agree across the pool; raises ValueError naming the first that does not."""
    pool = list(pool)
    if not pool:
        raise ValueError("the parameter pool is empty")
    ref = pool[0]
    for k, p in enumerate(pool[1:], start=1):
        for name in BATCH_WIDE_FIELDS:
            if getattr(p, name) != getattr(ref, name):
                raise ValueError("EnvParams.%s must be the same for the whole batch: set 0 has %r, set %d has %r"
                                 % (name, getattr(ref, name), k, getattr(p, name)))
    return pool


def build_env_rows(pool, noise_parameters, params_ids, n_envs):
    """Validate a pool and build the per-env rows.

    :param pool: sequence of EnvParams
    :param noise_parameters: one dict alpha1..alpha6 / None for every set, or a sequence with one per set
    :param params_ids: [n_envs] indices into the pool, or None for e % len(pool)
    :return: EnvRows
    """
    pool = check_pool(pool)
    noise = normalize_noise(len(pool), noise_parameters)
    n = int(n_envs)
    ids = (np.arange(n) % len(pool)) if params_ids is None else np.asarray(params_ids)
    if ids.shape != (n,) or not np.issubdtype(ids.dtype, np.integer):
        raise ValueError("params_ids must be %d integers" % n)
    ids = ids.astype(np.int64)
    if n and (ids.min() < 0 or ids.max() >= len(pool)):
        raise ValueError("params_ids must lie in [0, %d)" % len(pool))
    set_f = np.zeros((nat.EP_F_ROWS, len(pool)), dtype=np.float64)
    set_i = np.zeros((nat.EP_I_ROWS, len(pool)), dtype=np.int32)
    for k, (p, nz) in enumerate(zip(pool, noise)):
        delays = (p.control_delay, p.pose_delay, p.state_delay)
        for name, d in zip(("control_delay", "pose_delay", "state_delay"), delays):
            if int(d) != d or not 0 <= int(d) < MAX_DELAY:
                raise ValueError("EnvParams.%s of set %d must be an integer in [0, %d), got %r" % (name, k, MAX_DELAY, d))
        if int(p.iteration_timeout) != p.iteration_timeout or int(p.iteration_timeout) <= 0:
            raise ValueError("EnvParams.iteration_timeout of set %d must be a positive integer, got %r" % (k, p.iteration_timeout))
        rp = p.reward_provider_params
        set_f[nat.EP_F_SP, k] = rp.spatial_precision
        set_f[nat.EP_F_AP, k] = rp.angular_precision
        set_f[nat.EP_F_PM, k] = rp.spatial_progress_multiplier
        if nz is not None:
            alphas = [float(nz['alpha%d' % (j + 1)]) for j in range(6)]
            if not all(a >= 0.0 for a in alphas):          # (also refuses NaN)
                raise ValueError("noise alphas of set %d must be >= 0, got %r" % (k, alphas))
            set_f[nat.EP_F_ALPHA:nat.EP_F_ALPHA + 6, k] = alphas
        set_i[nat.EP_I_DELAY_CONTROL:nat.EP_I_DELAY_STATE + 1, k] = delays
        set_i[nat.EP_I_TIMEOUT, k] = p.iteration_timeout
        set_i[nat.EP_I_NOISE_ON, k] = 0 if nz is None else 1
    f = np.ascontiguousarray(set_f[:, ids])
    i = np.ascontiguousarray(set_i[:, ids])
    # over the whole pool, not only the sets in use: a reset may move an env to any set of the pool
    caps = tuple(int(set_i[r].max()) for r in (nat.EP_I_DELAY_CONTROL, nat.EP_I_DELAY_POSE, nat.EP_I_DELAY_STATE))
    return EnvRows(f, i, caps)
