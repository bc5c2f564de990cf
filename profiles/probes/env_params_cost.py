"""What per-env parameters (BcgEnvRows) cost per step.

    python profiles/probes/env_params_cost.py --tag r3a [--out PATH]

Three batches of the bench.py configs[2] workload (aisle worlds, delays 2/1/1, PlanEnv's default noise, egocentric
observation, auto-reset), at 65 536 and at 8 192 envs:
  none   one EnvParams: the batch-wide path, no rows
  one    params=[ep]: the same setting through the per-env rows
  pool4  four sets that differ in delays (2,1,1) / (0,0,0) / (1,2,0) / (3,0,2), noise and tolerances, assigned e % 4
Per-step time from CUDA events over `--steps` warm steps, the variants alternated over `--rounds` rounds (median and
spread reported).  Writes profiles/<tag>_env_params_cost.txt (or --out) with the card name and power limit of the run.
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from bc_gym_planning_env_b200.envs.base.params import EnvParams, RewardParams  # noqa: E402
from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool  # noqa: E402
from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE, VecPlanEnv  # noqa: E402


def pool4():
    return ([EnvParams(control_delay=2, pose_delay=1, state_delay=1),
             EnvParams(goal_spat_dist=0.2, goal_ang_dist=np.pi / 8, iteration_timeout=150),
             EnvParams(control_delay=1, pose_delay=2, state_delay=0,
                       reward_provider_params=RewardParams(spatial_precision=1.0, angular_precision=np.pi / 2,
                                                           spatial_progress_multiplier=0.5)),
             EnvParams(control_delay=3, pose_delay=0, state_delay=2)],
            [DEFAULT_NOISE, None, {k: 4 * v for k, v in DEFAULT_NOISE.items()}, DEFAULT_NOISE])


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "nvidia-smi not available (%s)" % torch.cuda.get_device_name()


def time_steps(env, acts, steps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for t in range(steps):
        env.step(acts[t % len(acts)])
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="r3")
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="65536,8192")
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--pool", type=int, default=256)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("env_params_cost needs a CUDA device")
    ep = EnvParams(control_delay=2, pose_delay=1, state_delay=1)
    costmaps, paths = random_aisle_pool(args.pool, 10000, ep)
    sets, noise = pool4()
    lines = ["# per-step time of per-env parameter rows (profiles/probes/env_params_cost.py)",
             "# card: %s" % card(),
             "# workload: bench.py configs[2] (aisle pool of %d maps, private copies, delays 2/1/1, default noise, ego, auto-reset)"
             % args.pool,
             "# %d warm-up + %d timed steps per variant per round, variants alternated over %d rounds; ms per step"
             % (args.warmup, args.steps, args.rounds)]
    for n in [int(x) for x in args.sizes.split(",")]:
        kw = dict(n_envs=n, seed=1234, auto_reset=True, with_ego=True, private_map_copies=True)
        envs = {"none": VecPlanEnv(costmaps, paths, ep, noise_parameters=DEFAULT_NOISE, **kw),
                "one": VecPlanEnv(costmaps, paths, [ep], noise_parameters=DEFAULT_NOISE, **kw),
                "pool4": VecPlanEnv(costmaps, paths, sets, noise_parameters=noise, **kw)}
        lo, hi = envs["none"].action_bounds()
        gen = torch.Generator(device="cuda")
        gen.manual_seed(5)
        acts = torch.rand((16, n, 2), generator=gen, device="cuda") * torch.tensor(hi - lo, device="cuda") + torch.tensor(lo, device="cuda")
        for env in envs.values():
            time_steps(env, acts, args.warmup)
        times = {k: [] for k in envs}
        for r in range(args.rounds):
            order = list(envs) if r % 2 == 0 else list(reversed(list(envs)))
            for k in order:
                times[k].append(time_steps(envs[k], acts, args.steps))
        base = float(np.median(times["none"]))
        lines.append("")
        lines.append("n_envs %d" % n)
        for k, v in times.items():
            med = float(np.median(v))
            lines.append("  %-6s median %.4f ms  min %.4f  max %.4f  (vs none: %+.4f ms, %+.1f %%)   rounds: %s"
                         % (k, med, min(v), max(v), med - base, 100 * (med - base) / base, " ".join("%.4f" % x for x in v)))
        del envs
        torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n"
    out = args.out or os.path.join(ROOT, "profiles", "%s_env_params_cost.txt" % args.tag)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
