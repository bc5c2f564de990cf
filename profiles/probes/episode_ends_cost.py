"""What episode ends (episode_ends=True) cost per step.

    python profiles/probes/episode_ends_cost.py --tag r3d [--out PATH]

Two batches of the bench.py configs[2] workload (aisle worlds, delays 2/1/1, PlanEnv's default noise, egocentric
observation, auto-reset), at 65 536 and at 8 192 envs:
  off   episode_ends=False: the parent's step
  on    episode_ends=True: reason bytes, final rows and final crops (capacity n_envs)
Per-step time from CUDA events over `--steps` warm steps, the variants alternated over `--rounds` rounds (median and
spread reported), then, untimed, the mean number of episode ends per step of the `on` batch.  Writes
profiles/<tag>_episode_ends_cost.txt (or --out) with the card name and power limit of the run.
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from bc_gym_planning_env_b200.envs.base.params import EnvParams  # noqa: E402
from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool  # noqa: E402
from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE, VecPlanEnv  # noqa: E402


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


def ends_per_step(env, acts, steps):
    total = torch.zeros((), dtype=torch.int64, device=env.device)
    for t in range(steps):
        env.step(acts[t % len(acts)])
        total += env.final_observation().count
    return int(total) / steps


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
        raise SystemExit("episode_ends_cost needs a CUDA device")
    ep = EnvParams(control_delay=2, pose_delay=1, state_delay=1)
    costmaps, paths = random_aisle_pool(args.pool, 10000, ep)
    lines = ["# per-step time of episode ends (profiles/probes/episode_ends_cost.py)",
             "# card: %s" % card(),
             "# workload: bench.py configs[2] (aisle pool of %d maps, private copies, delays 2/1/1, default noise, ego, auto-reset)"
             % args.pool,
             "# %d warm-up + %d timed steps per variant per round, variants alternated over %d rounds; ms per step"
             % (args.warmup, args.steps, args.rounds)]
    for n in [int(x) for x in args.sizes.split(",")]:
        kw = dict(n_envs=n, seed=1234, auto_reset=True, with_ego=True, private_map_copies=True, noise_parameters=DEFAULT_NOISE)
        envs = {"off": VecPlanEnv(costmaps, paths, ep, **kw), "on": VecPlanEnv(costmaps, paths, ep, episode_ends=True, **kw)}
        lo, hi = envs["off"].action_bounds()
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
        base = float(np.median(times["off"]))
        lines.append("")
        lines.append("n_envs %d   (episode ends per step, mean over %d untimed steps of `on`: %.1f)"
                     % (n, args.steps, ends_per_step(envs["on"], acts, args.steps)))
        for k, v in times.items():
            med = float(np.median(v))
            lines.append("  %-4s median %.4f ms  min %.4f  max %.4f  (vs off: %+.4f ms, %+.1f %%)   rounds: %s"
                         % (k, med, min(v), max(v), med - base, 100 * (med - base) / base, " ".join("%.4f" % x for x in v)))
        del envs
        torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n"
    out = args.out or os.path.join(ROOT, "profiles", "%s_episode_ends_cost.txt" % args.tag)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
