"""Per-step time of the headline step with a footprint whose mask rows take two words (footprint_scale 1.5 at 0.03 m:
88-row masks up to ~100 px wide), the workload on which every collision check runs collide_thread's loop.

    python profiles/probes/wide_footprint_cost.py [--libs NAME=PATH,NAME=PATH] [--rounds 5] [--out PATH]

The batch is bench.py's headline batch at footprint_scale 1.5: 65 536 envs on 2 048 random aisle maps, delays 2/1/1,
PlanEnv's odometry noise, auto-reset, egocentric observation; eight seeded action sets.  A round is `--warmup` steps,
then `--steps` steps between two CUDA events (ms per step).  With --libs every round runs each library (BCG_B200_LIB)
in a process of its own, the order alternating from round to round; without it, one round of the tree's own build.
Writes the median, spread and rounds per library, with the card name and power limit of the run, to --out (default
profiles/wide_footprint_cost.txt).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        import torch
        return "nvidia-smi not available (%s)" % torch.cuda.get_device_name()


def one_round(args):
    """ms per step of one round of the loaded library, and the episodes a collision ended per timed step"""
    import torch
    from bc_gym_planning_env_b200 import _native as nat
    from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
    from bc_gym_planning_env_b200.vec_env import VecPlanEnv
    import bench
    if not torch.cuda.is_available():
        raise SystemExit("wide_footprint_cost needs a CUDA device")
    params = bench.aisle_params()
    costmaps, paths = random_aisle_pool(2048, 10000, params)
    env = VecPlanEnv(costmaps, paths, params, n_envs=args.envs, seed=1234, auto_reset=True, device="cuda:0",
                     private_map_copies=True, with_ego=True, footprint_scale=args.scale)
    actions = bench.random_actions(env, "cuda:0", 4321)
    for w in range(args.warmup):
        env.step(actions[w % len(actions)])
    env.episode_stats(reset=True)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for k in range(args.steps):
        env.step(actions[k % len(actions)])
    stop.record()
    stop.synchronize()
    ms = start.elapsed_time(stop) / args.steps
    collided = float(env.episode_stats()[nat.STAT_NAMES.index("collided")])
    env.check_status()
    return {"ms_per_step": ms, "collisions_per_step": collided / args.steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--libs", default=None, help="NAME=PATH,...: libraries to alternate (default: the tree's own build)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--scale", type=float, default=1.5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wide_footprint_cost.txt"))
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        print(json.dumps(one_round(args)))
        return
    libs = [kv.split("=", 1) for kv in args.libs.split(",")] if args.libs else [["tree", ""]]
    worker = [sys.executable, os.path.abspath(__file__), "--worker", "--steps", str(args.steps), "--warmup",
              str(args.warmup), "--envs", str(args.envs), "--scale", str(args.scale)]
    rounds = {name: [] for name, _ in libs}
    for r in range(args.rounds if args.libs else 1):
        for name, path in (libs if r % 2 == 0 else libs[::-1]):
            env = dict(os.environ)
            if path:
                env["BCG_B200_LIB"] = os.path.abspath(path)
            out = subprocess.run(worker, env=env, stdout=subprocess.PIPE, text=True, check=True).stdout
            rounds[name].append(json.loads(out.strip().splitlines()[-1]))
    lines = ["# per-step time at footprint_scale %g (profiles/probes/wide_footprint_cost.py)" % args.scale,
             "# card: %s" % card(),
             "# workload: bench.py's headline batch (%d envs, 2 048 random aisle maps at 0.03 m, delays 2/1/1, odometry noise, "
             "auto-reset, egocentric observation) with footprint_scale %g" % (args.envs, args.scale),
             "# %d warm-up + %d timed steps per round (CUDA events), one process per library and round, order alternating"
             % (args.warmup, args.steps)]
    for name, got in rounds.items():
        ms = [g["ms_per_step"] for g in got]
        lines.append("%-8s median %.4f ms  min %.4f  max %.4f  episodes ended by a collision per step %.1f   rounds: %s"
                     % (name, float(np.median(ms)), min(ms), max(ms), got[0]["collisions_per_step"],
                        " ".join("%.4f" % x for x in ms)))
    text = "\n".join(lines) + "\n"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
