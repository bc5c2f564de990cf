"""Step and kernel times of two builds of the library on the bench.py configs[2] workload, alternated round by round.

    python profiles/probes/cell_index_cost.py --base LIB_A --new LIB_B [--tag r3b] [--out PATH]

LIB_A / LIB_B are libbcg_b200.so builds (for example the parent commit's, built with csrc/build.py into
csrc/variants/, against the current one).  Each round runs one child process per build (the library is loaded once per
process, via BCG_B200_LIB), in alternating order; a child times, at every size of --sizes, `--steps` warm steps of the
aisle workload (pool of --pool host maps, private copies, delays 2/1/1, default noise, egocentric observation,
auto-reset) with CUDA events around the whole loop, then per-kernel times from events between the kernels
(VecPlanEnv.step_timed, every step of a second loop).  Reports medians and the spread over the rounds, the extra HBM of
the tile-summary arena, and the card's name, power limit and clocks read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def child(sizes, steps, warmup, pool):
    sys.path.insert(0, ROOT)
    import torch
    from bc_gym_planning_env_b200.envs.base.params import EnvParams
    from bc_gym_planning_env_b200.envs.synth_turn_env import random_aisle_pool
    from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE, VecPlanEnv
    ep = EnvParams(control_delay=2, pose_delay=1, state_delay=1)
    costmaps, paths = random_aisle_pool(pool, 10000, ep)
    out = {}
    for n in sizes:
        env = VecPlanEnv(costmaps, paths, ep, n_envs=n, seed=1234, auto_reset=True, with_ego=True, private_map_copies=True,
                         noise_parameters=DEFAULT_NOISE)
        lo, hi = env.action_bounds()
        gen = torch.Generator(device="cuda")
        gen.manual_seed(5)
        acts = torch.rand((16, n, 2), generator=gen, device="cuda") * torch.tensor(hi - lo, device="cuda") + torch.tensor(lo, device="cuda")
        for t in range(warmup):
            env.step(acts[t % 16])
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for t in range(steps):
            env.step(acts[t % 16])
        b.record()
        b.synchronize()
        step_ms = a.elapsed_time(b) / steps
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        for e in evs:
            e.record()
        k = {"move": [], "reward": [], "ego": []}
        for t in range(min(steps, 100)):
            env.step_timed(acts[t % 16], evs)
            evs[4].synchronize()
            k["move"].append(evs[1].elapsed_time(evs[2]))
            k["reward"].append(evs[2].elapsed_time(evs[3]))
            k["ego"].append(evs[3].elapsed_time(evs[4]))
        env.check_status()
        out[str(n)] = {"step": step_ms, **{kk: float(np.mean(v)) for kk, v in k.items()},
                       "sum_arena_bytes_per_env": env.occ_sum_arena.numel() * 4 / n,
                       "handed_over": int(env._ego_list[n])}
        del env
        torch.cuda.empty_cache()
    print("RESULT " + json.dumps(out))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "nvidia-smi not available"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", help="library of the baseline build")
    ap.add_argument("--new", help="library of the build under test")
    ap.add_argument("--tag", default="r3")
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="65536,8192")
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--pool", type=int, default=256)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    sizes = [int(x) for x in args.sizes.split(",")]
    if args.child:
        return child(sizes, args.steps, args.warmup, args.pool)
    libs = {"base": os.path.abspath(args.base), "new": os.path.abspath(args.new)}
    res = {k: [] for k in libs}
    cards = [card()]
    for r in range(args.rounds):
        for name in (["base", "new"] if r % 2 == 0 else ["new", "base"]):
            cmd = [sys.executable, os.path.abspath(__file__), "--child", "--sizes", args.sizes, "--steps", str(args.steps),
                   "--warmup", str(args.warmup), "--pool", str(args.pool)]
            p = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, BCG_B200_LIB=libs[name]))
            line = [x for x in p.stdout.splitlines() if x.startswith("RESULT ")]
            if p.returncode != 0 or not line:
                raise SystemExit("child %s failed:\n%s\n%s" % (name, p.stdout[-3000:], p.stderr[-3000:]))
            res[name].append(json.loads(line[0][7:]))
        cards.append(card())
    lines = ["# two builds alternated over %d rounds (profiles/probes/cell_index_cost.py)" % args.rounds,
             "# card (name, power limit, SM clock, max SM clock) before the first and after every round:"]
    lines += ["#   " + c for c in cards]
    lines.append("# workload: bench.py configs[2] (aisle pool of %d maps, private copies, delays 2/1/1, default noise, ego, "
                 "auto-reset); %d warm-up + %d timed steps per size and round; kernels: mean of 100 step_timed steps"
                 % (args.pool, args.warmup, args.steps))
    lines.append("# base: %s" % args.base)
    lines.append("# new:  %s" % args.new)
    for n in sizes:
        lines.append("")
        lines.append("n_envs %d" % n)
        base_step = float(np.median([x[str(n)]["step"] for x in res["base"]]))
        for name in libs:
            rows = [x[str(n)] for x in res[name]]
            for key in ("step", "ego", "move", "reward"):
                v = [row[key] for row in rows]
                med = float(np.median(v))
                extra = ("   (vs base: %+.1f %%)" % (100 * (med - base_step) / base_step)) if key == "step" else ""
                lines.append("  %-4s %-6s median %.4f ms  min %.4f  max %.4f%s   rounds: %s"
                             % (name, key, med, min(v), max(v), extra, " ".join("%.4f" % x for x in v)))
            lines.append("  %-4s tile-summary arena %.0f bytes per env, envs handed to the dense kernel (last step) %d"
                         % (name, rows[0]["sum_arena_bytes_per_env"], rows[-1]["handed_over"]))
    text = "\n".join(lines) + "\n"
    out = args.out or os.path.join(ROOT, "profiles", "%s_cell_index_cost.txt" % args.tag)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
