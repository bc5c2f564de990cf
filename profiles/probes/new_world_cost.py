"""What auto-reset into a new world (auto_reset='new_world') costs per step, against the other two ways to run episodes.

    python profiles/probes/new_world_cost.py --tag r3e [--out PATH] [--variants same,new,host]

VecRandomAisleTurnEnv batches (device-drawn aisle worlds, 0.03 m, delays 2/1/1, PlanEnv's default noise, egocentric
observation), at 65 536 and at 8 192 envs.  One batch per size, built with auto_reset='new_world', runs every variant
(BcgParams.auto_reset is read at every step; the other modes ignore the world generator):
  same  auto_reset=True: the in-kernel reset restarts the env's current world
  new   auto_reset='new_world': reward_kernel lists the done envs, regenerate_kernel gives them new worlds in the step
  host  auto_reset=False and `reset(done)` after every step: a masked generation launch plus a whole-batch observe_ego
Per-step time from CUDA events over `--steps` warm steps (host: the step and the reset), the variants alternated over
`--rounds` rounds (median and spread reported).  Then, untimed, the mean number of done envs per step of each variant,
and a torch.profiler capture of `--profile-steps` steps of `new` for the time of each kernel (regenerate_kernel's own).
Writes profiles/<tag>_new_world_cost.txt (or --out) with the card name and power limit of the run.
"""
import argparse
import os
import re
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from bc_gym_planning_env_b200 import _native as nat  # noqa: E402
from bc_gym_planning_env_b200.envs.base.params import EnvParams  # noqa: E402
from bc_gym_planning_env_b200.vec_aisle_env import VecRandomAisleTurnEnv  # noqa: E402
from bc_gym_planning_env_b200.vec_env import DEFAULT_NOISE  # noqa: E402

MODES = {"same": 1, "new": nat.AUTO_RESET_NEW_WORLD, "host": 0}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "nvidia-smi not available (%s)" % torch.cuda.get_device_name()


def run(env, mode, acts, steps, count=None):
    env._c_params.auto_reset = MODES[mode]
    for t in range(steps):
        env.step(acts[t % len(acts)])
        if mode == "host":
            env.reset(env.done)
        if count is not None:
            count += env.done.sum()


def time_steps(env, mode, acts, steps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    run(env, mode, acts, steps)
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / steps


def kernel_times(env, acts, steps):
    """mean device time (ms) per step of every kernel of `steps` steps of the new-world mode, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    env._c_params.auto_reset = MODES["new"]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run(env, "new", acts, steps)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        m = re.search(r"(\w+_kernel)", ev.key)
        t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        if m and t > 0:
            out[m.group(1)] = out.get(m.group(1), 0.0) + t / 1000.0 / steps
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="r3")
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="65536,8192")
    ap.add_argument("--variants", default="same,new,host")
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--profile-steps", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("new_world_cost needs a CUDA device")
    variants = args.variants.split(",")
    ep = EnvParams(control_delay=2, pose_delay=1, state_delay=1)
    lines = ["# per-step time of the three ways to run episodes on device-drawn worlds (profiles/probes/new_world_cost.py)",
             "# card: %s" % card(),
             "# workload: VecRandomAisleTurnEnv, 0.03 m, delays 2/1/1, iteration_timeout %d, default noise, egocentric "
             "observation, uniform random actions" % ep.iteration_timeout,
             "# %d warm-up + %d timed steps per variant per round, variants alternated over %d rounds; ms per step"
             % (args.warmup, args.steps, args.rounds)]
    for n in [int(x) for x in args.sizes.split(",")]:
        env = VecRandomAisleTurnEnv(n, ep, seed=1234, auto_reset='new_world', with_ego=True, noise_parameters=DEFAULT_NOISE)
        lo, hi = env.action_bounds()
        gen = torch.Generator(device="cuda")
        gen.manual_seed(5)
        acts = torch.rand((16, n, 2), generator=gen, device="cuda") * torch.tensor(hi - lo, device="cuda") + torch.tensor(lo, device="cuda")
        times = {k: [] for k in variants}
        for r in range(args.rounds):
            order = variants if r % 2 == 0 else list(reversed(variants))
            for k in order:
                run(env, k, acts, args.warmup)
                times[k].append(time_steps(env, k, acts, args.steps))
        lines.append("")
        lines.append("n_envs %d" % n)
        base = float(np.median(times[variants[0]]))
        for k, v in times.items():
            med = float(np.median(v))
            cnt = torch.zeros((), dtype=torch.int64, device="cuda")
            run(env, k, acts, args.steps, cnt)
            lines.append("  %-4s median %.4f ms  min %.4f  max %.4f  (vs %s: %+.4f ms)  done envs per step %.1f   rounds: %s"
                         % (k, med, min(v), max(v), variants[0], med - base, int(cnt) / args.steps, " ".join("%.4f" % x for x in v)))
        if "new" in variants and args.profile_steps > 0:
            kt = kernel_times(env, acts, args.profile_steps)
            lines.append("  kernels of `new`, ms per step (torch.profiler, %d steps): %s"
                         % (args.profile_steps, ", ".join("%s %.4f" % (k, v) for k, v in sorted(kt.items(), key=lambda x: -x[1]))))
        env.check_status()
        del env
        torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n"
    out = args.out or os.path.join(ROOT, "profiles", "%s_new_world_cost.txt" % args.tag)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as fh:
        fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
