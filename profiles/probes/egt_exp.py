"""A/B of the egocentric kernels on the bench workload (run on the GPU box):
    python profiles/probes/egt_exp.py
sparse = ego_sparse_kernel (default); dense = ego_tiles_kernel for every env (BCG_EGO_KERNEL=dense)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for name, kernel in (("sparse", None), ("dense", "dense")):
    env = dict(os.environ)
    if kernel:
        env["BCG_EGO_KERNEL"] = kernel
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "50", "--warmup", "5", "--e2e-steps", "2",
                          "--cpu-seconds", "0.1", "--gen-envs", "0"], env=env, capture_output=True, text=True)
    try:
        d = json.loads(out.stdout.strip().splitlines()[-1])
        ego = [v for k, v in d["kernels_ms"].items() if k.startswith("ego_")][0]
        print("%-8s ego_ms %.4f step_ms %.4f value %.4g" % (name, ego, d["ms_per_step"], d["value"]), flush=True)
    except Exception:
        print(name, "failed", out.stderr[-800:], flush=True)
