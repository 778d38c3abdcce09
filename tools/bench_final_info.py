"""mt_step against mt_step_final (the ending envs' final observation, return and length) on the per-step workloads.

    python tools/bench_final_info.py [--steps K] [--regions R] [--rounds N] [--out FILE.json]

Workloads (mt_step with HBM actions, 2^20 envs, auto-reset, horizon 1000, after a 200-step burn-in so that the envs
are spread over their episodes and resets happen at their steady rate every step):
  ref_x10_fp32   reference arm, X = 10, fp32 observations
  ref_x10_fp16   reference arm, X = 10, binary16 observations
  ur5_x20_fp32   UR5 preset, X = 20
Each region is K steps with fresh actions every step, replayed as one K-node CUDA graph (device events); R regions per
run, median and best region reported.  The two calls alternate step, final, step, final, ... (--rounds pairs), with ONE
handle alive at a time: handles in one process share the 126 MB L2.  The spread of a call is the difference between
its runs' medians.  The GPU's name and power limit are read (nvidia-smi, read-only) in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from manytor_b200 import UR5_ARM, REFERENCE_ARM, BatchedEnvs  # noqa: E402
from tools.bench_obs_dtype import BURN_IN, HORIZON, N, entry, gpu_info, graph_regions  # noqa: E402


def run(arm, x, dtype, final, K, R):
    env = BatchedEnvs(N, x, arm=arm, device=0, auto_reset=True, horizon=HORIZON, seed=7, obs_dtype=dtype)
    env.reset()
    env.rollout_random(BURN_IN, write_obs=False)
    torch.cuda.synchronize()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(11)
    acts = [torch.randint(-180, 180, (N, arm.n_joints), device="cuda", generator=gen).float() for _ in range(K)]
    s0 = env.stats()
    times = graph_regions(env, lambda k: [env.step(acts[i], final=final) for i in range(k)], K, R)
    s1 = env.stats()
    return times, env.bytes_per_env_step(True, True), (s1["episodes"] - s0["episodes"]) / (s1["env_steps"] - s0["env_steps"]), env


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=100, help="K: steps per timed region")
    ap.add_argument("--regions", type=int, default=10, help="R: timed regions per run")
    ap.add_argument("--rounds", type=int, default=2, help="mt_step / mt_step_final pairs per workload")
    ap.add_argument("--out", default=None, help="write the JSON here as well")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_final_info.py needs a CUDA device"
    K, R = args.steps, args.regions
    workloads = {
        "ref_x10_fp32": (REFERENCE_ARM, 10, torch.float32),
        "ref_x10_fp16": (REFERENCE_ARM, 10, torch.float16),
        "ur5_x20_fp32": (UR5_ARM, 20, torch.float32),
    }
    result = {"gpu": gpu_info(), "n_envs": N, "horizon": HORIZON, "burn_in": BURN_IN, "steps_per_region": K,
              "regions": R, "rounds": args.rounds,
              "method": "alternating mt_step / mt_step_final handles, one alive at a time; K-step CUDA graph of fresh "
                        "actions per region; median and best region per run",
              "workloads": {}}
    for name, (arm, x, dtype) in workloads.items():
        runs = {"step": [], "step_final": []}
        for _ in range(args.rounds):
            for label, final in (("step", False), ("step_final", True)):
                times, b, reset_rate, env = run(arm, x, dtype, final, K, R)
                e = entry(times, b, K)
                e["episodes_per_env_step"] = reset_rate
                runs[label].append(e)
                env.close()
                del env
                torch.cuda.synchronize()
        w = {}
        for label, rs in runs.items():
            meds = [r["us_per_step_median"] for r in rs]
            w[label] = {"runs": rs, "us_per_step_median_of_runs": float(np.median(meds)),
                        "run_to_run_spread_us": max(meds) - min(meds)}
        w["final_over_step"] = w["step_final"]["us_per_step_median_of_runs"] / w["step"]["us_per_step_median_of_runs"]
        result["workloads"][name] = w
        print(f"{name:13s} mt_step {w['step']['us_per_step_median_of_runs']:8.2f} us (spread "
              f"{w['step']['run_to_run_spread_us']:.2f})  mt_step_final {w['step_final']['us_per_step_median_of_runs']:8.2f} us "
              f"(spread {w['step_final']['run_to_run_spread_us']:.2f})  ratio {w['final_over_step']:.4f}", flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({k: {"step_us": v["step"]["us_per_step_median_of_runs"],
                          "step_final_us": v["step_final"]["us_per_step_median_of_runs"],
                          "ratio": v["final_over_step"]} for k, v in result["workloads"].items()}))


if __name__ == "__main__":
    main()
