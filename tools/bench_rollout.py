"""Trajectory rollouts (mt_rollout) against the per-step path and the last-step-only rollout.

    python tools/bench_rollout.py [--steps K] [--regions R] [--rounds N] [--out FILE.json]

2^20 envs, auto-reset with horizon 1000 after a burn-in, for the reference arm at X = 10 and the UR5 preset at X = 20.
Each region is ONE call of K steps (default 64) captured as a CUDA graph and timed by device events; R regions per
run, median and best region reported, the workloads alternating for --rounds rounds on one handle per arm.  The
caller's action buffer is refilled with fresh values (a device copy) outside the timed region before every region.
  a_actions_per_step      mt_rollout(actions), MT_ROLLOUT_PERSISTENT=0: K mt_step launches into the slices
  b_actions_persistent    mt_rollout(actions), one launch of the multi-step rollout kernel
  c_random_last_step      mt_rollout_random(K): the same kernel keeping only the last step's outputs
  d_draws_trajectory      mt_rollout(NULL), every step kept, drawn_dev = NULL
  d_draws_recorded        mt_rollout(NULL) with drawn_dev: the drawn actions kept as well
Algorithmic bytes per env-step (state = 2 (4J + 8) B, read and written once per call):
  b, d   4J (caller actions read, or draws written; none for d without drawn_dev) + 12X + 5 (6X + 5 in binary16)
         + (state + 12X) / K
  c      12X + 5 + (state + 12X) / K
  a      mt_bytes_per_env_step(actions from HBM, obs written): the per-step path moves the whole state every step
The GPU's name and power limit are read (nvidia-smi, read-only) in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_obs_dtype import gpu_info  # noqa: E402
from manytor_b200 import REFERENCE_ARM, UR5_ARM, BatchedEnvs, Trajectory  # noqa: E402

N = 1 << 20
HORIZON = 1000
BURN_IN = 200
WORKLOADS = ("a_actions_per_step", "b_actions_persistent", "c_random_last_step", "d_draws_trajectory",
             "d_draws_recorded")


def algorithmic_bytes(env, name, K):
    J, X = env.j, env.x
    obs = (6 if env.obs_dtype == torch.float16 else 12) * X
    once = (2 * (4 * J + 8) + 12 * X) / K
    if name == "a_actions_per_step":
        return float(env.bytes_per_env_step(True, True))
    per_step = {"b_actions_persistent": 4 * J, "c_random_last_step": 0, "d_draws_trajectory": 0,
                "d_draws_recorded": 4 * J}[name]
    return per_step + obs + 5 + once


def regions(env, body, refill, R):
    """R timed replays of one captured call (device events), each after a refill of the action buffer; ms, sorted."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        body()                                            # warm-up: kernel attributes, launch shapes, NVRTC
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        body()
    g.replay()                                            # the first replay uploads the graph
    torch.cuda.synchronize()
    out = []
    for r in range(R):
        refill(r)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return sorted(out)


def run_arm(arm, x, K, R, rounds):
    env = BatchedEnvs(N, x, arm=arm, device=0, auto_reset=True, horizon=HORIZON, seed=7)
    env.reset()
    env.rollout_random(BURN_IN, write_obs=False)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    pool = [torch.rand((K, N, env.j), device="cuda", generator=gen) * 360.0 - 180.0 for _ in range(2)]
    acts = torch.empty_like(pool[0])
    refill = lambda r: acts.copy_(pool[r % 2])
    out = Trajectory(torch.empty((K, N, 3 * x), device="cuda"), torch.empty((K, N), device="cuda"),
                     torch.empty((K, N), dtype=torch.uint8, device="cuda"), None)
    drawn = torch.empty((K, N, env.j), device="cuda")
    bodies = {
        "a_actions_per_step": lambda: env.rollout(acts, out=out),
        "b_actions_persistent": lambda: env.rollout(acts, out=out),
        "c_random_last_step": lambda: env.rollout_random(K),
        "d_draws_trajectory": lambda: env.rollout(n_steps=K, out=out),
        "d_draws_recorded": lambda: env.rollout(n_steps=K, record_actions=True, out=out._replace(actions=drawn)),
    }
    runs = {w: [] for w in WORKLOADS}
    for _ in range(rounds):
        for w in WORKLOADS:
            if w == "a_actions_per_step":
                os.environ["MT_ROLLOUT_PERSISTENT"] = "0"     # read at every call: the capture takes the per-step path
            try:
                l0 = env.launch_count
                times = regions(env, bodies[w], refill, R)
                launches_warm_and_capture = env.launch_count - l0
            finally:
                os.environ.pop("MT_ROLLOUT_PERSISTENT", None)
            med, best = times[(len(times) - 1) // 2], times[0]
            b = algorithmic_bytes(env, w, K)
            runs[w].append({"us_per_step_median": 1e3 * med / K, "us_per_step_best": 1e3 * best / K,
                            "env_steps_per_s": N * K / (med * 1e-3), "bytes_per_env_step": b,
                            "algorithmic_gbs": N * K * b / (med * 1e-3) / 1e9,
                            "launches_per_call": launches_warm_and_capture // 2, "regions_ms": times})
    res = {}
    for w, rs in runs.items():
        meds = [r["us_per_step_median"] for r in rs]
        m = float(np.median(meds))
        res[w] = {"runs": rs, "us_per_step_median_of_runs": m, "run_to_run_spread_us": max(meds) - min(meds),
                  "env_steps_per_s": N / (m * 1e-6), "bytes_per_env_step": rs[0]["bytes_per_env_step"],
                  "launches_per_call": rs[0]["launches_per_call"]}
        print(f"{arm is REFERENCE_ARM and 'ref' or 'ur5'} x={x} {w:22s} {m:8.2f} us/step (spread {res[w]['run_to_run_spread_us']:.2f})"
              f"  {res[w]['env_steps_per_s']:.3e} env-steps/s  {res[w]['bytes_per_env_step']:.1f} B/env-step", flush=True)
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=64, help="K: steps per call (one call per timed region)")
    ap.add_argument("--regions", type=int, default=10, help="R: timed regions per run")
    ap.add_argument("--rounds", type=int, default=2, help="runs of every workload, alternating")
    ap.add_argument("--out", default=None, help="write the JSON here as well")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_rollout.py needs a CUDA device"
    result = {"gpu": gpu_info(), "n_envs": N, "steps_per_call": args.steps, "regions": args.regions,
              "rounds": args.rounds,
              "method": "one K-step call per CUDA-graph region, device events; action buffer refilled by a device copy "
                        "outside every timed region; workloads alternate on one handle per arm; median and best region "
                        "per run, median of runs and run-to-run spread",
              "arms": {}}
    for name, arm, x in (("reference_x10", REFERENCE_ARM, 10), ("ur5_x20", UR5_ARM, 20)):
        result["arms"][name] = run_arm(arm, x, args.steps, args.regions, args.rounds)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({a: {w: round(v["us_per_step_median_of_runs"], 2) for w, v in r.items()}
                      for a, r in result["arms"].items()}))


if __name__ == "__main__":
    main()
