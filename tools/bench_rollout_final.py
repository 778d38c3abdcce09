"""Trajectory rollouts with final outputs (mt_rollout_final) against plain trajectory rollouts (mt_rollout) and against
K mt_step_final launches into the same slices.

    python tools/bench_rollout_final.py [--steps K] [--regions R] [--rounds N] [--out FILE.json]

2^20 envs, auto-reset with obs_after_reset = 1 (the Gymnasium adapter's setting), for the reference arm at X = 10 and
the UR5 preset at X = 20, each at two horizons: bench_rollout.py's 1000, and 8, where about one env in eight ends
every step, to bound the cost of the rare path when resets are not rare.  After a burn-in the envs are spread over
their episodes.  Each region is ONE call of K steps (default 64) captured as a CUDA graph and timed by device events;
R regions per run, median and best region reported, the workloads alternating for --rounds rounds on one handle per
(arm, horizon).  The caller's action buffer is refilled with fresh values (a device copy) outside the timed region
before every region.
  actions_rollout          mt_rollout(actions): one launch of the multi-step rollout kernel
  actions_rollout_final    mt_rollout_final(actions): the same launch with the final slices
  actions_step_final       mt_rollout_final(actions), MT_ROLLOUT_PERSISTENT=0: K mt_step_final launches into the slices
  draws_rollout            mt_rollout(NULL): in-kernel draws, drawn_dev = NULL
  draws_rollout_final      mt_rollout_final(NULL)
  draws_step_final         mt_rollout_final(NULL), MT_ROLLOUT_PERSISTENT=0: K x (draw + mt_step_final launch)
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
from bench_rollout import BURN_IN, HORIZON, N, regions  # noqa: E402
from manytor_b200 import REFERENCE_ARM, UR5_ARM, BatchedEnvs, FinalInfo, Trajectory  # noqa: E402

RESET_HEAVY_HORIZON = 8
WORKLOADS = ("actions_rollout", "actions_rollout_final", "actions_step_final", "draws_rollout", "draws_rollout_final",
             "draws_step_final")
PER_STEP = ("actions_step_final", "draws_step_final")


def run_arm(arm, x, horizon, K, R, rounds):
    env = BatchedEnvs(N, x, arm=arm, device=0, auto_reset=True, obs_after_reset=True, horizon=horizon, seed=7)
    env.reset()
    env.rollout_random(BURN_IN, write_obs=False)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    pool = [torch.rand((K, N, env.j), device="cuda", generator=gen) * 360.0 - 180.0 for _ in range(2)]
    acts = torch.empty_like(pool[0])
    refill = lambda r: acts.copy_(pool[r % 2])
    out = Trajectory(torch.empty((K, N, 3 * x), device="cuda"), torch.empty((K, N), device="cuda"),
                     torch.empty((K, N), dtype=torch.uint8, device="cuda"), None)
    fin = FinalInfo(torch.empty((K, N, 3 * x), device="cuda"), torch.empty((K, N), device="cuda"),
                    torch.empty((K, N), dtype=torch.int32, device="cuda"))
    bodies = {
        "actions_rollout": lambda: env.rollout(acts, out=out),
        "actions_rollout_final": lambda: env.rollout(acts, out=out, final=True, final_out=fin),
        "actions_step_final": lambda: env.rollout(acts, out=out, final=True, final_out=fin),
        "draws_rollout": lambda: env.rollout(n_steps=K, out=out),
        "draws_rollout_final": lambda: env.rollout(n_steps=K, out=out, final=True, final_out=fin),
        "draws_step_final": lambda: env.rollout(n_steps=K, out=out, final=True, final_out=fin),
    }
    runs = {w: [] for w in WORKLOADS}
    for _ in range(rounds):
        for w in WORKLOADS:
            if w in PER_STEP:
                os.environ["MT_ROLLOUT_PERSISTENT"] = "0"     # read at every call: the capture takes the per-step path
            try:
                l0 = env.launch_count
                s0 = env.stats()
                times = regions(env, bodies[w], refill, R)
                s1 = env.stats()
                launches_warm_and_capture = env.launch_count - l0
            finally:
                os.environ.pop("MT_ROLLOUT_PERSISTENT", None)
            med, best = times[(len(times) - 1) // 2], times[0]
            runs[w].append({"us_per_step_median": 1e3 * med / K, "us_per_step_best": 1e3 * best / K,
                            "env_steps_per_s": N * K / (med * 1e-3),
                            "episodes_per_env_step": (s1["episodes"] - s0["episodes"]) / (s1["env_steps"] - s0["env_steps"]),
                            "launches_per_call": launches_warm_and_capture // 2, "regions_ms": times})
    res = {}
    for w, rs in runs.items():
        meds = [r["us_per_step_median"] for r in rs]
        m = float(np.median(meds))
        res[w] = {"runs": rs, "us_per_step_median_of_runs": m, "run_to_run_spread_us": max(meds) - min(meds),
                  "env_steps_per_s": N / (m * 1e-6), "episodes_per_env_step": rs[-1]["episodes_per_env_step"],
                  "launches_per_call": rs[0]["launches_per_call"]}
    for mode in ("actions", "draws"):
        base = res[f"{mode}_rollout"]["us_per_step_median_of_runs"]
        res[f"{mode}_final_over_rollout"] = res[f"{mode}_rollout_final"]["us_per_step_median_of_runs"] / base
        res[f"{mode}_step_final_over_rollout_final"] = (res[f"{mode}_step_final"]["us_per_step_median_of_runs"]
                                                        / res[f"{mode}_rollout_final"]["us_per_step_median_of_runs"])
    tag = f"{'ref' if arm is REFERENCE_ARM else 'ur5'} x={x} horizon={horizon}"
    for w in WORKLOADS:
        print(f"{tag} {w:22s} {res[w]['us_per_step_median_of_runs']:8.2f} us/step (spread "
              f"{res[w]['run_to_run_spread_us']:.2f})  {res[w]['episodes_per_env_step']:.4f} episodes/env-step", flush=True)
    print(f"{tag} final/plain: actions {res['actions_final_over_rollout']:.4f}  draws {res['draws_final_over_rollout']:.4f}",
          flush=True)
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=64, help="K: steps per call (one call per timed region)")
    ap.add_argument("--regions", type=int, default=10, help="R: timed regions per run")
    ap.add_argument("--rounds", type=int, default=2, help="runs of every workload, alternating")
    ap.add_argument("--out", default=None, help="write the JSON here as well")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_rollout_final.py needs a CUDA device"
    result = {"gpu": gpu_info(), "n_envs": N, "steps_per_call": args.steps, "regions": args.regions,
              "rounds": args.rounds, "burn_in": BURN_IN, "obs_after_reset": True,
              "method": "one K-step call per CUDA-graph region, device events; action buffer refilled by a device copy "
                        "outside every timed region; workloads alternate on one handle per arm and horizon; median and "
                        "best region per run, median of runs and run-to-run spread",
              "arms": {}}
    for name, arm, x in (("reference_x10", REFERENCE_ARM, 10), ("ur5_x20", UR5_ARM, 20)):
        for horizon in (HORIZON, RESET_HEAVY_HORIZON):
            result["arms"][f"{name}_horizon{horizon}"] = run_arm(arm, x, horizon, args.steps, args.regions, args.rounds)
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({a: {w: round(v["us_per_step_median_of_runs"], 2) for w, v in r.items() if isinstance(v, dict)}
                      for a, r in result["arms"].items()}))


if __name__ == "__main__":
    main()
