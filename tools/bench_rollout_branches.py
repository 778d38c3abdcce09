"""Branch rollouts (mt_rollout_branches) against what a planner does without them.

    python tools/bench_rollout_branches.py [--regions R] [--rounds N] [--out FILE.json]

An open-loop planner scores C candidate action sequences of K steps from each of N envs.  Here N = 4096 sources x
C = 256 candidates = M = 2^20 branches, K in {16, 64}, for the reference arm at X = 10 and the UR5 preset at X = 20.  The
sources run under auto-reset with horizon 1000 and are burnt in for 200 random steps, so that they are spread over
their episodes.  Workloads, each timed as one eager call per region by device events (median of R regions, a run per
round, the workloads alternating):
  branches        rollout_branches(actions, src, gamma, write_obs=False): one launch
  branches_obs    the same with write_obs=True (obs2 of each branch's last step)
  today           what a user does without it, on a twin handle of M envs created once (auto_reset off):
                  get_state + get_points(zero_dead=False) of the sources, a torch gather by src, set_state + set_points
                  of the twin (each synchronises), rollout(actions, write_obs=False), then the first-done scan and
                  the discounted sum in torch
The two give identical (ret, length, done), asserted once per (arm, K) before timing.  The action buffer is the same
for every region: its 2^20 x K x 4J bytes (1 to 1.6 GB) are far beyond the 126 MB L2.  The GPU's name and power limit
are read (nvidia-smi, read-only) in the same run.
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
from manytor_b200 import REFERENCE_ARM, UR5_ARM, BatchedEnvs, Branches  # noqa: E402

N_SRC, C = 4096, 256
M = N_SRC * C
HORIZON, BURN_IN, GAMMA = 1000, 200, 0.99
WORKLOADS = ("branches", "branches_obs", "today")


def today(env, twin, src, actions, gamma):
    """The per-branch answer without mt_rollout_branches: copy the sources into a twin, roll it, scan the slices."""
    st = env.get_state()
    pts = env.get_points(zero_dead=False)
    twin.set_state(goals=st["goals"][src], alive=st["alive"][src], total_reward=st["total_reward"][src],
                   ep_len=st["ep_len"][src])
    twin.set_points(pts[src])
    traj = twin.rollout(actions, write_obs=False)
    k = actions.shape[0]
    steps = torch.arange(k, device="cuda")[:, None]
    first = torch.where(traj.done != 0, steps, k).min(dim=0).values
    length = torch.where(first < k, first + 1, k).to(torch.int32)
    rows = torch.arange(M, device="cuda")
    done = torch.where(first < k, traj.done[(length - 1).long(), rows], 0).to(torch.uint8)
    ret = torch.zeros(M, device="cuda")
    d = torch.ones((), device="cuda")
    g = torch.tensor(gamma, dtype=torch.float32, device="cuda")
    for s in range(k):
        ret = torch.where(s < length, ret + d * traj.reward[s], ret)
        d = d * g
    return ret, length, done


def timed(body, R):
    body()                                                # warm-up: kernel attributes, launch shapes
    torch.cuda.synchronize()
    out = []
    for _ in range(R):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        body()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return sorted(out)


def run_arm(arm, x, K, R, rounds):
    env = BatchedEnvs(N_SRC, x, arm=arm, device=0, auto_reset=True, horizon=HORIZON, seed=7)
    env.reset()
    env.rollout_random(BURN_IN, write_obs=False)
    twin = BatchedEnvs(M, x, arm=arm, device=0, auto_reset=False, horizon=HORIZON, seed=7)
    twin.reset()
    src = torch.arange(N_SRC, device="cuda").repeat_interleave(C)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    acts = torch.rand((K, M, env.j), device="cuda", generator=gen) * 360.0 - 180.0
    out = Branches(torch.empty(M, device="cuda"), torch.empty(M, dtype=torch.int32, device="cuda"),
                   torch.empty(M, dtype=torch.uint8, device="cuda"), None)
    out_obs = out._replace(obs=torch.empty((M, 3 * x), device="cuda"))
    got = env.rollout_branches(acts, src, gamma=GAMMA, out=out)
    ref = today(env, twin, src, acts, GAMMA)
    torch.cuda.synchronize()
    for u, v in zip(got[:3], ref):
        assert torch.equal(u.view(torch.int32) if u.dtype == torch.float32 else u,
                           v.view(torch.int32) if v.dtype == torch.float32 else v), "branches and today's path differ"
    ended = int((got.done != 0).sum())
    bodies = {"branches": lambda: env.rollout_branches(acts, src, gamma=GAMMA, out=out),
              "branches_obs": lambda: env.rollout_branches(acts, src, gamma=GAMMA, write_obs=True, out=out_obs),
              "today": lambda: today(env, twin, src, acts, GAMMA)}
    runs = {w: [] for w in WORKLOADS}
    for _ in range(rounds):
        for w in WORKLOADS:
            times = timed(bodies[w], R)
            runs[w].append({"ms_median": times[(len(times) - 1) // 2], "ms_best": times[0], "regions_ms": times})
    res = {"branches_ended": ended, "identical_to_today": True}
    for w, rs in runs.items():
        med = float(np.median([r["ms_median"] for r in rs]))
        res[w] = {"runs": rs, "ms_median_of_runs": med,
                  "run_to_run_spread_ms": max(r["ms_median"] for r in rs) - min(r["ms_median"] for r in rs),
                  "ps_per_branch_step": 1e9 * med / (M * K), "branch_steps_per_s": M * K / (med * 1e-3)}
    res["today_over_branches"] = res["today"]["ms_median_of_runs"] / res["branches"]["ms_median_of_runs"]
    res["obs_over_no_obs"] = res["branches_obs"]["ms_median_of_runs"] / res["branches"]["ms_median_of_runs"]
    tag = f"{'ref' if arm is REFERENCE_ARM else 'ur5'} x={x} K={K}"
    for w in WORKLOADS:
        print(f"{tag} {w:13s} {res[w]['ms_median_of_runs']:9.3f} ms/call  {res[w]['ps_per_branch_step']:8.1f} ps per "
              f"branch-step (spread {res[w]['run_to_run_spread_ms']:.3f} ms)", flush=True)
    print(f"{tag} today/branches {res['today_over_branches']:.2f}  obs/no-obs {res['obs_over_no_obs']:.3f}", flush=True)
    env.close()
    twin.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--regions", type=int, default=10, help="R: timed regions per run")
    ap.add_argument("--rounds", type=int, default=2, help="runs of every workload, alternating")
    ap.add_argument("--steps", type=int, nargs="+", default=[16, 64], help="K values")
    ap.add_argument("--out", default=None, help="write the JSON here as well")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_rollout_branches.py needs a CUDA device"
    result = {"gpu": gpu_info(), "sources": N_SRC, "candidates": C, "branches": M, "horizon": HORIZON,
              "burn_in": BURN_IN, "gamma": GAMMA, "regions": args.regions, "rounds": args.rounds,
              "method": "one eager call per region, device events; median and best region per run, median of runs and "
                        "run-to-run spread; workloads alternate on one source handle and one twin per arm and K",
              "arms": {}}
    for name, arm, x in (("reference_x10", REFERENCE_ARM, 10), ("ur5_x20", UR5_ARM, 20)):
        for K in args.steps:
            result["arms"][f"{name}_K{K}"] = run_arm(arm, x, K, args.regions, args.rounds)
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({a: {w: round(v["ps_per_branch_step"], 1) for w, v in r.items() if isinstance(v, dict)}
                      for a, r in result["arms"].items()}))


if __name__ == "__main__":
    main()
