"""Branch rollouts with in-kernel draws (mt_rollout_branches_random) against a caller that materialises the draws.

    python tools/bench_rollout_branches_random.py [--regions R] [--rounds N] [--calls C] [--out FILE.json]

Random shooting: C = 256 candidates of K steps from each of 4096 sources (M = 2^20 branches), K in {16, 64}, for the
reference arm at X = 10 and the UR5 preset at X = 20, every action drawn from the environment's random policy (integer
degrees uniform on [-180, 180)).  Every path ends with the planner's choice: the best candidate per source by return
and its first action.  Paths:
  a_draws    rollout_branches(None, src, n_steps=K, draw_key=key) with a device key advanced by K per call (key.add_),
             argmax per source, branch_actions(best, key, 1)
  b_randint  what a caller does without draws: torch.randint(low, high, (K, M, J)).float() every call, then
             rollout_branches(actions, src), argmax per source, the first action gathered from the buffer
  c_fixed    b without the generation: rollout_branches on one fixed buffer (the kernel-only lower bound of b)
Monte-Carlo values: M = 2^20 playouts (256 per source) of K = 1000 steps, paths a and b, with
torch.cuda.max_memory_allocated over one call of each (the sources' own state excluded) -- the memory a path needs.
The sources run under auto-reset with horizon 1000 and are burnt in for 200 random steps, so that they are spread over
their episodes (playouts truncate at the horizon).  Before timing, once per (arm, K): path a's (ret, length, done) equal
rollout_branches fed the buffer branch_actions(arange(M), key, K) regenerates -- the c_fixed buffer.
Timing: C calls per region between two device events, median of R regions per run, a run of every path per round, the
paths alternating; per-path HBM footprints far beyond the 126 MB L2 (c's buffer is 2^20 x K x 4J bytes).  The GPU's name
and power limit are read (nvidia-smi, read-only) in the same run.
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
LOW, HIGH = -180, 180
SHOOTING = ("a_draws", "b_randint", "c_fixed")
PLAYOUTS = ("a_draws", "b_randint")


def source_handle(arm, x):
    env = BatchedEnvs(N_SRC, x, arm=arm, device=0, auto_reset=True, horizon=HORIZON, seed=7, action_low=LOW,
                      action_high=HIGH)
    env.reset()
    env.rollout_random(BURN_IN, write_obs=False)
    torch.cuda.synchronize()
    return env


def best_of(ret):
    """The best candidate of each source: a branch id."""
    return ret.view(N_SRC, C).argmax(dim=1) + torch.arange(N_SRC, device="cuda") * C


def timed(body, R, calls):
    body()                                                # warm-up: kernel attributes, launch shapes, allocator
    torch.cuda.synchronize()
    out = []
    for _ in range(R):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            body()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / calls)
    return sorted(out)


def peak_bytes(body):
    """Device memory one call allocates at its peak, beyond what was allocated before it."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    body()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def paths(env, src, K, key, out, fixed):
    j = env.j

    def a_draws():
        r = env.rollout_branches(None, src, gamma=GAMMA, out=out, n_steps=K, draw_key=key)
        first = env.branch_actions(best_of(r.ret), key, 1)
        key.add_(K)
        return first

    def b_randint():
        acts = torch.randint(LOW, HIGH, (K, M, j), device="cuda").float()
        r = env.rollout_branches(acts, src, gamma=GAMMA, out=out)
        return acts[0].index_select(0, best_of(r.ret))

    def c_fixed():
        r = env.rollout_branches(fixed, src, gamma=GAMMA, out=out)
        return fixed[0].index_select(0, best_of(r.ret))

    return {"a_draws": a_draws, "b_randint": b_randint, "c_fixed": c_fixed}


def assert_equivalent(env, src, K, key, out):
    """Path a's outputs equal rollout_branches fed the regenerated draws; returns that buffer and the ended count."""
    got = env.rollout_branches(None, src, gamma=GAMMA, out=out, n_steps=K, draw_key=key)
    got = [t.clone() for t in got[:3]]
    fixed = env.branch_actions(torch.arange(M, device="cuda"), key, K)
    want = env.rollout_branches(fixed, src, gamma=GAMMA)
    torch.cuda.synchronize()
    for u, v in zip(got, want[:3]):
        assert torch.equal(u.view(torch.int32) if u.dtype == torch.float32 else u,
                           v.view(torch.int32) if v.dtype == torch.float32 else v), "draws and fed draws differ"
    return fixed, int((got[2] != 0).sum()), float(got[1].float().mean())


def summarise(runs, K):
    res = {}
    for w, rs in runs.items():
        med = float(np.median([r["ms_median"] for r in rs]))
        res[w] = {"runs": rs, "ms_median_of_runs": med,
                  "run_to_run_spread_ms": max(r["ms_median"] for r in rs) - min(r["ms_median"] for r in rs),
                  "ps_per_branch_step": 1e9 * med / (M * K), "branch_steps_per_s": M * K / (med * 1e-3)}
    return res


def run_arm(arm, x, K, R, rounds, calls, workloads, tag):
    env = source_handle(arm, x)
    src = torch.arange(N_SRC, device="cuda").repeat_interleave(C)
    out = Branches(torch.empty(M, device="cuda"), torch.empty(M, dtype=torch.int32, device="cuda"),
                   torch.empty(M, dtype=torch.uint8, device="cuda"), None)
    key = torch.tensor([12345], dtype=torch.int64, device="cuda")
    fixed, ended, mean_len = assert_equivalent(env, src, K, key, out)
    bodies = paths(env, src, K, key, out, fixed)
    if "c_fixed" not in workloads:
        del fixed                                         # the playout shape: path a holds no K x M buffer
        bodies.pop("c_fixed")
    mem = {}
    for w in workloads:
        mem[w] = peak_bytes(bodies[w])
    runs = {w: [] for w in workloads}
    for _ in range(rounds):
        for w in workloads:
            times = timed(bodies[w], R, calls)
            runs[w].append({"ms_median": times[(len(times) - 1) // 2], "ms_best": times[0], "regions_ms": times})
    res = {"branches_ended": ended, "mean_length": mean_len, "identical_to_fed_draws": True, **summarise(runs, K)}
    for w in workloads:
        res[w]["peak_alloc_bytes_per_call"] = mem[w]
    a = res["a_draws"]["ms_median_of_runs"]
    res["b_over_a"] = res["b_randint"]["ms_median_of_runs"] / a
    if "c_fixed" in res:
        res["a_over_c"] = a / res["c_fixed"]["ms_median_of_runs"]
    res["memory_b_over_a"] = mem["b_randint"] / max(mem["a_draws"], 1)
    for w in workloads:
        print(f"{tag} {w:10s} {res[w]['ms_median_of_runs']:9.3f} ms/call  {res[w]['ps_per_branch_step']:7.1f} ps per "
              f"branch-step (spread {res[w]['run_to_run_spread_ms']:.3f} ms)  peak {mem[w] / 2 ** 20:9.1f} MiB", flush=True)
    print(f"{tag} b/a {res['b_over_a']:.3f}" + (f"  a/c {res['a_over_c']:.3f}" if "a_over_c" in res else ""), flush=True)
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--regions", type=int, default=10, help="R: timed regions per run")
    ap.add_argument("--rounds", type=int, default=2, help="runs of every path, alternating")
    ap.add_argument("--calls", type=int, default=4, help="calls per timed region (shooting; playouts take 1)")
    ap.add_argument("--steps", type=int, nargs="+", default=[16, 64], help="K values of the shooting workload")
    ap.add_argument("--playout-steps", type=int, default=1000, help="K of the Monte-Carlo workload (0: skip it)")
    ap.add_argument("--out", default=None, help="write the JSON here as well")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_rollout_branches_random.py needs a CUDA device"
    result = {"gpu": gpu_info(), "sources": N_SRC, "candidates": C, "branches": M, "horizon": HORIZON,
              "burn_in": BURN_IN, "gamma": GAMMA, "action_range": [LOW, HIGH], "regions": args.regions,
              "rounds": args.rounds, "calls_per_region": args.calls,
              "method": "device events around `calls` eager calls per region; median and best region per run, median "
                        "of runs and run-to-run spread; paths alternate on one source handle per arm and K; peak "
                        "allocation of one call by torch.cuda.max_memory_allocated",
              "shooting": {}, "playouts": {}}
    for name, arm, x in (("reference_x10", REFERENCE_ARM, 10), ("ur5_x20", UR5_ARM, 20)):
        for K in args.steps:
            result["shooting"][f"{name}_K{K}"] = run_arm(arm, x, K, args.regions, args.rounds, args.calls, SHOOTING,
                                                         f"shoot {name} K={K}")
            torch.cuda.empty_cache()
        if args.playout_steps:
            K = args.playout_steps
            result["playouts"][f"{name}_K{K}"] = run_arm(arm, x, K, max(3, args.regions // 2), args.rounds, 1,
                                                         PLAYOUTS, f"playout {name} K={K}")
            torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({kind: {a: {w: round(v["ps_per_branch_step"], 1) for w, v in r.items() if isinstance(v, dict)}
                             for a, r in result[kind].items()} for kind in ("shooting", "playouts")}))


if __name__ == "__main__":
    main()
