"""fp32 against binary16 observations (mt_config.obs_dtype) on the workloads whose cost is the observations.

    python tools/bench_obs_dtype.py [--steps K] [--regions R] [--rounds N] [--out FILE.json]

Workloads, each timed like bench.py's headline (K steps per timed region as one K-node CUDA graph, R regions, median
and best region reported):
  step_ref_x10      mt_step, HBM actions, 2^20 envs, reference arm, X = 10, auto-reset, horizon 1000, after burn-in
  rollout_k64       mt_rollout_random(64) on the same handle shape: one launch of the multi-step rollout kernel
  host_staged       mt_step_host, 2^20 envs, staged through device buffers (MT_HOST_ZEROCOPY=0)
  host_zero_copy    mt_step_host, 2^20 envs, the kernel on the pinned buffers (MT_HOST_ZEROCOPY=1)
  step_ur5_x20      mt_step, HBM actions, 2^20 envs, UR5 preset, X = 20
mt_step_host is synchronous and cannot be captured: its regions are K calls timed by the host clock.

Formats alternate fp32, fp16, fp32, fp16, ... (--rounds pairs), with ONE handle alive at a time: handles in one
process share the 126 MB L2, so a second resident handle would change what is measured.  The spread of a format is
the difference between its runs' medians (run-to-run, same process).  GB/s is algorithmic: env-steps times
mt_bytes_per_env_step of the handle.  The GPU's name and power limit are read (nvidia-smi, read-only) in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from manytor_b200 import UR5_ARM, REFERENCE_ARM, BatchedEnvs  # noqa: E402

N = 1 << 20
HORIZON = 1000
BURN_IN = 200


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:                              # the measurement still stands; say what is missing
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({ex})"}


def make_env(arm, x, dtype, seed=7):
    env = BatchedEnvs(N, x, arm=arm, device=0, auto_reset=True, horizon=HORIZON, seed=seed, obs_dtype=dtype)
    env.reset()
    env.rollout_random(BURN_IN, write_obs=False)           # envs spread over their episodes
    torch.cuda.synchronize()
    return env


def graph_regions(env, body, K, R):
    """R timed replays of one K-step CUDA graph (device events), after warm-up; ms per region, sorted."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        body(3)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        body(K)
    g.replay()                                            # the first replay uploads the graph
    torch.cuda.synchronize()
    out = []
    for _ in range(R):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return sorted(out)


def run_step(arm, x, dtype, K, R):
    env = make_env(arm, x, dtype)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(11)
    acts = [torch.randint(-180, 180, (N, arm.n_joints), device="cuda", generator=gen).float() for _ in range(K)]
    times = graph_regions(env, lambda k: [env.step(acts[i]) for i in range(k)], K, R)
    return times, env.bytes_per_env_step(True, True), env


def run_rollout(dtype, K, R):
    env = make_env(REFERENCE_ARM, 10, dtype)
    times = graph_regions(env, lambda k: env.rollout_random(k), K, R)
    return times, env.bytes_per_env_step(False, True), env


def run_host(zero_copy, dtype, K, R):
    os.environ["MT_HOST_ZEROCOPY"] = "1" if zero_copy else "0"   # read at the handle's first step_host
    try:
        env = make_env(REFERENCE_ARM, 10, dtype)
        rs = np.random.RandomState(5)
        acts = [env.pinned(f"a{i}", (N, 4), np.float32) for i in range(4)]
        for a in acts:
            a[:] = rs.randint(-180, 180, size=a.shape)
        for i in range(8):                                # warm-up: allocations, first touch
            env.step_host(acts[i % 4])
        assert env.host_step_mode == ("zero-copy" if zero_copy else "staged")
        out = []
        for _ in range(R):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(K):
                env.step_host(acts[i % 4])                # synchronous
            out.append((time.perf_counter() - t0) * 1e3)
        return sorted(out), env.bytes_per_env_step(True, True), env
    finally:
        os.environ.pop("MT_HOST_ZEROCOPY", None)


def entry(times, bytes_per, K, pcie_bytes=None):
    med, best = times[(len(times) - 1) // 2], times[0]
    e = {"us_per_step_median": 1e3 * med / K, "us_per_step_best": 1e3 * best / K,
         "env_steps_per_s": N * K / (med * 1e-3), "bytes_per_env_step": bytes_per,
         "algorithmic_gbs": N * K * bytes_per / (med * 1e-3) / 1e9, "regions_ms": times}
    if pcie_bytes is not None:
        e["pcie_bytes_per_env_step"] = pcie_bytes
        e["pcie_gbs"] = N * K * pcie_bytes / (med * 1e-3) / 1e9
    return e


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=100, help="K: steps per timed region (device workloads)")
    ap.add_argument("--host-steps", type=int, default=20, help="K of the mt_step_host workloads")
    ap.add_argument("--regions", type=int, default=10, help="R: timed regions per run")
    ap.add_argument("--rounds", type=int, default=2, help="fp32/fp16 pairs per workload")
    ap.add_argument("--out", default=None, help="write the JSON here as well")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_obs_dtype.py needs a CUDA device"
    K, R = args.steps, args.regions
    workloads = {
        "step_ref_x10": (K, lambda dt: run_step(REFERENCE_ARM, 10, dt, K, R), None),
        "rollout_k64": (64, lambda dt: run_rollout(dt, 64, R), None),
        "host_staged": (args.host_steps, lambda dt: run_host(False, dt, args.host_steps, R), True),
        "host_zero_copy": (args.host_steps, lambda dt: run_host(True, dt, args.host_steps, R), True),
        "step_ur5_x20": (K, lambda dt: run_step(UR5_ARM, 20, dt, K, R), None),
    }
    result = {"gpu": gpu_info(), "n_envs": N, "regions": R, "rounds": args.rounds,
              "method": "alternating fp32 / fp16 handles, one alive at a time; K-step CUDA graph per region "
                        "(host workloads: K synchronous calls, host clock); median and best region per run",
              "workloads": {}}
    for name, (k, run, host) in workloads.items():
        runs = {"fp32": [], "fp16": []}
        for _ in range(args.rounds):
            for label, dt in (("fp32", torch.float32), ("fp16", torch.float16)):
                times, b, env = run(dt)
                pcie = (4 * 4 + 3 * env.x * (2 if dt == torch.float16 else 4) + 5) if host else None
                runs[label].append(entry(times, b, k, pcie))
                env.close()
                del env
                torch.cuda.synchronize()
        w = {"steps_per_region": k}
        for label, rs in runs.items():
            meds = [r["us_per_step_median"] for r in rs]
            w[label] = {"runs": rs, "us_per_step_median_of_runs": float(np.median(meds)),
                        "run_to_run_spread_us": max(meds) - min(meds)}
        w["fp16_speedup"] = w["fp32"]["us_per_step_median_of_runs"] / w["fp16"]["us_per_step_median_of_runs"]
        result["workloads"][name] = w
        print(f"{name:15s} fp32 {w['fp32']['us_per_step_median_of_runs']:9.2f} us (spread {w['fp32']['run_to_run_spread_us']:.2f})"
              f"  fp16 {w['fp16']['us_per_step_median_of_runs']:9.2f} us (spread {w['fp16']['run_to_run_spread_us']:.2f})"
              f"  x{w['fp16_speedup']:.3f}", flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({k: {"fp32_us": v["fp32"]["us_per_step_median_of_runs"], "fp16_us": v["fp16"]["us_per_step_median_of_runs"],
                          "speedup": v["fp16_speedup"]} for k, v in result["workloads"].items()}))


if __name__ == "__main__":
    main()
