#!/usr/bin/env python
"""Benchmark of the ManyTor step loop on B200 (contract: see the task README / DESIGN.md).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input: ONE
fused-kernel launch advancing every env of the shard by one env-step, actions
read from HBM, observations/reward/done written to HBM, on-device auto-reset with
objective refresh (BASELINE.json configs[2]: 4-joint arm, 2^20 envs per GPU, x=10,
1000-step horizon).  N>1 runs under torchrun, one rank per GPU, envs sharded
(weak scaling, 2^20 per GPU, configs[3]); the only collective is one all-reduce of
the episode statistics at the end of the timed region.

`--impl reference` times the reference's own CPU implementation on all host cores:
oracle/_ref (the unmodified reference, byte-compiled by oracle/make_ref.py in the
build container; it travels to the GPU box with the snapshot) in a test_multi.py
loop, or -- when that was never built -- the vectorised numpy port in oracle/.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 1 << 20
OBJ = 10
HORIZON = 1000
SEED = 20201
METRIC = "env-steps/s"
WORKLOAD = "4-joint reference arm, 2^20 envs per GPU, x=10 objectives, 1000-step horizon, on-device auto-reset + objective refresh (BASELINE configs[2]/[3])"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------
# clocks during the timed region
# ----------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, period_ms: int = 200):
        self.gpu, self.proc, self.lines, self.period_ms = gpu_index, None, [], int(period_ms)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", str(self.period_ms)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm_sorted = sorted(sm)
        return {"sm_mhz": sm_sorted[len(sm_sorted) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------
# CPU legs (the ONLY place bench.py touches oracle/)
# ----------------------------------------------------------------------------
def _oracle_worker_init(n_envs, x, seed):
    global _W
    import numpy as np
    from oracle import OracleEnvs
    rng = np.random.RandomState(seed)
    env = OracleEnvs(n_envs, x)
    v = rng.normal(size=(n_envs, x, 3))
    v /= np.linalg.norm(v, axis=-1, keepdims=True)
    v[..., 2] = np.abs(v[..., 2])
    env.reset(points=v * (51.3 * rng.uniform(size=(n_envs, x, 1)) ** (1 / 3)))
    _W = (env, rng)


def _oracle_worker_step(_):
    env, rng = _W
    import numpy as np
    r = env.step(rng.randint(-180, 180, size=(env.n, 4)))
    if r.done.any():                                   # refresh like test_single.py:20-21,32
        v = rng.normal(size=(env.n, env.x, 3))
        v /= np.linalg.norm(v, axis=-1, keepdims=True)
        v[..., 2] = np.abs(v[..., 2])
        env.reset(mask=r.done, points=v * (51.3 * rng.uniform(size=(env.n, env.x, 1)) ** (1 / 3)))
    return int(r.reward.sum())


REF_SHAPE = (8, 8)        # Multienv((8,8), 10): SURVEY.md section 8(d)(i)


def _ref_worker_init(seed):
    """One process = the reference's own Multienv (oracle/_ref: the unmodified manytor.py, byte-compiled)."""
    global _R
    import numpy as np
    from oracle import make_ref
    ref = make_ref.load()
    np.random.seed(seed)
    me = ref.Multienv(env_shape=REF_SHAPE, obj_number=OBJ)
    me.reset()
    _R = (me, [0])


def _ref_worker_step(_):
    me, count = _R
    me.step(me.action_sample())                        # test_multi.py:20-21
    count[0] += 1
    if count[0] % 50 == 0:                             # test_multi.py:8,34: max_steps = 50, then reset()
        me.reset()
    return me.env_number


def cpu_baseline_single_core(budget_s: float = 10.0) -> dict:
    """The CPU figures the metric string asks for, on ONE core of this box:
    (i) the unmodified reference's Multienv loop (oracle/_ref, test_multi.py shape) -- kind "reference";
    (ii) the vectorised fp64 numpy oracle at N = 4096 ("host numpy") and the scalar loop port."""
    import numpy as np
    from oracle import make_ref
    n = 4096
    _oracle_worker_init(n, OBJ, 1)
    _oracle_worker_step(0)
    t0, steps = time.perf_counter(), 0
    while time.perf_counter() - t0 < budget_s:
        _oracle_worker_step(0)
        steps += 1
    dt = time.perf_counter() - t0
    port = {"value": n * steps / dt, "sample": f"oracle/manytor_oracle.py (vectorised fp64 numpy restatement of manytor.py:175-260), "
            f"{n} envs x {steps} steps, x={OBJ}, random integer actions, {dt:.1f}s on 1 core"}
    out = None
    if make_ref.load() is not None:
        _ref_worker_init(0)
        t1, rsteps = time.perf_counter(), 0
        while time.perf_counter() - t1 < budget_s:
            _ref_worker_step(0)
            rsteps += 1
        dtr = time.perf_counter() - t1
        ne = REF_SHAPE[0] * REF_SHAPE[1]
        out = {"value": ne * rsteps / dtr, "unit": METRIC, "cores": 1, "kind": "reference",
               "sample": f"oracle/_ref (the unmodified reference, byte-compiled by oracle/make_ref.py): Multienv({REF_SHAPE}, {OBJ}), "
                         f"reset() every 50 steps, {rsteps} x step(action_sample()) as in test_multi.py:11-34, no render, {dtr:.1f}s on 1 core",
               "numpy_port_value": port["value"], "numpy_port_sample": port["sample"]}
    else:
        out = {"value": port["value"], "unit": METRIC, "cores": 1, "kind": "port", "sample": port["sample"],
               "note": "oracle/_ref not present on this box: the reference itself was not timed"}
    return out


def config1_latency(steps: int = 1000) -> dict:
    """BASELINE configs[0] through the drop-in: ONE env, x = 10, `steps` x step(action_sample()) via
    manytor_b200.manytor.Environment (reset on done, test_single.py:17-21) -- a latency figure, not throughput."""
    import manytor_b200.manytor as tor
    env = tor.Environment(OBJ, seed=SEED)
    env.reset()
    for _ in range(20):
        env.step(env.action_sample())
    t0 = time.perf_counter()
    for _ in range(steps):
        _, _, done = env.step(env.action_sample())
        if done:
            env.reset()
    dt = time.perf_counter() - t0
    return {"workload": "configs[0]: Environment(10), 1000 x step(action_sample()), reset on done", "steps": steps,
            "env_steps_per_s": steps / dt, "us_per_step": 1e6 * dt / steps,
            "note": "each iteration = action_sample() on the host (np.random, like the reference), then ONE mt_step_host call (upload, kernel, read-back) through ctypes; launch-latency bound"}


def run_reference_arm(args) -> None:
    """`--impl reference`: the reference's own CPU implementation of the path on all host cores --
    oracle/_ref (the unmodified reference) when it was built, else the numpy port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import make_ref
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    procs = max(1, min(cores, 64))
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    ctx = mp.get_context("fork")
    use_ref = make_ref.load() is not None and not args.reference_port
    if use_ref:
        per = REF_SHAPE[0] * REF_SHAPE[1]
        pools = [ctx.Pool(1, initializer=_ref_worker_init, initargs=(100 + i,)) for i in range(procs)]
        fn = _ref_worker_step
        kind = "reference"
        sample = (f"oracle/_ref (the unmodified reference, byte-compiled): {procs} processes x Multienv({REF_SHAPE}, {OBJ}) "
                  f"x {args.steps} steps of step(action_sample()) (test_multi.py:11-34, no render)")
    else:
        per = 4096
        pools = [ctx.Pool(1, initializer=_oracle_worker_init, initargs=(per, OBJ, 100 + i)) for i in range(procs)]
        fn = _oracle_worker_step
        kind = "port"
        sample = (f"oracle/manytor_oracle.py (vectorised fp64 numpy port of the reference step, pinned to the "
                  f"reference's golden traces), {procs} processes x {per} envs x {args.steps} steps, x={OBJ}")

    def step_all():
        rs = [p.apply_async(fn, (0,)) for p in pools]
        return [r.get() for r in rs]

    for _ in range(max(args.warmup, 1)):
        step_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_all()
    dt = time.perf_counter() - t0
    for p in pools:
        p.terminate()
    value = procs * per * args.steps / dt
    line = {"impl": "reference", "impl_class": "cpu", "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "note": "CPU arm: each step = one env-step of a bounded sample "
                       f"({procs} x {per} envs) of the workload; throughput is per env-step, so the sample size does not enter the ratio"},
            "cpu_baseline": {"value": value, "unit": METRIC, "cores": procs, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _RESULT_LINE.append(json.dumps(line))


# ----------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------
DUMP_ENVS = 1 << 18       # 2^18 envs x (30 obs + reward + done) x 4 B = 32 MiB


def dump_sample(n: int):
    """The envs `--dump-outputs` writes: the same seeded sample of DUMP_ENVS of the n envs in every run, ascending."""
    import numpy as np
    return np.sort(np.random.RandomState(0).choice(n, size=min(n, DUMP_ENVS), replace=False))


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """`--dump-outputs`: write each output of the last timed step as out_dir/<name>.npy (float32), rows dump_sample(n),
    so that two builds can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    sel = torch.from_numpy(dump_sample(outputs["reward"].shape[0])).to(outputs["reward"].device)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, sel).float().cpu().numpy())


def run_gpu(args) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist
    import manytor_b200
    from manytor_b200 import BatchedEnvs, distributed as mtd

    rank, world, local = mtd.init_from_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    manytor_b200.load_library()
    cores = mtd.bind_to_gpu_numa(local) if world > 1 else None      # keep pinned buffers on the GPU's NUMA node

    n = ENVS_PER_GPU
    base = rank * n
    env = BatchedEnvs(n, OBJ, device=local, env_id_base=base, horizon=HORIZON, auto_reset=True, seed=SEED)
    env.reset()
    reducer = mtd.StatsReducer(dev)                   # N > 1: the library's own kernel over NVLink peer memory, else NCCL
    K, W, R = args.steps, max(args.warmup, 3), max(args.repeats, 1)
    stream = torch.cuda.current_stream(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED + rank)
    # One action buffer per timed AND per warm-up step, refilled with fresh uniform integer degrees before
    # every repeat: no env ever sees an action twice, i.e. the timed steps ARE a random-action rollout.
    n_buf = min(K + W, 2048)
    actions = [torch.empty((n, 4), device=dev, dtype=torch.float32) for _ in range(n_buf)]

    def refill():
        for a in actions:
            a.copy_(torch.randint(-180, 180, (n, 4), device=dev, generator=gen))

    def barrier():
        if world > 1:
            dist.barrier()

    def fence():
        torch.cuda.synchronize(); barrier(); torch.cuda.synchronize()

    # ---- steady state: clock warm-up, then burn-in with in-kernel random actions (never cycled) ---------
    t_warm = time.perf_counter()
    while time.perf_counter() - t_warm < args.clock_warm_s:          # same kernel family, obs written: clocks/power settle
        env.rollout_random(200, write_obs=True)
        torch.cuda.synchronize()
    # The warm-up ran for a wall-clock time, so it left the envs after a varying number of steps: start over
    # from the seed, so that the timed steps see the same state and actions in every run with the same arguments.
    env.set_seed(SEED)
    env.reset()
    env.clear_stats()
    env.rollout_random(args.burn_in, write_obs=False)
    refill()
    torch.cuda.synchronize()

    last = []                                         # outputs of the latest step (buffers every step rewrites)

    def step_fn(i):
        last[:] = env.step(actions[i % n_buf])

    def capture(body):
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(stream)
            with torch.cuda.stream(side):
                body(True)
            stream.wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                body(False)
            return g
        except Exception as ex:
            print(f"bench: CUDA graph capture failed ({ex}); timing stream launches", file=sys.stderr)
            return None

    # The K timed steps are K launches of the step kernel either way; by default they are submitted as ONE
    # K-node CUDA graph (each node its own action buffer), which is how an RL loop that graphs policy + env
    # drives it and removes the ~3 us per-launch gap of stream launches from Python.
    graph = None if args.no_graph else capture(lambda warm: [step_fn(W + i) for i in range(3 if warm else K)])
    sampler = ClockSampler(local, args.clock_period_ms) if rank == 0 and args.clock_period_ms > 0 else None
    if sampler:
        sampler.start()

    def timed_region(replay, eager):
        """W warm-up steps, then EXACTLY K steps + the end-of-rollout statistics all-reduce, on the device clock."""
        for i in range(W):
            step_fn(i)
        fence()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        if replay is not None:
            replay.replay()
        else:
            eager()
        e1.record(stream)
        st = reducer.reduce(env)                      # end-of-rollout statistics + the one collective (config 4)
        e2.record(stream)
        fence()
        return e0.elapsed_time(e2), e0.elapsed_time(e1), st

    if graph is not None:
        graph.replay()                                # untimed: the first replay uploads the graph
        torch.cuda.synchronize()
    l0 = env.launch_count
    reps = []
    for r in range(R):
        if r:
            refill()                                  # fresh random actions for every repeat (untimed)
        ms_all, ms_k, st = timed_region(graph, lambda: [step_fn(W + i) for i in range(K)])
        reps.append((mtd.max_over_ranks(ms_all, dev), mtd.max_over_ranks(ms_k, dev)))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("obs", "reward", "done"), last)))   # before other modes overwrite them
    stats = mtd.stats_dict(st)                        # burn-in + warm-ups + every timed repeat, all ranks
    launches_timed = (K + 1) if graph is not None else (env.launch_count - l0) // R - W
    order = sorted(range(R), key=lambda i: reps[i][0])
    med = order[(R - 1) // 2]                         # the (lower) median repeat IS the reported run
    ms_total, ms_kernels = reps[med]
    best_total = reps[order[0]][0]

    # ---- SURVEY config-3 protocol: in-kernel RNG actions, same repeats ---------------------------------
    def rand_mode(write_obs, persistent):
        """K x step(action_sample()) with in-kernel actions: as K launches of the step kernel, or as ONE launch of the
        multi-step rollout kernel (a tile's state stays in registers, its objectives in shared memory, for all K steps)."""
        os.environ["MT_ROLLOUT_PERSISTENT"] = "1" if persistent else "0"
        try:
            g = None if args.no_graph else capture(lambda warm: env.rollout_random(3 if warm else K, write_obs=write_obs))
            if g is not None:
                g.replay()
            out = []
            for r in range(R):
                env.rollout_random(W, write_obs=write_obs)
                fence()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                if g is not None:
                    g.replay()
                else:
                    env.rollout_random(K, write_obs=write_obs)
                e1.record(stream)
                fence()
                out.append(mtd.max_over_ranks(e0.elapsed_time(e1), dev))
        finally:
            os.environ.pop("MT_ROLLOUT_PERSISTENT", None)
        out.sort()
        return out

    peak, peak_src = peaks()

    def mode_entry(times, bytes_per):
        med_ms, best_ms = times[(len(times) - 1) // 2], times[0]
        return {"env_steps_per_s": world * n * K / (med_ms * 1e-3), "best_env_steps_per_s": world * n * K / (best_ms * 1e-3),
                "us_per_step_median": 1e3 * med_ms / K, "us_per_step_best": 1e3 * best_ms / K, "repeats": len(times),
                "bytes_per_env_step": bytes_per, "hbm_gbs": n * K * bytes_per / (med_ms * 1e-3) / 1e9,
                "frac_of_peak": n * K * bytes_per / (med_ms * 1e-3) / 1e9 / peak}

    X3 = 12 * OBJ
    modes = {
        "rollout_random_in_kernel_actions": mode_entry(rand_mode(True, False), env.bytes_per_env_step(False, True)),
        "rollout_random_no_obs_write": mode_entry(rand_mode(False, False), env.bytes_per_env_step(False, False)),
        # one launch for all K steps: per env-step only the outputs leave the SM (obs 12X + reward 4 + done 1), the
        # state (24 B read + 24 B written) and the objectives (12X read) move once per K steps
        "rollout_random_one_launch": mode_entry(rand_mode(True, True), X3 + 5 + (48 + X3) / K),
        "rollout_random_one_launch_no_obs_write": mode_entry(rand_mode(False, True), 5 + (48 + X3) / K),
    }
    for name in ("rollout_random_one_launch", "rollout_random_one_launch_no_obs_write"):
        modes[name]["note"] = ("mt_rollout_random(K) as ONE launch of rollout_kernel; bound by instruction issue / the fp32 pipe, "
                               "not by HBM: frac_of_peak is its (small) algorithmic traffic over the HBM peak")
    # the same steps as individual stream launches from Python (no graph)
    for i in range(W):
        step_fn(i)
    fence()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(K):
        step_fn(W + i)
    e1.record(stream)
    fence()
    modes["step_hbm_actions_stream_launches"] = mode_entry([mtd.max_over_ranks(e0.elapsed_time(e1), dev)], env.bytes_per_env_step(True, True))

    # K steps last only a few ms, far below nvidia-smi's sampling period: keep the same load running
    # (untimed) so the clock sampler sees what the timed regions ran under
    t_cont = time.perf_counter()
    while sampler and time.perf_counter() - t_cont < args.clock_probe_s:
        for i in range(200):
            step_fn(i)
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["note"] = (f"sampled every {args.clock_period_ms} ms from just before the first timed repeat, through the {R} timed "
                          f"regions of {ms_total:.1f} ms and the other modes, and over a {args.clock_probe_s:.1f} s untimed continuation of the same step loop")

    value = world * n * K / (ms_total * 1e-3)
    B = env.bytes_per_env_step(True, True)
    kernel_ms = ms_kernels / K
    achieved = B * n / (kernel_ms * 1e-3) / 1e9

    # ---- e2e: host buffers through the public API (H2D actions, D2H obs/reward/done) ----
    rs = np.random.RandomState(rank)
    e2e_steps = max(3, min(K, 10))
    e2e_acts = []                                           # one page-locked action buffer per timed step: fresh random actions
    for i in range(e2e_steps):
        a = env.pinned(f"actions{i}", (n, 4), np.float32)
        a[:] = rs.randint(-180, 180, size=(n, 4))
        e2e_acts.append(a)
    for i in range(8):                                      # untimed: the handle times both host-step variants on its first 6 calls
        env.step_host(e2e_acts[i % e2e_steps])
    torch.cuda.synchronize(); barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        obs_h, rew_h, done_h = env.step_host(e2e_acts[i])     # synchronous: results are in host memory
    torch.cuda.synchronize(); barrier()
    e2e_s = mtd.max_over_ranks(time.perf_counter() - t0, dev)
    e2e_value = world * n * e2e_steps / e2e_s
    h2d = n * 4 * 4
    d2h = n * (3 * OBJ * 4 + 4 + 1)
    # what the link can carry: the same bytes as bare pinned-memory copies, all ranks at once
    d_buf = torch.empty(d2h, dtype=torch.uint8, device=dev)
    h_buf = torch.empty(d2h, dtype=torch.uint8).pin_memory()
    h_buf.copy_(d_buf, non_blocking=True)
    torch.cuda.synchronize(); barrier()
    t0 = time.perf_counter()
    for _ in range(5):
        h_buf.copy_(d_buf, non_blocking=True)
    torch.cuda.synchronize(); barrier()
    d2h_s = mtd.max_over_ranks(time.perf_counter() - t0, dev) / 5
    ceiling = world * n / d2h_s                                 # env-steps/s if a step were ONLY its D2H read-back

    if rank == 0:
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        cpu = cpu_baseline_single_core() if world == 1 and not args.no_cpu else None
        cfg1 = config1_latency() if world == 1 and not args.no_cpu else None
        eps = max(stats["episodes"], 1)
        line = {
            "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": n, "n_joints": 4, "n_obj": OBJ, "horizon": HORIZON,
                       "terminate_on_ground": False, "auto_reset": True,
                       "actions": f"uniform integer degrees in [-180,180), read from HBM [N][4] fp32; {n_buf} distinct buffers "
                                  "(one per warm-up and timed step), refilled before every repeat: no action is ever replayed",
                       "submission": "one K-node CUDA graph" if graph is not None else "K stream launches",
                       "burn_in": f"{args.clock_warm_s:.1f} s of in-kernel random-action steps (clocks), then re-seed + reset and {args.burn_in} in-kernel random-action steps before the first repeat (steady state of the episode process)",
                       "repeats": f"{R} timed regions of exactly K steps each (W warm-up steps before each); value = the median region, best reported beside it",
                       "l2": f"working set {(n * (B + 8 * 4)) / 2**20:.0f} MiB per step > 126 MiB L2 (inputs larger than L2, no flush needed)",
                       "parallelism": f"env-sharded x{world}, no per-step collective, 1 stats all-reduce inside the timed region "
                                      f"(a stats kernel + the exchange of 64 B, the only thing that grows with N); collective path: {reducer.path}"},
            "repeats": {"n": R, "ms_per_step_all": [t / K for t, _ in reps], "median_ms_per_step": ms_total / K,
                        "best_ms_per_step": best_total / K, "best_value": world * n * K / (best_total * 1e-3)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per launch in steady state (mean of 20 consecutive warm launches under ncu --cache-control none), committed in profiles/traffic.json with the cold isolated-launch figure beside it (a constant of the kernel, NOT measured in this run)",
                         "peak_source": peak_src, "kernel": "mt::step_kernel<0,10,false,true>",
                         "algorithmic_bytes_per_env_step": B, "kernel_ms_per_launch": kernel_ms,
                         "envs_per_launch": n,
                         # the algorithmic count includes the 48 B/env-step of per-env state that the kernel keeps in
                         # L2 from launch to launch, so `frac` can pass 1; this is the DRAM side on its own: the
                         # steady-state traffic (streamed arrays only, no re-reads) over this run's kernel time
                         "dram_achieved": (traffic / kernel_ms / 1e6) if traffic else None,
                         "dram_frac": (traffic / kernel_ms / 1e6 / peak) if traffic else None},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": METRIC, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "api": "BatchedEnvs.step_host -> mt_step_host (pinned host buffers; staged = 16 chunks over 4 streams, zero-copy = one launch on the host buffers; the handle keeps whichever its first calls timed faster)",
                    "host_step_mode": env.host_step_mode,
                    "cpu_binding": f"{len(cores)} cores next to the GPU (NVML affinity)" if cores else "none",
                    "d2h_only_ceiling": ceiling, "frac_of_d2h_ceiling": e2e_value / ceiling,
                    "ceiling_note": f"bare pinned D2H of the same {d2h} B per step on all {world} ranks at once: "
                                    f"{d2h / d2h_s / 1e9:.1f} GB/s per GPU"},
            "gpu_launches": launches_timed,
            "clocks": clocks,
            "modes": modes,
            "config1_single_env": cfg1,
            "episode_stats": dict(stats, window="burn-in + warm-ups + all timed repeats (statistics cleared after reset)",
                                  terminated_fraction=stats["terminated"] / eps, catches_per_episode=stats["catches"] / eps,
                                  mean_episode_length=stats["length_sum"] / eps,
                                  ground_rate=stats["ground_steps"] / max(stats["env_steps"], 1)),
        }
        _RESULT_LINE.append(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_RESULT_LINE = []      # the one JSON line, printed by main() after stdout has been restored


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--clock-warm-s", type=float, default=1.0, help="untimed seconds of the step loop before warm-up")
    ap.add_argument("--clock-probe-s", type=float, default=1.0, help="untimed continuation for the clock sampler")
    ap.add_argument("--clock-period-ms", type=int, default=200, help="nvidia-smi sampling period (0 = no sampler)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="time K stream launches instead of one K-node CUDA graph")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--repeats", type=int, default=10, help="timed regions of K steps each; value = median, best beside it")
    ap.add_argument("--reference-port", action="store_true", help="--impl reference: time the numpy port even when oracle/_ref exists")
    # 20 horizons: episodes end at random steps (all objectives caught), so the wave of truncations that the common
    # start at step 0 sends every horizon has died out before the timed steps
    ap.add_argument("--burn-in", type=int, default=20 * HORIZON,
                    help="untimed random-action steps after the clock warm-up and the re-seeded reset, before the "
                         "warm-up steps of the first repeat, so that episodes reach their steady state")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's obs, reward and done (rank 0, a fixed sample "
                         f"of {DUMP_ENVS} envs) as DIR/<name>.npy in float32")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    # stdout carries exactly ONE line, the JSON result: anything a library writes to file descriptor 1 on the
    # way (NCCL prints its version there when the box sets NCCL_DEBUG) is sent to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        if args.impl == "reference":
            run_reference_arm(args)
        else:
            run_gpu(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if _RESULT_LINE:
        print(_RESULT_LINE[-1], flush=True)


if __name__ == "__main__":
    main()
