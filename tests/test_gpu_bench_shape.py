"""Oracle parity at the launch shape the benchmark times (-m gpu).

`launch_step` (mt_api.cu) gives a warp more than one tile only above 28 x 148 tiles = 132 608 envs
(16 x 148 tiles = 75 776 for the 16-warp generic kernels): below that every warp computes one tile and
the software pipeline of the step kernel -- next tile's scalars prefetched into registers, the second
objective buffer filled by TMA while the first is turned into observations, the tile queue in shared
memory, `sc = sn` -- never runs.  These tests put 2^18 .. 2^20 envs through the fp64 oracle
(manytor.py:175-260 restated, oracle/manytor_oracle.py) so that exactly that path is compared, with
in-kernel auto-reset + an uploaded objective stream, for the reference arm, the UR5 preset and an
NVRTC-specialised arm; and they check that one large handle equals many single-tile-per-warp handles bit
for bit.
"""
import json
import os

import numpy as np
import pytest

from oracle import ArmSpec as OArm, REFERENCE_ARM, UR5_ARM

from parity import ChunkedOracle, Report, _seed_late_episode, half_ball_points, lockstep_auto_reset

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def mt():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import manytor_b200
    manytor_b200.load_library()
    return manytor_b200


def _bench_shape_run(mt, n, x, steps, horizon, spec, arm, fk_mode, seed, scale=1.0, sets=3, alive_p=0.35):
    rs = np.random.RandomState(seed)
    stream = np.float32(half_ball_points(rs, (sets, n, x), radius=spec.radius)).astype(np.float64)
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, auto_reset=True, horizon=horizon, fk_mode=fk_mode, seed=seed)
    env.set_objective_stream(stream)
    env.reset()
    ora = ChunkedOracle(n, x, spec)
    ora.reset(points=stream[0])
    _seed_late_episode(env, ora, rs, n, x, horizon, alive_p)
    # objectives near the arm make catches (and therefore terminations) frequent enough to be seen in a few steps
    J = spec.n_joints
    rep, stats, slack, forked = lockstep_auto_reset(env, ora, spec, stream,
                                                    lambda t: rs.randint(-180, 180, size=(n, J)), steps, horizon,
                                                    check_points=True)
    s = env.stats()
    return rep, stats, slack, forked, s, ora


def _check(rep, stats, slack, forked, s, ora, n, steps):
    print(rep.summary(), "expected", stats, "device", s)
    assert rep.ok(), rep.notes[:5]
    assert rep.near_threshold <= max(4, int(rep.env_steps * 5e-6)), rep.summary()
    if not forked:
        assert rep.env_steps == n * steps
        for k, v in stats.items():
            assert abs(s[k] - v) <= (slack if k == "reward_sum" else 0), (k, s[k], v)
        assert s["live_reward_sum"] == int(ora.total_reward.sum())
    assert stats["episodes"] > 0 and stats["terminated"] > 0, "the run must exercise termination and truncation"


def _record(name, rep, n, steps, extra=None):
    """Leave the figures where the round's profiles are collected (gpurun_out/ travels back)."""
    try:
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        with open(os.path.join(ROOT, "gpurun_out", f"parity_bench_shape_{name}.json"), "w") as f:
            json.dump(dict(case=name, envs=n, steps=steps, env_steps=rep.env_steps, max_joint_err=rep.max_joint_err,
                           max_dist_err=rep.max_dist_err, max_angle_err_over_allowed=rep.max_angle_excess,
                           near_threshold_flips=rep.near_threshold, hard_mismatches=rep.hard_mismatch, **(extra or {})), f)
    except OSError:
        pass


@pytest.mark.parametrize("log2n,steps", [(19, 3), (20, 2)])
def test_reference_arm_at_benchmark_shape(mt, log2n, steps):
    """step_kernel<0,10,0,1>, one 28-warp block per SM, 4 (2^19) and 8 (2^20, the benchmark's size) tiles per
    warp: the pipelined path the bench times, against the oracle, through auto-reset."""
    n, x, horizon = 1 << log2n, 10, 50
    rep, stats, slack, forked, s, ora = _bench_shape_run(mt, n, x, steps, horizon, REFERENCE_ARM, mt.REFERENCE_ARM, 0,
                                                         seed=100 + log2n)
    _check(rep, stats, slack, forked, s, ora, n, steps)
    _record(f"ref_arm_2p{log2n}", rep, n, steps)


def test_ur5_preset_at_benchmark_shape(mt):
    """step_kernel<106,20,0,1> (config 5), 16-warp blocks: 2^18 envs = 8192 tiles = 3.5 tiles per warp."""
    n, x, steps, horizon = 1 << 18, 20, 2, 50
    rep, stats, slack, forked, s, ora = _bench_shape_run(mt, n, x, steps, horizon, UR5_ARM, mt.UR5_ARM, 0, seed=7)
    _check(rep, stats, slack, forked, s, ora, n, steps)
    _record("ur5_preset_2p18", rep, n, steps)


_CUSTOM_DH = ((0.0, np.pi / 2, 0.30, 0.0), (0.50, 0.0, 0.0, 0.2), (0.40, 0.3, 0.10, 0.0),
              (0.0, -np.pi / 2, 0.20, -np.pi / 2), (0.10, 0.0, 0.05, 0.0))


def test_nvrtc_arm_at_benchmark_shape(mt):
    """A user-supplied 5-joint table specialised at run time (fk_mode 3), multi-tile warps."""
    n, x, steps, horizon = 1 << 18, 12, 2, 50
    oarm = OArm(dh=_CUSTOM_DH, obs_frame=4, ground_frames=(4, 5), catch_frame=5, radius=0.9, catch_tol=0.15)
    arm = mt.ArmSpec(dh=_CUSTOM_DH, obs_frame=4, ground_frames=(4, 5), catch_frame=5, radius=0.9, catch_tol=0.15)
    rep, stats, slack, forked, s, ora = _bench_shape_run(mt, n, x, steps, horizon, oarm, arm, 3, seed=9)
    _check(rep, stats, slack, forked, s, ora, n, steps)
    _record("nvrtc_5joint_2p18", rep, n, steps)


@pytest.mark.parametrize("fk_mode", [3, 1])
def test_eight_joint_arm_at_benchmark_shape(mt, fk_mode):
    """The 8-joint table of tests/arms.py at X = 32 -- the largest tiles (12 KB per warp) of the 16-warp generic kernel,
    1.7 tiles per warp at 2^17 envs -- specialised at run time (fk_mode 3) and with the run-time table (fk_mode 1)."""
    from arms import arm_pair
    n, x, steps, horizon = 1 << 17, 32, 2, 50
    oarm, arm = arm_pair(8)
    # at X = 32 few envs are one catch from the end of their episode unless most objectives are already collected
    rep, stats, slack, forked, s, ora = _bench_shape_run(mt, n, x, steps, horizon, oarm, arm, fk_mode, seed=17,
                                                         alive_p=0.02)
    _check(rep, stats, slack, forked, s, ora, n, steps)
    _record(f"8joint_x32_fk{fk_mode}_2p17", rep, n, steps)


@pytest.mark.parametrize("rand", [True, False])
def test_one_large_handle_equals_many_small_ones(mt, rand):
    """2^18 envs in ONE handle (multi-tile warps, the tile queue, both objective buffers in turn) against
    the same envs in 64 handles of 4096 (one tile per warp, nothing pipelined): every output, the state,
    the objectives and the statistics must be bit-identical, through auto-reset with the on-device sampler."""
    import torch
    n, parts, x, k = 1 << 18, 64, 10, 18
    per = n // parts
    kw = dict(device=0, seed=77, auto_reset=True, horizon=5)
    whole = mt.BatchedEnvs(n, x, **kw)
    small = [mt.BatchedEnvs(per, x, env_id_base=i * per, **kw) for i in range(parts)]
    whole.reset()
    for p in small:
        p.reset()
    g = torch.Generator(device="cuda").manual_seed(5)
    for t in range(k):
        if rand:
            ow, rw, dw = whole.rollout_random(1)
            outs = [p.rollout_random(1) for p in small]
        else:
            a = torch.randint(-180, 180, (n, 4), device="cuda", generator=g).float()
            ow, rw, dw = whole.step(a)
            outs = [p.step(a[i * per:(i + 1) * per].contiguous()) for i, p in enumerate(small)]
        assert torch.equal(ow, torch.cat([o[0] for o in outs])), f"observations differ at step {t}"
        assert torch.equal(rw, torch.cat([o[1] for o in outs])) and torch.equal(dw, torch.cat([o[2] for o in outs]))
    sw = whole.get_state()
    ss = [p.get_state() for p in small]
    for key in sw:
        assert torch.equal(sw[key], torch.cat([q[key] for q in ss])), key
    assert torch.equal(whole.get_points(False), torch.cat([p.get_points(False) for p in small]))
    tw = whole.stats()
    ts = [p.stats() for p in small]
    for key in tw:
        assert tw[key] == sum(q[key] for q in ts), key
    assert tw["env_steps"] == n * k and tw["episodes"] >= n * (k // 5)


def test_bench_dump_outputs_are_reproducible(mt, tmp_path):
    """bench.py --dump-outputs: the outputs of the last timed step at the rows of bench.dump_sample -- equal to a replay
    of bench.py's seeded sequence through BatchedEnvs, identical in two runs whatever the wall-clock warm-up ran, and a
    different last step when --steps differs."""
    import subprocess
    import sys
    import torch
    import bench

    K, W, R, burn_in = 4, 3, 2, 300

    def run(name, steps, clock_warm_s):
        out = tmp_path / name
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(W),
               "--repeats", str(R), "--burn-in", str(burn_in), "--clock-warm-s", str(clock_warm_s), "--clock-probe-s", "0",
               "--clock-period-ms", "0", "--no-cpu", "--dump-outputs", str(out)]
        res = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp_path)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        files = sorted(p.name for p in out.iterdir())
        assert files == ["done.npy", "obs.npy", "reward.npy"], files
        assert sum((out / f).stat().st_size for f in files) <= 64 << 20
        return {f[:-4]: np.load(out / f) for f in files}, line

    (a, line), (b, _), (c, _) = run("a", K, 0.0), run("b", K, 0.5), run("c", K + 1, 0.0)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert not np.array_equal(a["obs"], c["obs"])

    # replay: re-seeded reset, burn-in, then the action buffers in bench.py's order -- with a CUDA graph, 3 steps while
    # capturing and one untimed replay of the K steps -- and per repeat a refill, W warm-up steps and the K timed steps
    n = bench.ENVS_PER_GPU
    env = mt.BatchedEnvs(n, bench.OBJ, device=0, horizon=bench.HORIZON, auto_reset=True, seed=bench.SEED)
    env.reset()
    env.set_seed(bench.SEED)
    env.reset()
    env.rollout_random(burn_in, write_obs=False)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(bench.SEED)
    actions = [torch.empty((n, 4), device="cuda", dtype=torch.float32) for _ in range(K + W)]

    def refill():
        for t in actions:
            t.copy_(torch.randint(-180, 180, (n, 4), device="cuda", generator=gen))

    refill()
    order = list(range(W, W + 3)) + list(range(W, W + K)) if line["config"]["submission"] == "one K-node CUDA graph" else []
    for r in range(R):
        if r:
            for i in order:
                out = env.step(actions[i])
            order = []
            refill()
        order += list(range(W + K))
    for i in order:
        out = env.step(actions[i])
    sel = torch.from_numpy(bench.dump_sample(n)).cuda()
    for name, t in zip(("obs", "reward", "done"), out):
        np.testing.assert_array_equal(a[name], t.index_select(0, sel).float().cpu().numpy(), err_msg=name)
    assert a["obs"].shape == (min(n, bench.DUMP_ENVS), 3 * bench.OBJ) and a["done"].any()
