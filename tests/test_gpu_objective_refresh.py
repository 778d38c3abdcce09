"""The objectives the device draws on reset, value by value against their fp64 restatement (-m gpu).

`sample_point` (mt_step.cuh) maps one Philox4x32-10 block keyed by (seed, global env id, episode x 32 + objective)
onto the upper half ball.  `reset_kernel` calls it one thread per env; `settle_step` calls it inside every step
kernel and the multi-step rollout kernel, one lane per objective.  `oracle.philox.device_points` restates it in
fp64, which makes a run with on-device objectives a function of (seed, env id) alone: these tests follow the device
through any number of in-kernel resets with nothing uploaded.

  a. mt_reset's objectives against the restatement: objective counts of both point layouts (compile-time and
     run-time X), two seeds, two shard bases, three radii, episodes 0..2, masked resets and re-seeding.
  b. The in-kernel refresh of every kernel that calls settle_step, without the oracle: with catch_tol = 0 nothing
     is ever caught, so every episode ends exactly at the horizon and each env's episode index is known.
  c. Lock step with the fp64 oracle and nothing uploaded: per-step launches, in-kernel actions, multi-step rollouts.
  d. The benchmark's launch shape and seed.
  e. The benchmark's burn-in protocol over several horizons for envs of its shard.
"""
import dataclasses
import json
import os
import subprocess

import numpy as np
import pytest

from oracle import REFERENCE_ARM, UR5_ARM
from oracle.philox import device_actions, device_points

from parity import (ChunkedOracle, Report, _seed_late_episode, lockstep_auto_reset, lockstep_chunked, philox_fresh,
                    point_tol_of)

pytestmark = pytest.mark.gpu

SEED_HI = 0x1234567890ABCDEF               # both key words non-zero
BASE_RANK3 = 3 * (1 << 20) + 5             # the shard of rank 3 of a 2^20-env-per-GPU run, shifted off a tile boundary


@pytest.fixture(scope="module")
def mt():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import manytor_b200
    manytor_b200.load_library()
    return manytor_b200


def _ulp(radius) -> float:
    return float(np.spacing(np.float32(radius)))


def _card():
    """Name and power limit of the card the figures were measured on."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out


def _record(name, fig):
    """Print a case's figures as one JSON line, and write them to $MANYTOR_FIGURES_DIR/objective_refresh_<name>.json
    when that variable names a directory (how profiles/r3_parity_philox_refresh.json is collected)."""
    fig = dict(case=name, card=_card(), **fig)
    print("figures", json.dumps(fig))
    out = os.environ.get("MANYTOR_FIGURES_DIR")
    if not out:
        return
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, f"objective_refresh_{name}.json"), "w") as f:
            json.dump(fig, f)
    except OSError:
        pass


def _figures(rep: Report, stats, spec, dropped=0):
    return dict(env_steps=rep.env_steps, max_point_err_ulps_of_R=rep.max_point_err / _ulp(spec.radius),
                max_joint_err=rep.max_joint_err, max_dist_err=rep.max_dist_err,
                max_angle_err_over_allowed=rep.max_angle_excess, hard_mismatches=rep.hard_mismatch,
                near_threshold_flips=rep.near_threshold, dropped_envs=int(dropped), refreshes=stats["episodes"],
                terminations=stats["terminated"], truncations=stats["episodes"] - stats["terminated"],
                catches=stats["catches"], ground_steps=stats["ground_steps"])


# --------------------------------------------------------------------------
# a. mt_reset
# --------------------------------------------------------------------------
def _arm(mt, name):
    from arms import arm_pair
    return {"ref": (mt.REFERENCE_ARM, 0), "ur5": (mt.UR5_ARM, 0), "j5": (arm_pair(5)[1], 1)}[name]


@pytest.mark.parametrize("arm_name", ["ref", "ur5", "j5"])
@pytest.mark.parametrize("x", [1, 2, 7, 10, 20, 31, 32])
def test_reset_objectives_match_restatement(mt, x, arm_name):
    """reset_kernel's objectives are device_points of (seed, env_id_base + i, episode) within 4 fp32 ulps of R per
    component, through repeated resets, a masked reset (only the masked envs move on an episode) and set_seed (back
    to episode 0, bit for bit)."""
    arm, fk_mode = _arm(mt, arm_name)
    n = 1000 + 13
    tol = point_tol_of(arm)
    worst, pole, pole_worst = 0.0, 0, 0.0
    for seed in (0, SEED_HI):
        for base in (0, BASE_RANK3):
            env = mt.BatchedEnvs(n, x, arm=arm, device=0, seed=seed, env_id_base=base, fk_mode=fk_mode)
            ids = base + np.arange(n)
            cur = np.zeros(n, dtype=np.int64)         # episode of the objectives the env holds
            count = np.zeros(n, dtype=np.int64)       # resets so far

            def check(prev=None, moved=None):
                nonlocal worst, pole, pole_worst
                dev = env.get_points(zero_dead=False).cpu().numpy()
                want = device_points(seed, ids, cur, x, arm.radius)
                err = np.abs(dev.astype(np.float64) - want).max(axis=-1)
                worst = max(worst, float(err.max()))
                ct = want[..., 2] / np.maximum(np.linalg.norm(want, axis=-1), 1e-300)
                at_pole = ct > 1 - 1e-4
                pole += int(at_pole.sum())
                pole_worst = max(pole_worst, float(err[at_pole].max()) if at_pole.any() else 0.0)
                assert err.max() <= tol, (seed, base, float(err.max()) / _ulp(arm.radius))
                if prev is not None:
                    np.testing.assert_array_equal(dev[~moved], prev[~moved])
                return dev

            snaps = []
            for _ in range(3):                                           # episodes 0, 1, 2
                env.reset()
                cur[:] = count
                count += 1
                snaps.append(check())
            mask = np.random.RandomState(x).rand(n) < 0.5
            env.reset(mask=mask)
            cur[mask] = count[mask]
            count[mask] += 1
            check(snaps[-1], mask)
            assert len(set(cur.tolist())) == 2                           # neighbours at different episodes
            env.set_seed(seed)
            env.reset()
            cur[:] = 0
            np.testing.assert_array_equal(check(), snaps[0])
    print(f"reset x={x} {arm_name}: max point error {worst / _ulp(arm.radius):.2f} ulps of R; "
          f"{pole} points with cos(theta) > 1 - 1e-4, worst {pole_worst / _ulp(arm.radius):.2f} ulps")


# --------------------------------------------------------------------------
# b. in-kernel refresh, no oracle
# --------------------------------------------------------------------------
def _no_catch(arm):
    return dataclasses.replace(arm, catch_tol=0.0)


_REFRESH = [  # id, arm name, x, fk_mode, mode, k, write_obs
    ("step_ref_x10", "ref", 10, 0, "step", 1, True),          # step_kernel<0,10,0,1>, HBM actions
    ("step_ref_x7", "ref", 7, 0, "step", 1, True),            # run-time X, single-point layout
    ("step_ref_x32", "ref", 32, 0, "step", 1, True),          # run-time X, pair layout, every lane draws
    ("rand1_ref_x10", "ref", 10, 0, "rollout", 1, True),      # the RAND step kernel
    ("rollout8_ref_x10_obs", "ref", 10, 0, "rollout", 8, True),
    ("rollout8_ref_x10_noobs", "ref", 10, 0, "rollout", 8, False),
    ("step_ur5_x20", "ur5", 20, 0, "step", 1, True),          # the UR5 preset
    ("step_j5_fk1", "j5", 9, 1, "step", 1, True),             # run-time DH table
    ("step_j5_fk3", "j5", 9, 3, "step", 1, True),             # NVRTC step kernel
    ("rollout5_j5_fk3", "j5", 9, 3, "rollout", 5, True),      # NVRTC rollout kernel
    ("host_ref_x10", "ref", 10, 0, "host", 1, True),          # step_host
]


@pytest.mark.parametrize("case,arm_name,x,fk_mode,mode,k,write_obs", _REFRESH, ids=[c[0] for c in _REFRESH])
def test_in_kernel_refresh_matches_restatement(mt, case, arm_name, x, fk_mode, mode, k, write_obs):
    """With catch_tol = 0 every episode ends exactly at the horizon h.  ep_len staggered over [0, h) -- whole warps
    in step, and warps of mixed phase -- gives every warp 0 .. 32 ending lanes per step, and env i holds the
    objectives of episode (e0_i + t) // h after t steps.  After every call the envs that were reset must hold
    device_points of that episode, and all others their objectives bit for bit.  A second handle that reaches the
    same episodes by host resets (reset_kernel) must hold the same bits."""
    arm = _no_catch(_arm(mt, arm_name)[0])
    n, h, seed, base = 2048 + 17, 4, SEED_HI, BASE_RANK3
    kw = dict(arm=arm, device=0, seed=seed, env_id_base=base, fk_mode=fk_mode, auto_reset=True, horizon=h)
    env = mt.BatchedEnvs(n, x, **kw)
    env.reset()
    rs = np.random.RandomState(len(case))
    e0 = rs.randint(0, h, size=n)
    warp = np.arange(n) // 32
    lockstep_warps = warp % 3 == 0
    e0[lockstep_warps] = (warp[lockstep_warps] // 3) % h                 # all 32 lanes end at the same step
    env.set_state(ep_len=e0.astype(np.int32))
    ids = base + np.arange(n)
    tol = point_tol_of(arm)
    prev = env.get_points(zero_dead=False).cpu().numpy()
    prev_ep = np.zeros(n, dtype=np.int64)
    assert np.abs(prev - device_points(seed, ids, prev_ep, x, arm.radius)).max() <= tol
    worst, refreshes, t = 0.0, 0, 0
    per_warp = set()
    for c in range(2 * h + 1 if k == 1 else 3):
        if mode == "step":
            env.step(rs.randint(-180, 180, size=(n, arm.n_joints)).astype(np.float32))
        elif mode == "host":
            env.step_host(rs.randint(-180, 180, size=(n, arm.n_joints)).astype(np.float32))
        else:
            env.rollout_random(k, write_obs=write_obs)
        t += k
        ep = (e0 + t) // h
        moved = ep != prev_ep
        pts = env.get_points(zero_dead=False).cpu().numpy()
        np.testing.assert_array_equal(pts[~moved], prev[~moved], err_msg=f"call {c}: objectives of running envs")
        err = np.abs(pts[moved].astype(np.float64) - device_points(seed, ids[moved], ep[moved], x, arm.radius)).max()
        worst = max(worst, float(err))
        assert err <= tol, f"call {c}: refreshed objectives off by {err / _ulp(arm.radius):.2f} ulps of R"
        refreshes += int((ep - prev_ep).sum())
        per_warp |= set(np.bincount(warp, weights=moved).astype(int).tolist())
        prev, prev_ep = pts, ep
    st = env.get_state()
    np.testing.assert_array_equal(st["ep_len"].cpu().numpy(), (e0 + t) % h)
    s = env.stats()
    assert s["episodes"] == refreshes and s["terminated"] == 0 and s["catches"] == 0, s
    if k == 1:
        assert {0, 32} <= per_warp and len(per_warp) > 4, sorted(per_warp)
    # the same episodes reached by host resets: reset_kernel and settle_step inline the same function
    other = mt.BatchedEnvs(n, x, **kw)
    other.reset()
    for j in range(1, int(ep.max()) + 1):
        other.reset(mask=ep >= j)
    np.testing.assert_array_equal(other.get_points(zero_dead=False).cpu().numpy(), prev)
    print(f"refresh {case}: {refreshes} refreshes over {t} steps, max point error "
          f"{worst / _ulp(arm.radius):.2f} ulps of R, ending lanes per warp {min(per_warp)}..{max(per_warp)}")


# --------------------------------------------------------------------------
# c. lock step with the fp64 oracle, nothing uploaded
# --------------------------------------------------------------------------
def _pair(mt, name):
    from arms import arm_pair
    return {"ref": (REFERENCE_ARM, mt.REFERENCE_ARM), "ur5": (UR5_ARM, mt.UR5_ARM)}.get(name) or arm_pair(int(name[1:]))


def _philox_setup(mt, spec, arm, n, x, horizon, fk_mode, seed, base, oar, alive_p, rs):
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, seed=seed, env_id_base=base, fk_mode=fk_mode, auto_reset=True,
                         horizon=horizon, obs_after_reset=oar)
    env.reset()                                                          # episode 0, drawn on the device
    ids = base + np.arange(n)
    ora = ChunkedOracle(n, x, spec)
    ora.reset(points=np.float32(device_points(seed, ids, 0, x, spec.radius)).astype(np.float64))
    if alive_p is not None:
        _seed_late_episode(env, ora, rs, n, x, horizon, alive_p)
    return env, ora, philox_fresh(seed, ids, x, spec.radius)


def _check_lockstep(env, rep, stats, slack, forked, spec):
    s = env.stats()
    print(rep.summary(), f"point err {rep.max_point_err / _ulp(spec.radius):.2f} ulps of R;",
          "forked" if forked else "", "expected", stats, "device", s)
    assert rep.ok(), rep.notes[:5]
    assert rep.near_threshold <= max(4, int(rep.env_steps * 5e-6)), rep.summary()
    if not forked:
        for key, v in stats.items():
            assert abs(s[key] - v) <= (slack if key == "reward_sum" else 0), (key, s[key], v)
    assert stats["terminated"] > 0 and stats["episodes"] > stats["terminated"], \
        "the run must see terminations, truncations and refreshes"


_LOCKSTEP = [  # id, arm, x, fk_mode, mode (step | rand1 | chunk<k>), obs_after_reset, alive_p
    ("ref_step", "ref", 10, 0, "step", False, 0.1),
    ("ref_step_oar", "ref", 10, 0, "step", True, 0.1),
    ("ref_rand1", "ref", 10, 0, "rand1", False, 0.1),
    ("ref_rand1_oar", "ref", 10, 0, "rand1", True, 0.1),
    ("ref_rollout8", "ref", 10, 0, "chunk8", False, 0.1),
    ("ref_rollout8_oar", "ref", 10, 0, "chunk8", True, 0.1),
    ("ur5_step", "ur5", 20, 0, "step", False, 0.1),
    ("j3_fk1_step", "j3", 5, 1, "step", False, 0.2),
    ("j8_fk3_step", "j8", 32, 3, "step", True, 0.02),
    ("j8_fk3_rollout4", "j8", 32, 3, "chunk4", True, 0.02),
]


@pytest.mark.parametrize("case,arm_name,x,fk_mode,mode,oar,alive_p", _LOCKSTEP, ids=[c[0] for c in _LOCKSTEP])
def test_lockstep_with_on_device_objectives(mt, case, arm_name, x, fk_mode, mode, oar, alive_p):
    """The oracle follows the device through in-kernel resets with objectives from device_points only: ragged N,
    a seed with high bits, the shard of rank 3, late-episode seeding, all eight statistics words exactly."""
    spec, arm = _pair(mt, arm_name)
    n, horizon, seed, base = 4096 + 17, 12, SEED_HI, BASE_RANK3
    rs = np.random.RandomState(len(case) + x)
    env, ora, fresh = _philox_setup(mt, spec, arm, n, x, horizon, fk_mode, seed, base, oar, alive_p, rs)
    ids = base + np.arange(n)
    J = spec.n_joints
    if mode.startswith("chunk"):
        k = int(mode[5:])
        rep, stats, dropped = lockstep_chunked(env, ora, spec, fresh, seed, k, 32 // k, horizon)
        _check_lockstep(env, rep, stats, 0, dropped.any(), spec)
        _record(case, _figures(rep, stats, spec, dropped.sum()))
        return
    if mode == "rand1":
        s0 = env.step_index
        step, acts = (lambda a: env.rollout_random(1)), (lambda t: device_actions(seed, ids, s0 + t, J))
    else:
        step, acts = None, (lambda t: rs.randint(-180, 180, size=(n, J)))
    rep, stats, slack, forked = lockstep_auto_reset(env, ora, spec, None, acts, 30, horizon, fresh=fresh,
                                                    device_step=step)
    _check_lockstep(env, rep, stats, slack, forked, spec)
    _record(case, _figures(rep, stats, spec))


# --------------------------------------------------------------------------
# d. the benchmark's shape
# --------------------------------------------------------------------------
def test_benchmark_shape_with_on_device_objectives(mt):
    """2^20 envs, X = 10, horizon 1000, bench.py's seed: two steps of step_kernel<0,10,0,1> with HBM actions (8 tiles
    per warp) and one rollout_random(2) (rollout_kernel<0,10,1>), every env seeded late in its episode so that the
    launches terminate, truncate and refresh."""
    import bench
    n, x, horizon, seed = 1 << 20, bench.OBJ, bench.HORIZON, bench.SEED
    spec, arm = REFERENCE_ARM, mt.REFERENCE_ARM
    rs = np.random.RandomState(1000)
    env, ora, fresh = _philox_setup(mt, spec, arm, n, x, horizon, 0, seed, 0, False, 0.35, rs)
    episode = np.ones(n, dtype=np.int64)
    rep, stats, slack, forked = lockstep_auto_reset(env, ora, spec, None,
                                                    lambda t: rs.randint(-180, 180, size=(n, 4)), 2, horizon,
                                                    fresh=fresh, episode=episode)
    dropped = np.zeros(n, dtype=bool)
    if not forked:                                   # a done flip leaves the two sides at different episodes
        rep, more, dropped = lockstep_chunked(env, ora, spec, fresh, seed, 2, 1, horizon, rep=rep, episode=episode)
        for key in stats:
            stats[key] = more[key] if key == "live_reward_sum" else stats[key] + more[key]
    _check_lockstep(env, rep, stats, slack, forked or dropped.any(), spec)
    _record("bench_shape_2p20", _figures(rep, stats, spec, dropped.sum()))


# --------------------------------------------------------------------------
# e. the burn-in protocol over several horizons
# --------------------------------------------------------------------------
def test_burn_in_protocol_over_several_horizons(mt):
    """bench.py's seed, horizon 1000, in-kernel actions and objectives, for 2048 envs of its rank-0 shard (the same
    global ids, so the same streams): 2500 steps of rollout_random(1) against the oracle at every step, every env
    through at least two episode ends.  Catches per episode and the terminated fraction are compared exactly,
    through the statistics."""
    import bench
    n, x, horizon, seed, steps = 2048, bench.OBJ, bench.HORIZON, bench.SEED, 2500
    base = bench.ENVS_PER_GPU // 2 + 12345
    spec, arm = REFERENCE_ARM, mt.REFERENCE_ARM
    env, ora, fresh = _philox_setup(mt, spec, arm, n, x, horizon, 0, seed, base, False, None, None)
    ids = base + np.arange(n)
    s0 = env.step_index
    rep, stats, slack, forked = lockstep_auto_reset(env, ora, spec, None, lambda t: device_actions(seed, ids, s0 + t, 4),
                                                    steps, horizon, fresh=fresh,
                                                    device_step=lambda a: env.rollout_random(1))
    _check_lockstep(env, rep, stats, slack, forked, spec)
    assert not forked and stats["episodes"] >= 2 * n
    print(f"burn-in: catches per episode {stats['catches'] / stats['episodes']:.4f}, "
          f"terminated fraction {stats['terminated'] / stats['episodes']:.4f}")
    _record("burn_in_2048x2500", dict(_figures(rep, stats, spec), catches_per_episode=stats["catches"] / stats["episodes"],
                                       terminated_fraction=stats["terminated"] / stats["episodes"]))
