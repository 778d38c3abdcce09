"""Trajectory rollouts (mt_rollout, BatchedEnvs.rollout) against one mt_step / rollout_random(1) call per step.

Every case runs twin handles with the same configuration and seed.  Slice s of a trajectory must equal, bit for bit,
what the s-th of K consecutive per-step calls returned; afterwards the state, objectives, statistics and step index
of the twins must be identical.  Each case runs under in-kernel auto-reset with a short horizon, so that resets with
their on-device objective refresh happen inside the rollout.
"""
import math
import os

import numpy as np
import pytest

from arms import arm_pair
from parity import ChunkedOracle, Report, lockstep_auto_reset, philox_fresh

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    return torch


def _arm(name):
    import manytor_b200 as mt
    if name == "ref":
        return mt.REFERENCE_ARM, 0
    if name == "ur5":
        return mt.UR5_ARM, 0
    kind, J = name.split("_j")                         # "rt_j7": run-time table, "jit_j5": NVRTC
    return arm_pair(int(J))[1], (1 if kind == "rt" else 3)


def handle(n, x, arm="ref", horizon=6, seed=11, **kw):
    from manytor_b200 import BatchedEnvs
    spec, fk_mode = _arm(arm)
    kw.setdefault("fk_mode", fk_mode)
    env = BatchedEnvs(n, x, arm=spec, device=0, auto_reset=True, horizon=horizon, seed=seed, **kw)
    env.reset()
    return env


def caller_actions(k, n, j, seed):
    """Continuous degrees, some out of the action range, some more than 540 degrees from any pose."""
    rs = np.random.RandomState(seed)
    a = rs.uniform(-180.0, 180.0, size=(k, n, j))
    a[:, ::7] *= 3.0                                                     # out of range
    a[:, 3::11] += rs.choice([-1.0, 1.0], size=a[:, 3::11].shape) * 1500.0   # > 540 degrees from the pose
    return _torch().tensor(a, dtype=_torch().float32, device="cuda")


def assert_twins(a, b):
    torch = _torch()
    torch.cuda.synchronize()
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert torch.equal(a.get_points(zero_dead=False), b.get_points(zero_dead=False))
    assert a.stats() == b.stats()
    assert a.step_index == b.step_index


def assert_slices(traj, per_step):
    torch = _torch()
    obs, rew, done = per_step
    if traj.obs is None:
        assert obs is None
    else:
        assert torch.equal(traj.obs.view(torch.int16 if traj.obs.dtype == torch.float16 else torch.int32),
                           obs.view(torch.int16 if obs.dtype == torch.float16 else torch.int32))
    assert torch.equal(traj.reward, rew)
    assert torch.equal(traj.done, done)


def step_each(env, actions, write_obs=True):
    """K mt_step calls (on a 16-byte aligned copy of each step's actions, as mt_step requires); each call's outputs
    are copied before the next one reuses the buffers."""
    outs = [tuple(o.clone() if o is not None else None for o in env.step(actions[s].clone(), write_obs=write_obs))
            for s in range(actions.shape[0])]
    st = lambda i: _torch().stack([o[i] for o in outs]) if outs[0][i] is not None else None
    return st(0), st(1), st(2)


@pytest.fixture
def per_step_path(monkeypatch):
    def use(on):
        if on:
            monkeypatch.setenv("MT_ROLLOUT_PERSISTENT", "0")
        else:
            monkeypatch.delenv("MT_ROLLOUT_PERSISTENT", raising=False)
    return use


# --------------------------------------------------------------------------
# 1. the caller's actions: persistent == per-step path == mt_step
# --------------------------------------------------------------------------
_CALLER = [  # id, arm, x, n, kw, persistent kernel available
    ("ref_x10", "ref", 10, 150003, {}, True),
    ("ref_x7_oar", "ref", 7, 5000, dict(obs_after_reset=True), True),
    ("ref_x32", "ref", 32, 33, {}, True),
    ("ur5_x20", "ur5", 20, 90001, {}, True),
    ("jit_j5_x12", "jit_j5", 12, 20000, {}, True),
    ("arms_j2_x1_misaligned", "jit_j2", 1, 9001, dict(fk_mode=0), True),
    ("jit_j8_x32", "jit_j8", 32, 4099, {}, True),
    ("rt_j7_x10", "rt_j7", 10, 3001, {}, False),
    ("ref_f16_aligned", "ref", 10, 40960, dict(obs_dtype="float16"), True),
    ("ref_f16_misaligned", "ref", 10, 40963, dict(obs_dtype="float16"), True),
    ("ref_no_obs", "ref", 10, 50001, dict(write_obs=False), True),
]


@pytest.mark.parametrize("case,arm,x,n,kw,persistent", _CALLER, ids=[c[0] for c in _CALLER])
def test_caller_actions_match_mt_step(case, arm, x, n, kw, persistent, per_step_path):
    torch = _torch()
    kw = dict(kw)
    write_obs = kw.pop("write_obs", True)
    if "obs_dtype" in kw:
        kw["obs_dtype"] = getattr(torch, kw["obs_dtype"])
    k = 24
    a, b, c = (handle(n, x, arm, **kw) for _ in range(3))
    acts = caller_actions(k, n, a.j, seed=n + x)
    l0 = a.launch_count
    traj = a.rollout(acts, write_obs=write_obs)
    assert a.launch_count - l0 == (math.ceil(k / 4096) if persistent else k)
    assert traj.actions is acts and traj.reward.shape == (k, n) and traj.done.dtype == torch.uint8
    per_step_path(True)
    l0 = b.launch_count
    trb = b.rollout(acts, write_obs=write_obs)
    assert b.launch_count - l0 == k
    per_step_path(False)
    ref = step_each(c, acts, write_obs)
    torch.cuda.synchronize()
    assert_slices(traj, ref)
    assert_slices(trb, ref)
    assert int((traj.done != 0).sum()) > 0                   # resets happened inside the rollout
    assert_twins(a, c)
    assert_twins(b, c)


# --------------------------------------------------------------------------
# 2. in-kernel actions: slices == rollout_random(1), draws == mt_sample_actions == the fp64 restatement
# --------------------------------------------------------------------------
@pytest.mark.parametrize("table", ["on", "off"])
@pytest.mark.parametrize("path", ["persistent", "per_step"])
@pytest.mark.parametrize("arm,x,n", [("ref", 10, 30011), ("ur5", 20, 12000), ("jit_j5", 12, 5003)])
def test_in_kernel_actions(arm, x, n, path, table, per_step_path, monkeypatch):
    torch = _torch()
    from oracle.philox import device_actions
    if table == "off":
        monkeypatch.setenv("MT_ACTION_TABLE", "0")
    k, seed = 20, 0x1234_5678_9ABC
    a, b, c = (handle(n, x, arm, seed=seed) for _ in range(3))
    s0 = a.step_index
    per_step_path(path == "per_step")
    traj = a.rollout(n_steps=k, record_actions=True)
    per_step_path(False)
    plain = handle(n, x, arm, seed=seed).rollout(n_steps=k)                     # drawn_dev = NULL
    obs, rew, done, drawn = [], [], [], []
    for s in range(k):
        drawn.append(b.sample_actions().clone())
        o, r, d = b.rollout_random(1)
        obs.append(o.clone()); rew.append(r.clone()); done.append(d.clone())
    c.rollout_random(k)
    torch.cuda.synchronize()
    assert_slices(traj, (torch.stack(obs), torch.stack(rew), torch.stack(done)))
    assert_slices(plain, (torch.stack(obs), torch.stack(rew), torch.stack(done)))
    assert plain.actions is None
    assert torch.equal(traj.actions, torch.stack(drawn))
    ids = np.arange(n)
    for s in (0, 1, k - 1):
        np.testing.assert_array_equal(traj.actions[s].cpu().numpy(), device_actions(seed, ids, s0 + s, a.j))
    assert_twins(a, b)
    assert_twins(a, c)


# --------------------------------------------------------------------------
# 3. chunk boundary: the second launch's slices land at the right offsets
# --------------------------------------------------------------------------
def test_chunk_boundary(per_step_path):
    torch = _torch()
    n, x = 96, 10
    k = 4100
    a, b = handle(n, x, horizon=9), handle(n, x, horizon=9)
    acts = caller_actions(k, n, 4, seed=5)
    l0 = a.launch_count
    traj = a.rollout(acts)
    assert a.launch_count - l0 == 2
    per_step_path(True)
    ref = b.rollout(acts)
    assert_slices(traj, (ref.obs, ref.reward, ref.done))
    assert_twins(a, b)
    # in-kernel draws over 4097 steps: the last chunk is one step, taken by the step kernel
    per_step_path(False)
    k = 4097
    trd = a.rollout(n_steps=k, record_actions=True)
    per_step_path(True)
    refd = b.rollout(n_steps=k, record_actions=True)
    assert_slices(trd, (refd.obs, refd.reward, refd.done))
    assert torch.equal(trd.actions, refd.actions)
    assert_twins(a, b)


# --------------------------------------------------------------------------
# 4. past 4 GiB of observations: 64-bit slice offsets
# --------------------------------------------------------------------------
def test_trajectory_past_4_gib(per_step_path):
    torch = _torch()
    n, x, k = 1 << 20, 10, 36
    assert (k - 1) * n * 3 * x * 4 > 1 << 32
    acts = caller_actions(k, n, 4, seed=9)
    a = handle(n, x, horizon=1000)
    traj = a.rollout(acts)
    torch.cuda.synchronize()
    last = traj.obs[-4:].clone(), traj.reward[-4:].clone(), traj.done[-4:].clone()
    del traj
    torch.cuda.empty_cache()
    b = handle(n, x, horizon=1000)
    per_step_path(True)
    ref = b.rollout(acts)
    torch.cuda.synchronize()
    assert torch.equal(last[0], ref.obs[-4:]) and torch.equal(last[1], ref.reward[-4:]) and torch.equal(last[2], ref.done[-4:])
    assert_twins(a, b)


# --------------------------------------------------------------------------
# 5. guard bands around every trajectory buffer at ragged N
# --------------------------------------------------------------------------
def _guarded(shape, dtype, pad=4096):
    torch = _torch()
    nbytes = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
    raw = torch.full((nbytes + 2 * pad,), 0xA5, dtype=torch.uint8, device="cuda")
    return raw, raw[pad:pad + nbytes].view(dtype).view(shape), pad


@pytest.mark.parametrize("path", ["persistent", "per_step"])
@pytest.mark.parametrize("mode", ["actions", "draws"])
@pytest.mark.parametrize("dtype", ["float32", "float16"])
def test_guard_bands(dtype, mode, path, per_step_path):
    torch = _torch()
    from manytor_b200 import Trajectory
    n, x, k = 1003, 10, 9                                    # N X % 4 = 2: misaligned slices (the per-lane path)
    obs_dtype = getattr(torch, dtype)
    a, b = handle(n, x, obs_dtype=obs_dtype), handle(n, x, obs_dtype=obs_dtype)
    shapes = dict(obs=((k, n, 3 * x), obs_dtype), reward=((k, n), torch.float32), done=((k, n), torch.uint8),
                  actions=((k, n, 4), torch.float32))
    g = {name: _guarded(*spec) for name, spec in shapes.items()}
    acts = caller_actions(k, n, 4, seed=3) if mode == "actions" else None
    out = Trajectory(g["obs"][1], g["reward"][1], g["done"][1], g["actions"][1] if mode == "draws" else None)
    per_step_path(path == "per_step")
    traj = a.rollout(acts, n_steps=k, record_actions=mode == "draws", out=out)
    per_step_path(False)
    ref = b.rollout(acts, n_steps=k, record_actions=mode == "draws")
    torch.cuda.synchronize()
    for name, (raw, view, pad) in g.items():
        if name == "actions" and mode == "actions":
            continue
        assert bool((raw[:pad] == 0xA5).all()) and bool((raw[-pad:] == 0xA5).all()), f"{name}: guard band written"
    assert_slices(traj, (ref.obs, ref.reward, ref.done))
    if mode == "draws":
        assert torch.equal(traj.actions, ref.actions)
    assert_twins(a, b)


# --------------------------------------------------------------------------
# 6. a captured rollout replayed with refilled actions
# --------------------------------------------------------------------------
def test_cuda_graph_replay():
    torch = _torch()
    from manytor_b200 import Trajectory
    n, x, k = 20000, 10, 16
    a, b = handle(n, x), handle(n, x)
    acts = caller_actions(k, n, 4, seed=1)
    out = Trajectory(torch.empty((k, n, 3 * x), device="cuda"), torch.empty((k, n), device="cuda"),
                     torch.empty((k, n), dtype=torch.uint8, device="cuda"), None)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                          # warm-up: kernel attributes and launch shapes
        a.rollout(acts, out=out)
    torch.cuda.current_stream().wait_stream(side)
    b.rollout(acts)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        a.rollout(acts, out=out)
    for r in range(3):
        acts.copy_(caller_actions(k, n, 4, seed=100 + r))
        idx = a.step_index
        graph.replay()
        ref = b.rollout(acts)
        torch.cuda.synchronize()
        assert_slices(out, (ref.obs, ref.reward, ref.done))
        assert a.step_index == idx + k
        assert_twins(a, b)


# --------------------------------------------------------------------------
# 7. oracle parity: every slice of a 64-step trajectory of continuous caller actions
# --------------------------------------------------------------------------
def test_oracle_parity_of_every_slice():
    torch = _torch()
    import manytor_b200 as mt
    from oracle import REFERENCE_ARM
    from oracle.philox import device_points
    n, x, k, horizon, seed = 4096, 10, 64, 12, 0xBEEF
    a, b = handle(n, x, horizon=horizon, seed=seed), handle(n, x, horizon=horizon, seed=seed)
    ora = ChunkedOracle(n, x, REFERENCE_ARM)
    ora.reset(points=np.float32(device_points(seed, np.arange(n), 0, x, REFERENCE_ARM.radius)).astype(np.float64))
    rs = np.random.RandomState(2)
    acts = rs.uniform(-180.0, 180.0, size=(k, n, 4)).astype(np.float32)
    traj = a.rollout(acts)
    t = iter(range(k))

    def device_step(act):
        # the twin steps with mt_step (the state the lock-step loop reads back); what is compared is the slice
        s = next(t)
        o, r, d = b.step(act.astype(np.float32))
        assert_slices(type(traj)(traj.obs[s:s + 1], traj.reward[s:s + 1], traj.done[s:s + 1], None),
                      (o[None], r[None], d[None]))
        return traj.obs[s], traj.reward[s], traj.done[s]

    rep, stats, slack, forked = lockstep_auto_reset(b, ora, REFERENCE_ARM, None, lambda s: acts[s], k, horizon,
                                                    rep=Report(), fresh=philox_fresh(seed, np.arange(n), x,
                                                                                     REFERENCE_ARM.radius),
                                                    device_step=device_step)
    print(rep.summary(), "forked" if forked else "")
    assert rep.ok(), rep.notes[:5]
    assert rep.hard_mismatch == 0
    assert forked or next(t, None) is None                  # every slice was compared unless a flip forked the run
