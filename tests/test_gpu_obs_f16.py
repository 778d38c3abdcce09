"""Binary16 observations (mt_config.obs_dtype = MT_OBS_F16) against a twin fp32 handle.

The twin has the same configuration and seed and is driven with the same actions, so every fp16 observation must be
the fp32 one rounded to nearest even, bit for bit (`obs32.half()`), and everything else -- rewards, done flags, the
full state, the objectives, the step index and all eight statistics words -- must be identical.  The fp32 path is
checked against the fp64 oracle elsewhere; this pins the new format to it exactly.

Below 132 608 envs every warp of the step kernel computes one tile and its software pipeline never runs, so the
benchmark shapes are covered too (2^20 envs of the reference arm, the 16-warp single-buffer UR5 shape, the rollout
kernel at 2^20).
"""
import ctypes as C
import types

import numpy as np
import pytest

from arms import arm_pair
from parity import _seed_late_episode

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
    kind, J = name.split("_j")                         # "rt_j5": run-time table, "jit_j5": NVRTC
    return arm_pair(int(J))[1], (1 if kind == "rt" else 3)


def twins(n, x, arm="ref", **kw):
    """An fp32 and an fp16 handle with the same configuration and seed, both reset."""
    torch = _torch()
    from manytor_b200 import BatchedEnvs
    spec, fk_mode = _arm(arm)
    kw.setdefault("fk_mode", fk_mode)
    a = BatchedEnvs(n, x, arm=spec, device=0, obs_dtype=torch.float32, **kw)
    b = BatchedEnvs(n, x, arm=spec, device=0, obs_dtype=torch.float16, **kw)
    a.reset()
    b.reset()
    return a, b


def assert_obs_twin(o32, o16):
    torch = _torch()
    assert o32.dtype == torch.float32 and o16.dtype == torch.float16 and o16.shape == o32.shape
    want = o32.half().view(torch.int16)
    got = o16.view(torch.int16)
    bad = int((want != got).sum())
    assert bad == 0, f"{bad} fp16 observations differ from the fp32 twin's rounded to nearest even"


def assert_same(t32, t16):
    torch = _torch()
    assert torch.equal(t32, t16)


def assert_state_twin(a, b):
    torch = _torch()
    torch.cuda.synchronize()
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert torch.equal(a.get_points(zero_dead=False), b.get_points(zero_dead=False))
    assert a.step_index == b.step_index
    assert a.stats() == b.stats()


def actions_for(n, j, rs, fractional):
    act = rs.randint(-180, 180, size=(n, j)).astype(np.float32)
    if fractional:
        act += rs.rand(n, j).astype(np.float32)
    return act


def step_twins(a, b, act):
    torch = _torch()
    t = torch.from_numpy(act).cuda()
    o32, r32, d32 = (v.clone() for v in a.step(t))
    o16, r16, d16 = b.step(t)
    assert_obs_twin(o32, o16)
    assert_same(r32, r16)
    assert_same(d32, d16)


# ---- per-step mt_step --------------------------------------------------------------------------------------------
ARM_CASES = [("ref", 10), ("ref", 20), ("ref", 1), ("ref", 7), ("ref", 32), ("ur5", 10),
             ("rt_j5", 10), ("jit_j5", 10), ("jit_j8", 7)]


@pytest.mark.parametrize("obs_after_reset", [0, 1])
@pytest.mark.parametrize("n", [1, 31, 33, 257, 4097])
@pytest.mark.parametrize("arm,x", ARM_CASES)
def test_step_matches_fp32_twin(arm, x, n, obs_after_reset):
    a, b = twins(n, x, arm, auto_reset=True, horizon=3, obs_after_reset=bool(obs_after_reset), seed=n + x)
    rs = np.random.RandomState(n * 7 + x)
    for i in range(8):                                    # integer and fractional actions; resets every 3 steps
        step_twins(a, b, actions_for(n, a.j, rs, fractional=i % 2 == 1))
    assert_state_twin(a, b)
    assert a.stats()["episodes"] >= n


# ---- in-kernel actions ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [33, 4097])
@pytest.mark.parametrize("arm,x", [("ref", 10), ("ref", 7), ("ur5", 20), ("jit_j5", 10), ("rt_j5", 10)])
def test_rollout_random_matches_fp32_twin(arm, x, n):
    """rollout_random(1) (step kernel), rollout_random(K >= 2) (multi-step rollout kernel; per-step launches for the
    run-time table)."""
    a, b = twins(n, x, arm, auto_reset=True, horizon=4, obs_after_reset=True, seed=5)
    for k in (1, 5, 2, 7):
        o32, r32, d32 = (v.clone() for v in a.rollout_random(k))
        o16, r16, d16 = b.rollout_random(k)
        assert_obs_twin(o32, o16)
        assert_same(r32, r16)
        assert_same(d32, d16)
    assert_state_twin(a, b)
    assert a.stats()["episodes"] >= n


# ---- read-back and the Gymnasium adapter --------------------------------------------------------------------------------
def test_observe_and_returnable_reset():
    torch = _torch()
    a, b = twins(1000, 10, "ref", seed=3)
    assert_obs_twin(a.reset(returnable=True).clone(), b.reset(returnable=True))
    rs = np.random.RandomState(0)
    for _ in range(3):
        step_twins(a, b, actions_for(1000, 4, rs, fractional=True))
        assert_obs_twin(a.observe(), b.observe())
        out = torch.empty((1000, 30), dtype=torch.float16, device="cuda")
        assert b.observe(out=out) is out
        assert_obs_twin(a.observe(), out)
    with pytest.raises(ValueError):
        b.observe(out=torch.empty((1000, 30), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        a.observe(out=torch.empty((1000, 30), dtype=torch.float16, device="cuda"))


def test_vector_env_returns_fp16():
    torch = _torch()
    from manytor_b200 import ManyTorVectorEnv
    va = ManyTorVectorEnv(777, 10, max_episode_steps=5, device=0, seed=9)
    vb = ManyTorVectorEnv(777, 10, max_episode_steps=5, device=0, seed=9, obs_dtype=torch.float16)
    oa, _ = va.reset(seed=4)
    ob, _ = vb.reset(seed=4)
    assert_obs_twin(oa.clone(), ob)
    for _ in range(12):
        act = va.sample_actions()
        assert torch.equal(act, vb.sample_actions())
        oa, ra, ta, ua, _ = va.step(act)
        oa = oa.clone()
        ob, rb, tb, ub, _ = vb.step(act)
        assert_obs_twin(oa, ob)
        assert torch.equal(ra, rb) and torch.equal(ta, tb) and torch.equal(ua, ub)
    assert va.episode_statistics() == vb.episode_statistics()


# ---- host path -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("write_obs", [True, False])
@pytest.mark.parametrize("zero_copy", ["0", "1"])
def test_step_host_matches_fp32_twin(zero_copy, write_obs, monkeypatch):
    monkeypatch.setenv("MT_HOST_ZEROCOPY", zero_copy)       # read at a handle's first step_host
    n = 3000
    a, b = twins(n, 10, "ref", auto_reset=True, horizon=5, seed=2)
    rs = np.random.RandomState(1)
    for i in range(8):
        act = actions_for(n, 4, rs, fractional=i % 2 == 1)
        oa, ra, da = (None if v is None else v.copy() for v in a.step_host(act, write_obs=write_obs))
        ob, rb, db = b.step_host(act, write_obs=write_obs)
        if write_obs:
            assert oa.dtype == np.float32 and ob.dtype == np.float16 and ob.shape == oa.shape
            np.testing.assert_array_equal(oa.astype(np.float16).view(np.uint16), ob.view(np.uint16))
        else:
            assert oa is None and ob is None
        np.testing.assert_array_equal(ra, rb)
        np.testing.assert_array_equal(da, db)
    assert b.host_step_mode == {"0": "staged", "1": "zero-copy"}[zero_copy]
    assert_state_twin(a, b)


# ---- the benchmark shapes ------------------------------------------------------------------------------------------------
def _late_twins(n, x, arm, horizon, seed):
    a, b = twins(n, x, arm, auto_reset=True, horizon=horizon, seed=seed)
    for env in (a, b):                                    # the same late-episode state in both
        stub = types.SimpleNamespace(spec=types.SimpleNamespace(n_joints=env.j), bounds=(), parts=())
        _seed_late_episode(env, stub, np.random.RandomState(seed), n, x, horizon)
    return a, b


def test_benchmark_shape_reference_arm():
    """2^20 envs, X = 10, horizon 1000 (8 tiles per warp: the two-buffer pipeline runs), seeded late in their episodes."""
    a, b = _late_twins(1 << 20, 10, "ref", 1000, seed=20)
    rs = np.random.RandomState(2)
    for i in range(3):
        step_twins(a, b, actions_for(1 << 20, 4, rs, fractional=i == 1))
    assert_state_twin(a, b)
    assert a.stats()["episodes"] > 1000


def test_benchmark_shape_ur5_single_buffer():
    """UR5 preset at X = 20: 16-warp blocks with one tile buffer per warp, 163 840 envs = 2.2 tiles per warp."""
    n = 163840
    a, b = _late_twins(n, 20, "ur5", 40, seed=21)
    rs = np.random.RandomState(3)
    for i in range(3):
        step_twins(a, b, actions_for(n, 6, rs, fractional=i == 1))
    assert_state_twin(a, b)
    assert a.stats()["episodes"] > 100


def test_benchmark_shape_rollout_kernel():
    a, b = _late_twins(1 << 20, 10, "ref", 1000, seed=22)
    for k in (3, 2):
        o32, r32, d32 = (v.clone() for v in a.rollout_random(k))
        o16, r16, d16 = b.rollout_random(k)
        assert_obs_twin(o32, o16)
        assert_same(r32, r16)
        assert_same(d32, d16)
    assert_state_twin(a, b)
    assert a.stats()["episodes"] > 1000


# ---- raw C calls into sentinel-filled allocations -------------------------------------------------------------------------
G = 4096                                                  # guard elements on each side (16-byte multiples)
SENT16 = 0x7E55                                           # a NaN bit pattern no observation has


def _guarded(count, dtype, fill):
    torch = _torch()
    t = torch.full((count + 2 * G,), fill, dtype=dtype, device="cuda")
    return t, t[G:G + count]


def _check_guarded(whole, inner, fill):
    torch = _torch()
    torch.cuda.synchronize()
    assert bool((whole[:G] == fill).all()) and bool((whole[-G:] == fill).all()), "write outside the buffer"
    assert bool((inner != fill).all()), "element left unwritten"


@pytest.mark.parametrize("first", ["f32", "f16"])
@pytest.mark.parametrize("J", [5, 8])
def test_nvrtc_cache_keeps_formats_apart(J, first):
    """Two NVRTC handles with the same DH table in one process, one per format: each kernel writes its own format
    (a shared cache entry would write fp32 rows into the fp16 buffer, twice its size)."""
    torch = _torch()
    from manytor_b200 import BatchedEnvs, _lib
    lib = _lib.load()
    n, x = 1000, 10
    spec = arm_pair(J)[1]
    dtypes = [torch.float32, torch.float16] if first == "f32" else [torch.float16, torch.float32]
    envs = {}
    for dt in dtypes:                                     # the first handle's kernel is compiled and cached first
        envs[dt] = BatchedEnvs(n, x, arm=spec, device=0, fk_mode=3, seed=J, auto_reset=True, horizon=3, obs_dtype=dt)
        envs[dt].reset()
    whole, obs16 = _guarded(n * 3 * x, torch.int16, SENT16)
    rs = np.random.RandomState(J)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for i in range(4):
        act = torch.from_numpy(actions_for(n, J, rs, fractional=i % 2 == 1)).cuda()
        o32, r32, d32 = (v.clone() for v in envs[torch.float32].step(act))
        r16, d16 = torch.empty_like(r32), torch.empty_like(d32)
        _lib.check(lib.mt_step(envs[torch.float16]._h, C.c_void_p(act.data_ptr()), C.c_void_p(obs16.data_ptr()),
                               C.c_void_p(r16.data_ptr()), C.c_void_p(d16.data_ptr()), None, stream))
        _check_guarded(whole, obs16, SENT16)
        assert_obs_twin(o32, obs16.view(torch.float16).reshape(n, 3 * x))
        assert_same(r32, r16)
        assert_same(d32, d16)


@pytest.mark.parametrize("x", [7, 10, 20])
@pytest.mark.parametrize("n", [1, 31, 33, 95, 1000, 4097])
def test_f16_outputs_stay_inside_their_buffers(n, x):
    """Every fp16 output lands inside N * 3X halves of a sentinel-filled allocation and fills them: mt_step,
    mt_rollout_random(1) (step kernel), mt_rollout_random(3) (rollout kernel) and mt_observe."""
    torch = _torch()
    from manytor_b200 import BatchedEnvs, _lib
    lib = _lib.load()
    env = BatchedEnvs(n, x, device=0, auto_reset=True, horizon=4, obs_after_reset=True, seed=n, obs_dtype=torch.float16)
    env.reset()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())
    act = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    rew = torch.empty((n,), dtype=torch.float32, device="cuda")
    done = torch.empty((n,), dtype=torch.uint8, device="cuda")
    calls = {
        "step": lambda o: lib.mt_step(env._h, p(act), p(o), p(rew), p(done), None, stream),
        "rollout1": lambda o: lib.mt_rollout_random(env._h, 1, p(o), p(rew), p(done), stream),
        "rollout3": lambda o: lib.mt_rollout_random(env._h, 3, p(o), p(rew), p(done), stream),
        "observe": lambda o: lib.mt_observe(env._h, p(o), stream),
    }
    for it in range(3):
        for name, call in calls.items():
            whole, obs = _guarded(n * 3 * x, torch.int16, SENT16)
            _lib.check(lib.mt_sample_actions(env._h, p(act), stream))
            _lib.check(call(obs))
            _check_guarded(whole, obs, SENT16)


def test_bytes_per_env_step_and_config():
    from manytor_b200 import _lib
    a, b = twins(64, 10, "ref")
    assert a.bytes_per_env_step() == 309 and b.bytes_per_env_step() == 249      # 12J + 24X + 21, 12J + 18X + 21
    assert a.bytes_per_env_step(False, False) == b.bytes_per_env_step(False, False)
    for env, want in ((a, _lib.MT_OBS_F32), (b, _lib.MT_OBS_F16)):
        cfg = _lib.MtConfig()
        _lib.check(_lib.load().mt_get_config(env._h, C.byref(cfg)))
        assert cfg.obs_dtype == want
