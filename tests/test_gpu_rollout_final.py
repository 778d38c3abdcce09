"""Trajectory rollouts with final outputs (mt_rollout_final, BatchedEnvs.rollout(final=True)) against one
mt_step_final call per step.

Every case runs twin handles with the same configuration and seed, and prefills every final array with the bit
pattern 0xA5 in each byte.  Slice s of every output must equal, bit for bit, what the s-th of K consecutive
mt_step_final calls returns; the rows of final slice s where done[s] == 0 must still hold the prefill; afterwards
the state, objectives, statistics and step index of the twins must be identical.  Every case runs under in-kernel
auto-reset with a short horizon, so that episodes end inside the rollout.
"""
import math

import numpy as np
import pytest

from arms import arm_pair
from parity import Report, compare_obs, compare_step, half_ball_points

pytestmark = pytest.mark.gpu

FILL = 0xA5


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


def handle(n, x, arm="ref", horizon=6, seed=11, reset=True, burn_in=0, **kw):
    """burn_in: in-kernel random steps after the reset, so that the envs are spread over their episodes."""
    from manytor_b200 import BatchedEnvs
    spec, fk_mode = _arm(arm)
    kw.setdefault("fk_mode", fk_mode)
    kw.setdefault("auto_reset", True)
    env = BatchedEnvs(n, x, arm=spec, device=0, horizon=horizon, seed=seed, **kw)
    if reset:
        env.reset()
    if burn_in:
        env.rollout_random(burn_in, write_obs=False)
    return env


def caller_actions(k, n, j, seed):
    """Continuous degrees, some out of the action range, some more than 540 degrees from any pose."""
    rs = np.random.RandomState(seed)
    a = rs.uniform(-180.0, 180.0, size=(k, n, j))
    a[:, ::7] *= 3.0
    a[:, 3::11] += rs.choice([-1.0, 1.0], size=a[:, 3::11].shape) * 1500.0
    return _torch().tensor(a, dtype=_torch().float32, device="cuda")


def bits(t):
    torch = _torch()
    return t.view(torch.int16 if t.dtype == torch.float16 else torch.int32)


def filled(env, k):
    """A FinalInfo of (K, N) slices, every byte FILL."""
    torch = _torch()
    from manytor_b200 import FinalInfo
    fin = FinalInfo(torch.empty((k, env.n, 3 * env.x), dtype=env.obs_dtype, device="cuda"),
                    torch.empty((k, env.n), device="cuda"), torch.empty((k, env.n), dtype=torch.int32, device="cuda"))
    for t in fin:
        t.view(torch.uint8).fill_(FILL)
    return fin


def fill_bits(t):
    torch = _torch()
    return bits(torch.full_like(t, 0).view(torch.uint8).fill_(FILL).view(t.dtype))


def assert_twins(a, b):
    torch = _torch()
    torch.cuda.synchronize()
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert torch.equal(a.get_points(zero_dead=False), b.get_points(zero_dead=False))
    assert a.stats() == b.stats()
    assert a.step_index == b.step_index


def assert_traj(traj, ref):
    torch = _torch()
    assert torch.equal(bits(traj.obs), bits(ref.obs))
    assert torch.equal(traj.reward, ref.reward)
    assert torch.equal(traj.done, ref.done)


def assert_final_equal(fa, fb):
    """Two FinalInfos bit for bit, filled rows included."""
    torch = _torch()
    for u, v in zip(fa, fb):
        assert torch.equal(bits(u), bits(v))


def assert_final_matches_steps(fin, done, per_step):
    """Slice s of `fin` against the FinalInfo of the s-th mt_step_final call: the rows where done[s] != 0 equal,
    every other row still FILL."""
    torch = _torch()
    for s, step_fin in enumerate(per_step):
        ended = done[s] != 0
        for name, u, v in zip(fin._fields, fin, step_fin):
            assert torch.equal(bits(u[s][ended]), bits(v[ended])), (name, s)
            assert torch.equal(bits(u[s][~ended]), fill_bits(u[s][~ended])), (name, s)


def step_final_each(env, actions):
    """K mt_step_final calls; each call's outputs are copied before the next one reuses the buffers."""
    torch = _torch()
    obs, rew, done, fins = [], [], [], []
    for s in range(actions.shape[0]):
        o, r, d, f = env.step(actions[s].clone(), final=True)
        obs.append(o.clone()); rew.append(r.clone()); done.append(d.clone())
        fins.append(tuple(t.clone() for t in f))
    from manytor_b200 import Trajectory
    return Trajectory(torch.stack(obs), torch.stack(rew), torch.stack(done), None), fins


def sampled_step_final_each(env, k):
    """K x (sample_actions + mt_step_final)."""
    torch = _torch()
    acts = torch.empty((k, env.n, env.j), device="cuda")
    obs, rew, done, fins = [], [], [], []
    for s in range(k):
        a = env.sample_actions()
        acts[s].copy_(a)
        o, r, d, f = env.step(a, final=True)
        obs.append(o.clone()); rew.append(r.clone()); done.append(d.clone())
        fins.append(tuple(t.clone() for t in f))
    from manytor_b200 import Trajectory
    return Trajectory(torch.stack(obs), torch.stack(rew), torch.stack(done), acts), fins


@pytest.fixture
def per_step_path(monkeypatch):
    def use(on):
        if on:
            monkeypatch.setenv("MT_ROLLOUT_PERSISTENT", "0")
        else:
            monkeypatch.delenv("MT_ROLLOUT_PERSISTENT", raising=False)
    return use


def rollout_final(env, actions=None, k=None, record=False, fin=None, **kw):
    fin = fin if fin is not None else filled(env, k if actions is None else actions.shape[0])
    traj, f = env.rollout(actions, n_steps=k, record_actions=record, final=True, final_out=fin, **kw)
    assert f is fin
    return traj, f


# --------------------------------------------------------------------------
# 1. the caller's actions: persistent == per-step path == K mt_step_final calls
# --------------------------------------------------------------------------
_CALLER = [  # id, arm, x, n, kw, persistent kernel available
    ("ref_x10", "ref", 10, 40003, {}, True),
    ("ref_x1", "ref", 1, 20000, {}, True),
    ("ref_x7", "ref", 7, 5001, {}, True),
    ("ur5_x20", "ur5", 20, 30011, {}, True),
    ("jit_j5_x12", "jit_j5", 12, 9001, {}, True),
    ("rt_j7_x10", "rt_j7", 10, 3001, {}, False),
    ("arms_j2_x1_misaligned", "jit_j2", 1, 9001, dict(fk_mode=0), True),
    ("ref_f16_aligned", "ref", 10, 40960, dict(obs_dtype="float16"), True),
    ("ref_f16_misaligned", "ref", 10, 40963, dict(obs_dtype="float16"), True),
]


@pytest.mark.parametrize("oar", [True, False], ids=["obs_after_reset", "obs2"])
@pytest.mark.parametrize("case,arm,x,n,kw,persistent", _CALLER, ids=[c[0] for c in _CALLER])
def test_caller_actions_match_mt_step_final(case, arm, x, n, kw, persistent, oar, per_step_path):
    torch = _torch()
    kw = dict(kw)
    if "obs_dtype" in kw:
        kw["obs_dtype"] = getattr(torch, kw["obs_dtype"])
    k = 24
    a, b, c = (handle(n, x, arm, obs_after_reset=oar, **kw) for _ in range(3))
    acts = caller_actions(k, n, a.j, seed=n + x)
    l0 = a.launch_count
    traj, fin = rollout_final(a, acts)
    assert a.launch_count - l0 == (math.ceil(k / 4096) if persistent else k)
    assert traj.actions is acts and fin.obs.shape == (k, n, 3 * x) and fin.episode_length.shape == (k, n)
    per_step_path(True)
    l0 = b.launch_count
    trb, fib = rollout_final(b, acts)
    assert b.launch_count - l0 == k
    per_step_path(False)
    ref, fins = step_final_each(c, acts)
    torch.cuda.synchronize()
    assert_traj(traj, ref)
    assert_traj(trb, ref)
    assert_final_matches_steps(fin, ref.done, fins)
    assert_final_equal(fin, fib)
    assert int((traj.done != 0).sum()) > 0
    assert_twins(a, c)
    assert_twins(b, c)


# --------------------------------------------------------------------------
# 2. in-kernel draws: trajectory == mt_rollout, final rows == K x (sample_actions + mt_step_final)
# --------------------------------------------------------------------------
@pytest.mark.parametrize("table", ["on", "off"])
@pytest.mark.parametrize("path", ["persistent", "per_step"])
@pytest.mark.parametrize("arm,x,n", [("ref", 10, 30011), ("ur5", 20, 12000), ("jit_j5", 12, 5003), ("rt_j7", 10, 3001)])
def test_in_kernel_draws(arm, x, n, path, table, per_step_path, monkeypatch):
    torch = _torch()
    if table == "off":
        monkeypatch.setenv("MT_ACTION_TABLE", "0")
    k, seed = 20, 0x1234_5678_9ABC
    a, a2, b, c = (handle(n, x, arm, seed=seed, obs_after_reset=True) for _ in range(4))
    per_step_path(path == "per_step")
    traj, fin = rollout_final(a, k=k, record=True)
    tr2, fi2 = rollout_final(a2, k=k)                                    # drawn_dev = NULL
    per_step_path(False)
    plain = b.rollout(n_steps=k, record_actions=True)
    ref, fins = sampled_step_final_each(c, k)
    torch.cuda.synchronize()
    assert_traj(traj, plain)
    assert_traj(tr2, plain)
    assert tr2.actions is None
    assert torch.equal(traj.actions, plain.actions) and torch.equal(traj.actions, ref.actions)
    assert_traj(ref, plain)                       # a table lookup is the kernel's own sin / cos
    assert_final_matches_steps(fin, plain.done, fins)
    assert_final_equal(fin, fi2)
    assert int((traj.done != 0).sum()) > 0
    for e in (a2, b, c):
        assert_twins(a, e)


# --------------------------------------------------------------------------
# 3. final_obs == the obs slices of an obs_after_reset = 0 twin
# --------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["persistent", "per_step"])
@pytest.mark.parametrize("arm,x,n,dtype", [("ref", 10, 20011, "float32"), ("ur5", 20, 7001, "float32"),
                                           ("ref", 10, 20011, "float16")])
def test_final_obs_is_obs2(arm, x, n, dtype, path, per_step_path):
    torch = _torch()
    obs_dtype = getattr(torch, dtype)
    k = 16
    a = handle(n, x, arm, obs_after_reset=True, obs_dtype=obs_dtype)
    z = handle(n, x, arm, obs_after_reset=False, obs_dtype=obs_dtype)
    acts = caller_actions(k, n, a.j, seed=4)
    per_step_path(path == "per_step")
    traj, fin = rollout_final(a, acts)
    per_step_path(False)
    ref = z.rollout(acts)
    torch.cuda.synchronize()
    assert torch.equal(traj.done, ref.done) and torch.equal(traj.reward, ref.reward)
    ended = traj.done != 0
    assert int(ended.sum()) > 0
    assert torch.equal(bits(fin.obs[ended]), bits(ref.obs[ended]))
    assert torch.equal(bits(traj.obs[~ended]), bits(ref.obs[~ended]))      # obs_after_reset changes ended rows only


# --------------------------------------------------------------------------
# 4. returns and lengths against a host accumulation from get_state(); the statistics identity
# --------------------------------------------------------------------------
def host_check(env, traj, fin, state0, stats0):
    """Accumulate the trajectory's rewards from the state before the call and compare at every done."""
    torch = _torch()
    torch.cuda.synchronize()
    ret = state0["total_reward"].cpu().numpy().astype(np.float32)
    length = state0["ep_len"].cpu().numpy().astype(np.int64)
    rew, done = traj.reward.cpu().numpy(), traj.done.cpu().numpy()
    fr, fl = fin.episode_return.cpu().numpy(), fin.episode_length.cpu().numpy()
    ep_max = 65535 if (env.x <= 16 or env.cfg.horizon == 0 or env.cfg.horizon >= (1 << (32 - env.x))) else (1 << (32 - env.x)) - 1
    sums = dict(episodes=0, reward_sum=0, length_sum=0)
    for s in range(rew.shape[0]):
        ret = ret + rew[s]
        length = np.minimum(length + 1, ep_max)
        e = done[s] != 0
        np.testing.assert_array_equal(fr[s][e], ret[e], err_msg=f"return at s={s}")
        np.testing.assert_array_equal(fl[s][e], length[e], err_msg=f"length at s={s}")
        sums["episodes"] += int(e.sum())
        sums["reward_sum"] += int(fr[s][e].astype(np.int64).sum())
        sums["length_sum"] += int(fl[s][e].astype(np.int64).sum())
        ret[e] = 0.0
        length[e] = 0
    st = env.get_state()
    np.testing.assert_array_equal(st["total_reward"].cpu().numpy(), ret)
    np.testing.assert_array_equal(st["ep_len"].cpu().numpy(), length)
    s1 = env.stats()
    for k, v in sums.items():
        assert s1[k] - stats0[k] == v, k
    return sums["episodes"], length


@pytest.mark.parametrize("path", ["persistent", "per_step"])
@pytest.mark.parametrize("case", ["packed", "wide", "saturated_x4", "saturated_x20"])
def test_returns_and_lengths_on_the_host(case, path, per_step_path):
    n, k = 4096, 24
    if case == "packed":                                  # X = 20, horizon 7: the counter shares the alive word
        env = handle(n, 20, horizon=7, burn_in=3)
    elif case == "wide":                                  # X = 20, horizon 65535: the counter has its own array
        env = handle(n, 20, horizon=65535)
        env.set_state(ep_len=65535 - np.random.RandomState(1).randint(1, 2 * k, size=n).astype(np.int32))
    else:                                                 # no horizon: the counter saturates at 65535
        x = 4 if case == "saturated_x4" else 20
        env = handle(n, x, horizon=0, terminate_on_ground=True)
        env.set_state(ep_len=np.full(n, 65530, np.int32))
    state0, stats0 = env.get_state(), env.stats()
    acts = caller_actions(k, n, env.j, seed=7) if case != "packed" else None
    per_step_path(path == "per_step")
    traj, fin = rollout_final(env, acts, k=k)
    per_step_path(False)
    ended, length = host_check(env, traj, fin, state0, stats0)
    assert ended > 0
    if case.startswith("saturated"):
        assert bool((fin.episode_length[traj.done != 0] == 65535).any())   # episodes that ended at the maximum
    if case == "wide":
        assert int(((traj.done & 2) != 0).sum()) > 0


# --------------------------------------------------------------------------
# 5. chunk boundary: episodes that end at s = 4095 and s = 4096
# --------------------------------------------------------------------------
def test_chunk_boundary(per_step_path):
    torch = _torch()
    n, x, k, horizon = 1024, 32, 4100, 2048
    a, b = handle(n, x, horizon=horizon), handle(n, x, horizon=horizon)
    ep = np.where(np.arange(n) % 2 == 0, 0, horizon - 1).astype(np.int32)    # truncations at 2047 / 4095 and 0 / 2048 / 4096
    a.set_state(ep_len=ep)
    b.set_state(ep_len=ep)
    state0, stats0 = a.get_state(), a.stats()
    acts = caller_actions(k, n, 4, seed=5)
    l0 = a.launch_count
    traj, fin = rollout_final(a, acts)
    assert a.launch_count - l0 == 2
    per_step_path(True)
    trb, fib = rollout_final(b, acts)
    per_step_path(False)
    torch.cuda.synchronize()
    assert_traj(traj, trb)
    assert_final_equal(fin, fib)
    assert int((traj.done[4095] != 0).sum()) > 0 and int((traj.done[4096] != 0).sum()) > 0
    host_check(a, traj, fin, state0, stats0)
    assert_twins(a, b)


# --------------------------------------------------------------------------
# 6. final rows more than 4 GiB past the base: 64-bit slice offsets
# --------------------------------------------------------------------------
def test_final_obs_past_4_gib(per_step_path):
    torch = _torch()
    n, x, k = 1 << 20, 10, 36
    assert (k - 1) * n * 3 * x * 4 > 1 << 32
    acts = caller_actions(k, n, 4, seed=9)
    a = handle(n, x, horizon=1000, burn_in=2000, obs_after_reset=True)
    traj, fin = rollout_final(a, acts)
    torch.cuda.synchronize()
    last = [t[-2:].clone() for t in (traj.obs, traj.reward, traj.done, *fin)]
    del traj, fin
    torch.cuda.empty_cache()
    b = handle(n, x, horizon=1000, burn_in=2000, obs_after_reset=True)
    per_step_path(True)
    trb, fib = rollout_final(b, acts)
    per_step_path(False)
    torch.cuda.synchronize()
    ref = [t[-2:] for t in (trb.obs, trb.reward, trb.done, *fib)]
    for u, v in zip(last, ref):
        assert torch.equal(bits(u) if u.dtype != torch.uint8 else u, bits(v) if v.dtype != torch.uint8 else v)
    ended = last[2] != 0
    assert int(ended[-1].sum()) > 100                        # rows past 4 GiB were written
    assert not torch.equal(bits(last[3][ended]), fill_bits(last[3][ended]))
    assert_twins(a, b)


# --------------------------------------------------------------------------
# 7. guard bands around every output at N = 33 and N = 1000
# --------------------------------------------------------------------------
def _guarded(shape, dtype, pad=4096):
    torch = _torch()
    nbytes = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
    raw = torch.full((nbytes + 2 * pad,), FILL, dtype=torch.uint8, device="cuda")
    return raw, raw[pad:pad + nbytes].view(dtype).view(shape), pad


@pytest.mark.parametrize("path", ["persistent", "per_step"])
@pytest.mark.parametrize("mode", ["actions", "draws"])
@pytest.mark.parametrize("dtype", ["float32", "float16"])
@pytest.mark.parametrize("n", [33, 1000])
def test_guard_bands(n, dtype, mode, path, per_step_path):
    torch = _torch()
    from manytor_b200 import FinalInfo, Trajectory
    x, k = 10, 9
    obs_dtype = getattr(torch, dtype)
    a, b = (handle(n, x, obs_dtype=obs_dtype, obs_after_reset=True, horizon=4) for _ in range(2))
    shapes = dict(obs=((k, n, 3 * x), obs_dtype), reward=((k, n), torch.float32), done=((k, n), torch.uint8),
                  actions=((k, n, 4), torch.float32), fobs=((k, n, 3 * x), obs_dtype),
                  fret=((k, n), torch.float32), flen=((k, n), torch.int32))
    g = {name: _guarded(*spec) for name, spec in shapes.items()}
    acts = caller_actions(k, n, 4, seed=3) if mode == "actions" else None
    out = Trajectory(g["obs"][1], g["reward"][1], g["done"][1], g["actions"][1] if mode == "draws" else None)
    fout = FinalInfo(g["fobs"][1], g["fret"][1], g["flen"][1])
    per_step_path(path == "per_step")
    traj, fin = a.rollout(acts, n_steps=k, record_actions=mode == "draws", out=out, final=True, final_out=fout)
    per_step_path(False)
    trb, fib = rollout_final(b, acts, k=k, record=mode == "draws")
    torch.cuda.synchronize()
    for name, (raw, view, pad) in g.items():
        if name == "actions" and mode == "actions":
            continue
        assert bool((raw[:pad] == FILL).all()) and bool((raw[-pad:] == FILL).all()), f"{name}: guard band written"
    assert_traj(traj, trb)
    assert_final_equal(fin, fib)
    if mode == "draws":
        assert torch.equal(traj.actions, trb.actions)
    assert int((traj.done != 0).sum()) > 0
    assert_twins(a, b)


# --------------------------------------------------------------------------
# 8. the benchmark's launch shape after a burn-in: persistent == per-step path
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["actions", "draws"])
def test_benchmark_launch_shape(mode, per_step_path):
    torch = _torch()
    n, x, k = 1 << 20, 10, 8
    a, b = (handle(n, x, horizon=1000, seed=7, burn_in=2000, obs_after_reset=True) for _ in range(2))
    acts = None
    if mode == "actions":
        gen = torch.Generator(device="cuda")
        gen.manual_seed(5)
        acts = torch.randint(-180, 180, (k, n, 4), device="cuda", generator=gen).float()
    traj, fin = rollout_final(a, acts, k=k)
    per_step_path(True)
    trb, fib = rollout_final(b, acts, k=k)
    per_step_path(False)
    torch.cuda.synchronize()
    assert_traj(traj, trb)
    assert_final_equal(fin, fib)
    n_term, n_trunc = int(((traj.done & 1) != 0).sum()), int(((traj.done & 2) != 0).sum())
    assert n_term > 0 and n_trunc > 0 and n_term + n_trunc > 100 * k
    assert_twins(a, b)


# --------------------------------------------------------------------------
# 9. a captured rollout(final=True) replayed with refilled actions == an eager twin
# --------------------------------------------------------------------------
def test_cuda_graph_replay():
    torch = _torch()
    from manytor_b200 import Trajectory
    n, x, k = 20000, 10, 16
    a, b = handle(n, x, obs_after_reset=True), handle(n, x, obs_after_reset=True)
    acts = caller_actions(k, n, 4, seed=1)
    out = Trajectory(torch.empty((k, n, 3 * x), device="cuda"), torch.empty((k, n), device="cuda"),
                     torch.empty((k, n), dtype=torch.uint8, device="cuda"), None)
    fa, fb = filled(a, k), filled(b, k)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                          # warm-up: kernel attributes and launch shapes
        a.rollout(acts, out=out, final=True, final_out=fa)
    torch.cuda.current_stream().wait_stream(side)
    b.rollout(acts, final=True, final_out=fb)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        a.rollout(acts, out=out, final=True, final_out=fa)
    for r in range(3):
        acts.copy_(caller_actions(k, n, 4, seed=100 + r))
        idx = a.step_index
        graph.replay()
        ref, _ = b.rollout(acts, final=True, final_out=fb)
        torch.cuda.synchronize()
        assert_traj(out, ref)
        assert_final_equal(fa, fb)
        assert int((ref.done != 0).sum()) > 0
        assert a.step_index == idx + k
        assert_twins(a, b)


# --------------------------------------------------------------------------
# 10. the oracle: final observation, return and length of every episode that ends in a lock-step run
# --------------------------------------------------------------------------
def test_final_values_against_oracle():
    torch = _torch()
    import manytor_b200 as mt
    from oracle import OracleEnvs, REFERENCE_ARM
    n, x, horizon, k, sets = 1024, 4, 12, 60, 8
    rs = np.random.RandomState(8)
    stream = np.float32(half_ball_points(rs, (sets, n, x))).astype(np.float64)
    env = mt.BatchedEnvs(n, x, device=0, horizon=horizon, auto_reset=True, seed=1)
    env.set_objective_stream(stream)
    env.reset()
    acts = rs.randint(-180, 180, size=(k, n, 4)).astype(np.float64)
    traj, fin = rollout_final(env, torch.as_tensor(acts, dtype=torch.float32, device="cuda"))
    torch.cuda.synchronize()
    obs_all, rew_all, done_all = traj.obs.cpu().numpy(), traj.reward.cpu().numpy(), traj.done.cpu().numpy()
    fo_all, fr_all, fl_all = (t.cpu().numpy() for t in fin)
    ora = OracleEnvs(n, x)
    ora.reset(points=stream[0])
    episode = np.ones(n, dtype=np.int64)
    rep = Report()
    n_ended, forked = 0, False
    for s in range(k):
        alive_before, points_before = ora.alive.copy(), ora.points.copy()
        o, rew, done = obs_all[s], rew_all[s], done_all[s]
        r = ora.step(acts[s])
        want_trunc = (ora.ep_len >= horizon) & ~r.done
        ended = r.done | want_trunc
        near = (r.ground_margin < 1e-3) | (np.where(alive_before, np.abs(r.catch_margin), np.inf).min(axis=1) < 1e-3)
        ok = (rew.astype(np.int64) == r.reward) & ((done & 1).astype(bool) == r.done) & ((done & 2).astype(bool) == want_trunc)
        assert (ok | near).all(), "flags differ away from a threshold"
        if not ok.all():
            forked = True                                   # a near-threshold flip forked the run: stop comparing
            break
        # (the device's alive words are not kept per step; the flags and observations are compared)
        compare_step(rep, REFERENCE_ARM, ora, r, points_before, alive_before, o, rew, done, r.alive)
        if ended.any():
            e = ended
            compare_obs(rep, REFERENCE_ARM, r.frames[e, REFERENCE_ARM.obs_frame], points_before[e], alive_before[e],
                        fo_all[s][e], r.obs[e])
            np.testing.assert_array_equal(fr_all[s][e], np.float32(ora.total_reward[e]))
            np.testing.assert_array_equal(fl_all[s][e], ora.ep_len[e])
            n_ended += int(e.sum())
            ora.reset(mask=e, points=stream[episode % sets, np.arange(n)])
            episode[e] += 1
    assert rep.ok(), rep.notes[:5]
    assert forked or n_ended >= n * (k // horizon)


# --------------------------------------------------------------------------
# 11. state errors of the C ABI
# --------------------------------------------------------------------------
def test_state_errors():
    torch = _torch()
    n, x, k = 64, 10, 3
    obs = torch.empty((k, n, 3 * x), device="cuda")
    rew = torch.empty((k, n), device="cuda")
    done = torch.empty((k, n), dtype=torch.uint8, device="cuda")
    fo = torch.empty((k, n, 3 * x), device="cuda")
    fr = torch.empty((k, n), device="cuda")
    fl = torch.empty((k, n), dtype=torch.int32, device="cuda")
    act = torch.zeros((k, n, 4), device="cuda")

    def call(env, steps=k):
        p = env._p
        return env._lib.mt_rollout_final(env._h, steps, p(act), None, p(obs), p(rew), p(done), p(fo), p(fr), p(fl),
                                         env._stream())

    plain = handle(n, x, auto_reset=False)
    assert call(plain) == -1                               # MT_ERR_INVALID
    assert b"auto_reset" in plain._lib.mt_last_error()
    with pytest.raises(ValueError, match="auto_reset"):
        plain.rollout(act, final=True)
    fresh = handle(n, x, reset=False)
    assert call(fresh) == -4                               # MT_ERR_STATE
    assert b"before mt_reset" in fresh._lib.mt_last_error()
    fresh.reset()
    idx = fresh.step_index
    assert call(fresh, 0) == 0                             # n_steps = 0 does nothing
    assert fresh.step_index == idx
    assert call(fresh) == 0
    torch.cuda.synchronize()
    assert fresh.step_index == idx + k
