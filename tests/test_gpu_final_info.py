"""What an ending episode leaves behind (mt_step_final, BatchedEnvs.step(final=True), ManyTorVectorEnv(final_info=True)).

With auto_reset the step kernel resets an env that ends in the same launch; mt_step_final also writes, for exactly the
envs with done != 0, the observation that closed the episode (obs2 of the ending step), the episode's return and its
length.  Every case runs twin handles with the same configuration and seed: everything mt_step computes must be
identical bit for bit, the final observation must be the obs2 row a handle with obs_after_reset = 0 returns, and the
rows of envs that did not end must keep their contents.
"""
import numpy as np
import pytest

from arms import arm_pair
from parity import Report, alive_bits_to_matrix, compare_obs, compare_step, half_ball_points

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


def caller_actions(n, j, rs):
    """Continuous degrees, some out of the action range, some far from any pose."""
    a = rs.uniform(-180.0, 180.0, size=(n, j))
    a[::7] *= 3.0
    return _torch().tensor(a, dtype=_torch().float32, device="cuda")


def bits(t):
    torch = _torch()
    return t.view(torch.int16 if t.dtype == torch.float16 else torch.int32)


def assert_twins(a, b):
    torch = _torch()
    torch.cuda.synchronize()
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert torch.equal(a.get_points(zero_dead=False), b.get_points(zero_dead=False))
    assert a.stats() == b.stats()
    assert a.step_index == b.step_index


def run_twins(n, x, arm, oar, steps, horizon=6, seed=11, actions=None, **kw):
    """Handle `a` steps with final=True beside `b` (mt_step, same configuration) and `c` (mt_step, obs_after_reset = 0).
    Checks every step; returns the observed (terminations, truncations)."""
    torch = _torch()
    a = handle(n, x, arm, horizon, seed, obs_after_reset=oar, **kw)
    b = handle(n, x, arm, horizon, seed, obs_after_reset=oar, **kw)
    c = handle(n, x, arm, horizon, seed, obs_after_reset=False, **kw) if oar else None
    rs = np.random.RandomState(n + x)
    s0 = a.stats()
    sums = dict(episodes=0, reward_sum=0, length_sum=0)
    n_term = n_trunc = 0
    prev = None
    for t in range(steps):
        act = actions(t) if actions is not None else caller_actions(n, a.j, rs)
        before = b.get_state()
        o, r, d, fin = a.step(act, final=True)
        ob, rb, db = b.step(act)
        torch.cuda.synchronize()
        assert torch.equal(bits(o), bits(ob)) and torch.equal(r, rb) and torch.equal(d, db), t
        ended = d != 0
        if c is not None:
            oc, rc, dc = c.step(act)
            assert torch.equal(rc, r) and torch.equal(dc, d)
            want = oc
        else:
            want = o
        assert torch.equal(bits(fin.obs[ended]), bits(want[ended])), t
        # return and length: the episode's state before the step plus this step
        assert torch.equal(fin.episode_return[ended], before["total_reward"][ended] + r[ended]), t
        assert torch.equal(fin.episode_length[ended], before["ep_len"][ended] + 1), t
        if prev is not None:                                   # rows of envs that went on keep their contents
            go = ~ended
            assert torch.equal(bits(fin.obs[go]), bits(prev[0][go]))
            assert torch.equal(bits(fin.episode_return[go]), bits(prev[1][go]))       # bits: never-written rows may hold NaNs
            assert torch.equal(fin.episode_length[go], prev[2][go])
        prev = tuple(v.clone() for v in fin)
        sums["episodes"] += int(ended.sum())
        sums["reward_sum"] += int(fin.episode_return[ended].double().sum())
        sums["length_sum"] += int(fin.episode_length[ended].long().sum())
        n_term += int(((d & 1) != 0).sum())
        n_trunc += int(((d & 2) != 0).sum())
    assert_twins(a, b)
    if c is not None:
        assert_twins(a, c)
    s1 = a.stats()
    for k, v in sums.items():                                  # the statistics identity
        assert s1[k] - s0[k] == v, k
    return n_term, n_trunc


# --------------------------------------------------------------------------
# 1. twin handles: mt_step_final == mt_step, final_obs == the obs2 rows
# --------------------------------------------------------------------------
_CASES = [  # id, arm, x, n
    ("ref_x10", "ref", 10, 40003),
    ("ref_x1", "ref", 1, 20000),
    ("ref_x7", "ref", 7, 5001),
    ("ur5_x20", "ur5", 20, 30011),
    ("jit_j5_x12", "jit_j5", 12, 9001),
    ("rt_j7_x10", "rt_j7", 10, 3001),
]


@pytest.mark.parametrize("oar", [True, False], ids=["obs_after_reset", "obs2"])
@pytest.mark.parametrize("case,arm,x,n", _CASES, ids=[c[0] for c in _CASES])
def test_twins_bit_for_bit(case, arm, x, n, oar):
    n_term, n_trunc = run_twins(n, x, arm, oar, steps=20)
    assert n_trunc > 0
    if x == 1:
        assert n_term > 0                                      # episodes also end by collecting everything


# --------------------------------------------------------------------------
# 2. binary16: final_obs16 == final_obs32.half()
# --------------------------------------------------------------------------
@pytest.mark.parametrize("arm,x,n", [("ref", 10, 20003), ("ur5", 20, 7001)])
def test_f16_final_obs_is_the_rounded_f32(arm, x, n):
    torch = _torch()
    a = handle(n, x, arm, obs_after_reset=True, obs_dtype=torch.float16)
    b = handle(n, x, arm, obs_after_reset=True)
    rs = np.random.RandomState(3)
    ended_total = 0
    for t in range(15):
        act = caller_actions(n, a.j, rs)
        o16, r16, d16, f16 = a.step(act, final=True)
        o32, r32, d32, f32 = b.step(act, final=True)
        torch.cuda.synchronize()
        assert torch.equal(bits(o16), bits(o32.half())) and torch.equal(r16, r32) and torch.equal(d16, d32)
        ended = d32 != 0
        ended_total += int(ended.sum())
        assert torch.equal(bits(f16.obs[ended]), bits(f32.obs[ended].half())), t
        assert torch.equal(f16.episode_return[ended], f32.episode_return[ended])
        assert torch.equal(f16.episode_length[ended], f32.episode_length[ended])
    assert ended_total > 0
    assert_twins(a, b)


# --------------------------------------------------------------------------
# 3. the oracle: final observation, return and length of every ended episode
# --------------------------------------------------------------------------
@pytest.mark.parametrize("iface,x", [("batched", 4), ("vector_env", 1), ("vector_env", 4)])
def test_final_values_against_oracle(iface, x):
    torch = _torch()
    import manytor_b200 as mt
    from oracle import OracleEnvs, REFERENCE_ARM
    n, horizon, steps, sets = 1024, 12, 60, 8
    rs = np.random.RandomState(4 + x)
    stream = np.float32(half_ball_points(rs, (sets, n, x))).astype(np.float64)
    if iface == "vector_env":
        venv = mt.ManyTorVectorEnv(n, x, max_episode_steps=horizon, seed=1, final_info=True)
        env = venv.envs
        env.set_objective_stream(stream)
        venv.reset()
    else:
        env = mt.BatchedEnvs(n, x, device=0, horizon=horizon, auto_reset=True, seed=1)
        env.set_objective_stream(stream)
        env.reset()
    ora = OracleEnvs(n, x)
    ora.reset(points=stream[0])
    episode = np.ones(n, dtype=np.int64)
    rep = Report()
    n_ended = 0
    for t in range(steps):
        act = rs.randint(-180, 180, size=(n, 4)).astype(np.float64)
        alive_before, points_before = ora.alive.copy(), ora.points.copy()
        a = torch.as_tensor(act, dtype=torch.float32, device="cuda")
        if iface == "vector_env":
            o, rew, term, trunc, info = venv.step(a)
            assert set(info) == {"final_obs", "_final_obs", "episode", "_episode"}
            assert set(info["episode"]) == {"r", "l"}
            mask = term | trunc
            assert torch.equal(info["_final_obs"], mask) and torch.equal(info["_episode"], mask)
            assert info["final_obs"].shape == (n, 3 * x) and info["final_obs"].is_cuda
            assert info["episode"]["r"].dtype == torch.float32 and info["episode"]["l"].dtype == torch.int32
            fo, fr, fl = info["final_obs"], info["episode"]["r"], info["episode"]["l"]
            done = (term.to(torch.uint8) | (trunc.to(torch.uint8) << 1))
        else:
            o, rew, done, fin = env.step(a, final=True)
            fo, fr, fl = fin
        o, rew, done = o.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()
        fo, fr, fl = fo.cpu().numpy(), fr.cpu().numpy(), fl.cpu().numpy()
        r = ora.step(act)
        want_trunc = (ora.ep_len >= horizon) & ~r.done
        ended = r.done | want_trunc
        near = (r.ground_margin < 1e-3) | (np.where(alive_before, np.abs(r.catch_margin), np.inf).min(axis=1) < 1e-3)
        ok = (rew.astype(np.int64) == r.reward) & ((done & 1).astype(bool) == r.done) & ((done & 2).astype(bool) == want_trunc)
        assert (ok | near).all(), "flags differ away from a threshold"
        if not ok.all():
            pytest.skip("a near-threshold flip forked the episode structure; covered by the lock-step tests")
        st = env.get_state()
        dev_alive = np.where(ended[:, None], r.alive, alive_bits_to_matrix(st["alive"].cpu().numpy(), x))
        obs_rows = ~ended if iface == "vector_env" else None                 # obs_after_reset: ended rows are new
        compare_step(rep, REFERENCE_ARM, ora, r, points_before, alive_before, o, rew, done, dev_alive, obs_rows=obs_rows)
        if ended.any():
            e = ended
            compare_obs(rep, REFERENCE_ARM, r.frames[e, REFERENCE_ARM.obs_frame], points_before[e], alive_before[e],
                        fo[e], r.obs[e])
            np.testing.assert_array_equal(fr[e], np.float32(ora.total_reward[e]))   # before the oracle's reset
            np.testing.assert_array_equal(fl[e], ora.ep_len[e])
            n_ended += int(e.sum())
            ora.reset(mask=e, points=stream[episode % sets, np.arange(n)])
            episode[e] += 1
    assert rep.ok(), rep.notes[:5]
    assert n_ended >= n * (steps // horizon)
    s = env.stats()
    assert s["episodes"] == n_ended


# --------------------------------------------------------------------------
# 5. rows of envs that go on, and the bytes around the buffers, are not touched
# --------------------------------------------------------------------------
SENTINEL = 0xA5


def _guarded(shape, dtype, pad=4096):
    torch = _torch()
    nbytes = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
    raw = torch.full((nbytes + 2 * pad,), SENTINEL, dtype=torch.uint8, device="cuda")
    return raw, raw[pad:pad + nbytes].view(dtype).view(shape), pad


@pytest.mark.parametrize("dtype", ["float32", "float16"])
@pytest.mark.parametrize("n", [33, 1000])
def test_untouched_rows_and_guard_bands(n, dtype):
    torch = _torch()
    x = 10
    obs_dtype = getattr(torch, dtype)
    a = handle(n, x, obs_after_reset=True, obs_dtype=obs_dtype, horizon=4)
    b = handle(n, x, obs_after_reset=False, obs_dtype=obs_dtype, horizon=4)
    g = dict(obs=_guarded((n, 3 * x), obs_dtype), ret=_guarded((n,), torch.float32), len=_guarded((n,), torch.int32))
    raw_rows = {k: raw[pad:-pad].view(n, -1) for k, (raw, _, pad) in g.items()}
    obs = torch.empty((n, 3 * x), dtype=obs_dtype, device="cuda")
    rew = torch.empty((n,), device="cuda")
    done = torch.empty((n,), dtype=torch.uint8, device="cuda")
    rs = np.random.RandomState(7)
    ever = torch.zeros(n, dtype=torch.bool, device="cuda")
    prev = {k: v.clone() for k, v in raw_rows.items()}
    for t in range(12):
        act = caller_actions(n, 4, rs)
        rc = a._lib.mt_step_final(a._h, a._p(act), a._p(obs), a._p(rew), a._p(done), None, a._p(g["obs"][1]),
                                  a._p(g["ret"][1]), a._p(g["len"][1]), a._stream())
        assert rc == 0, a._lib.mt_last_error()
        ob, rb, db = b.step(act)
        torch.cuda.synchronize()
        assert torch.equal(db, done) and torch.equal(rb, rew)
        ended = done != 0
        ever |= ended
        for k, (raw, view, pad) in g.items():
            assert bool((raw[:pad] == SENTINEL).all()) and bool((raw[-pad:] == SENTINEL).all()), f"{k}: guard band written"
            assert torch.equal(raw_rows[k][~ended], prev[k][~ended]), f"{k}: a row of an env that went on was written"
            assert bool((raw_rows[k][~ever] == SENTINEL).all())
        assert torch.equal(bits(g["obs"][1][ended]), bits(ob[ended]))
        prev = {k: v.clone() for k, v in raw_rows.items()}
    assert bool(ever.any())


# --------------------------------------------------------------------------
# 6. the benchmark's launch shape: 2^20 envs after the burn-in (multi-tile warps, in-kernel resets every step)
# --------------------------------------------------------------------------
def test_benchmark_launch_shape():
    torch = _torch()
    n, x, k = 1 << 20, 10, 8
    gen = torch.Generator(device="cuda")
    gen.manual_seed(5)
    acts = [torch.randint(-180, 180, (n, 4), device="cuda", generator=gen).float() for _ in range(k)]
    # a burn-in past the horizon: episodes then end by truncation as well as by termination in every step
    n_term, n_trunc = run_twins(n, x, "ref", True, steps=k, horizon=1000, seed=7, actions=lambda t: acts[t], burn_in=2000)
    assert n_term > 0 and n_trunc > 0 and n_term + n_trunc > 100 * k


# --------------------------------------------------------------------------
# 7. the episode-length counter at its maximum
# --------------------------------------------------------------------------
@pytest.mark.parametrize("x", [4, 20])
def test_counter_at_its_maximum(x):
    torch = _torch()
    n = 64
    env = handle(n, x, horizon=65535)
    env.set_state(ep_len=np.full(n, 65534, np.int32))
    o, r, d, fin = env.step(caller_actions(n, 4, np.random.RandomState(1)), final=True)
    torch.cuda.synchronize()
    assert bool((d != 0).all())                            # 65535 steps: every episode ends, most by truncation
    assert int(((d & 2) != 0).sum()) > n // 2
    assert bool((fin.episode_length == 65535).all())
    assert bool((env.get_state()["ep_len"] == 0).all())


# --------------------------------------------------------------------------
# 8. a captured mt_step_final replayed N times == N eager calls
# --------------------------------------------------------------------------
def test_cuda_graph_replay():
    torch = _torch()
    n, x = 20000, 10
    a, b = handle(n, x, obs_after_reset=True), handle(n, x, obs_after_reset=True)
    rs = np.random.RandomState(2)
    act = caller_actions(n, 4, rs)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                          # warm-up: kernel attributes, launch shapes, buffers
        a.step(act, final=True)
    torch.cuda.current_stream().wait_stream(side)
    b.step(act, final=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = a.step(act, final=True)
    for rep in range(4):
        act.copy_(caller_actions(n, 4, rs))
        idx = a.step_index
        graph.replay()
        o, r, d, fin = b.step(act, final=True)
        torch.cuda.synchronize()
        assert a.step_index == idx + 1
        assert torch.equal(out[0], o) and torch.equal(out[1], r) and torch.equal(out[2], d)
        ended = d != 0
        for u, v in zip(out[3], fin):
            assert torch.equal(u[ended], v[ended])
        assert_twins(a, b)


# --------------------------------------------------------------------------
# 9. state errors of the C ABI
# --------------------------------------------------------------------------
def test_state_errors():
    torch = _torch()
    n, x = 64, 10
    obs = torch.empty((n, 3 * x), device="cuda")
    rew = torch.empty((n,), device="cuda")
    done = torch.empty((n,), dtype=torch.uint8, device="cuda")
    fo = torch.empty((n, 3 * x), device="cuda")
    fr = torch.empty((n,), device="cuda")
    fl = torch.empty((n,), dtype=torch.int32, device="cuda")
    act = torch.zeros((n, 4), device="cuda")

    def call(env):
        p = env._p
        return env._lib.mt_step_final(env._h, p(act), p(obs), p(rew), p(done), None, p(fo), p(fr), p(fl), env._stream())

    plain = handle(n, x, auto_reset=False)
    assert call(plain) == -1                               # MT_ERR_INVALID
    assert b"auto_reset" in plain._lib.mt_last_error()
    with pytest.raises(ValueError, match="auto_reset"):
        plain.step(act, final=True)
    fresh = handle(n, x, reset=False)
    assert call(fresh) == -4                               # MT_ERR_STATE
    assert b"before mt_reset" in fresh._lib.mt_last_error()
    fresh.reset()
    assert call(fresh) == 0
    torch.cuda.synchronize()
