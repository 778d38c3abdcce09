"""In-kernel branch draws (mt_rollout_branches_random, mt_branch_actions; BatchedEnvs.rollout_branches with draw_key and
BatchedEnvs.branch_actions).

- Draws: branch_actions equals oracle.philox.device_actions at step index key + first_step + s for the branch id, over
  keys at the 32-bit carry and the 64-bit wrap, ids past 2^31, J = 2 .. 8 and three action ranges, and equals
  sample_actions of an env_id_base = 0 handle at that step index.
- Equivalence: rollout_branches(prefix, draw_key=key, n_steps=K) equals, bit for bit, rollout_branches fed
  cat(prefix, branch_actions(arange(M), key, K - P, first_step=P)) -- mt_rollout_branches, itself tested against a twin
  handle in tests/test_gpu_rollout_branches.py.  Every output buffer is prefilled with the byte 0xA5.
- A branch's outputs depend on (src[m], m, key) only; the handle is untouched; CUDA-graph replay with a device key;
  no-op and state errors; 2^20 branches.
"""

import numpy as np
import pytest

from arms import arm_pair
from oracle.philox import device_actions

pytestmark = pytest.mark.gpu

FILL = 0xA5
HORIZON = 12
U64 = 1 << 64


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


def handle(n, x, arm="ref", obs="f32", tog=False, horizon=HORIZON, seed=11, burn_in=5, reset=True, low=-180, high=180):
    """A source handle: n envs burnt in with `burn_in` random steps; env n // 2 then sits at horizon - 1 (horizon > 0)."""
    torch = _torch()
    from manytor_b200 import BatchedEnvs
    spec, fk_mode = _arm(arm)
    env = BatchedEnvs(n, x, arm=spec, device=0, horizon=horizon, seed=seed, fk_mode=fk_mode, auto_reset=True,
                      terminate_on_ground=tog, obs_dtype=torch.float16 if obs == "f16" else torch.float32,
                      action_low=low, action_high=high)
    if reset:
        env.reset()
        if burn_in:
            env.rollout_random(burn_in, write_obs=False)
        if horizon > 0:
            el = env.get_state()["ep_len"]
            el[n // 2] = horizon - 1
            env.set_state(ep_len=el)
    return env


def caller_actions(k, m, j, seed):
    """Continuous degrees, some out of the action range, some more than 540 degrees from any pose."""
    rs = np.random.RandomState(seed)
    a = rs.uniform(-180.0, 180.0, size=(k, m, j))
    a[:, ::7] *= 3.0
    a[:, 3::11] += rs.choice([-1.0, 1.0], size=a[:, 3::11].shape) * 1500.0
    return _torch().tensor(a, dtype=_torch().float32, device="cuda")


def bits(t):
    torch = _torch()
    if t.dtype == torch.float16:
        return t.view(torch.int16)
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def filled(env, m, write_obs):
    torch = _torch()
    from manytor_b200 import Branches
    out = Branches(torch.empty(m, device="cuda"), torch.empty(m, dtype=torch.int32, device="cuda"),
                   torch.empty(m, dtype=torch.uint8, device="cuda"),
                   torch.empty((m, 3 * env.x), dtype=env.obs_dtype, device="cuda") if write_obs else None)
    for t in out:
        if t is not None:
            t.view(torch.uint8).fill_(FILL)
    return out


def same(u, v):
    for a, b in zip(u, v):
        assert (a is None) == (b is None)
        if a is not None:
            assert _torch().equal(bits(a), bits(b))


def oracle_draws(env, ids, key, first, k):
    """(k, R, J) of device_actions for the branch ids (int64 bit patterns) at step index key + first + s mod 2^64."""
    cfg = env.cfg
    u = np.asarray(ids, dtype=np.int64).view(np.uint64)
    return np.stack([device_actions(cfg.seed, u, (key + first + s) % U64, env.j, cfg.action_low, cfg.action_high)
                     for s in range(k)]).astype(np.float32)


def check_fed(env, src, prefix, k, key, gamma, write_obs):
    """rollout_branches with draws against rollout_branches fed cat(prefix, branch_actions(...)); returns the outputs."""
    torch = _torch()
    m = env.n if src is None else len(src)
    p = 0 if prefix is None else prefix.shape[0]
    got = filled(env, m, write_obs)
    l0 = env.launch_count
    r = env.rollout_branches(prefix, src, gamma=gamma, write_obs=write_obs, out=got, n_steps=k, draw_key=key)
    assert r is got and env.launch_count == l0 + 1
    drawn = env.branch_actions(torch.arange(m, device="cuda"), key, k - p, first_step=p)
    fed = torch.cat([prefix, drawn]) if p else drawn
    want = env.rollout_branches(fed, src, gamma=gamma, write_obs=write_obs, out=filled(env, m, write_obs))
    torch.cuda.synchronize()
    same(got, want)
    return got


def sources(kind, n, rs):
    torch = _torch()
    if kind == "identity":
        return None
    if kind == "cand":                                 # C = 3 candidates per env, then 5 more: M = 3N + 5
        s = np.concatenate([np.repeat(np.arange(n), 3), rs.randint(0, n, size=5)])
    elif kind == "oob":                                # repeats, and sources outside [0, N)
        s = rs.randint(0, n, size=301)
        s[[0, 31, 32, 150, 300]] = [-1, n, 2 ** 40, -(2 ** 40), 2 ** 31]
    else:
        s = rs.randint(0, n, size=int(kind.split("_")[1]))
    return torch.tensor(s, dtype=torch.int64, device="cuda")


CONFIGS = [  # arm, X, observations, terminate_on_ground
    ("ref", 10, "f32", False), ("ref", 20, "f16", True), ("ref", 7, "off", True), ("ref", 32, "f32", False),
    ("ur5", 10, "f16", False), ("ur5", 20, "f32", True), ("ur5", 7, "off", False),
    ("rt_j7", 7, "f32", True), ("rt_j7", 32, "off", False), ("rt_j7", 10, "f16", False),
    ("jit_j5", 10, "f32", True), ("jit_j5", 20, "f16", False), ("jit_j5", 32, "off", True),
]
RUNS = [  # gamma, K, P (the prefix), sources (identity: M = N; cand: M = 3N + 5; rand_M: M random; oob: out of range)
    (1.0, 17, 0, "identity"), (0.99, 64, 32, "cand"), (0.0, 2, 1, "rand_33"), (0.99, 40, 1, "oob"),
    (0.97, 16, 16, "rand_1000"), (1.0, 64, 0, "rand_1"), (0.9, 33, 0, "cand"),
]


@pytest.mark.parametrize("table", ["table", "no_table"])
@pytest.mark.parametrize("arm, x, obs, tog", CONFIGS)
def test_draws_equal_branches_fed_their_actions(arm, x, obs, tog, table, monkeypatch):
    """Every configuration of the branch tests, with a prefix of P in {0, 1, K/2, K} steps, with and without the
    per-block sin / cos table (MT_ACTION_TABLE=0, set before the handle's first launch)."""
    torch = _torch()
    if table == "no_table":
        monkeypatch.setenv("MT_ACTION_TABLE", "0")
    n = 1000
    env = handle(n, x, arm, obs, tog)
    rs = np.random.RandomState(5)
    ends = []
    for i, (gamma, k, p, kind) in enumerate(RUNS):
        src = sources(kind, n, rs)
        m = n if src is None else len(src)
        prefix = caller_actions(p, m, env.j, 100 + i) if p else None
        got = check_fed(env, src, prefix, k, 7919 * i + 3, gamma, obs != "off")
        ends.append(got.done)
        if kind == "oob":
            bad = torch.tensor([0, 31, 32, 150, 300], device="cuda")
            assert bool(got.ret[bad].isnan().all()) and bool((got.length[bad] == -1).all())
            if obs != "off":
                assert bool((got.obs[bad].view(torch.uint8) == FILL).all())
    assert bool((torch.cat(ends) != 0).any())          # branches end inside the rollout


@pytest.mark.parametrize("arm, low, high", [("ref", -30, 30), ("ref", 0, 1000), ("ur5", 0, 1000), ("rt_j7", -30, 30),
                                            ("ref", 10, 100), ("ref", -100, -10), ("ur5", 10, 100), ("rt_j7", -100, -10)])
def test_draws_equal_fed_branches_in_other_action_ranges(arm, low, high):
    """[0, 1000) has no table (more than 720 values) and moves joints by up to 1000 degrees, which sends a reference-arm
    warp down its general sub-pose path; the padding lanes of a partial tile draw nothing there either.  [10, 100) and
    [-100, -10) have a table that does not hold 0, the action of a padding lane: every M here is off a tile boundary, so
    the last tile's padding lanes evaluate their zeros as the fed call does, without a table."""
    env = handle(997, 10, arm, "f32", tog=True, low=low, high=high)
    rs = np.random.RandomState(3)
    for i, (gamma, k, p, kind) in enumerate(RUNS[:4]):
        src = sources(kind, env.n, rs)
        m = env.n if src is None else len(src)
        prefix = caller_actions(p, m, env.j, 7 + i) if p else None
        check_fed(env, src, prefix, k, 2 ** 63 + 11 * i, gamma, True)


def test_views_off_the_alignment_are_copied():
    """Sources, a prefix and branch ids given as device views that start off the library's 16-byte alignment (e.g.
    best[1:]) give what their aligned copies give."""
    torch = _torch()
    env = handle(500, 10, "ref", "f32", tog=True)
    rs = np.random.RandomState(12)
    m, p, k = 333, 3, 20
    src_all = torch.tensor(rs.randint(0, env.n, size=m + 1), dtype=torch.int64, device="cuda")
    flat = caller_actions(1, 1, p * m * env.j + 1, 13).reshape(-1)
    src, prefix = src_all[1:], flat[1:].view(p, m, env.j)
    assert src.data_ptr() % 16 != 0 and prefix.data_ptr() % 16 != 0
    got = env.rollout_branches(prefix, src, gamma=0.99, write_obs=True, n_steps=k, draw_key=77)
    got = [t.clone() for t in got]
    want = env.rollout_branches(prefix.clone(), src.clone(), gamma=0.99, write_obs=True, n_steps=k, draw_key=77)
    torch.cuda.synchronize()
    same(got, want)
    ids = src_all[1:8]
    assert torch.equal(env.branch_actions(ids, 77, 2), env.branch_actions(ids.clone(), 77, 2))


KEYS = [0, 2 ** 32 - 1, 2 ** 62, U64 - 3]
IDS = [0, 31, 32, 2 ** 31 - 1, 2 ** 40, 5, 2 ** 32, -1, -(2 ** 63), 2 ** 63 - 1]


@pytest.mark.parametrize("arm, low, high", [
    ("ref", -180, 180), ("rt_j2", -30, 30), ("rt_j5", 0, 1000), ("rt_j8", -180, 180), ("ur5", 0, 1000)])
def test_branch_actions_equal_the_oracle(arm, low, high):
    """J in {2, 4, 5, 6, 8}; keys at the 32-bit carry and the 64-bit wrap (key + s passes 2^64 - 1 within a call); int
    keys mod 2^64 and device keys; a seed set with set_seed; no reset needed."""
    torch = _torch()
    env = handle(64, 10, arm, reset=False, low=low, high=high)
    env.set_seed(2 ** 40 + 12345)
    ids = torch.tensor(IDS, dtype=torch.int64, device="cuda")
    for key in KEYS:
        for first, k in ((0, 6), (3, 4)):
            want = oracle_draws(env, IDS, key, first, k)
            got = env.branch_actions(ids, key, k, first_step=first)
            np.testing.assert_array_equal(got.cpu().numpy(), want)
            signed = key - U64 if key >= 2 ** 63 else key
            dev = torch.tensor([signed], dtype=torch.int64, device="cuda")
            out = torch.full((k, len(IDS), env.j), 7.0, device="cuda")
            assert env.branch_actions(ids, dev, k, first_step=first, out=out) is out
            np.testing.assert_array_equal(out.cpu().numpy(), want)
            np.testing.assert_array_equal(env.branch_actions(IDS, key + U64, k, first).cpu().numpy(), want)
            np.testing.assert_array_equal(env.branch_actions(IDS, signed, k, first).cpu().numpy(), want)
    assert int(np.unique(oracle_draws(env, IDS, 5, 0, 8)).size) > 1


@pytest.mark.parametrize("arm", ["ref", "rt_j5", "ur5"])
def test_branch_actions_equal_sample_actions(arm):
    """Slice s of branch_actions(arange(N), key, K) is sample_actions() of an env_id_base = 0 handle at step index
    key + s (the step index stops at 2^62, so these keys stay below it)."""
    torch = _torch()
    n, k = 300, 5
    env = handle(n, 10, arm, reset=False)
    for key in (0, 2 ** 32 - 2, 2 ** 62 - k):
        got = env.branch_actions(torch.arange(n, device="cuda"), key, k)
        for s in range(k):
            env.step_index = key + s
            assert torch.equal(env.sample_actions(), got[s])


@pytest.mark.parametrize("arm, x", [("ref", 10), ("ref", 20), ("ur5", 10), ("rt_j7", 7)])
def test_a_branch_depends_on_its_source_id_and_key_only(arm, x):
    """Branch m of two calls with different M and other sources agrees wherever src[m] agrees.  (In-range draws from
    in-range poses: the reference arm's warp-wide choice of sub-pose path then never depends on the neighbours.)"""
    torch = _torch()
    n, key = 1000, 2 ** 35 + 17
    env = handle(n, x, arm, "f32", tog=True, horizon=30)
    rs = np.random.RandomState(11)
    a = torch.tensor(rs.randint(0, n, size=1500), dtype=torch.int64, device="cuda")
    b = torch.tensor(rs.randint(0, n, size=4003), dtype=torch.int64, device="cuda")
    keep = torch.tensor(rs.rand(1500) < 0.5, device="cuda")
    b[:1500] = torch.where(keep, a, b[:1500])
    ra = env.rollout_branches(None, a, gamma=0.99, write_obs=True, n_steps=24, draw_key=key)
    rb = env.rollout_branches(None, b, gamma=0.99, write_obs=True, n_steps=24, draw_key=key)
    torch.cuda.synchronize()
    for u, v in zip(ra, rb):
        assert torch.equal(bits(u)[keep], bits(v[:1500])[keep])
    assert bool((ra.done[keep] != 0).any())
    # another key draws other actions
    rc = env.rollout_branches(None, a, gamma=0.99, write_obs=True, n_steps=24, draw_key=key + 24)
    assert not torch.equal(bits(rc.obs), bits(ra.obs))


def _assert_same_handle(a, b):
    torch = _torch()
    torch.cuda.synchronize()
    sa, sb = a.get_state(), b.get_state()
    for key in sa:
        assert torch.equal(sa[key], sb[key]), key
    assert torch.equal(a.get_points(zero_dead=False), b.get_points(zero_dead=False))
    assert a.stats() == b.stats()
    assert a.step_index == b.step_index


@pytest.mark.parametrize("arm, x, obs", [("ref", 10, "f32"), ("ur5", 20, "f16"), ("rt_j7", 7, "f32"), ("jit_j5", 10, "off")])
def test_the_handle_is_untouched_and_continues(arm, x, obs):
    torch = _torch()
    n = 777
    a, b = handle(n, x, arm, obs, tog=True), handle(n, x, arm, obs, tog=True)
    _assert_same_handle(a, b)
    rs = np.random.RandomState(2)
    for i, (gamma, k, p, kind) in enumerate(RUNS):
        src = sources(kind, n, rs)
        m = n if src is None else len(src)
        prefix = caller_actions(p, m, a.j, 40 + i) if p else None
        a.rollout_branches(prefix, src, gamma=gamma, write_obs=obs != "off", n_steps=k, draw_key=100 * i)
        a.branch_actions(torch.arange(m, device="cuda"), 100 * i, k)
    _assert_same_handle(a, b)
    ta, tb = a.rollout(n_steps=20, write_obs=obs != "off"), b.rollout(n_steps=20, write_obs=obs != "off")
    for u, v in zip(ta, tb):
        if u is not None:
            assert torch.equal(bits(u), bits(v))
    _assert_same_handle(a, b)


@pytest.mark.parametrize("obs, p", [("f32", 0), ("off", 5)])
def test_cuda_graph_replay_with_a_device_key(obs, p):
    """A graph that captures the call and key.add_(K): replay r equals the eager call with key0 + r K."""
    torch = _torch()
    n, k, key0, replays = 640, 24, 2 ** 64 - 30, 4        # the key wraps past 2^64 between replays
    env = handle(n, 10, "ref", obs, tog=True)
    rs = np.random.RandomState(4)
    src = torch.tensor(rs.randint(0, n, size=2 * n + 3), dtype=torch.int64, device="cuda")
    m, wobs = len(src), obs != "off"
    prefix = caller_actions(p, m, env.j, 6) if p else None
    ids = src[:7].clone()
    eager = []
    for r in range(replays):
        out = env.rollout_branches(prefix, src, gamma=0.97, write_obs=wobs, n_steps=k, draw_key=key0 + r * k)
        first = env.branch_actions(ids, key0 + r * k, 1)
        eager.append(([t.clone() if t is not None else None for t in out], first.clone()))
    key = torch.tensor([key0 - U64], dtype=torch.int64, device="cuda")
    out = filled(env, m, wobs)
    first = torch.empty((1, 7, env.j), device="cuda")
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env.rollout_branches(prefix, src, gamma=0.97, write_obs=wobs, out=out, n_steps=k, draw_key=key)
        env.branch_actions(ids, key, 1, out=first)
        key.add_(k)
    for r in range(replays):
        g.replay()
        torch.cuda.synchronize()
        same(out, eager[r][0])
        assert torch.equal(first, eager[r][1])
    assert int(key) == key0 + replays * k - U64


def test_nothing_to_do_and_state_errors():
    torch = _torch()
    from manytor_b200 import MantorLibraryError
    from manytor_b200 import _lib
    env = handle(64, 10, "ref", "f32")
    for k, src in ((0, None), (5, np.zeros(0, np.int64))):
        m = 64 if src is None else 0
        out = filled(env, m, True)
        env.rollout_branches(None, src, write_obs=True, out=out, n_steps=k, draw_key=1)
        torch.cuda.synchronize()
        for t in out:
            assert bool((t.view(torch.uint8) == FILL).all())
    # the same through the C ABI, with real buffers
    out = filled(env, 64, True)
    src = torch.arange(64, device="cuda")
    key = torch.zeros(1, dtype=torch.int64, device="cuda")
    pre = caller_actions(2, 64, env.j, 1)
    acts = torch.full((3, 64, env.j), 7.0, device="cuda")
    l0 = env.launch_count
    for k, p, m in ((0, 0, 64), (4, 2, 0), (4, 0, 0)):
        assert env._lib.mt_rollout_branches_random(env._h, k, p, m, src.data_ptr(), pre.data_ptr() if p else None,
                                                   key.data_ptr(), 1.0, out.ret.data_ptr(), out.length.data_ptr(),
                                                   out.done.data_ptr(), out.obs.data_ptr(), None) == 0
    for k, r in ((0, 64), (3, 0)):
        assert env._lib.mt_branch_actions(env._h, key.data_ptr(), 0, k, r, src.data_ptr(), acts.data_ptr(), None) == 0
    torch.cuda.synchronize()
    assert env.launch_count == l0
    for t in out:
        assert bool((t.view(torch.uint8) == FILL).all())
    assert bool((acts == 7.0).all())
    fresh = handle(64, 10, "ref", "f32", reset=False)
    with pytest.raises(MantorLibraryError, match="mt_rollout_branches_random before mt_reset"):
        fresh.rollout_branches(None, src, n_steps=4, draw_key=0)
    assert fresh._lib.mt_rollout_branches_random(fresh._h, 4, 0, 64, src.data_ptr(), None, key.data_ptr(), 1.0,
                                                 out.ret.data_ptr(), out.length.data_ptr(), out.done.data_ptr(), None,
                                                 None) == -4   # MT_ERR_STATE
    assert _lib.load().mt_last_error() == b"mt_rollout_branches_random before mt_reset"
    # branch_actions needs no reset
    assert tuple(fresh.branch_actions(src, 0, 2).shape) == (2, 64, 4)


@pytest.mark.parametrize("p", [0, 16])
def test_benchmark_shape(p):
    """4096 sources x 256 candidates = 2^20 branches, K = 64, burnt in with horizon 1000, against the fed call."""
    torch = _torch()
    n, c, k = 4096, 256, 64
    env = handle(n, 10, "ref", "f32", horizon=1000, burn_in=200)
    src = torch.arange(n, device="cuda").repeat_interleave(c)
    prefix = None
    if p:
        gen = torch.Generator(device="cuda")
        gen.manual_seed(1)
        prefix = torch.rand((p, n * c, 4), device="cuda", generator=gen) * 360.0 - 180.0
    got = check_fed(env, src, prefix, k, 2 ** 33 + 1, 0.99, True)
    assert bool((got.done != 0).any()) and bool((got.length == k).any())
