"""Branch rollouts (mt_rollout_branches, BatchedEnvs.rollout_branches) against a twin handle stepped with the same actions.

The expectation of every case comes from a twin handle of M envs with the source's configuration and auto_reset=False:
its goals, alive words, total rewards, episode lengths and raw objectives are gathered from the source handle by `src`,
and it is stepped K times with the same actions (mt_rollout, bit for bit K mt_step calls).  Its outputs give each
branch's length T (the first done step + 1, or K), the done byte of that step, the discounted return in the fp32 order
of the header (d_0 = 1, d_{s+1} = d_s gamma, G += d_s r_s) and obs2 at step T - 1.  Everything is compared bit for bit.
Branches of an NVRTC handle run the run-time-table kernel, so their twin is the run-time-table handle of the same table.
Sources are burnt in under auto-reset with a short horizon, so that branches end inside the rollout; one source sits at
horizon - 1 and truncates at step 0.  Every output buffer is prefilled with the byte 0xA5.
"""

import numpy as np
import pytest

from arms import arm_pair

pytestmark = pytest.mark.gpu

FILL = 0xA5
HORIZON = 12


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


def _dtype(obs):
    torch = _torch()
    return torch.float16 if obs == "f16" else torch.float32


def handle(n, x, arm="ref", obs="f32", tog=False, horizon=HORIZON, seed=11, auto_reset=True, burn_in=5, reset=True):
    """A source handle: n envs burnt in with `burn_in` random steps; env n // 2 then sits at horizon - 1 (horizon > 0)."""
    from manytor_b200 import BatchedEnvs
    spec, fk_mode = _arm(arm)
    env = BatchedEnvs(n, x, arm=spec, device=0, horizon=horizon, seed=seed, fk_mode=fk_mode, auto_reset=auto_reset,
                      terminate_on_ground=tog, obs_dtype=_dtype(obs))
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


def twin_of(env, src):
    """A handle of len(src) envs, auto_reset off, whose env m holds the state and raw objectives of env src[m].  The twin
    of an NVRTC handle (fk_mode=3) takes the run-time table (fk_mode=1): branches of such a handle run the run-time-table
    kernel, whose positions may differ in the last bits from the NVRTC-specialised ones."""
    from manytor_b200 import BatchedEnvs
    torch = _torch()
    cfg = env.cfg
    fk_mode = 1 if cfg.fk_mode == 3 else cfg.fk_mode
    twin = BatchedEnvs(len(src), env.x, arm=env.arm, device=0, horizon=cfg.horizon, seed=cfg.seed, fk_mode=fk_mode,
                       auto_reset=False, terminate_on_ground=bool(cfg.terminate_on_ground), obs_dtype=env.obs_dtype)
    twin.reset()
    st = env.get_state()
    pts = env.get_points(zero_dead=False)
    s = src.to(torch.int64)
    twin.set_state(goals=st["goals"][s], alive=st["alive"][s], total_reward=st["total_reward"][s], ep_len=st["ep_len"][s])
    twin.set_points(pts[s])
    return twin


def expected(env, src, actions, gamma, write_obs):
    """(ret, length, done, obs or None, reward at the ending step) from a twin, for the sources inside [0, N); the
    others are computed from env 0, as the kernel computes them (their rows are checked separately)."""
    torch = _torch()
    k, m = actions.shape[0], actions.shape[1]
    src = torch.arange(env.n, device="cuda") if src is None else torch.as_tensor(src, device="cuda").to(torch.int64)
    ok = (src >= 0) & (src < env.n)
    twin = twin_of(env, torch.where(ok, src, torch.zeros_like(src)))
    traj = twin.rollout(actions, write_obs=write_obs)
    twin.close()
    steps = torch.arange(k, device="cuda")[:, None].expand(k, m)
    ended = traj.done != 0
    first = torch.where(ended, steps, torch.full_like(steps, k)).min(dim=0).values
    any_end = first < k
    length = torch.where(any_end, first + 1, torch.full_like(first, k)).to(torch.int32)
    last = (length - 1).long()
    rows = torch.arange(m, device="cuda")
    done = torch.where(any_end, traj.done[last, rows], torch.zeros_like(traj.done[0]))
    ret = torch.zeros(m, dtype=torch.float32, device="cuda")
    d = torch.ones((), dtype=torch.float32, device="cuda")
    g = torch.tensor(gamma, dtype=torch.float32, device="cuda")
    for s in range(k):
        ret = torch.where(s < length, ret + d * traj.reward[s], ret)
        d = d * g
    obs = traj.obs[last, rows] if write_obs else None
    return ret, length, done, obs, traj.reward[last, rows], ok


def check(env, src, actions, gamma, write_obs):
    """Run rollout_branches into prefilled buffers and compare with the twin; returns (done, reward at the end)."""
    torch = _torch()
    m = actions.shape[1]
    out = filled(env, m, write_obs)
    l0 = env.launch_count
    got = env.rollout_branches(actions, src, gamma=gamma, write_obs=write_obs, out=out)
    torch.cuda.synchronize()
    assert got is out
    assert env.launch_count == l0 + 1
    ret, length, done, obs, r_end, ok = expected(env, src, actions, gamma, write_obs)
    assert torch.equal(bits(got.ret[ok]), bits(ret[ok]))
    assert torch.equal(got.length[ok], length[ok])
    assert torch.equal(got.done[ok], done[ok])
    assert bool(got.ret[~ok].isnan().all())
    assert bool((got.length[~ok] == -1).all()) and bool((got.done[~ok] == 0).all())
    if write_obs:
        assert torch.equal(bits(got.obs[ok]), bits(obs[ok]))
        assert bool((got.obs[~ok].view(torch.uint8) == FILL).all())
    return done[ok], r_end[ok], length[ok]


def sources(kind, n, rs):
    torch = _torch()
    if kind == "identity":
        return None
    if kind == "cand":                                 # C = 3 candidates per env, then 5 more: M = 3N + 5
        s = np.concatenate([np.repeat(np.arange(n), 3), rs.randint(0, n, size=5)])
    else:
        s = rs.randint(0, n, size=int(kind.split("_")[1]))
    return torch.tensor(s, dtype=torch.int64, device="cuda")


CONFIGS = [  # arm, X, observations, terminate_on_ground
    ("ref", 10, "f32", False), ("ref", 20, "f16", True), ("ref", 7, "off", True), ("ref", 32, "f32", False),
    ("ur5", 10, "f16", False), ("ur5", 20, "f32", True), ("ur5", 7, "off", False),
    ("rt_j7", 7, "f32", True), ("rt_j7", 32, "off", False), ("rt_j7", 10, "f16", False),
    ("jit_j5", 10, "f32", True), ("jit_j5", 20, "f16", False), ("jit_j5", 32, "off", True),
]
RUNS = [  # gamma, K, sources (identity: M = N; cand: M = 3N + 5; rand_M: M random sources with repeats)
    (1.0, 17, "identity"), (0.99, 64, "cand"), (0.0, 2, "rand_33"), (0.99, 1, "rand_1000"), (1.0, 64, "rand_1"),
]


@pytest.mark.parametrize("arm, x, obs, tog", CONFIGS)
def test_branches_match_a_twin(arm, x, obs, tog):
    torch = _torch()
    n = 1000
    env = handle(n, x, arm, obs, tog)
    rs = np.random.RandomState(5)
    ends = []
    for i, (gamma, k, kind) in enumerate(RUNS):
        src = sources(kind, n, rs)
        m = n if src is None else len(src)
        done, _, length = check(env, src, caller_actions(k, m, env.j, 100 + i), gamma, obs != "off")
        ends.append(done)
        if kind == "identity":
            assert int(length[n // 2]) == 1 and int(done[n // 2]) != 0     # the source at horizon - 1
    assert bool((torch.cat(ends) != 0).any())          # branches end inside the rollout (kinds: test_every_kind_of_ending)


def _prime_catches(env, actions, envs):
    """Leave only objective 0 alive in each of `envs`, placed on the catch frame of its branch's first action."""
    torch = _torch()
    catcher = env.joints_of(actions[0])[:, env.arm.catch_frame - 1]
    pts = env.get_points(zero_dead=False)
    st = env.get_state()
    idx = torch.tensor(envs, device="cuda")
    pts[idx, 0] = catcher[idx]
    st["alive"][idx] = 1
    env.set_points(pts)
    env.set_state(alive=st["alive"])


@pytest.mark.parametrize("arm", ["ref", "ur5", "rt_j7", "jit_j5"])
def test_every_kind_of_ending(arm):
    """Branches end on the ground (terminate_on_ground), by truncation at the horizon, and by catching every objective;
    the others run all K steps.  Each kind gets the handle where it is certain to occur: UR5 under terminate_on_ground,
    for one, ends nearly every branch on the ground before any horizon."""
    n, k = 999, 17
    ground = handle(n, 10, arm, "f32", tog=True)
    done, r_end, _ = check(ground, None, caller_actions(k, n, ground.j, 3), 0.99, True)
    assert bool((((done & 1) != 0) & (r_end == -1.0)).any()), "no branch ended on the ground"
    trunc = handle(n, 10, arm, "f32", tog=False)
    done, _, _ = check(trunc, None, caller_actions(k, n, trunc.j, 5), 0.99, True)
    assert bool((done == 2).any()), "no branch was truncated"
    free = handle(n, 10, arm, "f32", tog=False, horizon=0)
    actions = caller_actions(k, n, free.j, 4)
    _prime_catches(free, actions, list(range(1, n, 37)))
    done, _, length = check(free, None, actions, 0.99, True)
    assert bool((done == 1).any()), "no branch ended by catching everything"
    assert bool((done == 0).any()) and bool((length[done == 0] == k).all())


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
    for i, (gamma, k, kind) in enumerate(RUNS):
        src = sources(kind, n, rs)
        m = n if src is None else len(src)
        a.rollout_branches(caller_actions(k, m, a.j, 40 + i), src, gamma=gamma, write_obs=obs != "off")
    _assert_same_handle(a, b)
    acts = caller_actions(20, n, a.j, 9)
    ta, tb = a.rollout(acts, write_obs=obs != "off"), b.rollout(acts, write_obs=obs != "off")
    for u, v in zip(ta, tb):
        if u is not None:
            assert torch.equal(bits(u), bits(v))
    _assert_same_handle(a, b)


def test_out_of_range_sources():
    torch = _torch()
    n = 500
    env = handle(n, 10, "ref", "f32", tog=True)
    rs = np.random.RandomState(8)
    src = torch.tensor(rs.randint(0, n, size=300), dtype=torch.int64, device="cuda")
    bad = torch.tensor([0, 31, 32, 150, 299], device="cuda")
    src[bad] = torch.tensor([-1, n, 2 ** 40, -(2 ** 40), 2 ** 31], dtype=torch.int64, device="cuda")
    check(env, src, caller_actions(17, 300, env.j, 1), 0.99, True)
    check(env, src, caller_actions(3, 300, env.j, 2), 1.0, False)


def test_nothing_to_do_and_state_errors():
    torch = _torch()
    from manytor_b200 import MantorLibraryError
    from manytor_b200 import _lib
    env = handle(64, 10, "ref", "f32")
    for k, m in ((0, 64), (5, 0)):
        out = filled(env, m, True)
        env.rollout_branches(caller_actions(k, m, env.j, 1), None if m == 64 else np.zeros(0, np.int64), write_obs=True,
                             out=out)
        torch.cuda.synchronize()
        for t in out:
            assert bool((t.view(torch.uint8) == FILL).all())
    # the same through the C ABI, with real buffers
    out = filled(env, 64, True)
    src = torch.arange(64, device="cuda")
    acts = caller_actions(4, 64, env.j, 1)
    l0 = env.launch_count
    for k, m in ((0, 64), (4, 0)):
        assert env._lib.mt_rollout_branches(env._h, k, m, src.data_ptr(), acts.data_ptr(), 1.0, out.ret.data_ptr(),
                                            out.length.data_ptr(), out.done.data_ptr(), out.obs.data_ptr(), None) == 0
    torch.cuda.synchronize()
    assert env.launch_count == l0
    for t in out:
        assert bool((t.view(torch.uint8) == FILL).all())
    fresh = handle(64, 10, "ref", "f32", reset=False)
    with pytest.raises(MantorLibraryError, match="mt_rollout_branches before mt_reset"):
        fresh.rollout_branches(acts, src)
    assert fresh._lib.mt_rollout_branches(fresh._h, 4, 64, src.data_ptr(), acts.data_ptr(), 1.0, out.ret.data_ptr(),
                                          out.length.data_ptr(), out.done.data_ptr(), None, None) == -4   # MT_ERR_STATE
    assert _lib.load().mt_last_error() == b"mt_rollout_branches before mt_reset"


@pytest.mark.parametrize("obs", ["f32", "off"])
def test_cuda_graph_replay_equals_eager(obs):
    torch = _torch()
    n, k = 640, 24
    env = handle(n, 10, "ref", obs, tog=True)
    rs = np.random.RandomState(4)
    src = torch.tensor(rs.randint(0, n, size=2 * n + 3), dtype=torch.int64, device="cuda")
    acts = caller_actions(k, len(src), env.j, 6)
    eager = env.rollout_branches(acts, src, gamma=0.97, write_obs=obs != "off")
    eager = [t.clone() if t is not None else None for t in eager]
    out = filled(env, len(src), obs != "off")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        env.rollout_branches(acts, src, gamma=0.97, write_obs=obs != "off", out=out)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for t in out:
        if t is not None:
            t.view(torch.uint8).fill_(FILL)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env.rollout_branches(acts, src, gamma=0.97, write_obs=obs != "off", out=out)
    g.replay()
    torch.cuda.synchronize()
    for u, v in zip(out, eager):
        if u is not None:
            assert torch.equal(bits(u), bits(v))


def test_benchmark_shape():
    """4096 sources x 256 candidates = 2^20 branches, K = 64, burnt in with horizon 1000, against the twin."""
    torch = _torch()
    n, c, k = 4096, 256, 64
    env = handle(n, 10, "ref", "f32", horizon=1000, burn_in=200)
    src = torch.arange(n, device="cuda").repeat_interleave(c)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1)
    acts = torch.rand((k, n * c, 4), device="cuda", generator=gen) * 360.0 - 180.0
    done, _, length = check(env, src, acts, 0.99, True)
    assert bool((done != 0).any()) and bool((length == k).any())
