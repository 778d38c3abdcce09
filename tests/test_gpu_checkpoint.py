"""A checkpoint restored into a fresh handle continues bit for bit (-m gpu).

A checkpoint holds what include/manytor_b200.h lists next to mt_set_points: the config, get_state() (goals, alive,
total_reward, ep_len and the per-env reset counts that key the objective sampler and pick the objective stream's
set), the raw objectives and the step index.  Handle A runs on from the checkpoint; handle B, created with the same
config, reset and restored, makes the same calls.  Every output of every call, the final state and the statistics
gathered since the checkpoint must be the same bits on both.

  a. every driver (step with caller / sampled actions, rollout_random, rollout with caller / drawn actions and with
     final outputs, step(final=True), step_host) x the on-device sampler and a 3-set objective stream x every layout
     of the state: compile-time and run-time X, ep_len in bits 16-31, in bits 20-31 and in the wide counters array,
     binary16 observations, the UR5 preset, NVRTC and run-time DH tables, obs_after_reset both ways; ragged N off a
     tile boundary.
  b. re-sharded resume: one handle into two split off a warp boundary, and two into one.
  c. arbitrary reset counts (random, around 2^27 where count*32 wraps, 2^32 - 1 which wraps to 0) followed through
     several in-kernel resets against the fp64 restatement of the sampler.
  d. the reset counts against a plain count: done flags, masked resets, set_seed, masked set_state, guard bands.
  e. the benchmark's shape.
"""
import numpy as np
import pytest

from oracle import REFERENCE_ARM
from oracle.philox import device_points

from parity import ChunkedOracle, _seed_late_episode, half_ball_points, lockstep_auto_reset, lockstep_chunked, \
    philox_fresh

pytestmark = pytest.mark.gpu

SEED_HI = 0x1234567890ABCDEF               # both key words non-zero
BASE_RANK3 = 3 * (1 << 20) + 5             # the shard of rank 3 of a 2^20-env-per-GPU run, shifted off a tile boundary
N = 1000 + 13                              # not a multiple of 32
H = 4                                      # horizon: every env ends an episode at least every 4 steps
K = 3                                      # steps per rollout call (the multi-step kernel)
ADDITIVE = ("env_steps", "episodes", "terminated", "reward_sum", "length_sum", "catches", "ground_steps")


@pytest.fixture(scope="module")
def mt():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import manytor_b200
    manytor_b200.load_library()
    return manytor_b200


def _torch():
    import torch
    return torch


def _bits(t):
    """A tensor as integers of its width, so that equality is bit equality."""
    torch = _torch()
    t = t.contiguous()
    return t.view({4: torch.int32, 2: torch.int16}[t.element_size()]) if t.is_floating_point() else t


def _assert_same(u, v, what):
    torch = _torch()
    assert u.shape == v.shape and u.dtype == v.dtype, (what, u.shape, v.shape, u.dtype, v.dtype)
    eq = _bits(u) == _bits(v)
    if not bool(eq.all()):
        rows = torch.nonzero(~eq.reshape(eq.shape[0], -1).all(dim=1)).flatten() if eq.dim() else None
        raise AssertionError(f"{what}: differs (first rows {rows[:5].tolist() if rows is not None else ''})")


def _counts(env):
    """The reset counts as unsigned integers."""
    return env.get_state()["resets"].cpu().numpy().view(np.uint32).astype(np.int64)


def checkpoint(env):
    return dict(state={k: v.clone() for k, v in env.get_state().items()},
                points=env.get_points(zero_dead=False).clone(), step_index=env.step_index, stats=env.stats())


def restore(mt, ck, n, x, stream=None, **kw):
    """A fresh handle with the same config: reset (which advances the counts), then every part of the checkpoint."""
    env = mt.BatchedEnvs(n, x, **kw)
    if stream is not None:
        env.set_objective_stream(stream)
    env.reset()
    env.set_state(**ck["state"])
    env.set_points(ck["points"])
    env.step_index = ck["step_index"]
    return env


def _slice(ck, a, b):
    return dict(state={k: v[a:b] for k, v in ck["state"].items()}, points=ck["points"][a:b],
                step_index=ck["step_index"], stats=None)


def _join(cks):
    torch = _torch()
    assert len({c["step_index"] for c in cks}) == 1
    return dict(state={k: torch.cat([c["state"][k] for c in cks]) for k in cks[0]["state"]},
                points=torch.cat([c["points"] for c in cks]), step_index=cks[0]["step_index"], stats=None)


def assert_same_state(a, b, what=""):
    sa, sb = a.get_state(), b.get_state()
    assert set(sa) == {"goals", "alive", "total_reward", "ep_len", "resets"}
    for k in sa:
        _assert_same(sa[k], sb[k], f"{what} state {k}")
    _assert_same(a.get_points(zero_dead=False), b.get_points(zero_dead=False), f"{what} points")
    assert a.step_index == b.step_index


def assert_stats_since(a, ck_stats, b):
    """B's additive statistics are A's change since the checkpoint; the in-progress sum is A's."""
    sa, sb = a.stats(), b.stats()
    for k in ADDITIVE:
        assert sb[k] == sa[k] - ck_stats[k], (k, sb[k], sa[k], ck_stats[k])
    assert sb["live_reward_sum"] == sa["live_reward_sum"]


# --------------------------------------------------------------------------
# a. every driver x objectives x layouts
# --------------------------------------------------------------------------
LAYOUTS = [  # id, arm, x, fk_mode, obs dtype, obs_after_reset
    ("ref_x10", "ref", 10, 0, "float32", False),            # compile-time X, ep_len in bits 16-31
    ("ref_x10_oar", "ref", 10, 0, "float32", True),
    ("ref_x7_f16", "ref", 7, 0, "float16", False),          # run-time X, binary16 observations
    ("ref_x20_oar", "ref", 20, 0, "float32", True),         # ep_len in bits 20-31 (horizon <= 4095)
    ("ref_x32", "ref", 32, 0, "float32", False),            # ep_len in the counters array
    ("ur5_x10", "ur5", 10, 0, "float32", False),            # the UR5 preset
    ("j5_fk3_x9_oar", "j5", 9, 3, "float32", True),         # NVRTC step and rollout kernels
    ("j5_fk1_x9", "j5", 9, 1, "float16", False),            # run-time DH table: rollouts take one step kernel per step
]
DRIVERS = ["step", "sample_step", "rollout_random", "rollout_actions", "rollout_drawn", "rollout_final", "step_final",
           "step_host"]
SINGLE = {"step", "sample_step", "step_final", "step_host"}


def _arm(mt, name):
    from arms import arm_pair
    return {"ref": mt.REFERENCE_ARM, "ur5": mt.UR5_ARM, "j5": arm_pair(5)[1]}[name]


def _kw(mt, layout, seed=SEED_HI, base=BASE_RANK3):
    _, arm, x, fk_mode, dtype, oar = layout
    return x, dict(arm=_arm(mt, arm), device=0, seed=seed, env_id_base=base, fk_mode=fk_mode, auto_reset=True,
                   horizon=H, obs_after_reset=oar, obs_dtype=getattr(_torch(), dtype))


def _final_rows(fin, done):
    ended = done != 0
    return dict(final_obs=fin.obs[ended], final_return=fin.episode_return[ended],
                final_length=fin.episode_length[ended])


def _drive(env, driver, acts, t):
    """One call of `driver`; `acts` (K, N, J) are the call's caller actions (single-step drivers use slice 0).
    Returns the call's outputs, cloned; FinalInfo rows only where an episode ended (the others keep old contents)."""
    torch = _torch()
    if driver == "step":
        o, r, d = env.step(acts[0])
        out = dict(obs=o, reward=r, done=d)
    elif driver == "sample_step":
        a = env.sample_actions()
        o, r, d = env.step(a)
        out = dict(actions=a, obs=o, reward=r, done=d)
    elif driver == "step_final":
        o, r, d, fin = env.step(acts[0], final=True)
        out = dict(obs=o, reward=r, done=d, **_final_rows(fin, d))
    elif driver == "step_host":
        o, r, d = env.step_host(acts[0].cpu().numpy())
        out = dict(obs=torch.from_numpy(o.copy()), reward=torch.from_numpy(r.copy()), done=torch.from_numpy(d.copy()))
    elif driver == "rollout_random":
        o, r, d = env.rollout_random(K)
        out = dict(obs=o, reward=r, done=d)
    elif driver == "rollout_actions":
        tr = env.rollout(acts)
        out = dict(obs=tr.obs, reward=tr.reward, done=tr.done)
    elif driver == "rollout_drawn":
        tr = env.rollout(n_steps=K, record_actions=True)
        out = dict(obs=tr.obs, reward=tr.reward, done=tr.done, actions=tr.actions)
    else:                                                    # rollout_final: caller actions and in-kernel draws in turn
        tr, fin = env.rollout(acts, final=True) if t % 2 == 0 else env.rollout(n_steps=K, record_actions=True,
                                                                                  final=True)
        out = dict(obs=tr.obs, reward=tr.reward, done=tr.done, **_final_rows(fin, tr.done))
        if tr.actions is not None:
            out["actions"] = tr.actions
    return {k: v.clone() for k, v in out.items()}


def _burn_in(env, rs, n, j, steps=13):
    """Every env through several episodes, with counts that differ between envs: staggered episode lengths, two
    masked resets and caller actions."""
    torch = _torch()
    env.reset()
    env.set_state(ep_len=rs.randint(0, H, size=n).astype(np.int32))
    for t in range(steps):
        if t in (4, 9):
            env.reset(mask=rs.rand(n) < 0.3)
        env.step(torch.as_tensor(rs.randint(-180, 180, size=(n, j)), dtype=torch.float32, device="cuda"))


@pytest.mark.parametrize("objectives", ["sampler", "stream3"])
@pytest.mark.parametrize("driver", DRIVERS)
@pytest.mark.parametrize("layout", LAYOUTS, ids=[c[0] for c in LAYOUTS])
def test_restored_handle_continues_bit_for_bit(mt, layout, driver, objectives):
    torch = _torch()
    x, kw = _kw(mt, layout)
    j = kw["arm"].n_joints
    rs = np.random.RandomState(len(layout[0]) * 31 + DRIVERS.index(driver))
    stream = None
    if objectives == "stream3":                              # set e mod 3 for the e-th reset of an env
        stream = torch.tensor(half_ball_points(rs, (3, N, x), kw["arm"].radius), dtype=torch.float32, device="cuda")
    a = mt.BatchedEnvs(N, x, **kw)
    if stream is not None:
        a.set_objective_stream(stream)
    _burn_in(a, rs, N, j)
    ck = checkpoint(a)
    c0 = ck["state"]["resets"].cpu().numpy().view(np.uint32)
    assert c0.min() >= 3 and len(set(c0.tolist())) >= 3, "the checkpoint must hold varied reset counts"
    calls = 9 if driver in SINGLE else 4
    acts = [torch.as_tensor(rs.randint(-180, 180, size=(K, N, j)), dtype=torch.float32, device="cuda")
            for _ in range(calls)]
    want = [_drive(a, driver, acts[t], t) for t in range(calls)]
    b = restore(mt, ck, N, x, stream=stream, **kw)
    for t in range(calls):
        got = _drive(b, driver, acts[t], t)
        assert set(got) == set(want[t])
        for k in want[t]:
            _assert_same(want[t][k], got[k], f"call {t} {k}")
    assert_same_state(a, b)
    assert_stats_since(a, ck["stats"], b)
    assert (_counts(b) - c0 >= 2).all(), "every env must refresh its objectives after the restore"


# --------------------------------------------------------------------------
# b. re-sharded resume
# --------------------------------------------------------------------------
def _draws(env, t):
    """In-kernel draws: rollout_random(K) and rollout(n_steps=K) in turn."""
    if t % 2 == 0:
        return [v.clone() for v in env.rollout_random(K)]
    tr = env.rollout(n_steps=K, record_actions=True)
    return [tr.obs.clone(), tr.reward.clone(), tr.done.clone(), tr.actions.clone()]


@pytest.mark.parametrize("oar", [False, True])
def test_resharded_resume(mt, oar):
    """One handle of N envs checkpointed and restored as two shards split at a non-multiple of 32 (the second with
    env_id_base = base + cut), then two shards restored as one: with in-kernel draws and the sampler, every env
    depends on its global id alone, so the joined continuations equal the uninterrupted run bit for bit."""
    torch = _torch()
    n, cut, x = 2000 + 7, 1000 + 13, 10
    kw = dict(device=0, seed=SEED_HI, auto_reset=True, horizon=H, obs_after_reset=oar)
    calls = 4

    def run(envs):
        """`calls` calls on every shard; per call, each output joined over the shards along the env axis."""
        res = []
        for t in range(calls):
            per = [_draws(e, t) for e in envs]
            # rollout(n_steps=K) returns (K, N, ...) slices, rollout_random(K) the last step's (N, ...)
            res.append([torch.cat(vals, dim=1 if t % 2 else 0) for vals in zip(*per)])
        return res

    def compare(want, got, what):
        for t, (u, v) in enumerate(zip(want, got)):
            for i, (p, q) in enumerate(zip(u, v)):
                _assert_same(p, q, f"{what} call {t} output {i}")

    def join_state(envs):
        sts = [e.get_state() for e in envs]
        return ({k: torch.cat([s[k] for s in sts]) for k in sts[0]},
                torch.cat([e.get_points(zero_dead=False) for e in envs]))

    rs = np.random.RandomState(11)
    # one -> two
    one = mt.BatchedEnvs(n, x, env_id_base=BASE_RANK3, **kw)
    one.reset()
    one.set_state(ep_len=rs.randint(0, H, size=n).astype(np.int32))
    one.reset(mask=rs.rand(n) < 0.3)
    one.rollout_random(11)
    ck = checkpoint(one)
    two = [restore(mt, _slice(ck, 0, cut), cut, x, env_id_base=BASE_RANK3, **kw),
           restore(mt, _slice(ck, cut, n), n - cut, x, env_id_base=BASE_RANK3 + cut, **kw)]
    compare(run([one]), run(two), "one -> two")
    st, pts = join_state(two)
    for k, v in one.get_state().items():
        _assert_same(v, st[k], f"one -> two state {k}")
    _assert_same(one.get_points(zero_dead=False), pts, "one -> two points")
    s1, s2 = one.stats(), [e.stats() for e in two]
    for k in ADDITIVE:
        assert sum(s[k] for s in s2) == s1[k] - ck["stats"][k], k
    assert sum(s["live_reward_sum"] for s in s2) == s1["live_reward_sum"]
    assert all(e.step_index == one.step_index for e in two)

    # two -> one
    two = [mt.BatchedEnvs(cut, x, env_id_base=BASE_RANK3, **kw),
           mt.BatchedEnvs(n - cut, x, env_id_base=BASE_RANK3 + cut, **kw)]
    ep = rs.randint(0, H, size=n).astype(np.int32)
    mask = rs.rand(n) < 0.3
    for e, (lo, hi) in zip(two, ((0, cut), (cut, n))):
        e.reset()
        e.set_state(ep_len=ep[lo:hi])
        e.reset(mask=mask[lo:hi])
        e.rollout_random(11)
    cks = [checkpoint(e) for e in two]
    one = restore(mt, _join(cks), n, x, env_id_base=BASE_RANK3, **kw)
    compare(run(two), run([one]), "two -> one")
    st, pts = join_state(two)
    for k, v in one.get_state().items():
        _assert_same(st[k], v, f"two -> one state {k}")
    _assert_same(pts, one.get_points(zero_dead=False), "two -> one points")
    s1, s2 = one.stats(), [e.stats() for e in two]
    for k in ADDITIVE:
        assert s1[k] == sum(s[k] - c["stats"][k] for s, c in zip(s2, cks)), k
    assert s1["live_reward_sum"] == sum(s["live_reward_sum"] for s in s2)


# --------------------------------------------------------------------------
# c. arbitrary reset counts against the fp64 restatement
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["step", "rollout4"])
def test_set_reset_counts_against_restatement(mt, mode):
    """Reset counts set to arbitrary values -- random, around 2^27 (where count*32 wraps mod 2^32) and 2^32 - 1 and
    2^32 - 2 (the count wraps to 0 on a following reset) -- key the objectives of every later in-kernel reset: the
    oracle follows the device with device_points of the plain count, within point_tol_of, with no hard mismatch."""
    spec, arm = REFERENCE_ARM, mt.REFERENCE_ARM
    n, x, horizon, seed, base = 4096 + 17, 10, H, SEED_HI, BASE_RANK3
    rs = np.random.RandomState(5 + len(mode))
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, seed=seed, env_id_base=base, auto_reset=True, horizon=horizon)
    env.reset()
    ids = base + np.arange(n)
    ora = ChunkedOracle(n, x, spec)
    ora.reset(points=np.float32(device_points(seed, ids, 0, x, spec.radius)).astype(np.float64))
    _seed_late_episode(env, ora, rs, n, x, horizon, 0.1)
    kind = np.arange(n) % 8
    counts = rs.randint(0, 2 ** 32, size=n, dtype=np.int64)
    counts[kind == 1] = (1 << 27) - 3 + rs.randint(0, 4, size=int((kind == 1).sum()))
    counts[kind == 2] = 2 ** 32 - 1
    counts[kind == 3] = 2 ** 32 - 2
    counts[kind == 4] = 0
    env.set_state(resets=counts)
    np.testing.assert_array_equal(_counts(env), counts)
    episode = counts.copy()
    fresh = philox_fresh(seed, ids, x, spec.radius)
    if mode == "step":
        rep, stats, _, forked = lockstep_auto_reset(env, ora, spec, None, lambda t: rs.randint(-180, 180, size=(n, 4)),
                                                    12, horizon, fresh=fresh, episode=episode)
        assert not forked, "a near-threshold flip changed which envs reset"
        keep = np.ones(n, dtype=bool)
    else:
        rep, stats, dropped = lockstep_chunked(env, ora, spec, fresh, seed, 4, 3, horizon, episode=episode)
        keep = ~dropped
    print(rep.summary(), f"max point error {rep.max_point_err:.3e}")
    assert rep.ok(), rep.notes[:5]
    assert keep.sum() >= n - 8, "too many envs lost to near-threshold flips"
    np.testing.assert_array_equal(_counts(env)[keep], (episode & 0xFFFFFFFF)[keep])
    assert (episode - counts >= 3)[keep].all(), "every env must pass several in-kernel resets"
    assert (episode[kind == 2] >= 2 ** 32).all() and (episode[kind == 1] >= 1 << 27).all()   # both wraps were crossed


# --------------------------------------------------------------------------
# d. the reset counts against a plain count
# --------------------------------------------------------------------------
def test_reset_counts_follow_a_plain_count(mt):
    torch = _torch()
    n, x = N, 10
    rs = np.random.RandomState(3)
    env = mt.BatchedEnvs(n, x, device=0, seed=3, env_id_base=BASE_RANK3, auto_reset=True, horizon=5)
    assert (_counts(env) == 0).all()                                # a new handle has had no reset
    env.reset()
    assert (_counts(env) == 1).all()
    env.set_state(ep_len=rs.randint(0, 5, size=n).astype(np.int32))      # envs end at different steps
    # every done != 0 of a trajectory is one in-kernel reset
    c0 = _counts(env)
    tr = env.rollout(n_steps=23, record_actions=True)
    ends = (tr.done != 0).sum(dim=0).cpu().numpy()
    np.testing.assert_array_equal(_counts(env) - c0, ends)
    c0 = _counts(env)
    ends = np.zeros(n, dtype=np.int64)
    for _ in range(8):                                                  # 31 steps in all: not a multiple of 5
        ends += env.step(env.sample_actions())[2].cpu().numpy() != 0
    np.testing.assert_array_equal(_counts(env) - c0, ends)
    assert ends.max() > 0 and len(set(_counts(env).tolist())) > 1
    # a masked reset adds exactly one to the masked envs
    c0 = _counts(env)
    mask = rs.rand(n) < 0.4
    env.reset(mask=mask)
    np.testing.assert_array_equal(_counts(env), c0 + mask)
    # set_state(resets=..., mask=...) writes the masked envs only, and nothing else
    c0 = _counts(env)
    before = {k: v.clone() for k, v in env.get_state().items()}
    pts = env.get_points(zero_dead=False).clone()
    new = rs.randint(0, 2 ** 32, size=n, dtype=np.int64)
    m2 = rs.rand(n) < 0.5
    env.set_state(resets=new, mask=m2)
    np.testing.assert_array_equal(_counts(env), np.where(m2, new, c0))
    after = env.get_state()
    for k in ("goals", "alive", "total_reward", "ep_len"):
        _assert_same(before[k], after[k], k)
    _assert_same(pts, env.get_points(zero_dead=False), "points")
    env.set_state(resets=torch.from_numpy(new.astype(np.uint32).view(np.int32)).cuda())   # int32 bits, as get_state has them
    np.testing.assert_array_equal(_counts(env), new)
    # the getter writes exactly N words
    pad, fill = 4096, 0xA5
    raw = torch.full((4 * n + 2 * pad,), fill, dtype=torch.uint8, device="cuda")
    view = raw[pad:pad + 4 * n].view(torch.int32)
    assert env._lib.mt_get_reset_counts(env._h, view.data_ptr(), None) == 0
    torch.cuda.synchronize()
    assert bool((raw[:pad] == fill).all()) and bool((raw[-pad:] == fill).all()), "guard band written"
    np.testing.assert_array_equal(view.cpu().numpy().view(np.uint32), new)
    # set_seed zeroes the counts
    env.set_seed(9)
    assert (_counts(env) == 0).all()


# --------------------------------------------------------------------------
# e. the benchmark's shape
# --------------------------------------------------------------------------
def test_benchmark_shape(mt):
    """2^20 envs, X = 10, horizon 1000, bench.py's seed: staggered episode lengths and a burn-in with rollout_random
    (every env past one or two episode ends), checkpoint, restore, then two
    step calls (several tiles per warp) and one rollout_random(8) (the multi-step kernel), bit-equal to the original."""
    import bench
    torch = _torch()
    n, x = 1 << 20, bench.OBJ
    kw = dict(device=0, seed=bench.SEED, auto_reset=True, horizon=bench.HORIZON)
    a = mt.BatchedEnvs(n, x, **kw)
    a.reset()
    a.set_state(ep_len=np.random.RandomState(19).randint(0, bench.HORIZON, size=n).astype(np.int32))
    a.rollout_random(1500, write_obs=False)
    ck = checkpoint(a)
    c0 = ck["state"]["resets"].cpu().numpy().view(np.uint32)
    assert c0.min() >= 2 and c0.max() > c0.min()
    rs = np.random.RandomState(20)
    acts = [torch.as_tensor(rs.randint(-180, 180, size=(n, 4)), dtype=torch.float32, device="cuda") for _ in range(2)]
    want = [[v.clone() for v in a.step(act)] for act in acts] + [[v.clone() for v in a.rollout_random(8)]]
    b = restore(mt, ck, n, x, **kw)
    got = [[v.clone() for v in b.step(act)] for act in acts] + [[v.clone() for v in b.rollout_random(8)]]
    for t, (u, v) in enumerate(zip(want, got)):
        for name, p, q in zip(("obs", "reward", "done"), u, v):
            _assert_same(p, q, f"call {t} {name}")
    assert_same_state(a, b)
    assert_stats_since(a, ck["stats"], b)
