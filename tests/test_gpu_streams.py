"""Handles driven from non-default streams, and several handles running at once on one GPU (-m gpu).

RL code steps its environments on a side stream so that they overlap with the learner, keeps train and eval
environments as two handles on one device, and replays CUDA graphs captured on a pool stream.  PyTorch's pool
streams are non-blocking: the legacy default stream, on which the library's synchronous calls run, does not wait
for them.  BatchedEnvs therefore makes its synchronous calls wait for the handle's last non-default stream.

The expected value of a case comes from a twin handle wherever possible: same configuration, seed and env_id_base,
driven the same way on the default stream with a host synchronisation after every call (the rest of the suite pins
those paths to the oracle).  To make a wrong order show every time, the work under test is queued behind a bounded
delay (torch.cuda._sleep) on its stream, and every such case asserts that the stream was still busy when the call
under test was issued, so that no case can pass without exercising the order.

  a. each synchronous call (stats, step_index get / set, fetch_env, step_host staged and zero-copy, the vector
     env's episode_statistics, set_seed, the drop-in Environment / Multienv) issued right after side-stream work
     sees that work;
  b. every asynchronous entry point stays on the stream it is called on (fp32 and fp16 observations);
  c. six handles of different kernels (closed form, UR5 preset, NVRTC, run-time table, fp16 with small blocks, and
     a twin of the first) on their own streams with no host synchronisation between them, each bit-equal to the
     same handle run alone;
  d. lock step with the fp64 oracle while four handles run concurrently, with auto-reset and on-device objectives;
  e. step_host of one handle while another runs a long rollout_random on a side stream;
  f. a graph captured on a side stream and replayed on another non-default stream.
"""
import numpy as np
import pytest

from arms import arm_pair
from oracle import REFERENCE_ARM as ORACLE_REF, UR5_ARM as ORACLE_UR5
from oracle.philox import device_actions, device_points
from parity import ChunkedOracle, Report, _seed_late_episode, lockstep_auto_reset, philox_fresh

pytestmark = pytest.mark.gpu

SEED = 0x1234567890ABCDEF
BASE = 3 * (1 << 20) + 5            # env_id_base off a tile boundary
HORIZON = 12
DELAY = 80_000_000                  # torch.cuda._sleep cycles: about 40 ms at the B200's 1.965 GHz boost clock


def _torch():
    import torch
    return torch


@pytest.fixture(scope="module")
def mt():
    torch = _torch()
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import manytor_b200
    manytor_b200.load_library()
    return manytor_b200


@pytest.fixture
def side():
    """A pool stream (non-blocking, like every torch.cuda.Stream) ordered after what the test set up so far."""
    torch = _torch()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    yield s
    torch.cuda.synchronize()


def delay():
    """A bounded delay on the current stream: work queued behind it runs tens of milliseconds later."""
    _torch().cuda._sleep(DELAY)


def assert_busy(stream, what=""):
    assert not stream.query(), f"{what}: the stream finished its work before the call under test: the case would prove nothing"


def handle(mt, n=4096 + 17, x=10, arm=None, reset=True, **kw):
    kw.setdefault("auto_reset", True)
    kw.setdefault("horizon", HORIZON)
    env = mt.BatchedEnvs(n, x, arm=arm or mt.REFERENCE_ARM, device=0, seed=SEED, env_id_base=BASE, **kw)
    if reset:
        env.reset()
    return env


def twins(mt, burn_in=5, **kw):
    """Two identical handles, spread over their episodes by `burn_in` in-kernel steps."""
    a, b = handle(mt, **kw), handle(mt, **kw)
    for h in (a, b):
        h.rollout_random(burn_in, write_obs=False)
    _torch().cuda.synchronize()
    return a, b


def actions(n, j, seed, k=None):
    """Continuous degrees on the device, some outside the action range."""
    torch = _torch()
    rs = np.random.RandomState(seed)
    a = rs.uniform(-180.0, 180.0, size=((k,) if k else ()) + (n, j))
    a[..., ::7, :] *= 3.0
    return torch.tensor(a, dtype=torch.float32, device="cuda")


def ids_of(env):
    return np.uint64(env.cfg.env_id_base) + np.arange(env.n, dtype=np.uint64)


def state_of(env):
    """Everything a handle holds, read after a device synchronisation: state, objectives, statistics, step index."""
    torch = _torch()
    torch.cuda.synchronize()
    st = {k: v.cpu().numpy() for k, v in env.get_state().items()}
    st["points"] = env.get_points(zero_dead=False).cpu().numpy()
    st["stats"] = env.stats()
    st["step_index"] = env.step_index
    return st


def assert_same_state(a, b, what=""):
    sa, sb = state_of(a), state_of(b)
    for k in sa:
        if isinstance(sa[k], np.ndarray):
            np.testing.assert_array_equal(sa[k], sb[k], err_msg=f"{what} {k}")
        else:
            assert sa[k] == sb[k], (what, k, sa[k], sb[k])


def as_numpy(out):
    """Flatten (nested tuples of) tensors / arrays into a list of numpy copies."""
    torch = _torch()
    if out is None:
        return [None]
    if isinstance(out, torch.Tensor):
        return [out.cpu().numpy()]
    if isinstance(out, np.ndarray):
        return [out.copy()]
    if isinstance(out, dict):
        return [v for k in sorted(out) for v in as_numpy(out[k])]
    if isinstance(out, (tuple, list)):
        return [v for o in out for v in as_numpy(o)]
    return [out]


def assert_same(got, want, what=""):
    got, want = as_numpy(got), as_numpy(want)
    assert len(got) == len(want), what
    for i, (g, w) in enumerate(zip(got, want)):
        if isinstance(w, np.ndarray):
            np.testing.assert_array_equal(g, w, err_msg=f"{what} output {i}")
        else:
            assert g == w, (what, i, g, w)


def clone(out):
    """Copies of a call's tensors, taken on the current stream (step outputs are buffers the next step reuses)."""
    torch = _torch()
    if isinstance(out, torch.Tensor):
        return out.clone()
    if isinstance(out, tuple):
        return type(out)(*(clone(o) for o in out)) if hasattr(out, "_fields") else tuple(clone(o) for o in out)
    if isinstance(out, dict):
        return {k: clone(v) for k, v in out.items()}
    return out


def ended_only(out):
    """A final=True result with the FinalInfo rows of envs that did not end zeroed (those rows keep whatever an
    earlier call left there).  torch.where, not boolean indexing: no host synchronisation on a busy stream."""
    torch = _torch()
    if isinstance(out[0], tuple):                           # rollout: (Trajectory, FinalInfo)
        done, fin = out[0].done, out[1]
    else:                                                   # step: (obs, reward, done, FinalInfo)
        done, fin = out[2], out[-1]
    m = done != 0
    fin = type(fin)(torch.where(m[..., None], fin.obs, torch.zeros_like(fin.obs)),
                    torch.where(m, fin.episode_return, torch.zeros_like(fin.episode_return)),
                    torch.where(m, fin.episode_length, torch.zeros_like(fin.episode_length)))
    return out[:-1] + (fin,)


# --------------------------------------------------------------------------
# a. synchronous calls after side-stream work
# --------------------------------------------------------------------------
def _side_step(env, side, act):
    torch = _torch()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        delay()
        env.step(act)


def case_stats(mt, side, monkeypatch):
    a, b = twins(mt)
    act = actions(a.n, a.j, 1)
    b.step(act)
    want = b.stats()
    _side_step(a, side, act)
    assert_busy(side)
    assert a.stats() == want
    assert_same_state(a, b)


def case_step_index_get(mt, side, monkeypatch):
    a, b = twins(mt)
    act = actions(a.n, a.j, 2)
    b.step(act)
    want = b.step_index
    _side_step(a, side, act)
    assert_busy(side)
    assert a.step_index == want
    assert_same_state(a, b)


def case_step_index_set(mt, side, monkeypatch):
    """The setter after a side-stream rollout: the rollout draws at the old index, and the index ends as set."""
    torch = _torch()
    a, b = twins(mt)
    old, new = b.step_index, 1 << 40
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        delay()
        rec = a.rollout(n_steps=1, record_actions=True)
    assert_busy(side)
    a.step_index = new
    torch.cuda.synchronize()
    assert a.step_index == new
    np.testing.assert_array_equal(rec.actions[0].cpu().numpy(), device_actions(SEED, ids_of(a), old, a.j))


def case_sample_after_set(mt, side, monkeypatch):
    """A side-stream draw right after the setter draws at the new index."""
    torch = _torch()
    a, b = twins(mt)
    new = (1 << 40) + 3
    _side_step(a, side, actions(a.n, a.j, 3))
    assert_busy(side)
    a.step_index = new
    with torch.cuda.stream(side):
        drawn = a.sample_actions()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(drawn.cpu().numpy(), device_actions(SEED, ids_of(a), new, a.j))
    assert a.step_index == new


def case_fetch_env(mt, side, monkeypatch):
    a, b = twins(mt)
    act = actions(a.n, a.j, 4)
    b.step(act)
    rows = [0, 1, 777, a.n - 1]
    want = [b.fetch_env(i) for i in rows]
    _side_step(a, side, act)
    assert_busy(side)
    got = [a.fetch_env(i) for i in rows]
    st = state_of(a)
    for i, g, w in zip(rows, got, want):
        assert_same(g, w, f"env {i}")
        np.testing.assert_array_equal(g["goals"], st["goals"][i])
        assert np.float32(g["total_reward"]) == st["total_reward"][i]
        alive = int(st["alive"][i]) & 0xFFFFFFFF
        np.testing.assert_array_equal(g["alives"], [(alive >> p) & 1 for p in range(a.x)])


def _case_step_host(zero_copy):
    def case(mt, side, monkeypatch):
        monkeypatch.setenv("MT_HOST_ZEROCOPY", zero_copy)    # read by each handle's first step_host
        a, b = twins(mt)
        act = actions(a.n, a.j, 5)
        host = np.random.RandomState(6).randint(-180, 180, size=(a.n, a.j)).astype(np.float32)
        b.step(act)
        want = as_numpy(b.step_host(host))
        _side_step(a, side, act)
        assert_busy(side)
        got = a.step_host(host)
        assert_same(got, want)
        assert a.host_step_mode == b.host_step_mode == {"0": "staged", "1": "zero-copy"}[zero_copy]
        assert_same_state(a, b)
    return case


def case_episode_statistics(mt, side, monkeypatch):
    torch = _torch()
    envs = [mt.ManyTorVectorEnv(4096 + 17, 10, max_episode_steps=4, seed=SEED, env_id_base=BASE) for _ in range(2)]
    for v in envs:
        v.reset(seed=SEED)
        v.envs.rollout_random(3, write_obs=False)
    act = actions(envs[0].num_envs, 4, 7)
    envs[1].step(act)
    want = envs[1].episode_statistics()
    assert want["episodes"] > 0
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        delay()
        envs[0].step(act)
    assert_busy(side)
    assert envs[0].episode_statistics() == want


def case_set_seed(mt, side, monkeypatch):
    torch = _torch()
    a, b = twins(mt)
    act = actions(a.n, a.j, 8)
    b.step(act)
    b.set_seed(5)
    _side_step(a, side, act)
    assert_busy(side)
    a.set_seed(5)
    assert_same_state(a, b)
    with torch.cuda.stream(side):
        got = a.sample_actions()
    assert_same(got, b.sample_actions())


def case_dropin_multienv(mt, side, monkeypatch):
    torch = _torch()
    import manytor_b200.manytor as tor

    def run(env, stream):                           # stream None: the default stream, no delay
        rs = np.random.RandomState(9)
        out = []
        torch.cuda.synchronize()                    # the handle's creation
        with torch.cuda.stream(stream):
            if stream is not None:
                delay()
            env.reset()
            for t in range(4):
                act = rs.randint(-180, 180, size=(env.env_number, 4)).astype(np.float32)
                if stream is not None and t == 0:
                    assert_busy(stream)
                out += as_numpy(env.step(act))
                out += [np.array(v) for i in (0, 5, env.env_number - 1) for v in
                        (env.environment[i].goals, env.environment[i].alives, env.environment[i].points,
                         env.environment[i].joints_coordinates, env.environment[i].total_reward)]
        return out

    want = run(tor.Multienv((3, 7), 10, as_lists=False, seed=SEED, horizon=3, auto_reset=True), None)
    got = run(tor.Multienv((3, 7), 10, as_lists=False, seed=SEED, horizon=3, auto_reset=True), side)
    assert_same(got, want)


def case_dropin_environment(mt, side, monkeypatch):
    torch = _torch()
    import manytor_b200.manytor as tor

    def run(env, stream):
        rs = np.random.RandomState(10)
        out = []
        torch.cuda.synchronize()                    # the handle's creation
        with torch.cuda.stream(stream):
            if stream is not None:
                delay()
            env.reset()
            for t in range(6):
                if stream is not None and t == 0:
                    assert_busy(stream)
                out += as_numpy(env.step(rs.randint(-180, 180, size=4)))
                out += [np.array(v) for v in (env.goals, env.alives, env.points, env.joints_coordinates,
                                              env.total_reward)]
        return out

    want = run(tor.Environment(10, index=3, seed=SEED), None)
    got = run(tor.Environment(10, index=3, seed=SEED), side)
    assert_same(got, want)


_SYNC_CASES = {
    "stats": case_stats,
    "step_index_get": case_step_index_get,
    "step_index_set": case_step_index_set,
    "sample_after_set": case_sample_after_set,
    "fetch_env": case_fetch_env,
    "step_host_staged": _case_step_host("0"),
    "step_host_zero_copy": _case_step_host("1"),
    "episode_statistics": case_episode_statistics,
    "set_seed": case_set_seed,
    "dropin_multienv": case_dropin_multienv,
    "dropin_environment": case_dropin_environment,
}


@pytest.mark.parametrize("case", sorted(_SYNC_CASES))
def test_synchronous_call_sees_side_stream_work(mt, side, monkeypatch, case):
    _SYNC_CASES[case](mt, side, monkeypatch)


# --------------------------------------------------------------------------
# b. asynchronous entry points stay on their stream
# --------------------------------------------------------------------------
def _async_segments(n, j):
    """(name, fn(env, check)): a state-changing call and the calls under test; `check()` marks the point where the
    stream must still be busy (before set_state, which synchronises its stream)."""
    torch = _torch()
    k = 5
    act = actions(n, j, 11)
    traj = actions(n, j, 12, k)
    mask = torch.tensor(np.random.RandomState(13).rand(n) < 0.4, device="cuda")
    goals = actions(n, j, 14)
    words = torch.tensor(np.random.RandomState(15).randint(1, 1 << 10, size=n), dtype=torch.int32, device="cuda")
    total = torch.full((n,), -3.0, device="cuda")
    ep_len = torch.tensor(np.random.RandomState(16).randint(0, HORIZON, size=n), dtype=torch.int32, device="cuda")

    def then(*calls):
        def fn(e, check):
            out = tuple(clone(c(e)) for c in calls)
            check()
            return out
        return fn

    def set_state(e, check):
        out = clone(e.step(act))
        check()
        e.set_state(goals=goals, alive=words, total_reward=total, ep_len=ep_len, mask=mask)
        return out, clone(e.get_state()), clone(e.observe())

    return [
        ("reset(mask), observe", then(lambda e: e.reset(mask=mask), lambda e: e.observe())),
        ("step(joints=True), observe", then(lambda e: e.step(act, joints=True), lambda e: e.observe())),
        ("step, step(final=True)", then(lambda e: e.step(traj[0]), lambda e: ended_only(e.step(traj[1], final=True)))),
        ("sample_actions, rollout_random", then(lambda e: e.sample_actions(), lambda e: e.rollout_random(k))),
        ("rollout(actions)", then(lambda e: e.rollout(traj), lambda e: e.get_state())),
        ("rollout(draws)", then(lambda e: e.rollout(n_steps=k, record_actions=True), lambda e: e.get_state())),
        ("rollout(actions, final=True)", then(lambda e: ended_only(e.rollout(traj, final=True)), lambda e: e.get_points())),
        ("rollout(draws, final=True)",
         then(lambda e: ended_only(e.rollout(n_steps=k, record_actions=True, final=True)),
              lambda e: e.get_points(zero_dead=False))),
        ("step, get_state, get_points", then(lambda e: e.step(act), lambda e: e.get_state(),
                                             lambda e: e.get_points(zero_dead=False))),
        ("rollout_random, stats_tensor, clear_stats, stats_tensor",
         then(lambda e: e.rollout_random(3), lambda e: e.stats_tensor(), lambda e: e.clear_stats(),
              lambda e: e.step(act), lambda e: e.stats_tensor())),
        ("step, set_state", set_state),
    ]


@pytest.mark.parametrize("obs_dtype", ["float32", "float16"])
def test_asynchronous_calls_stay_on_their_stream(mt, side, obs_dtype):
    """On a busy side stream, each state-changing call and the calls after it give what the twin gives on the
    default stream: an internal launch or copy on another stream would run ahead of the delay and differ."""
    torch = _torch()
    a, b = twins(mt, obs_dtype=getattr(torch, obs_dtype))
    segs = _async_segments(a.n, a.j)
    # a warm-up pass on both, `a` on the side stream: no allocation (PyTorch caches blocks per stream) and no first
    # launch of a kernel happens behind the delay
    for h, s in ((a, side), (b, None)):
        with torch.cuda.stream(s):
            for _, fn in segs:
                fn(h, lambda: None)
                torch.cuda.synchronize()
    assert_same_state(a, b, "warm-up")
    for what, fn in segs:
        want = as_numpy(fn(b, torch.cuda.synchronize))
        torch.cuda.synchronize()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            delay()
            got = fn(a, lambda: assert_busy(side, what))
        torch.cuda.synchronize()
        assert_same(got, want, what)
    assert_same_state(a, b)


# --------------------------------------------------------------------------
# c. handles side by side, each on its own stream
# --------------------------------------------------------------------------
def _side_by_side_handles(mt):
    """(name, constructor): reference arm filling every SM, UR5 preset, NVRTC, run-time table (per-step rollouts),
    fp16 with small blocks, and a twin of the first."""
    torch = _torch()
    j5, j7 = arm_pair(5)[1], arm_pair(7)[1]
    return [
        ("ref_x10_2p18", lambda: handle(mt, 1 << 18, 10)),
        ("ur5_x20", lambda: handle(mt, 40000 + 3, 20, arm=mt.UR5_ARM)),
        ("nvrtc_j5_x12", lambda: handle(mt, 30000 + 7, 12, arm=j5, fk_mode=3)),
        ("table_j7_x9", lambda: handle(mt, 20000 + 9, 9, arm=j7, fk_mode=1)),
        ("f16_x7_4097", lambda: handle(mt, 4097, 7, obs_dtype=torch.float16)),
        ("ref_x10_2p18_twin", lambda: handle(mt, 1 << 18, 10)),
    ]


def _mixed_sequence(env, k=5):
    """Inputs of the mixed call sequence of one handle, made on the current stream."""
    torch = _torch()
    seed = env.n + env.x
    # one tensor per call: a slice of a larger one need not be 16-byte aligned
    return dict(act=[actions(env.n, env.j, seed + i) for i in range(2)],
                traj=[actions(env.n, env.j, seed + 2 + i, k) for i in range(2)],
                mask=torch.tensor(np.random.RandomState(seed).rand(env.n) < 0.3, device="cuda"), k=k)


def _run_mixed(env, inp):
    """step, step(final=True), rollout(K), rollout(K, final=True), rollout_random(7), reset(mask), sample_actions:
    one generator step per call, every output cloned on the current stream."""
    yield clone(env.step(inp["act"][0]))
    yield clone(ended_only(env.step(inp["act"][1], final=True)))
    yield clone(env.rollout(inp["traj"][0]))
    yield clone(ended_only(env.rollout(inp["traj"][1], final=True)))
    yield clone(env.rollout_random(7))
    env.reset(mask=inp["mask"])
    yield clone(env.observe())
    yield clone(env.sample_actions())


def test_handles_side_by_side(mt):
    """Six handles on six streams, their calls interleaved with no host synchronisation: each one's outputs, state,
    objectives, eight statistics words and step index equal the same handle run alone, bit for bit."""
    torch = _torch()
    makers = _side_by_side_handles(mt)
    alone = {}
    for name, make in makers:
        env = make()
        inp = _mixed_sequence(env)
        outs = []
        for o in _run_mixed(env, inp):
            torch.cuda.synchronize()
            outs.append(as_numpy(o))
        alone[name] = (outs, state_of(env))
        env.close()
    envs = [(name, make()) for name, make in makers]
    streams = [torch.cuda.Stream() for _ in envs]
    inputs = [_mixed_sequence(env) for _, env in envs]
    gens = []
    for s, (_, env), inp in zip(streams, envs, inputs):
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            torch.cuda._sleep(DELAY // 4)                # every stream starts once the calls are queued
        gens.append(_run_mixed(env, inp))
    outs = [[] for _ in envs]
    while True:
        more = False
        for i, (s, g) in enumerate(zip(streams, gens)):
            with torch.cuda.stream(s):
                o = next(g, None)
            if o is not None:
                outs[i].append(o)
                more = True
        if not more:
            break
    torch.cuda.synchronize()
    for (name, env), got in zip(envs, outs):
        want, st = alone[name]
        assert len(got) == len(want), name
        for c, (g, w) in enumerate(zip(got, want)):
            assert_same(g, w, f"{name} call {c}")
        got_st = state_of(env)
        for key in st:
            assert_same(got_st[key], st[key], f"{name} {key}")
    # the two identical handles, against each other
    assert_same(outs[0], outs[-1], "twins")
    assert_same(state_of(envs[0][1]), state_of(envs[-1][1]), "twins' state")


# --------------------------------------------------------------------------
# d. lock step with the oracle while the handles run concurrently
# --------------------------------------------------------------------------
def _lockstep_handles(mt):
    """(oracle spec, arm, X, fk_mode, alive_p): closed form, UR5 preset, NVRTC, run-time table."""
    return [(ORACLE_REF, mt.REFERENCE_ARM, 10, 0, 0.1), (ORACLE_UR5, mt.UR5_ARM, 20, 0, 0.1),
            (*arm_pair(5), 12, 3, 0.1), (*arm_pair(7), 9, 1, 0.1)]


def test_oracle_lockstep_under_concurrency(mt):
    """Each iteration launches one step on every handle's stream, synchronises once, and compares each handle with
    its own fp64 oracle (auto-reset, objectives drawn on the device): the same bar as the single-handle lock step."""
    torch = _torch()
    n, steps = 4096 + 17, 30
    runs = []
    for i, (spec, arm, x, fk_mode, alive_p) in enumerate(_lockstep_handles(mt)):
        base = BASE + 100003 * i
        env = mt.BatchedEnvs(n, x, arm=arm, device=0, seed=SEED, env_id_base=base, fk_mode=fk_mode, auto_reset=True,
                             horizon=HORIZON)
        env.reset()
        ids = base + np.arange(n)
        ora = ChunkedOracle(n, x, spec)
        ora.reset(points=np.float32(device_points(SEED, ids, 0, x, spec.radius)).astype(np.float64))
        rs = np.random.RandomState(20 + i)
        _seed_late_episode(env, ora, rs, n, x, HORIZON, alive_p)
        acts = rs.randint(-180, 180, size=(steps, n, spec.n_joints)).astype(np.float32)
        runs.append(dict(env=env, ora=ora, spec=spec, x=x, fresh=philox_fresh(SEED, ids, x, spec.radius),
                         acts=acts, dev_acts=[torch.tensor(a, device="cuda") for a in acts], stream=torch.cuda.Stream(),
                         rep=Report(), episode=np.ones(n, dtype=np.int64), stats=None, slack=0, forked=False))
    torch.cuda.synchronize()
    for t in range(steps):
        live = [r for r in runs if not r["forked"] and r["rep"].ok()]
        for r in live:
            r["stream"].wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(r["stream"]):
                r["out"] = r["env"].step(r["dev_acts"][t])
        torch.cuda.synchronize()
        for r in live:
            rep, stats, slack, forked = lockstep_auto_reset(
                r["env"], r["ora"], r["spec"], None, lambda _: r["acts"][t], 1, HORIZON, rep=r["rep"],
                fresh=r["fresh"], device_step=lambda a: r["out"], episode=r["episode"])
            if r["stats"] is None:
                r["stats"] = stats
            else:
                for key in stats:
                    r["stats"][key] = stats[key] if key == "live_reward_sum" else r["stats"][key] + stats[key]
            r["slack"] += slack
            r["forked"] = forked
    for i, r in enumerate(runs):
        rep, stats, s = r["rep"], r["stats"], r["env"].stats()
        print(f"handle {i}:", rep.summary(), "forked" if r["forked"] else "", "expected", stats, "device", s)
        assert rep.ok(), (i, rep.notes[:5])
        assert rep.near_threshold <= max(4, int(rep.env_steps * 5e-6)), (i, rep.summary())
        if not r["forked"]:
            for key, v in stats.items():
                assert abs(s[key] - v) <= (r["slack"] if key == "reward_sum" else 0), (i, key, s[key], v)
        assert stats["terminated"] > 0 and stats["episodes"] > stats["terminated"], \
            (i, "the run must see terminations, truncations and refreshes")


# --------------------------------------------------------------------------
# e. step_host of one handle while another runs on a side stream
# --------------------------------------------------------------------------
@pytest.mark.parametrize("zero_copy", ["0", "1"])
def test_step_host_beside_a_long_rollout(mt, side, monkeypatch, zero_copy):
    """The host step's internal streams and launch tickets belong to its handle: host steps of one handle, issued
    while another handle's long rollout_random runs on a side stream, neither wait for it nor disturb it."""
    torch = _torch()
    monkeypatch.setenv("MT_HOST_ZEROCOPY", zero_copy)
    a, a_alone = twins(mt)
    b, b_alone = handle(mt, 1 << 18, 10), handle(mt, 1 << 18, 10)
    rs = np.random.RandomState(30)
    host = [rs.randint(-180, 180, size=(a.n, a.j)).astype(np.float32) for _ in range(4)]
    for h in (a, a_alone):                          # first call: streams, buffers, the variant
        h.step_host(host[0])
    b_alone.rollout_random(256)
    want = [as_numpy(a_alone.step_host(act)) for act in host[1:]]
    torch.cuda.synchronize()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        delay()
        b.rollout_random(256)
    got = [as_numpy(a.step_host(act)) for act in host[1:]]
    assert_busy(side)                               # the host steps ran while the rollout was still queued
    for c, (g, w) in enumerate(zip(got, want)):
        assert_same(g, w, f"host step {c}")
    assert a.host_step_mode == {"0": "staged", "1": "zero-copy"}[zero_copy]
    assert_same_state(a, a_alone, "host-stepped handle")
    assert_same_state(b, b_alone, "rollout handle")


# --------------------------------------------------------------------------
# f. a graph captured on a side stream, replayed on another non-default stream
# --------------------------------------------------------------------------
def test_graph_replay_on_a_side_stream(mt, side):
    """The wrapper cannot see a replay: after current_stream().wait_stream(replay stream), stats() and step_index
    read what the replays did.  The replays are checked against eager calls of a twin."""
    torch = _torch()
    a, b = twins(mt)
    act = actions(a.n, a.j, 40)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                   # warm-up: kernel attributes, launch shapes, buffers
        a.step(act)
        a.rollout_random(3)
    torch.cuda.current_stream().wait_stream(side)
    b.step(act)
    b.rollout_random(3)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = a.step(act)
        a.rollout_random(3)
    replay = torch.cuda.Stream()
    for rep in range(3):
        act.copy_(actions(a.n, a.j, 41 + rep))
        b.step(act)
        want_out = clone(b.rollout_random(3))              # the step's buffers hold the rollout's last step
        torch.cuda.synchronize()
        want_stats, want_index = b.stats(), b.step_index
        replay.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(replay):
            delay()
            graph.replay()
        torch.cuda.current_stream().wait_stream(replay)
        assert_busy(replay)
        assert a.stats() == want_stats, rep
        assert a.step_index == want_index, rep
        assert_same(out[:3], want_out, f"replay {rep}")
        assert_same_state(a, b, f"replay {rep}")
