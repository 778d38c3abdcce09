"""The device-side bookkeeping of every launch: step index, env-step count and launch count (-m gpu).

The step index (StepParams::ctrl) and the statistics live in device memory and each kernel advances them itself
(launch_ticket, mt_step.cuh): every warp bumps its block's count once it has read the step index, the block's last
warp takes the launch's ticket, and the launch's last block adds P.advance to the index and the launch's env-steps
to the statistics.  CUDA-graph replays, the in-kernel action stream keyed by (seed, env id, step index), the
4096-step chunks of mt_rollout_random, the overlapping chunk launches of the staged mt_step_host and checkpoints
all rest on it.

  a. Every launch shape plan_launch makes (1, 2, 3 and the largest number of warps per block, blocks with idle
     warps, ragged last tiles) through every launch path, on five kinds of handle.  After each call the step index,
     env_steps and the launch count must be exactly what the call implies, the in-kernel actions must have been
     keyed by the right step index (the goals hold the last step's action), and the statistics words must follow in
     closed form from the horizon; the multi-step rollout kernel must be bit-identical to per-step launches.
  b. The same without a host synchronisation between launches (programmatic dependent launch lets the next grid
     start early), and a chunked rollout replayed from a CUDA graph.
  c. A step index that crosses 2^32 inside one launch.
  d. The top of the accepted range, 2^62, and the refusal of anything above it.

Shard sizes are derived from the device's SM count S, so the shapes hold on any SM count.
"""
import contextlib
import dataclasses
import os
import time
from typing import NamedTuple

import numpy as np
import pytest

from oracle.philox import device_actions

pytestmark = pytest.mark.gpu

SEED = 0x1234567890ABCDEF          # both key words non-zero
BASE = (1 << 32) - 50              # the env ids of a shard of more than 50 envs cross 2^32
HORIZON = 7                        # coprime to the 4096-step chunk: episodes end at every phase of a chunk
TOP = 1 << 62                      # MT_STEP_INDEX_MAX
LONG_K_MAX_ENVS = 16384            # rollouts of thousands of steps only on shards up to this size


@pytest.fixture(scope="module")
def mt():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import manytor_b200
    manytor_b200.load_library()
    return manytor_b200


@contextlib.contextmanager
def _env(**kv):
    """Set (or, for None, remove) environment variables the library reads, for the duration of the block."""
    old = {k: os.environ.get(k) for k in kv}
    try:
        for k, v in kv.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _sms() -> int:
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# --------------------------------------------------------------------------
# handles and launch shapes
# --------------------------------------------------------------------------
class Kind(NamedTuple):
    arm: object
    x: int
    fk_mode: int
    f16: bool
    max_wpb: int           # kMaxWarpsRefArm or kMaxWarpsGeneric: X is small enough that shared memory allows it
    rollout_kernel: bool   # mt_rollout_random(k >= 2) is one launch per 4096 steps (else one launch per step)


def _kind(mt, name) -> Kind:
    from arms import arm_pair
    j5 = arm_pair(5)[1]
    return {
        "ref": Kind(mt.REFERENCE_ARM, 10, 0, False, 28, True),       # built-in kernels, compile-time X
        "ref_f16": Kind(mt.REFERENCE_ARM, 7, 0, True, 28, True),     # built-in binary16 kernels, run-time X
        "ur5": Kind(mt.UR5_ARM, 10, 0, False, 16, True),             # the UR5 preset
        "j5_fk3": Kind(j5, 7, 3, False, 16, True),                   # NVRTC kernels of a 5-joint table
        "j5_fk1": Kind(j5, 7, 1, False, 16, False),                  # run-time DH table: one launch per step
    }[name]


def _handle(mt, kind: Kind, n, *, stats_config=False):
    """A reset handle.  Plain configuration: no auto-reset, no horizon, so the goals after a call are the last
    step's action.  Statistics configuration: nothing is ever caught (catch_tol = 0), auto-reset at the horizon."""
    import torch
    arm = dataclasses.replace(kind.arm, catch_tol=0.0) if stats_config else kind.arm
    with _env(MT_DISABLE_JIT="1" if kind.fk_mode == 0 else None):     # built-in kernels for fk_mode 0
        env = mt.BatchedEnvs(n, kind.x, arm=arm, device=0, seed=SEED, env_id_base=BASE, fk_mode=kind.fk_mode,
                             auto_reset=stats_config, horizon=HORIZON if stats_config else 0,
                             terminate_on_ground=False, obs_dtype=torch.float16 if kind.f16 else torch.float32)
    env.reset()
    return env


def launch_shape(tiles, sms, max_wpb):
    """(warps per block, blocks, warps without a first tile) of a launch over `tiles` tiles (plan_launch, mt_api.cu)."""
    wpb = min(max(-(-tiles // sms), 1), max_wpb)
    grid = min(-(-tiles // wpb), sms)
    return wpb, grid, max(grid * wpb - tiles, 0)


# name -> (N from (S, max_wpb), (warps per block, warps without a tile) it must give)
SHAPES = {
    "n1": (lambda s, m: 1, lambda s, m: (1, 0)),
    "n33": (lambda s, m: 33, lambda s, m: (1, 0)),                               # two blocks of one warp
    "w2_full": (lambda s, m: 64 * s, lambda s, m: (2, 0)),                       # 2S tiles, every block full
    "w2_idle": (lambda s, m: 32 * (2 * s - 2) + 7, lambda s, m: (2, 1)),         # 2S - 1 tiles: the last block holds one
    "w3": (lambda s, m: 96 * s - 31, lambda s, m: (3, 0)),                       # last tile holds one env
    "wmax": (lambda s, m: 32 * m * s - 5, lambda s, m: (m, 0)),
    "wmax_idle": (lambda s, m: 32 * (m * (s - 1) + 1) - 9, lambda s, m: (m, m - 1)),  # m - 1 blocks with an idle warp
}


def _shape_n(name, kind: Kind) -> int:
    s = _sms()
    n_of, want = SHAPES[name]
    n = n_of(s, kind.max_wpb)
    wpb, grid, idle = launch_shape(-(-n // 32), s, kind.max_wpb)
    assert (wpb, idle) == want(s, kind.max_wpb) and grid <= s, (name, n, wpb, grid, idle)
    return n


def _staged_chunks(tiles) -> int:
    """Launches of one staged mt_step_host call (mt_api.cu: up to 16 chunks of whole tiles)."""
    chunks = 1 if tiles < 16 else 16
    per = -(-tiles // chunks)
    return -(-tiles // per)


def _launches(op, k, n, persistent, host_mode):
    if op == "step":
        return 1
    if op == "host":
        return _staged_chunks(-(-n // 32)) if host_mode == "0" else 1
    # one launch per full or partial 4096-step chunk; a remainder of one step is one launch of the step kernel
    return -(-k // 4096) if persistent else k


def _calls(n):
    if n <= LONG_K_MAX_ENVS:
        ks = (4095, 4096, 4097, 8193)
    else:
        ks = (3,)
    return [("step", 1), ("rand", 1), ("rand", 2), ("host", 1)] + [("rand", k) for k in ks] + [("host", 1)]


def _bits(a):
    """Host copy of a tensor or array, floats as their bit patterns (so -0.0 != 0.0 and NaN == NaN)."""
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.array(a, copy=True)
    return a.view(f"u{a.itemsize}") if a.dtype.kind == "f" else a


def _call(env, op, k, actions):
    with_obs = env.step_host(actions) if op == "host" else (env.step(actions) if op == "step" else env.rollout_random(k))
    return [_bits(t) for t in with_obs]


def _snapshot(env):
    st = env.get_state()
    return ({key: _bits(v) for key, v in st.items()}, _bits(env.get_points(zero_dead=False)), env.stats(), env.step_index)


def _assert_same(a, b, what):
    for u, v in zip(a, b):
        np.testing.assert_array_equal(u, v, err_msg=what)


def _assert_actions(env, ids, step, what):
    """The goals hold the actions of `step`, and mt_sample_actions draws those of `step + 1`."""
    J = env.j
    goals = env.get_state()["goals"].cpu().numpy()
    np.testing.assert_array_equal(goals, device_actions(SEED, ids, step, J).astype(np.float32),
                                  err_msg=f"{what}: goals are not the actions of step {step}")
    np.testing.assert_array_equal(env.sample_actions().cpu().numpy(), device_actions(SEED, ids, step + 1, J).astype(np.float32),
                                  err_msg=f"{what}: mt_sample_actions at step {step + 1}")


def _staggered_ep_len(n, seed):
    """Episode lengths over [0, h): whole warps in phase and warps of mixed phase."""
    rs = np.random.RandomState(seed)
    e0 = rs.randint(0, HORIZON, size=n)
    warp = np.arange(n) // 32
    lockstep = warp % 3 == 0
    e0[lockstep] = (warp[lockstep] // 3) % HORIZON
    return e0


# --------------------------------------------------------------------------
# a. every launch shape, every launch path
# --------------------------------------------------------------------------
_KINDS = ("ref", "ref_f16", "ur5", "j5_fk3", "j5_fk1")


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kind_name", _KINDS)
def test_bookkeeping_at_every_launch_shape(mt, kind_name, shape):
    """mt_step, rollout_random(1) (the step kernel with in-kernel actions), rollout_random(k) across the 4096-step
    chunks, and the staged and zero-copy mt_step_host, one after the other on one handle.

    Plain configuration, host steps staged: after every call the step index and env_steps are exact, the launch count
    grew by the call's launches, the goals are the restated actions of the call's last step and mt_sample_actions
    draws those of the next.  Statistics configuration, host steps zero-copy, beside a twin that takes one launch per
    step (MT_ROLLOUT_PERSISTENT=0): episodes, length_sum, catches, terminated and ep_len follow in closed form from
    the horizon, reward_sum + live_reward_sum = -ground_steps, and the twin's outputs, state, objectives, statistics
    and step index are bit-identical."""
    kind = _kind(mt, kind_name)
    n = _shape_n(shape, kind)
    calls = _calls(n)
    ids = BASE + np.arange(n)
    t0 = time.perf_counter()

    # plain configuration
    env = _handle(mt, kind, n)
    s = 0
    for c, (op, k) in enumerate(calls):
        what = f"{kind_name} {shape} n={n} call {c}: {op}({k})"
        actions = None
        if op == "step":
            actions = env.sample_actions()
        elif op == "host":
            actions = device_actions(SEED, ids, s, env.j).astype(np.float32)
        l0 = env.launch_count
        with _env(MT_HOST_ZEROCOPY="0"):
            _call(env, op, k, actions)
        launched = env.launch_count - l0
        s += k
        assert launched == _launches(op, k, n, kind.rollout_kernel, "0"), (what, launched)
        assert env.step_index == s, (what, env.step_index, s)
        assert env.stats()["env_steps"] == n * s, (what, env.stats())
        _assert_actions(env, ids, s - 1, what)
    assert env.host_step_mode == "staged"

    # statistics configuration, and the same calls as one launch per step
    env = _handle(mt, kind, n, stats_config=True)
    twin = _handle(mt, kind, n, stats_config=True)
    e0 = _staggered_ep_len(n, len(shape) + len(kind_name))
    env.set_state(ep_len=e0.astype(np.int32))
    twin.set_state(ep_len=e0.astype(np.int32))
    rs = np.random.RandomState(n)
    t = 0
    for c, (op, k) in enumerate(calls):
        what = f"{kind_name} {shape} n={n} statistics call {c}: {op}({k})"
        host_actions = rs.randint(-180, 180, size=(n, env.j)).astype(np.float32)
        outs, snaps = [], []
        for h, persistent in ((env, "1"), (twin, "0")):
            actions = h.sample_actions() if op == "step" else host_actions
            l0 = h.launch_count
            with _env(MT_HOST_ZEROCOPY="1", MT_ROLLOUT_PERSISTENT=persistent):
                outs.append(_call(h, op, k, actions))
            launched = h.launch_count - l0
            assert launched == _launches(op, k, n, kind.rollout_kernel and persistent == "1", "1"), (what, persistent, launched)
            snaps.append(_snapshot(h))
        t += k
        state, _, st, index = snaps[0]
        assert index == t, (what, index)
        episodes = int(((e0 + t) // HORIZON).sum())
        assert st["env_steps"] == n * t, (what, st)
        assert st["episodes"] == episodes and st["length_sum"] == episodes * HORIZON, (what, st, episodes)
        assert st["catches"] == 0 and st["terminated"] == 0, (what, st)
        assert st["reward_sum"] + st["live_reward_sum"] == -st["ground_steps"], (what, st)
        np.testing.assert_array_equal(state["ep_len"], (e0 + t) % HORIZON, err_msg=what)
        _assert_same(outs[0], outs[1], f"{what}: outputs of the last step differ from per-step launches")
        for key in state:
            np.testing.assert_array_equal(state[key], snaps[1][0][key], err_msg=f"{what}: {key} differs from per-step launches")
        np.testing.assert_array_equal(snaps[0][1], snaps[1][1], err_msg=f"{what}: objectives differ from per-step launches")
        assert snaps[0][2:] == snaps[1][2:], (what, snaps[0][2:], snaps[1][2:])
    assert env.host_step_mode == "zero-copy"
    if n * t >= 100_000:
        assert st["ground_steps"] > 0 and st["episodes"] > 0, st
    print(f"bookkeeping {kind_name} {shape}: n={n}, {t} steps per handle, {time.perf_counter() - t0:.2f} s")


# --------------------------------------------------------------------------
# b. no host synchronisation between launches; a chunked rollout in a CUDA graph
# --------------------------------------------------------------------------
@pytest.mark.parametrize("kind_name,shape", [("ref", "n33"), ("ref", "w2_idle"), ("ur5", "w2_full"), ("j5_fk3", "w2_idle")])
def test_mixed_calls_without_host_sync(mt, kind_name, shape):
    """50 calls enqueued on one stream with no synchronisation in between: mt_step (on fresh or earlier draws of
    mt_sample_actions), rollout_random(1), rollout_random(3), rollout_random(4097) and mt_sample_actions.  Afterwards
    the step index, env_steps, the launch count, the goals and every draw must be what the sequence implies."""
    import torch
    kind = _kind(mt, kind_name)
    n = _shape_n(shape, kind)
    ids = BASE + np.arange(n)
    env = _handle(mt, kind, n)
    torch.cuda.synchronize()
    rs = np.random.RandomState(n)
    seq = [str(v) for v in rs.choice(["step", "r1", "r3", "sample"], size=50)]
    for i in (7, 23, 41):
        seq[i] = "r4097"
    s, launches, last, draws = 0, 0, None, []
    l0 = env.launch_count
    for op in seq:
        if op == "sample":
            draws.append((env.sample_actions(), s))
            launches += 1
        elif op == "step":
            if draws and rs.rand() < 0.5:
                a, at = draws[rs.randint(len(draws))]                    # an earlier draw
            else:
                a, at = env.sample_actions(), s
                draws.append((a, at))
                launches += 1
            env.step(a)
            last, s, launches = at, s + 1, launches + 1
        else:
            k = int(op[1:])
            env.rollout_random(k)
            last, s, launches = s + k - 1, s + k, launches + _launches("rand", k, n, kind.rollout_kernel, None)
    torch.cuda.synchronize()
    assert env.launch_count - l0 == launches
    assert env.step_index == s and env.stats()["env_steps"] == n * s, (env.step_index, s)
    for a, at in draws:
        np.testing.assert_array_equal(a.cpu().numpy(), device_actions(SEED, ids, at, env.j).astype(np.float32),
                                      err_msg=f"draw at step {at}")
    goals = env.get_state()["goals"].cpu().numpy()
    np.testing.assert_array_equal(goals, device_actions(SEED, ids, last, env.j).astype(np.float32))


def test_graph_replay_of_a_chunked_rollout(mt):
    """rollout_random(4097) captured once (a 4096-step rollout launch and one step-kernel launch) and replayed twice
    must equal two eager calls: outputs of the last step, state, objectives, statistics and step index."""
    import torch
    kind = _kind(mt, "ref")
    n = _shape_n("w2_idle", kind)
    ids = BASE + np.arange(n)
    eager = _handle(mt, kind, n)
    for _ in range(2):
        want = [_bits(v) for v in eager.rollout_random(4097)]
    cap = _handle(mt, kind, n)
    cap._out_buffers(True, False)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = cap.rollout_random(4097)
    assert cap.step_index == 0 and cap.stats()["env_steps"] == 0         # capture ran nothing
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    _assert_same([_bits(v) for v in out], want, "replayed outputs differ from the eager calls")
    a, b = _snapshot(cap), _snapshot(eager)
    for key in a[0]:
        np.testing.assert_array_equal(a[0][key], b[0][key], err_msg=key)
    np.testing.assert_array_equal(a[1], b[1])
    assert a[2:] == b[2:] and a[3] == 2 * 4097 and a[2]["env_steps"] == 2 * 4097 * n, (a[2:], b[2:])
    _assert_actions(cap, ids, 2 * 4097 - 1, "graph replay")


# --------------------------------------------------------------------------
# c. the high word of the step index
# --------------------------------------------------------------------------
@pytest.mark.parametrize("kind_name", ["ref", "ur5", "j5_fk3"])
def test_step_index_crossing_2_32(mt, kind_name):
    """draw_actions XORs the index's high word into the stream tag of both Philox blocks (J > 4 uses the second),
    and the rollout kernel forms step0 + s in 64 bits.  rollout_random(5) from 2^32 - 2 crosses 2^32 in one launch;
    one launch per step must give the same bits, and mt_sample_actions must match the restatement above 2^32."""
    kind = _kind(mt, kind_name)
    n = _shape_n("w2_idle", kind)
    ids = BASE + np.arange(n)
    start = (1 << 32) - 2
    runs = []
    for persistent in ("1", "0"):
        env = _handle(mt, kind, n)
        env.step_index = start
        l0 = env.launch_count
        with _env(MT_ROLLOUT_PERSISTENT=persistent):
            out = [_bits(v) for v in env.rollout_random(5)]
        assert env.launch_count - l0 == (1 if persistent == "1" else 5)
        assert env.step_index == start + 5 and env.stats()["env_steps"] == 5 * n
        _assert_actions(env, ids, start + 4, f"persistent={persistent}")
        runs.append((out, _snapshot(env)))
        for v in ((1 << 32) - 1, 1 << 32, (1 << 33) + 7):
            env.step_index = v
            np.testing.assert_array_equal(env.sample_actions().cpu().numpy(),
                                          device_actions(SEED, ids, v, env.j).astype(np.float32), err_msg=f"step {v}")
    (oa, sa), (ob, sb) = runs
    _assert_same(oa, ob, "rollout kernel and per-step launches differ across 2^32")
    for key in sa[0]:
        np.testing.assert_array_equal(sa[0][key], sb[0][key], err_msg=key)
    np.testing.assert_array_equal(sa[1], sb[1])
    assert sa[2:] == sb[2:]


# --------------------------------------------------------------------------
# d. the top of the range
# --------------------------------------------------------------------------
def test_top_of_the_step_index_range(mt, monkeypatch):
    """The largest accepted index, 2^62, at the 28-warp reference shape (an even number of warps per block, every
    warp with a tile): rollout_random(1) and rollout_random(3) advance the index and count their env-steps.  Above
    2^62 mt_set_step_index returns MT_ERR_INVALID and leaves the index alone, and the Python setter raises ValueError
    for -1 and for 2^62 + 1 before it calls the library (it used to store them modulo 2^64)."""
    from manytor_b200 import _lib
    kind = _kind(mt, "ref")
    s = _sms()
    n = 28 * s * 32 + 5
    assert launch_shape(-(-n // 32), s, 28) == (28, s, 0)
    ids = BASE + np.arange(n)
    env = _handle(mt, kind, n)
    env.step_index = TOP
    done = 0
    for k in (1, 3):
        l0 = env.launch_count
        env.rollout_random(k)
        assert env.launch_count - l0 == 1
        done += k
        assert env.step_index == TOP + done and env.stats()["env_steps"] == n * done, (env.step_index - TOP, env.stats())
        _assert_actions(env, ids, TOP + done - 1, f"rollout_random({k}) at 2^62")
    lib = _lib.load()
    for v in (TOP + 1, 1 << 63, (1 << 64) - 1):
        assert lib.mt_set_step_index(env._h, v) == -1, v                  # MT_ERR_INVALID
        assert b"MT_STEP_INDEX_MAX" in lib.mt_last_error()
        assert env.step_index == TOP + done

    class NoLibrary:
        def __getattr__(self, name):
            raise AssertionError(f"the library was called: {name}")

    with monkeypatch.context() as m:
        m.setattr(env, "_lib", NoLibrary())
        for v in (-1, TOP + 1, 1 << 64):
            with pytest.raises(ValueError, match=r"step_index must be in \[0, 2\*\*62\]"):
                env.step_index = v
    assert env.step_index == TOP + done
