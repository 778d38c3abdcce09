"""The generic DH chain at every joint count it is built for (J = 2 .. 8), against the fp64 oracle (-m gpu).

mt_api.cu instantiates `step_kernel<J, 0, ...>` and the helper kernels for each J, and NVRTC folds a user's table into a
`Preset<1000 + J>` (fk_mode 3, or 0 with the usual frame selectors).  Per-J code sits in both: odd-J goal loads and
stores, J = 8 float2 rows, `jbuf[J * 3]`, `gn[J]`, `TileScalars<J>`, the J = 2 first-row shortcut of `subpose_zmin`,
the second Philox block of `draw_actions` (joints 4 .. 7), the 130-float fetch record at J = 8, X = 32.  The tables
(tests/arms.py) put every fold of `push_row`'s preset branch -- alpha = 0, +-pi/2, pi; offsets 0, +-pi/2, pi -- on an
inner row.
"""
import numpy as np
import pytest

from arms import JOINT_COUNTS, arm_pair, reach
from oracle import OracleEnvs, fk, fk_frames
from oracle.manytor_oracle import joints_coordinates

from parity import (REL_POS_TOL, Report, alive_bits_to_matrix, compare_obs, compare_step, half_ball_points, lockstep,
                    lockstep_auto_reset)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mt():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import manytor_b200
    manytor_b200.load_library()
    return manytor_b200


def _points(rs, shape, radius):
    """Half-ball objectives as the device stores them (fp32), in float64 for the oracle."""
    return np.float32(half_ball_points(rs, shape, radius=radius)).astype(np.float64)


def _actions(rs, n, J):
    """30 steps of integer degrees in [-180, 180), then 10 of fp32 targets in [-720, 720) (half-turn reduction)."""
    return lambda t: rs.randint(-180, 180, size=(n, J)) if t < 30 else np.float32(rs.uniform(-720, 720, size=(n, J)))


# --------------------------------------------------------------------------
# a. lock step with the oracle at every J, run-time table (fk_mode 1) and NVRTC (fk_mode 3)
# --------------------------------------------------------------------------
_X_OF = {2: 1, 3: 7, 4: 10, 5: 4, 6: 20, 7: 13, 8: 32}          # X = 1, odd, even, 10, 20 and the maximum 32
_LOCKSTEP = [(J, fk_mode, _X_OF[J], 25) for J in JOINT_COUNTS for fk_mode in (1, 3)] + [(3, 1, 7, 8), (8, 3, 32, 8)]


@pytest.mark.parametrize("J,fk_mode,x,substeps", _LOCKSTEP)
def test_lockstep_at_every_joint_count(mt, J, fk_mode, x, substeps):
    """n = 1000 + 7J (a ragged last tile), 40 steps with joint positions; substeps = 8 gives an odd count of interior
    sub-poses, the other pairing of the packed sub-pose loop.  Fresh objectives for envs that collected everything."""
    spec, arm = arm_pair(J, substeps=substeps)
    n = 1000 + 7 * J
    rs = np.random.RandomState(100 * J + 10 * fk_mode + substeps)
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=fk_mode, substeps=substeps, seed=J)
    ora = OracleEnvs(n, x, spec=spec)
    pts = _points(rs, (n, x), spec.radius)
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rep = lockstep(env, ora, spec, _actions(rs, n, J), 40, on_done=lambda t, done: _points(rs, (n, x), spec.radius))
    print(f"J={J} fk_mode={fk_mode} x={x} substeps={substeps}:", rep.summary())
    assert rep.ok(), rep.notes[:5]
    assert rep.near_threshold <= max(2, rep.env_steps // 500), rep.summary()
    assert rep.rewarded >= 100 and rep.ground >= 1000, rep.summary()        # catches and ground contacts were compared


# --------------------------------------------------------------------------
# b. frame selectors at the ends of the chain (run-time-select copies of generic_arm / subpose_zmin)
# --------------------------------------------------------------------------
_SELECTORS = [(2, 0, (1, 2), 1), (3, 1, (0, 3), 2), (8, 8, (1, 8), 7)]


@pytest.mark.parametrize("J,obs,ground,catch", _SELECTORS)
def test_frame_selectors_at_the_ends_of_the_chain(mt, J, obs, ground, catch):
    import torch
    spec, arm = arm_pair(J, obs_frame=obs, ground_frames=ground, catch_frame=catch)
    n, x = 600 + J, 6
    rs = np.random.RandomState(J)
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=1, seed=J)
    ora = OracleEnvs(n, x, spec=spec)
    pts = _points(rs, (n, x), spec.radius)
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rep = lockstep(env, ora, spec, _actions(rs, n, J), 40, on_done=lambda t, done: _points(rs, (n, x), spec.radius))
    print(f"J={J} obs={obs} ground={ground} catch={catch}:", rep.summary())
    assert rep.ok(), rep.notes[:5]
    assert rep.near_threshold <= max(2, rep.env_steps // 500), rep.summary()
    # only the usual selectors specialise: fk_mode 3 refuses, fk_mode 0 takes the run-time table path silently
    with pytest.raises(mt.MantorLibraryError, match="usual frame selectors"):
        mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=3)
    a = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=0, seed=3)
    b = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=1, seed=3)
    a.reset(); b.reset()
    for t in range(5):
        act = torch.as_tensor(rs.randint(-180, 180, size=(n, J)), dtype=torch.float32, device="cuda")
        for u, v in zip(a.step(act, joints=True), b.step(act, joints=True)):
            assert torch.equal(u, v)
    sa, sb = a.get_state(), b.get_state()
    for key in sa:
        assert torch.equal(sa[key], sb[key]), key


# --------------------------------------------------------------------------
# c. in-kernel auto-reset with an uploaded objective stream
# --------------------------------------------------------------------------
@pytest.mark.parametrize("J,fk_mode,x", [(2, 1, 2), (3, 3, 5), (7, 1, 3), (8, 3, 9)])
def test_auto_reset_at_joint_count(mt, J, fk_mode, x):
    n, sets, steps, horizon = 700 + J, 6, 40, 6
    spec, arm = arm_pair(J)
    rs = np.random.RandomState(J)
    stream = _points(rs, (sets, n, x), spec.radius)
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=fk_mode, auto_reset=True, horizon=horizon)
    env.set_objective_stream(stream)
    env.reset()                                           # takes set 0
    ora = OracleEnvs(n, x, spec=spec)
    ora.reset(points=stream[0])
    rep, stats, slack, forked = lockstep_auto_reset(env, ora, spec, stream,
                                                    lambda t: rs.randint(-180, 180, size=(n, J)), steps, horizon)
    s = env.stats()
    print(f"J={J} fk_mode={fk_mode} auto-reset:", rep.summary(), s)
    assert rep.ok(), rep.notes[:5]
    if not forked:
        for k, v in stats.items():
            assert abs(s[k] - v) <= (slack if k == "reward_sum" else 0), (k, s[k], v)
        assert s["live_reward_sum"] == int(ora.total_reward.sum())
    assert stats["episodes"] > n


# --------------------------------------------------------------------------
# d. the first observation of the next episode (obs_after_reset): anchor at the zero pose (fill_arm)
# --------------------------------------------------------------------------
@pytest.mark.parametrize("J,obs,ground,catch,fk_mode", [(2, None, None, None, 3), (8, None, None, None, 1),
                                                        (8, None, None, None, 3), (2, 0, (1, 2), 1, 1)])
def test_first_observation_after_reset(mt, J, obs, ground, catch, fk_mode):
    n, x, sets, steps, horizon = 900 + J, 5, 4, 14, 4
    spec, arm = arm_pair(J, obs_frame=obs, ground_frames=ground, catch_frame=catch)
    rs = np.random.RandomState(J + 50)
    stream = _points(rs, (sets, n, x), spec.radius)
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=fk_mode, auto_reset=True, horizon=horizon,
                         obs_after_reset=True)
    env.set_objective_stream(stream)
    env.reset()
    ora = OracleEnvs(n, x, spec=spec)
    ora.reset(points=stream[0])
    episode = np.ones(n, dtype=np.int64)
    rep, first = Report(), Report()
    for t in range(steps):
        act = rs.randint(-180, 180, size=(n, J)).astype(np.float64)
        alive_before, points_before = ora.alive.copy(), ora.points.copy()
        obs_, rew, done = (o.cpu().numpy() for o in env.step(act.astype(np.float32)))
        r = ora.step(act)
        ended = r.done | ((ora.ep_len >= horizon) & ~r.done)
        dev_alive = np.where(ended[:, None], r.alive, alive_bits_to_matrix(env.get_state()["alive"].cpu().numpy(), x))
        o_cmp = np.where(ended[:, None], np.float32(r.obs), obs_)      # rows that ended are compared below
        bad = compare_step(rep, spec, ora, r, points_before, alive_before, o_cmp, rew, done, dev_alive)
        assert rep.ok(), rep.notes[:5]
        if bad.any():
            break                 # a near-threshold flip changes which envs reset: the two sides part here
        if ended.any():
            fresh = stream[episode % sets, np.arange(n)]
            ora.reset(mask=ended, points=fresh)
            episode[ended] += 1
            want = ora.get_observations()                                # manytor.py:251-253 of the new episode
            anchor = fk_frames(np.zeros((int(ended.sum()), J)), spec)[:, spec.obs_frame]
            compare_obs(first, spec, anchor, ora.points[ended], ora.alive[ended], obs_[ended], want[ended])
            first.env_steps += int(ended.sum())
    print(f"J={J} obs={spec.obs_frame} first observations:", first.summary())
    assert first.ok(), first.notes[:5]
    assert first.env_steps >= n                            # every env started a new episode at least once


# --------------------------------------------------------------------------
# e. the helper kernels at every J
# --------------------------------------------------------------------------
@pytest.mark.parametrize("J", JOINT_COUNTS)
def test_helpers_at_every_joint_count(mt, J):
    import manytor_b200.manytor as tor
    spec, arm = arm_pair(J)
    tol = REL_POS_TOL * reach(spec.dh)
    rs = np.random.RandomState(J)
    m = 777
    goals = np.float32(rs.uniform(-720, 720, size=(m, J))).astype(np.float64)
    goals[:5] = rs.randint(-180, 180, size=(5, J))
    env = mt.BatchedEnvs(m, 7, arm=arm, device=0, seed=J)
    env.reset()
    # joints_coordinates (manytor.py:188-189) of arbitrary poses
    np.testing.assert_allclose(env.joints_of(goals).cpu().numpy(), joints_coordinates(goals, spec), rtol=0, atol=tol)
    # fk(mode) for every frame the chain has (manytor.py:35-53)
    for mode in range(1, J + 1):
        got = tor.fk(mode, goals, arm)
        want = fk(mode, goals, spec)
        np.testing.assert_allclose(got[:, :3, :3], want[:, :3, :3], rtol=0, atol=1e-5, err_msg=f"rotation of frame {mode}")
        np.testing.assert_allclose(got[:, :3, 3], want[:, :3, 3], rtol=0, atol=tol, err_msg=f"origin of frame {mode}")
        np.testing.assert_array_equal(got[:, 3], np.broadcast_to([0.0, 0.0, 0.0, 1.0], (m, 4)))
    # observe() after set_state: random poses and alive masks (manytor.py:141-153)
    alive = rs.rand(m, 7) > 0.3
    total = rs.randint(-40, 3, size=m).astype(np.float32)
    env.set_state(goals=np.float32(goals), alive=alive, total_reward=total)
    ora = OracleEnvs(m, 7, spec=spec)
    ora.reset(points=env.get_points(zero_dead=False).cpu().numpy().astype(np.float64))
    ora.goals, ora.alive = goals.copy(), alive.copy()
    want = ora.get_observations()
    rep = Report()
    compare_obs(rep, spec, fk_frames(goals, spec)[:, spec.obs_frame], ora.points, alive, env.observe().cpu().numpy(), want)
    assert rep.ok(), rep.notes[:5]
    if J % 2:
        # odd J: the state round trip through the scalar goal loads / stores
        ep = rs.randint(0, 65535, size=m).astype(np.int32)
        env.set_state(ep_len=ep)
        st = env.get_state()
        np.testing.assert_array_equal(st["goals"].cpu().numpy(), np.float32(goals))
        np.testing.assert_array_equal(alive_bits_to_matrix(st["alive"].cpu().numpy(), 7), alive)
        np.testing.assert_array_equal(st["total_reward"].cpu().numpy(), total)
        np.testing.assert_array_equal(st["ep_len"].cpu().numpy(), ep)


@pytest.mark.parametrize("J,x", [(8, 32), (3, 7)])
def test_fetch_env_record(mt, J, x):
    """mt_fetch_env copies J * 4 + 3X + 2 floats: 130 at J = 8, X = 32, the whole of the record."""
    spec, arm = arm_pair(J)
    n = 100
    rs = np.random.RandomState(x)
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, seed=1)
    env.reset()
    goals = np.float32(rs.uniform(-180, 180, size=(n, J)))
    alive = rs.rand(n, x) > 0.5
    total = rs.randint(-50, 5, size=n).astype(np.float32)
    env.set_state(goals=goals, alive=alive, total_reward=total)
    pts = env.get_points(zero_dead=False).cpu().numpy()
    for i in (0, 37, n - 1):
        f = env.fetch_env(i)
        np.testing.assert_array_equal(f["goals"], goals[i])
        np.testing.assert_array_equal(f["alives"], alive[i])
        np.testing.assert_array_equal(f["points"], np.where(alive[i][:, None], pts[i], 0.0))   # dead read as zeros
        assert f["total_reward"] == float(total[i])
        np.testing.assert_allclose(f["joints_coordinates"], joints_coordinates(goals[i].astype(np.float64), spec),
                                   rtol=0, atol=REL_POS_TOL * reach(spec.dh))


@pytest.mark.parametrize("J", [3, 7])
def test_step_host_equals_step_at_odd_joint_counts(mt, J):
    _, arm = arm_pair(J)
    n, x = 5000 + J, 9
    a = mt.BatchedEnvs(n, x, arm=arm, device=0, seed=3)
    b = mt.BatchedEnvs(n, x, arm=arm, device=0, seed=3)
    a.reset(); b.reset()
    rng = np.random.RandomState(J)
    for _ in range(5):
        act = rng.randint(-180, 180, size=(n, J)).astype(np.float32)
        oa, ra, da = a.step(act)
        ob, rb, db = b.step_host(act)
        np.testing.assert_array_equal(oa.cpu().numpy(), ob)
        np.testing.assert_array_equal(ra.cpu().numpy(), rb)
        np.testing.assert_array_equal(da.cpu().numpy(), db)
    sa, sb = a.get_state(), b.get_state()
    for key in sa:
        np.testing.assert_array_equal(sa[key].cpu().numpy(), sb[key].cpu().numpy(), err_msg=key)
