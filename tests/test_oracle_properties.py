"""Property tests of the CPU oracle (hypothesis): invariants the reference's geometry implies, used to
cross-check the restatement beyond the recorded traces."""
import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from oracle import OracleEnvs, REFERENCE_ARM, fk_frames, observations

angles = st.lists(st.floats(-720, 720, allow_nan=False, width=32), min_size=4, max_size=4)


@settings(max_examples=60, deadline=None)
@given(angles, st.floats(-360, 360))
def test_base_rotation_leaves_heights_and_lengths_alone(g, turn):
    """Joint 0 turns the arm about the vertical axis (DH row 1, manytor.py:42): z of every frame and all
    link lengths are unchanged, so the ground test never depends on it."""
    a = fk_frames(np.array(g, dtype=np.float64))
    g2 = list(g)
    g2[0] += turn
    b = fk_frames(np.array(g2, dtype=np.float64))
    np.testing.assert_allclose(a[:, 2], b[:, 2], atol=1e-9)
    np.testing.assert_allclose(np.linalg.norm(a, axis=1), np.linalg.norm(b, axis=1), atol=1e-9)


@settings(max_examples=60, deadline=None)
@given(angles)
def test_link_lengths_and_reach(g):
    fr = fk_frames(np.array(g, dtype=np.float64))
    assert abs(np.linalg.norm(fr[2] - fr[0]) - 4.3) < 1e-9            # frame 2 sits on top of the base column
    assert abs(np.linalg.norm(fr[3] - fr[2]) - 24.3) < 1e-9           # upper arm (manytor.py:46)
    assert abs(np.linalg.norm(fr[4] - fr[3]) - 27.0) < 1e-9           # forearm (manytor.py:48)
    assert np.linalg.norm(fr[4]) <= 4.3 + 24.3 + 27.0 + 1e-9


@settings(max_examples=40, deadline=None)
@given(st.integers(0, 2**31 - 1))
def test_observation_ranges_and_dead_objectives(seed):
    rng = np.random.RandomState(seed)
    n, x = 5, 6
    env = OracleEnvs(n, x)
    env.reset(points=rng.uniform(-40, 40, size=(n, x, 3)) * [1, 1, 0.5] + [0, 0, 20])
    r = env.step(rng.randint(-180, 180, size=(n, 4)))
    o = r.obs.reshape(n, x, 3)
    assert (o[..., 0] >= 0).all() and (o[..., 1:] >= 0).all() and (o[..., 1:] <= 90 + 1e-9).all()   # manytor.py:17-22
    assert set(np.unique(r.reward)) <= {-1, 0, 1}
    r2 = env.step(rng.randint(-180, 180, size=(n, 4)))
    dead_before = ~r.alive
    assert (r2.obs.reshape(n, x, 3)[dead_before] == 0).all()          # manytor.py:146-148
    assert (r2.alive <= r.alive).all()                                # objectives never come back without a reset
    assert ((r2.reward == 1) <= (r2.alive.sum(1) < r.alive.sum(1))).all()   # +1 only with a catch this step


@settings(max_examples=40, deadline=None)
@given(angles, angles)
def test_ground_flag_is_sticky_over_the_route(g, a):
    """neg is the OR over all 25 interpolated poses (manytor.py:183-192): it must be set whenever the
    end pose or the start pose is underground."""
    env = OracleEnvs(1, 1)
    env.reset(points=np.array([[[0.0, 0.0, 40.0]]]))
    env.step(np.array([g]))
    start = fk_frames(np.array(g, dtype=np.float64))
    end = fk_frames(np.array(a, dtype=np.float64))
    r = env.step(np.array([a]))
    under = min(start[3, 2], start[4, 2], end[3, 2], end[4, 2]) < 0
    assert (not under) or bool(r.neg[0])
    assert r.reward[0] == -1 if r.neg[0] else r.reward[0] in (0, 1)


@pytest.mark.parametrize("J", [2, 3, 8])
def test_frame_selectors_pick_the_frame_of_that_number(J):
    """Frame k is the origin after the first k DH rows (frame 0 the base): every selector in 0 .. J must observe from,
    and catch with, exactly fk_frames(goals)[:, k] -- including frame 1, which joints_coordinates has no row for."""
    import dataclasses
    from arms import arm_pair
    spec0, _ = arm_pair(J)
    rng = np.random.RandomState(J)
    n, x = 64, 5
    for f in range(J + 1):
        spec = dataclasses.replace(spec0, obs_frame=f, catch_frame=f)
        env = OracleEnvs(n, x, spec=spec)
        pts = rng.uniform(-1, 1, size=(n, x, 3)) * spec.radius
        env.reset(points=pts)
        np.testing.assert_array_equal(env.get_observations(),
                                      observations(fk_frames(np.zeros((n, J)), spec)[:, f], pts, np.ones((n, x), bool)))
        act = rng.randint(-180, 180, size=(n, J)).astype(np.float64)
        frames = fk_frames(act, spec)
        # objective 0 of every other env sits just inside the catch cube of frame f at the new pose
        env.points[::2, 0] = frames[::2, f] + 0.5 * spec.catch_tol
        points_before, alive_before = env.points.copy(), env.alive.copy()
        r = env.step(act)
        np.testing.assert_array_equal(r.obs, observations(frames[:, f], points_before, alive_before))
        caught = (np.abs(frames[:, f][:, None, :] - points_before) <= spec.catch_tol).all(axis=-1)
        np.testing.assert_array_equal(r.alive, alive_before & ~caught)
        assert caught[::2, 0].all()
        np.testing.assert_array_equal(env.get_observations(), observations(frames[:, f], env.points, env.alive))
    np.testing.assert_array_equal(r.frames, frames)                   # what the GPU comparisons read the anchor from
