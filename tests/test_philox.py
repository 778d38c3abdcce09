"""Known-answer vectors for the oracle's Philox4x32-10 (Random123 kat_vectors)."""
import numpy as np

from oracle.philox import device_actions, device_points, philox4x32_10


def _one(c, k):
    r = philox4x32_10(*[np.array([v], dtype=np.uint32) for v in c], *[np.array([v], dtype=np.uint32) for v in k])
    return [int(v[0]) for v in r]


def test_random123_known_answers():
    assert _one([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert _one([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert _one([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_action_map_range_and_uniformity():
    a = device_actions(42, np.arange(200000), 3, 4)
    assert a.min() == -180 and a.max() == 179          # manytor.py:216: integers on [-180, 180)
    counts = np.bincount((a + 180).ravel(), minlength=360)
    assert counts.min() > 0.9 * a.size / 360 and counts.max() < 1.1 * a.size / 360
    assert not np.array_equal(a, device_actions(42, np.arange(200000), 4, 4))
    np.testing.assert_array_equal(a[1000:2000], device_actions(42, np.arange(1000, 2000), 3, 4))  # shard-invariant


def test_device_points_lie_in_the_upper_half_ball():
    for radius in (51.3, 0.81725):
        big_r = float(np.float32(radius))
        p = device_points(0x1234567890ABCDEF, np.arange(20000) + (3 << 20) + 5, np.arange(20000) % 3, 32, radius)
        assert p.shape == (20000, 32, 3)
        assert (p[..., 2] >= 0).all() and (np.linalg.norm(p, axis=-1) <= big_r * (1 + 1e-12)).all()


def test_device_points_follow_the_reference_law():
    """Uniform in the upper half ball, as the reference's rejection sampler (manytor.py:228-239)."""
    from scipy import stats as sst
    from oracle.manytor_oracle import sample_points_reference_stream
    big_r = float(np.float32(51.3))
    p = device_points(5, np.arange(5000), 0, 10).reshape(-1, 3)
    r = np.linalg.norm(p, axis=1)
    assert sst.kstest((r / big_r) ** 3, "uniform").pvalue > 1e-3
    assert sst.kstest((np.arctan2(p[:, 1], p[:, 0]) + np.pi) / (2 * np.pi), "uniform").pvalue > 1e-3
    assert sst.kstest(p[:, 2] / r, "uniform").pvalue > 1e-3
    state = np.random.get_state()
    try:
        np.random.seed(11)
        ref = np.stack([sample_points_reference_stream(1)[0] for _ in range(4000)])
    finally:
        np.random.set_state(state)
    assert sst.ks_2samp(np.linalg.norm(ref, axis=1), r[:20000]).pvalue > 1e-3
    assert sst.ks_2samp(ref[:, 0], p[:20000, 0]).pvalue > 1e-3
    assert sst.ks_2samp(ref[:, 1], p[:20000, 1]).pvalue > 1e-3
    assert sst.ks_2samp(ref[:, 2], p[:20000, 2]).pvalue > 1e-3


def test_device_points_depend_on_every_key():
    """Seed lo / hi, env id lo / hi (ids >= 2^32), episode and objective index each change every point."""
    seed, gid, ep, x = 0x1234567890ABCDEF, (5 << 32) + 77, 3, 8
    base = device_points(seed, [gid], [ep], x)[0]
    variants = [device_points(seed ^ 1, [gid], [ep], x), device_points(seed ^ (1 << 40), [gid], [ep], x),
                device_points(seed, [gid ^ 1], [ep], x), device_points(seed, [gid ^ (1 << 33)], [ep], x),
                device_points(seed, [gid], [ep + 1], x)]
    for v in variants:
        assert (np.abs(v[0] - base).max(axis=-1) > 0).all()
    # objective p of episode e is counter e * 32 + p: objective 1 is a new block, not objective 0 again
    assert (np.abs(base[1:] - base[:1]).max(axis=-1) > 0).all()
    np.testing.assert_array_equal(device_points(seed, [gid], [ep], 32)[0, :x], base)   # X only truncates


def test_no_two_objectives_of_an_env_are_equal():
    p = device_points(20201, np.arange(4096), np.arange(4096) % 5, 32)
    d = np.abs(p[:, :, None, :] - p[:, None, :, :]).max(axis=-1)
    d[:, np.arange(32), np.arange(32)] = np.inf
    assert d.min() > 0
