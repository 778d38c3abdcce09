"""numpy Philox4x32-10 (Salmon, Moraes, Dror, Shaw, SC'11; Random123) and the
integer action map of the device path -- TEST INFRASTRUCTURE ONLY.

The reference draws actions from the global MT19937 stream
(``np.random.randint(-180, 180)``, manytor.py:215-217), which a GPU cannot
reproduce in lock step; the CUDA path uses a counter-based Philox stream keyed
by (seed, global env id, step index) instead.  This restates that stream in
integer arithmetic so tests can check the device's actions bit for bit, and
restates the objective map of the device's auto-reset (``device_points``) in
fp64 so tests can check the refreshed objectives value by value.
Pinned by the Random123 known-answer vectors in tests/test_philox.py.
"""
from __future__ import annotations

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
STREAM_ACTIONS = 0x41435431
STREAM_POINTS = 0x50545331
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised over equal-shaped uint32 arrays; returns 4 uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(v, dtype=np.uint32).copy() for v in (c0, c1, c2, c3))
    k0 = np.asarray(k0, dtype=np.uint32).copy()
    k1 = np.asarray(k1, dtype=np.uint32).copy()
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = M0 * c0.astype(np.uint64)
            p1 = M1 * c2.astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), (p0 & _MASK).astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), (p1 & _MASK).astype(np.uint32)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0 = (k0 + W0).astype(np.uint32)
            k1 = (k1 + W1).astype(np.uint32)
    return c0, c1, c2, c3


def device_actions(seed: int, env_ids: np.ndarray, step_index: int, n_joints: int = 4,
                   low: int = -180, high: int = 180) -> np.ndarray:
    """The (N, J) integer actions mt_sample_actions / mt_rollout_random draw at
    ``step_index`` (manytor_b200/csrc/mt_step.cuh: draw_actions)."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    lo = (env_ids & _MASK).astype(np.uint32)
    hi = (env_ids >> np.uint64(32)).astype(np.uint32)
    step_lo = np.uint32(step_index & 0xFFFFFFFF)
    step_hi = np.uint32((step_index >> 32) & 0xFFFFFFFF)
    k0 = np.full_like(lo, seed & 0xFFFFFFFF)
    k1 = np.full_like(lo, (seed >> 32) & 0xFFFFFFFF)
    span = np.uint64(high - low)
    out = np.zeros((env_ids.size, n_joints), dtype=np.int64)
    for chunk in range((n_joints + 3) // 4):
        tag = np.uint32((STREAM_ACTIONS + chunk) & 0xFFFFFFFF) ^ step_hi
        w = philox4x32_10(lo, hi, np.full_like(lo, step_lo), np.full_like(lo, tag), k0, k1)
        for i in range(4):
            j = chunk * 4 + i
            if j < n_joints:
                out[:, j] = low + ((w[i].astype(np.uint64) * span) >> np.uint64(32)).astype(np.int64)
    return out


def _u01(w: np.ndarray) -> np.ndarray:
    """mt_math.cuh ``uniform01``: the top 24 bits times 2^-24, exact in fp32 and fp64."""
    return (w >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


def device_points(seed: int, env_ids: np.ndarray, episodes, x: int, radius: float = 51.3) -> np.ndarray:
    """The (N, X, 3) objectives the device draws for the reset that starts episode ``episodes[i]`` of env
    ``env_ids[i]`` (manytor_b200/csrc/mt_step.cuh: sample_point, called by reset_kernel and settle_step),
    in fp64.  ``episodes`` is per env (or one value for all): the number of resets the env had before.

    Counter (gid lo, gid hi, episode * 32 + objective mod 2^32, STREAM_POINTS), key (seed lo, seed hi);
    words x, y, z of the block give r = min(R cbrt(1 - u01(x)), R), cos(theta) = u01(y) and
    phi = 2 pi u01(z), where R is the fp32 radius the config holds.  The device evaluates the same map in
    fp32 (cbrtf, sincospif, 1 - ct^2 as one FFMA), a few fp32 roundings of R from these values."""
    env_ids = np.asarray(env_ids, dtype=np.uint64).reshape(-1)
    n = env_ids.size
    ep = np.broadcast_to(np.asarray(episodes, dtype=np.uint64).reshape(-1), (n,))
    lo = np.repeat((env_ids & _MASK).astype(np.uint32)[:, None], x, axis=1)
    hi = np.repeat((env_ids >> np.uint64(32)).astype(np.uint32)[:, None], x, axis=1)
    ctr = ((ep[:, None] * np.uint64(32) + np.arange(x, dtype=np.uint64)[None, :]) & _MASK).astype(np.uint32)
    k0 = np.full_like(lo, seed & 0xFFFFFFFF)
    k1 = np.full_like(lo, (seed >> 32) & 0xFFFFFFFF)
    wx, wy, wz, _ = philox4x32_10(lo, hi, ctr, np.full_like(lo, STREAM_POINTS), k0, k1)
    big_r = float(np.float32(radius))
    r = np.minimum(big_r * np.cbrt(1.0 - _u01(wx)), big_r)
    ct = _u01(wy)
    st = np.sqrt(np.maximum(1.0 - ct * ct, 0.0))          # ct has 24 bits: ct^2 and 1 - ct^2 are exact here
    phi = 2.0 * np.pi * _u01(wz)
    return np.stack([r * st * np.cos(phi), r * st * np.sin(phi), r * ct], axis=-1)
