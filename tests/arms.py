"""One DH table for every joint count the generic chain is built for (J = 2 .. 8).

`step_kernel<J, ...>`, the helper kernels and the NVRTC `Preset<1000 + J>` are instantiated for each J;
these tables give each of them an arm to run.  Between them the snapped rows (cos / sin of alpha and of the
theta offset, as mt_api.cu's `snap` leaves them) cover every case that `push_row` folds at compile time --
alpha in {0, pi/2, -pi/2, pi} and general values, offsets in {0, +-pi/2, pi} and general values -- and a, d
negative, zero and positive.  tests/test_arm_tables.py asserts that coverage.

Frame selectors default to the usual ones (obs J-1, ground J-1 and J, catch J: the only ones NVRTC
specialises); radius = 0.8 reach and catch_tol scaled like the reference's 8.0 / 51.3.
"""
from __future__ import annotations

import math

from oracle import ArmSpec as OracleArm

PI = math.pi

# rows (a, alpha, d, theta offset), radians; an alpha on the LAST row moves no frame origin, so the
# folded alphas (pi above all) sit on inner rows where they matter
TABLES = {
    2: ((0.20, PI / 2, 0.40, 0.0), (0.45, PI, 0.0, PI / 2)),
    3: ((0.0, PI / 2, 0.25, 0.0), (-0.40, PI, 0.0, PI / 2), (0.30, 0.0, 0.05, 0.0)),
    4: ((0.05, -PI / 2, 0.30, PI), (0.35, 0.3, 0.0, -PI / 2), (0.25, PI / 2, -0.05, 0.0), (0.10, 0.0, 0.0, 0.4)),
    5: ((0.0, PI / 2, 0.20, 0.0), (0.40, 0.0, 0.0, 0.0), (-0.30, PI, 0.05, PI / 2), (0.0, -PI / 2, 0.10, 0.0),
        (0.10, 1.2, 0.0, 0.0)),
    6: ((0.0, PI / 2, 0.15, 0.0), (-0.35, 0.0, 0.0, -PI / 2), (-0.30, 0.0, 0.0, 0.0), (0.0, PI / 2, 0.10, PI),
        (0.0, -PI / 2, 0.08, 0.0), (0.05, 0.0, 0.06, 0.0)),
    7: ((0.0, -PI / 2, 0.20, 0.0), (0.30, PI / 2, 0.0, 0.0), (0.0, -PI / 2, 0.25, PI / 2), (0.20, PI, 0.0, 0.0),
        (0.0, PI / 2, -0.04, 0.0), (0.15, -0.8, 0.0, -PI / 2), (0.06, 0.0, 0.02, 0.3)),
    8: ((0.0, PI / 2, 0.10, 0.0), (0.25, 0.0, 0.0, PI / 2), (0.20, PI, 0.0, 0.0), (0.0, -PI / 2, 0.10, -PI / 2),
        (0.15, 0.5, -0.03, 0.0), (0.0, PI / 2, 0.05, PI), (0.08, -PI / 2, 0.0, 0.7), (0.05, 0.0, 0.03, 0.0)),
}


def reach(dh) -> float:
    return float(sum(abs(r[0]) + abs(r[2]) for r in dh))


def snap(v: float) -> float:
    """mt_api.cu's snap(): cos / sin within fp32 rounding of 0 or +-1 become exactly that."""
    return 0.0 if abs(v) < 5e-7 else ((1.0 if v > 0 else -1.0) if abs(abs(v) - 1.0) < 5e-7 else v)


def snapped_rows(dh):
    """(a, d, ca, sa, co, so) per row as the device holds them (fill_arm, after the fp32 round trip)."""
    import numpy as np
    out = []
    for a, alpha, d, off in dh:
        alpha, off = float(np.float32(alpha)), float(np.float32(off))
        out.append((float(np.float32(a)), float(np.float32(d)), snap(math.cos(alpha)), snap(math.sin(alpha)),
                    snap(math.cos(off)), snap(math.sin(off))))
    return out


def arm_pair(J: int, obs_frame=None, ground_frames=None, catch_frame=None, substeps: int = 25):
    """(oracle.ArmSpec, manytor_b200.ArmSpec) of the J-joint table; selectors default to the usual ones."""
    import manytor_b200
    dh = TABLES[J]
    radius = 0.8 * reach(dh)
    sel = dict(obs_frame=J - 1 if obs_frame is None else obs_frame,
               ground_frames=(J - 1, J) if ground_frames is None else tuple(ground_frames),
               catch_frame=J if catch_frame is None else catch_frame,
               radius=radius, catch_tol=radius * 8.0 / 51.3)
    return OracleArm(dh=dh, substeps=substeps, **sel), manytor_b200.ArmSpec(dh=dh, **sel)


JOINT_COUNTS = tuple(sorted(TABLES))
