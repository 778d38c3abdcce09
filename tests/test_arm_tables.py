"""The per-joint-count DH tables of tests/arms.py cover what the kernels fold (no GPU needed)."""
import math

import numpy as np

from arms import JOINT_COUNTS, TABLES, arm_pair, reach, snapped_rows


def test_one_table_per_generic_joint_count():
    assert JOINT_COUNTS == tuple(range(2, 9))                  # step_kernel<J, ...> for J = 2 .. 8 (mt_api.cu pick_kernel)
    for J in JOINT_COUNTS:
        ora, dev = arm_pair(J)
        assert ora.n_joints == dev.n_joints == J and ora.dh == dev.dh
        assert (ora.obs_frame, ora.ground_frames, ora.catch_frame) == (J - 1, (J - 1, J), J)
        assert (dev.obs_frame, dev.ground_frames, dev.catch_frame) == (J - 1, (J - 1, J), J)
        assert ora.radius == dev.radius == 0.8 * reach(TABLES[J])
        assert math.isclose(ora.catch_tol, ora.radius * 8.0 / 51.3) and ora.catch_tol == dev.catch_tol


def test_tables_cover_every_folded_case():
    """After snapping, the tables hold alpha in {0, pi/2, -pi/2, pi} and two general values, theta offsets in
    {0, +-pi/2, pi} and a general value, and negative, zero and positive a and d -- each fold of push_row's preset
    branch on an inner row, where it moves a frame origin (alpha of the last row moves none)."""
    alphas, offsets, a_signs, d_signs = set(), set(), set(), set()
    general_alpha, general_offset = set(), set()
    for J in JOINT_COUNTS:
        for i, (a, d, ca, sa, co, so) in enumerate(snapped_rows(TABLES[J])):
            a_signs.add(int(np.sign(a)))
            d_signs.add(int(np.sign(d)))
            if (co, so) in ((1.0, 0.0), (0.0, 1.0), (0.0, -1.0), (-1.0, 0.0)):
                offsets.add((co, so))
            else:
                general_offset.add((co, so))
            if i == J - 1:
                continue
            if (ca, sa) in ((1.0, 0.0), (0.0, 1.0), (0.0, -1.0), (-1.0, 0.0)):
                alphas.add((ca, sa))
            else:
                general_alpha.add((ca, sa))
    assert alphas == {(1.0, 0.0), (0.0, 1.0), (0.0, -1.0), (-1.0, 0.0)}
    assert len(general_alpha) >= 2
    assert offsets == {(1.0, 0.0), (0.0, 1.0), (0.0, -1.0), (-1.0, 0.0)}
    assert len(general_offset) >= 1
    assert a_signs == {-1, 0, 1} and d_signs == {-1, 0, 1}

