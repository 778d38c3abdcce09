"""Vectorised float64 numpy restatement of ManyTor's environment step loop.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``): the product path in
``manytor_b200/`` never imports this module.

Every function cites the reference lines (paths under ``/root/reference``) it
restates.  The arithmetic is kept literal -- real 4x4 DH matrices chained by
matrix products in float64, all 25 interpolated sub-poses evaluated in full --
so that it can be checked step-for-step against the unmodified reference
(``tests/golden/make_golden.py``) and then serve as the checker for the CUDA
path, which uses a closed-form fp32 formulation instead.

Batch convention: N lock-step environments, J joints, X objectives.
  goals   (N, J)  float64  joint targets in DEGREES (absolute, not deltas)
  points  (N, X, 3) float64
  alive   (N, X)  bool
Frames: frame 0 is the base; frame k is the origin after the first k DH rows.
The reference stacks ``joints_coordinates`` = [base, frame 2, frame 3, frame 4]
(manytor.py:188-189), observes from row 2 = frame 3 (manytor.py:143), tests the
ground on rows 2 and 3 = frames 3 and 4 (manytor.py:191) and catches with row
3 = frame 4 (manytor.py:162).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import NamedTuple, Optional, Sequence

import numpy as np


# --------------------------------------------------------------------------
# arm description (the reference hard-codes this inside fk(), manytor.py:42-48)
# --------------------------------------------------------------------------
@dataclass(frozen=True)
class ArmSpec:
    """DH table rows are (a, alpha, d, theta_offset); angles in radians."""

    dh: tuple                     # J rows of 4 floats
    obs_frame: int                # frame whose origin anchors observations
    ground_frames: tuple          # two frames whose z is tested against the ground
    catch_frame: int              # frame that catches objectives
    radius: float = 51.3          # objective half-ball radius       (manytor.py:231,236)
    catch_tol: float = 8.0        # per-axis inclusive catch tolerance (manytor.py:162)
    substeps: int = 25            # interpolated poses per step       (manytor.py:178)
    action_low: int = -180        # action_sample range               (manytor.py:216)
    action_high: int = 180

    @property
    def n_joints(self) -> int:
        return len(self.dh)

    def table(self) -> np.ndarray:
        return np.asarray(self.dh, dtype=np.float64).reshape(self.n_joints, 4)


# manytor.py:42-48 -- (a, alpha, d, theta offset)
REFERENCE_ARM = ArmSpec(
    dh=(
        (0.0, -np.pi / 2, 4.3, 0.0),
        (0.0, np.pi / 2, 0.0, 0.0),
        (0.0, -np.pi / 2, 24.3, 0.0),
        (27.0, np.pi / 2, 0.0, -np.pi / 2),
    ),
    obs_frame=3,
    ground_frames=(3, 4),
    catch_frame=4,
)

# BASELINE.json config 5: "generalised 6-DOF DH chain via pluggable FK
# (UR5-style params)".  The reference has no 6-DOF arm; these are the public
# UR5 DH figures in metres, with the frame selectors generalised as in
# SURVEY.md section 8(a-FK): obs = frame J-1, ground = frames J-1 and J,
# catch = frame J; radius = |a2|+|a3|, tolerance scaled like 8.0/51.3.
UR5_ARM = ArmSpec(
    dh=(
        (0.0, np.pi / 2, 0.089159, 0.0),
        (-0.425, 0.0, 0.0, 0.0),
        (-0.39225, 0.0, 0.0, 0.0),
        (0.0, np.pi / 2, 0.10915, 0.0),
        (0.0, -np.pi / 2, 0.09465, 0.0),
        (0.0, 0.0, 0.0823, 0.0),
    ),
    obs_frame=5,
    ground_frames=(5, 6),
    catch_frame=6,
    radius=0.81725,
    catch_tol=0.81725 * 8.0 / 51.3,
)


# --------------------------------------------------------------------------
# kinematics
# --------------------------------------------------------------------------
def dh(a, alfa, d, theta):
    """One 4x4 DH transform, batched over leading dims of ``theta``.

    Restates manytor.py:25-32 (standard DH: Rz(theta) Tz(d) Tx(a) Rx(alfa)).
    """
    theta = np.asarray(theta, dtype=np.float64)
    ct, st = np.cos(theta), np.sin(theta)
    ca, sa = np.cos(alfa), np.sin(alfa)
    m = np.zeros(theta.shape + (4, 4), dtype=np.float64)
    m[..., 0, 0] = ct
    m[..., 0, 1] = -st * ca
    m[..., 0, 2] = st * sa
    m[..., 0, 3] = a * ct
    m[..., 1, 0] = st
    m[..., 1, 1] = ct * ca
    m[..., 1, 2] = -ct * sa
    m[..., 1, 3] = a * st
    m[..., 2, 1] = sa
    m[..., 2, 2] = ca
    m[..., 2, 3] = d
    m[..., 3, 3] = 1.0
    return m


def _chain(spec: ArmSpec, goals_deg: np.ndarray, upto: int) -> list:
    """Prefix products T_1, T_1 T_2, ... of the first ``upto`` DH rows.

    manytor.py:39 converts degrees to radians per joint, :42-48 builds the
    rows (the offset is added to the already-converted angle), :50-52 chains
    them left to right starting from the identity.
    """
    goals_deg = np.asarray(goals_deg, dtype=np.float64)
    t = goals_deg * (math.pi / 180.0)            # math.radians, manytor.py:39
    tab = spec.table()
    out = []
    m = None
    for i in range(upto):
        a, alfa, d, off = tab[i]
        h = dh(a, alfa, d, t[..., i] + off)
        m = h if m is None else np.matmul(m, h)  # eye(4).dot(h) == h exactly
        out.append(m)
    return out


def fk(mode: int, goals, spec: ArmSpec = REFERENCE_ARM) -> np.ndarray:
    """4x4 transform of frame ``mode`` -- restates manytor.py:35-53."""
    return _chain(spec, np.asarray(goals, dtype=np.float64), mode)[-1]


def fk_frames(goals_deg, spec: ArmSpec = REFERENCE_ARM) -> np.ndarray:
    """Origins of frames 0..J, shape (..., J+1, 3).

    The reference evaluates ``fk(mode=i)[0:3, 3]`` for i = 2, 3, 4 and stacks
    them under a zero row (manytor.py:188-189); frame 1 is included here too so
    that generic arms can select any frame.
    """
    goals_deg = np.asarray(goals_deg, dtype=np.float64)
    mats = _chain(spec, goals_deg, spec.n_joints)
    out = np.zeros(goals_deg.shape[:-1] + (spec.n_joints + 1, 3), dtype=np.float64)
    for k, m in enumerate(mats):
        out[..., k + 1, :] = m[..., 0:3, 3]
    return out


def joints_coordinates(goals_deg, spec: ArmSpec = REFERENCE_ARM) -> np.ndarray:
    """The reference's ``joints_coordinates``: rows [base, frame 2 .. frame J]
    (manytor.py:188-189), shape (..., J, 3)."""
    fr = fk_frames(goals_deg, spec)
    return np.concatenate([fr[..., 0:1, :], fr[..., 2:, :]], axis=-2)


def r_theta(v1, v2):
    """Bearing angles in degrees of |v1 - v2| -- restates manytor.py:17-22.

    Vectorised over leading dims; both angles lie in [0, 90].
    """
    d = np.abs(np.asarray(v1, dtype=np.float64) - np.asarray(v2, dtype=np.float64))
    h_l = np.sqrt(d[..., 0] ** 2 + d[..., 1] ** 2)
    r = np.degrees(np.arctan2(d[..., 0], d[..., 1]))
    theta = np.degrees(np.arctan2(h_l, d[..., 2]))
    return r, theta


def observations(anchor: np.ndarray, points: np.ndarray, alive: np.ndarray) -> np.ndarray:
    """Observation vector (N, 3X) -- restates manytor.py:141-153.

    Per objective: [euclidean distance, r, theta] measured from ``anchor`` (the
    obs frame, i.e. the elbow for the reference arm, manytor.py:143), or three
    zeros when the objective is dead (manytor.py:146-148).
    """
    n, x, _ = points.shape
    mod = np.abs(anchor[:, None, :] - points)                       # manytor.py:150
    euc = np.sqrt(np.sqrt(mod[..., 0] ** 2 + mod[..., 1] ** 2) ** 2 + mod[..., 2] ** 2)  # :151
    r, theta = r_theta(anchor[:, None, :], points)                  # :152
    obs = np.stack([euc, r, theta], axis=-1)                        # (N, X, 3)
    obs = np.where(alive[..., None], obs, 0.0)
    return obs.reshape(n, 3 * x)


def _route(goals: np.ndarray, action: np.ndarray, num: int) -> np.ndarray:
    """``np.linspace(goals, action, num)`` per environment (manytor.py:182).

    numpy evaluates ``arange(num) * (delta / div) + start`` unless *any* joint
    of that call has a zero step, in which case it uses ``(arange(num) / div) *
    delta + start``; the last pose is pinned to ``action`` exactly.  The
    reference calls linspace once per env, so the any() is per env.
    """
    div = num - 1
    k = np.arange(num, dtype=np.float64).reshape(num, 1, 1)
    delta = action - goals
    step = delta / div
    a = k * step[None] + goals[None]
    b = (k / div) * delta[None] + goals[None]
    use_b = np.any(step == 0, axis=-1)                              # (N,)
    route = np.where(use_b[None, :, None], b, a)
    route[-1] = action
    return route                                                    # (num, N, J)


# --------------------------------------------------------------------------
# reference RNG streams (legacy global numpy MT19937)
# --------------------------------------------------------------------------
def sample_points_reference_stream(x: int, radius: float = 51.3) -> np.ndarray:
    """Draw X objectives exactly as the reference does -- manytor.py:228-241.

    Consumes the process-global ``np.random`` stream scalar by scalar, three
    uniforms per trial, accepting z >= 0 inside the ball.
    """
    pts = []
    while len(pts) < x:
        c = [np.random.uniform(-radius, radius) for _ in range(3)]
        if c[2] >= 0:
            value = math.sqrt(math.sqrt(c[0] ** 2 + c[1] ** 2) ** 2 + c[2] ** 2)
            if value <= radius:
                pts.append(c)
    return np.asarray(pts, dtype=np.float64).reshape(x, 3)


def action_sample_reference_stream(n_joints: int = 4, low: int = -180, high: int = 180) -> np.ndarray:
    """One ``action_sample()`` -- manytor.py:215-217 (integers, high exclusive)."""
    return np.asarray([np.random.randint(low=low, high=high, size=1)[0] for _ in range(n_joints)],
                      dtype=np.float64)


# --------------------------------------------------------------------------
# the batched environment
# --------------------------------------------------------------------------
class StepResult(NamedTuple):
    obs: np.ndarray            # (N, 3X) float64   obs2 of manytor.py:204
    reward: np.ndarray         # (N,)   int64 in {-1, 0, 1}
    done: np.ndarray           # (N,)   bool
    joints: np.ndarray         # (N, J, 3) joints_coordinates at the final pose
    alive: np.ndarray          # (N, X) bool after this step's catches
    neg: np.ndarray            # (N,)   bool ground flag (sticky over the 25 poses)
    ground_margin: np.ndarray  # (N,)   min |z| over sub-poses and ground frames
    catch_margin: np.ndarray   # (N, X) distance of the catch decision from flipping
    frames: np.ndarray         # (N, J+1, 3) origins of frames 0..J at the final pose, indexed by frame number


class OracleEnvs:
    """N independent reference environments advanced in lock step.

    State and transitions restate ``Environment`` (manytor.py:125-260); the N
    dimension replaces the sequential loop of ``Multienv`` (manytor.py:106-122).
    ``terminate_on_ground`` is the README's reading (README.md:44); the code's
    behaviour, and the default here, is False (SURVEY.md Q1).
    """

    def __init__(self, n_envs: int, obj_number: int = 10, spec: ArmSpec = REFERENCE_ARM,
                 terminate_on_ground: bool = False):
        self.n = int(n_envs)
        self.x = int(obj_number)
        self.spec = spec
        self.j = spec.n_joints
        self.terminate_on_ground = bool(terminate_on_ground)
        self.goals = np.zeros((self.n, self.j))                     # manytor.py:133
        self.alive = np.ones((self.n, self.x), dtype=bool)          # manytor.py:134
        self.points = np.zeros((self.n, self.x, 3))
        self.total_reward = np.zeros(self.n)                        # manytor.py:138
        self.ep_len = np.zeros(self.n, dtype=np.int64)
        self.joints = joints_coordinates(self.goals, spec)

    # -- frame helpers ------------------------------------------------------
    def _row(self, frame: int) -> int:
        """Row of ``joints_coordinates`` holding ``frame`` (row 0 = base, row r = frame r+1).

        Frame 1 has no row there (manytor.py:188-189): select it from ``StepResult.frames`` /
        ``fk_frames``, which are indexed by frame number and hold every frame."""
        if frame == 1:
            raise ValueError("joints_coordinates has no row for frame 1; index fk_frames / StepResult.frames instead")
        return 0 if frame == 0 else frame - 1

    # -- reset --------------------------------------------------------------
    def reset(self, mask: Optional[np.ndarray] = None, points: Optional[np.ndarray] = None,
              returnable: bool = False):
        """Restates ``Environment.reset`` (manytor.py:219-253) for the masked envs.

        ``points`` (N, X, 3) supplies the fresh objectives (rows outside the mask
        are ignored).  When omitted they are drawn from the reference's global
        ``np.random`` stream in env order, as ``Multienv.reset`` would
        (manytor.py:106-107).
        """
        if mask is None:
            mask = np.ones(self.n, dtype=bool)
        mask = np.asarray(mask, dtype=bool)
        idx = np.nonzero(mask)[0]
        self.goals[idx] = 0.0                                       # :220
        self.total_reward[idx] = 0.0                                # :221
        self.alive[idx] = True                                      # :222
        self.ep_len[idx] = 0
        if points is None:
            for i in idx:                                           # :228-241
                self.points[i] = sample_points_reference_stream(self.x, self.spec.radius)
        else:
            self.points[idx] = np.asarray(points, dtype=np.float64)[idx]
        self.joints = joints_coordinates(self.goals, self.spec)     # :224-225
        if returnable:                                              # :251-253
            return self.get_observations()
        return None

    def get_observations(self) -> np.ndarray:
        """manytor.py:141-153, including the side effect of zeroing dead points."""
        self.points[~self.alive] = 0.0                              # :148
        anchor = fk_frames(self.goals, self.spec)[:, self.spec.obs_frame]
        return observations(anchor, self.points, self.alive)

    # -- step ---------------------------------------------------------------
    def step(self, action) -> StepResult:
        """Restates ``Environment.step`` -> ``action`` -> ``is_done``
        (manytor.py:255-260, 175-213, 155-173)."""
        spec = self.spec
        action = np.asarray(action, dtype=np.float64).reshape(self.n, self.j)
        self.points[~self.alive] = 0.0                              # :256 -> :148 side effect
        initial = self.alive.copy()                                 # :180
        route = _route(self.goals, action, spec.substeps)           # :182

        ga, gb = spec.ground_frames
        neg = np.zeros(self.n, dtype=bool)
        margin = np.full(self.n, np.inf)
        for p in range(spec.substeps):                              # :183
            fr = fk_frames(route[p], spec)                          # :188
            za, zb = fr[:, ga, 2], fr[:, gb, 2]
            neg |= (za < 0) | (zb < 0)                              # :191-192
            margin = np.minimum(margin, np.minimum(np.abs(za), np.abs(zb)))
        self.goals = route[-1].copy()                               # :184 (last pose == action)
        self.joints = np.concatenate([fr[:, 0:1], fr[:, 2:]], axis=1)   # :189

        # anchor and catcher by frame number: joints_coordinates has no row for frame 1
        obs2 = observations(fr[:, spec.obs_frame], self.points, self.alive)  # :204

        ee = fr[:, spec.catch_frame]                                # :162
        dist = np.abs(ee[:, None, :] - self.points)                 # (N, X, 3)
        close = dist <= spec.catch_tol                              # math.isclose(abs_tol), rel term < 6e-8
        caught = close.all(axis=-1)                                 # :167
        self.alive = self.alive & ~caught                           # :168
        slack = spec.catch_tol - dist
        viol = np.where(slack < 0, -slack, -np.inf)
        catch_margin = np.where(caught, slack.min(axis=-1), viol.max(axis=-1))

        reward = np.where(initial.sum(axis=1) > self.alive.sum(axis=1), 1, 0)   # :208-209
        reward = np.where(neg, -1, reward).astype(np.int64)         # :211-212
        self.total_reward = self.total_reward + reward              # :258
        self.ep_len = self.ep_len + 1
        done = ~self.alive.any(axis=1)                              # :170-171, :259
        if self.terminate_on_ground:
            done = done | neg
        return StepResult(obs2, reward, done, self.joints.copy(), self.alive.copy(), neg,
                          margin, catch_margin, fr)

    # -- state exchange with the device path ---------------------------------
    def alive_mask_u32(self) -> np.ndarray:
        w = (1 << np.arange(self.x, dtype=np.uint64))
        return (self.alive.astype(np.uint64) * w).sum(axis=1).astype(np.uint32)
