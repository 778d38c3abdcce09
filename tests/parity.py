"""Lock-step comparison of the CUDA path with the CPU oracle.

Parity bar (BASELINE.json north_star): joint / end-effector positions within
1e-5 relative (of the arm's reach) in fp32; reward, catch events (alive mask)
and done flags bit-exact EXCEPT where a distance lies within `THRESH_TOL` of the
catch or ground threshold -- those cases are counted and reported, and the
device state is re-synchronised to the oracle so the rest of the run stays
comparable.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

REL_POS_TOL = 1e-5          # of reach
THRESH_TOL = 1e-3           # |distance - threshold| below which a flag flip is "near-threshold"
DIST_ATOL_REL = 2e-5        # distance observation, relative to reach
ANGLE_FLOOR_DEG = 1e-3      # angle observation floor; plus the conditioning term below


@dataclass
class Report:
    env_steps: int = 0
    max_joint_err: float = 0.0
    max_dist_err: float = 0.0
    max_angle_excess: float = 0.0      # worst (error / allowed)
    near_threshold: int = 0            # reported, allowed
    hard_mismatch: int = 0             # must stay 0
    rewarded: int = 0                  # env-steps with reward +1 (oracle): catches were compared
    ground: int = 0                    # env-steps with ground contact (oracle): the ground test was compared
    max_point_err: float = 0.0         # refreshed objectives against their fp64 restatement (Philox objectives)
    notes: list = field(default_factory=list)

    def ok(self) -> bool:
        return self.hard_mismatch == 0

    def summary(self) -> str:
        return (f"{self.env_steps} env-steps: joint err {self.max_joint_err:.2e}, dist err {self.max_dist_err:.2e}, "
                f"angle err/allowed {self.max_angle_excess:.2f}, near-threshold flips {self.near_threshold}, "
                f"hard mismatches {self.hard_mismatch}; events: reward +1 {self.rewarded}, ground {self.ground}")


def reach_of(spec) -> float:
    tab = spec.table()
    return float(np.abs(tab[:, 0]).sum() + np.abs(tab[:, 2]).sum())


def compare_step(rep: Report, spec, ora, r, points_before, alive_before, dev_obs, dev_reward, dev_done,
                 dev_alive, dev_joints=None, scale=None, obs_rows=None):
    """Compare one step.  `r` is the oracle StepResult; returns the bool mask of
    envs whose flags differ (all of them near-threshold, or hard_mismatch grows).
    The observations are compared on the rows `obs_rows` (default all; none when `dev_obs` is None)."""
    n, x = alive_before.shape
    reach = reach_of(spec)
    pos_tol = REL_POS_TOL * reach
    thr = THRESH_TOL * (reach / 55.6)
    rep.env_steps += n
    rep.rewarded += int((r.reward == 1).sum())
    rep.ground += int(r.neg.sum())

    if dev_joints is not None:
        je = np.abs(dev_joints.astype(np.float64) - r.joints).max()
        rep.max_joint_err = max(rep.max_joint_err, float(je))
        if je > pos_tol:
            rep.hard_mismatch += 1
            rep.notes.append(f"joint error {je:.3e} > {pos_tol:.3e}")

    # flags
    rew_bad = dev_reward.astype(np.int64) != r.reward
    done_bad = (dev_done & 1).astype(bool) != r.done
    alive_bad = (dev_alive != r.alive).any(axis=1)
    bad = rew_bad | done_bad | alive_bad
    cm = np.where(alive_before, np.abs(r.catch_margin), np.inf).min(axis=1)
    near = (r.ground_margin < thr) | (cm < thr)
    rep.near_threshold += int((bad & near).sum())
    hard = bad & ~near
    if hard.any():
        rep.hard_mismatch += int(hard.sum())
        i = int(np.nonzero(hard)[0][0])
        rep.notes.append(f"env {i}: reward dev {dev_reward[i]} ora {r.reward[i]}, done dev {dev_done[i]} ora {r.done[i]}, "
                         f"ground margin {r.ground_margin[i]:.3e}, catch margin {cm[i]:.3e}")

    # observations (computed from alive_before, which is kept in sync)
    if dev_obs is not None and (obs_rows is None or obs_rows.any()):
        o = slice(None) if obs_rows is None else obs_rows
        compare_obs(rep, spec, r.frames[o, spec.obs_frame], points_before[o], alive_before[o], dev_obs[o], r.obs[o])
    return bad


def compare_obs(rep: Report, spec, anchor, points, alive, dev_obs, ref_obs):
    """Compare observations (N, 3X) of objectives `points` (N, X, 3) seen from `anchor` (N, 3): distances within
    DIST_ATOL_REL of reach, bearings within the error a position error of REL_POS_TOL moves them by (plus a floor),
    dead objectives exactly zero.  Misses count as hard mismatches."""
    n, x = alive.shape
    reach = reach_of(spec)
    pos_tol = REL_POS_TOL * reach
    d = np.abs(anchor[:, None, :] - points)
    hxy = np.hypot(d[..., 0], d[..., 1])
    dist = np.sqrt(hxy ** 2 + d[..., 2] ** 2)
    o_dev = dev_obs.astype(np.float64).reshape(n, x, 3)
    o_ref = ref_obs.reshape(n, x, 3)
    de = np.abs(o_dev[..., 0] - o_ref[..., 0])
    rep.max_dist_err = max(rep.max_dist_err, float(de.max()))
    dist_tol = DIST_ATOL_REL * reach + pos_tol
    # an angle moves by ~ position error / lever arm; allow that plus a floor
    allow_r = np.degrees(pos_tol / np.maximum(hxy, 1e-9)) + ANGLE_FLOOR_DEG
    allow_t = np.degrees(pos_tol / np.maximum(dist, 1e-9)) + ANGLE_FLOOR_DEG
    er = np.abs(o_dev[..., 1] - o_ref[..., 1]) / np.minimum(allow_r, 90.0)
    et = np.abs(o_dev[..., 2] - o_ref[..., 2]) / np.minimum(allow_t, 90.0)
    ex = max(float(er.max()), float(et.max()))
    rep.max_angle_excess = max(rep.max_angle_excess, ex)
    if de.max() > dist_tol or ex > 1.0:
        rep.hard_mismatch += 1
        rep.notes.append(f"obs mismatch: dist err {de.max():.3e} (tol {dist_tol:.3e}), angle err/allowed {ex:.2f}")
    dead = ~alive
    if dead.any() and np.abs(o_dev[dead]).max() != 0.0:
        rep.hard_mismatch += 1
        rep.notes.append("dead objective did not read as zeros")


def alive_bits_to_matrix(words: np.ndarray, x: int) -> np.ndarray:
    w = words.astype(np.int64) & 0xFFFFFFFF
    return ((w[:, None] >> np.arange(x)[None, :]) & 1).astype(bool)


def lockstep(env, ora, spec, actions_fn, steps: int, on_done=None, rep: Report | None = None, joints=True):
    """Advance device `env` (BatchedEnvs) and oracle `ora` together for `steps`.

    actions_fn(t) -> (N, J) array.  on_done(t, done_mask) -> (N, X, 3) fresh
    points for the envs that ended (reset on both sides), or None for no reset.
    """
    rep = rep or Report()
    for t in range(steps):
        act = np.float32(np.asarray(actions_fn(t))).astype(np.float64)   # the device sees fp32 actions
        alive_before = ora.alive.copy()
        points_before = ora.points.copy()
        out = env.step(act.astype(np.float32), joints=joints)
        obs, rew, done = (o.cpu().numpy() for o in out[:3])
        jn = out[3].cpu().numpy() if joints else None
        r = ora.step(act)
        dev_alive = alive_bits_to_matrix(env.get_state()["alive"].cpu().numpy(), ora.x)
        bad = compare_step(rep, spec, ora, r, points_before, alive_before, obs, rew, done, dev_alive, jn)
        if bad.any():   # near-threshold flips: put the device back on the oracle's trajectory
            env.set_state(goals=ora.goals, alive=ora.alive, total_reward=ora.total_reward, mask=bad)
        if on_done is not None and r.done.any():
            fresh = on_done(t, r.done)
            if fresh is not None:
                ora.reset(mask=r.done, points=fresh)
                env.reset(mask=r.done)
                env.set_points(fresh, mask=r.done)
    return rep


class ChunkedOracle:
    """One OracleEnvs interface over several smaller ones (bounded temporaries at 2^18..2^20 envs).

    Exposes what `compare_step` / the lock-step loops use: n, x, spec, goals, alive, points,
    total_reward, ep_len, step(), reset()."""

    def __init__(self, n_envs: int, obj_number: int, spec, chunk: int = 1 << 16, **kw):
        from oracle import OracleEnvs
        self.n, self.x, self.spec = int(n_envs), int(obj_number), spec
        self.bounds = [(a, min(a + chunk, self.n)) for a in range(0, self.n, chunk)]
        self.parts = [OracleEnvs(b - a, obj_number, spec=spec, **kw) for a, b in self.bounds]

    def _cat(self, name):
        return np.concatenate([getattr(p, name) for p in self.parts], axis=0)

    goals = property(lambda self: self._cat("goals"))
    alive = property(lambda self: self._cat("alive"))
    points = property(lambda self: self._cat("points"))
    total_reward = property(lambda self: self._cat("total_reward"))
    ep_len = property(lambda self: self._cat("ep_len"))

    def reset(self, mask=None, points=None):
        for (a, b), p in zip(self.bounds, self.parts):
            p.reset(mask=None if mask is None else mask[a:b], points=None if points is None else points[a:b])

    def set_alive(self, alive):
        for (a, b), p in zip(self.bounds, self.parts):
            p.alive = np.array(alive[a:b], dtype=bool)

    def step(self, action):
        from oracle import StepResult
        rs = [p.step(action[a:b]) for (a, b), p in zip(self.bounds, self.parts)]
        return StepResult(*[np.concatenate([getattr(r, f) for r in rs], axis=0) for f in StepResult._fields])


def _seed_late_episode(env, ora, rs, n, x, horizon, alive_p=0.35):
    """Put every env somewhere inside an episode: random poses, a random subset of objectives already
    collected (many envs one catch away from termination), random episode lengths up to the horizon --
    so that the few steps of a test see terminations, truncations and fresh objectives.  `ora` is a
    ChunkedOracle."""
    goals = rs.randint(-180, 180, size=(n, ora.spec.n_joints)).astype(np.float64)
    alive = rs.rand(n, x) < alive_p
    alive[np.arange(n), rs.randint(0, x, size=n)] = True               # at least one objective alive
    total = -rs.randint(0, 40, size=n).astype(np.float64)
    ep = rs.randint(0, horizon, size=n)
    env.set_state(goals=goals.astype(np.float32), alive=alive, total_reward=total.astype(np.float32),
                  ep_len=ep.astype(np.int32))
    from oracle.manytor_oracle import joints_coordinates
    for (a, b), p in zip(ora.bounds, ora.parts):
        p.goals = goals[a:b].copy()
        p.alive = alive[a:b].copy()
        p.total_reward = total[a:b].copy()
        p.ep_len = ep[a:b].astype(np.int64)
        p.joints = joints_coordinates(p.goals, p.spec)


def point_tol_of(spec) -> float:
    """Tolerance of a device-drawn objective against its fp64 restatement (oracle.philox.device_points), per
    component: 4 fp32 ulps of the radius.  cbrtf and sincospif are within 1 ulp, the rest adds a few roundings,
    and 1 - ct^2 is one FFMA (no cancellation near the pole)."""
    return 4.0 * float(np.spacing(np.float32(spec.radius)))


def philox_fresh(seed: int, env_ids, x: int, radius: float):
    """`fresh(episode, ended)` for the loops below: the fp64 objectives (N, X, 3) the device draws for the reset that
    starts episode `episode[i]` of each ended env (rows outside `ended` are zeros)."""
    from oracle.philox import device_points
    env_ids = np.asarray(env_ids, dtype=np.uint64)

    def fresh(episode, ended):
        out = np.zeros((env_ids.size, x, 3))
        out[ended] = device_points(seed, env_ids[ended], episode[ended], x, radius)
        return out
    return fresh


def _zero_pose_obs(spec, points):
    """The first observation of an episode (obs_after_reset): objectives `points` (M, X, 3), all alive, seen from
    the obs frame at the zero pose.  Returns (anchor (M, 3), observations (M, 3X))."""
    from oracle.manytor_oracle import fk_frames, observations
    m, x = points.shape[:2]
    anchor = np.repeat(fk_frames(np.zeros((1, spec.n_joints)), spec)[:, spec.obs_frame], m, axis=0)
    return anchor, observations(anchor, points, np.ones((m, x), dtype=bool))


def _check_fresh_points(rep, dev, want, exact, tol):
    """Refreshed objectives: bit-exact against an uploaded stream, within `tol` of the fp64 restatement otherwise."""
    if exact:
        np.testing.assert_array_equal(dev, np.float32(want))
        return
    err = float(np.abs(dev.astype(np.float64) - want).max()) if dev.size else 0.0
    rep.max_point_err = max(rep.max_point_err, err)
    if err > tol:
        rep.hard_mismatch += 1
        rep.notes.append(f"refreshed objective off by {err:.3e} > {tol:.3e}")


def _new_stats():
    return dict(env_steps=0, episodes=0, terminated=0, reward_sum=0, length_sum=0, catches=0, ground_steps=0,
                live_reward_sum=0)


def _fold_ended(stats, x, r, ended, total, ep_len):
    stats["episodes"] += int(ended.sum())
    stats["terminated"] += int(r.done.sum())
    stats["reward_sum"] += int(total[ended].sum())
    stats["length_sum"] += int(ep_len[ended].sum())
    stats["catches"] += int((x - r.alive[ended].sum(axis=1)).sum())


def lockstep_auto_reset(env, ora, spec, stream, actions_fn, steps: int, horizon: int, rep: Report | None = None,
                        check_points: bool = True, fresh=None, device_step=None, episode=None):
    """Device auto-reset (in-kernel) against the oracle reset on the host with the same objectives.

    The fresh objectives of the e-th reset of an env come either from the uploaded `stream` (E, N, X, 3), set e mod E,
    which the device must copy bit for bit; or, with `stream` None, from `fresh(episode, ended)` -> (N, X, 3) fp64,
    the restated on-device draw (`philox_fresh`): the oracle resets with its fp32 rounding and the device's objectives
    must lie within `point_tol_of(spec)` of it.  `episode` (N,) counts each env's resets so far and is advanced in
    place; by default both sides have had exactly one (episode 0).  `device_step(act)` -> (obs, reward, done) advances the device (default `env.step`).  With
    obs_after_reset an ended env's observation is the first one of its next episode: it is compared with the
    oracle's observation of the fresh objectives from the zero pose.

    Returns (report, expected statistics (all eight words), reward slack, forked): a near-threshold catch/done flip
    changes WHICH envs reset, after which the two sides are no longer comparable -- the loop stops there and says
    so (`forked`)."""
    rep = rep or Report()
    n, x = ora.n, ora.x
    if stream is not None:
        sets = stream.shape[0]
        fresh = lambda ep, ended: stream[ep % sets, np.arange(n)]
    device_step = device_step or (lambda a: env.step(a.astype(np.float32)))
    oar = bool(env.cfg.obs_after_reset)
    tol = point_tol_of(spec)
    episode = np.ones(n, dtype=np.int64) if episode is None else episode      # resets so far
    stats = _new_stats()
    slack, forked = 0, False
    for t in range(steps):
        act = np.float32(np.asarray(actions_fn(t))).astype(np.float64)
        alive_before, points_before = ora.alive.copy(), ora.points.copy()
        obs, rew, done = (o.cpu().numpy() for o in device_step(act))
        r = ora.step(act)
        ep_len, total = ora.ep_len, ora.total_reward
        trunc = (ep_len >= horizon) & ~r.done if horizon > 0 else np.zeros(n, dtype=bool)
        ended = r.done | trunc
        st = env.get_state()
        dev_alive_after = alive_bits_to_matrix(st["alive"].cpu().numpy(), x)
        dev_alive = np.where(ended[:, None], r.alive, dev_alive_after)       # ended envs were reset on the device
        keep_obs = ~ended if oar else None
        bad = compare_step(rep, spec, ora, r, points_before, alive_before, obs, rew, done, dev_alive, None,
                           obs_rows=keep_obs)
        stats["env_steps"] += n
        stats["ground_steps"] += int(np.where(bad, rew == -1, r.neg).sum())   # the device's own flag where it flipped
        if not rep.ok():
            break
        if bad.any():
            fork = (((done & 1).astype(bool) != r.done) | (dev_alive != r.alive).any(axis=1)) & bad
            if fork.any():
                forked = True
                break
            slack += 2 * int((bad & ended).sum())
            if (bad & ~ended).any():
                env.set_state(total_reward=total, mask=bad & ~ended)
        assert np.array_equal((done & 2).astype(bool), trunc), "truncation flags differ"
        if ended.any():
            _fold_ended(stats, x, r, ended, total, ep_len)
            pts = fresh(episode, ended)
            ora.reset(mask=ended, points=np.float32(pts).astype(np.float64))
            episode[ended] += 1
            assert np.all(dev_alive_after[ended]) and np.all(st["goals"].cpu().numpy()[ended] == 0)
            assert np.all(st["ep_len"].cpu().numpy()[ended] == 0) and np.all(st["total_reward"].cpu().numpy()[ended] == 0)
            if check_points:
                _check_fresh_points(rep, env.get_points(zero_dead=False).cpu().numpy()[ended], pts[ended],
                                    stream is not None, tol)
            if oar:
                anchor, want = _zero_pose_obs(spec, ora.points[ended])
                compare_obs(rep, spec, anchor, ora.points[ended], np.ones((int(ended.sum()), x), dtype=bool),
                            obs[ended], want)
    stats["live_reward_sum"] = int(ora.total_reward.sum())
    return rep, stats, slack, forked


def _rows(r, keep):
    return type(r)(*[f[keep] for f in r])


def lockstep_chunked(env, ora, spec, fresh, seed: int, k: int, chunks: int, horizon: int, rep: Report | None = None,
                     write_obs: bool = True, episode=None):
    """`chunks` calls of env.rollout_random(k) (in-kernel actions, auto-reset, Philox objectives) against the oracle
    advanced k steps per call with the restated actions (oracle.philox.device_actions at env.step_index + s) and
    objectives (`fresh`, as in lockstep_auto_reset).  Only the last step of a call can be read back: its outputs
    are compared (compare_step), and so are the full state -- goals, alive words, total_reward and ep_len exactly
    -- and the objectives refreshed during the call.  `episode` is as in lockstep_auto_reset.

    A near-threshold flip inside a call cannot be re-synchronised.  Every env depends on its own id alone, so an
    env whose state differs after a call in which one of its margins came within THRESH_TOL is dropped from all
    later comparisons and counted as a near-threshold flip; a difference without such a margin is a hard mismatch.
    Returns (report, expected statistics, dropped mask): the statistics are comparable when nothing was dropped."""
    from oracle.philox import device_actions
    rep = rep or Report()
    n, x, J = ora.n, ora.x, spec.n_joints
    ids = np.uint64(env.cfg.env_id_base) + np.arange(n, dtype=np.uint64)
    oar = bool(env.cfg.obs_after_reset) and write_obs
    thr = THRESH_TOL * (reach_of(spec) / 55.6)
    tol = point_tol_of(spec)
    episode = np.ones(n, dtype=np.int64) if episode is None else episode
    keep = np.ones(n, dtype=bool)
    stats = _new_stats()
    s0 = env.step_index
    for c in range(chunks):
        out = env.rollout_random(k, write_obs=write_obs)
        obs = out[0].cpu().numpy() if write_obs else None
        rew, done = out[1].cpu().numpy(), out[2].cpu().numpy()
        near = np.zeros(n, dtype=bool)
        refreshed = np.zeros(n, dtype=bool)
        last_pts = np.zeros((n, x, 3))
        for s in range(k):
            act = device_actions(seed, ids, s0 + c * k + s, J).astype(np.float64)
            alive_before, points_before = ora.alive.copy(), ora.points.copy()
            r = ora.step(act)
            ep_len, total = ora.ep_len, ora.total_reward
            trunc = (ep_len >= horizon) & ~r.done if horizon > 0 else np.zeros(n, dtype=bool)
            ended = r.done | trunc
            cm = np.where(alive_before, np.abs(r.catch_margin), np.inf).min(axis=1)
            near |= (r.ground_margin < thr) | (cm < thr)
            stats["env_steps"] += n
            stats["ground_steps"] += int(r.neg.sum())
            if ended.any():
                _fold_ended(stats, x, r, ended, total, ep_len)
                pts = fresh(episode, ended)
                ora.reset(mask=ended, points=np.float32(pts).astype(np.float64))
                episode[ended] += 1
                refreshed |= ended
                last_pts[ended] = pts[ended]
        st = {key: v.cpu().numpy() for key, v in env.get_state().items()}
        dev_alive_after = alive_bits_to_matrix(st["alive"], x)
        differs = ((st["goals"] != np.float32(ora.goals)).any(axis=1) | (dev_alive_after != ora.alive).any(axis=1) |
                   (st["total_reward"] != np.float32(ora.total_reward)) | (st["ep_len"] != ora.ep_len)) & keep
        hard = differs & ~near
        if hard.any():
            rep.hard_mismatch += int(hard.sum())
            i = int(np.nonzero(hard)[0][0])
            rep.notes.append(f"call {c}: env {i} state differs with no margin near a threshold")
        rep.near_threshold += int((differs & near).sum())
        keep &= ~differs
        # the last step of the call, on the envs both sides still agree on
        dev_alive = np.where(ended[:, None], r.alive, dev_alive_after)
        rk = _rows(r, keep)
        compare_step(rep, spec, None, rk, points_before[keep], alive_before[keep], None if obs is None else obs[keep],
                     rew[keep], done[keep], dev_alive[keep], None, obs_rows=(~ended[keep] if oar else None))
        rep.env_steps += (k - 1) * int(keep.sum())
        if not np.array_equal((done[keep] & 2).astype(bool), trunc[keep]):
            rep.hard_mismatch += 1
            rep.notes.append(f"call {c}: truncation flags differ")
        if oar and (ended & keep).any():
            e = ended & keep
            anchor, want = _zero_pose_obs(spec, ora.points[e])
            compare_obs(rep, spec, anchor, ora.points[e], np.ones((int(e.sum()), x), dtype=bool), obs[e], want)
        sel = refreshed & keep
        if sel.any():
            _check_fresh_points(rep, env.get_points(zero_dead=False).cpu().numpy()[sel], last_pts[sel], False, tol)
    stats["live_reward_sum"] = int(ora.total_reward.sum())
    return rep, stats, ~keep


def half_ball_points(rs, shape, radius=51.3):
    """i.i.d. uniform points in the upper half ball (the law of manytor.py:228-239), vectorised."""
    v = rs.normal(size=tuple(shape) + (3,))
    v /= np.linalg.norm(v, axis=-1, keepdims=True)
    v[..., 2] = np.abs(v[..., 2])
    return v * (radius * rs.uniform(0, 1, size=tuple(shape) + (1,)) ** (1 / 3))
