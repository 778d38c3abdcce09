"""CUDA path vs the CPU oracle and the reference's golden traces (-m gpu).

Every call goes through the C ABI (manytor_b200._lib -> libmanytor_b200.so)."""
import numpy as np
import pytest

from oracle import OracleEnvs, REFERENCE_ARM, UR5_ARM, sample_points_reference_stream
from oracle.philox import device_actions

from parity import Report, alive_bits_to_matrix, compare_step, half_ball_points, lockstep, lockstep_auto_reset

pytestmark = pytest.mark.gpu

GOLDEN = ["single_x10_seed0", "multi_3x2_x7_seed1", "batch32_x10_seed2", "batch16_x2_seed3", "batch8_x10_seed4", "multi_default_1x2_x5_seed5"]


@pytest.fixture(scope="module")
def mt():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import manytor_b200
    manytor_b200.load_library()
    return manytor_b200


def ref_points(n, x, seed):
    st = np.random.get_state()
    np.random.seed(seed)
    pts = np.stack([sample_points_reference_stream(x) for _ in range(n)])
    np.random.set_state(st)
    return pts


# --------------------------------------------------------------------------
# golden traces of the unmodified reference
# --------------------------------------------------------------------------
@pytest.mark.parametrize("name", GOLDEN)
def test_golden_trace(mt, golden, name):
    g = golden(name)
    x = int(g["x"])
    T, n = g["reward"].shape
    env = mt.BatchedEnvs(n, x, device=0)
    ora = OracleEnvs(n, x)
    rep = Report()
    for t in range(T):
        m = ~np.isnan(g["fresh"][t, :, 0, 0])
        if m.any():
            fresh = np.nan_to_num(g["fresh"][t])
            ora.reset(mask=m, points=fresh)
            env.reset(mask=m)
            env.set_points(fresh, mask=m)
            if t == 0:
                o0 = env.observe().cpu().numpy()
                np.testing.assert_allclose(o0[:, 0::3], g["obs0"][:, 0::3], atol=2e-3)
        alive_before, points_before = ora.alive.copy(), ora.points.copy()
        obs, rew, done, jn = (o.cpu().numpy() for o in env.step(g["actions"][t].astype(np.float32), joints=True))
        r = ora.step(g["actions"][t])
        # the oracle equals the reference on this trace (tests/test_oracle_golden.py)
        assert np.array_equal(r.reward, g["reward"][t]) and np.array_equal(r.done, g["done"][t])
        dev_alive = alive_bits_to_matrix(env.get_state()["alive"].cpu().numpy(), x)
        bad = compare_step(rep, REFERENCE_ARM, ora, r, points_before, alive_before, obs, rew, done, dev_alive, jn)
        np.testing.assert_allclose(jn, g["joints"][t], atol=5.6e-4)
        if bad.any():
            env.set_state(goals=ora.goals, alive=ora.alive, total_reward=ora.total_reward, mask=bad)
    print(name, rep.summary())
    assert rep.ok(), rep.notes[:5]
    assert rep.near_threshold <= max(2, rep.env_steps // 500)


# --------------------------------------------------------------------------
# BASELINE.json config 2: 4096 lock-step envs, x = 10, fp32 parity vs numpy
# --------------------------------------------------------------------------
@pytest.mark.parametrize("steps", [1000])
def test_config2_4096_envs(mt, steps):
    n, x = 4096, 10
    env = mt.BatchedEnvs(n, x, device=0)
    ora = OracleEnvs(n, x)
    pts = ref_points(n, x, seed=11)                      # objectives from the reference's RNG, uploaded
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rng = np.random.RandomState(12)
    refresh = np.random.RandomState(13)

    def fresh(t, done):
        # refresh stream for envs that collected everything (reference distribution, vectorised)
        out = np.zeros((n, x, 3))
        for i in np.nonzero(done)[0]:
            k = 0
            while k < x:
                c = refresh.uniform(-51.3, 51.3, size=3)
                if c[2] >= 0 and np.sqrt((c ** 2).sum()) <= 51.3:
                    out[i, k] = c
                    k += 1
        return out

    rep = lockstep(env, ora, REFERENCE_ARM, lambda t: rng.randint(-180, 180, size=(n, 4)), steps, on_done=fresh)
    print("config2", rep.summary())
    assert rep.ok(), rep.notes[:5]
    assert rep.max_joint_err < 5.56e-4
    assert rep.near_threshold < rep.env_steps * 2e-4


def test_generic_chain_on_reference_arm(mt):
    """The pluggable DH-chain kernel (fk_mode=1) must agree with the oracle on the reference arm too."""
    n, x = 512, 10
    env = mt.BatchedEnvs(n, x, device=0, fk_mode=1)
    ora = OracleEnvs(n, x)
    pts = ref_points(n, x, seed=3)
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rng = np.random.RandomState(4)
    rep = lockstep(env, ora, REFERENCE_ARM, lambda t: rng.uniform(-180, 180, size=(n, 4)), 60)
    print("generic-on-ref", rep.summary())
    assert rep.ok(), rep.notes[:5]


@pytest.mark.parametrize("fk_mode", [0, 1])
def test_config5_ur5_six_dof(mt, fk_mode):
    """BASELINE.json config 5: 6-DOF UR5-style chain, x = 20.  fk_mode 0 picks the compile-time
    preset table (constant-folded chain), fk_mode 1 forces the run-time DH table path."""
    n, x = 1024, 20
    env = mt.BatchedEnvs(n, x, arm=mt.UR5_ARM, device=0, fk_mode=fk_mode)
    ora = OracleEnvs(n, x, spec=UR5_ARM)
    rng = np.random.RandomState(21)
    env.reset()
    pts = env.get_points(zero_dead=False).cpu().numpy().astype(np.float64)   # on-device sampler, downloaded
    assert (np.linalg.norm(pts, axis=-1) <= UR5_ARM.radius * (1 + 1e-6)).all() and (pts[..., 2] >= 0).all()
    ora.reset(points=pts)
    rep = lockstep(env, ora, UR5_ARM, lambda t: rng.randint(-180, 180, size=(n, 6)), 80)
    print("ur5", rep.summary())
    assert rep.ok(), rep.notes[:5]


@pytest.mark.parametrize("n,x", [(1, 10), (33, 1), (95, 7), (64, 32), (100, 5), (31, 20), (257, 4)])
def test_ragged_sizes(mt, n, x):
    """Tail tiles (N not a multiple of 32), single env, X = 1 / odd / 32 (max)."""
    env = mt.BatchedEnvs(n, x, device=0)
    ora = OracleEnvs(n, x)
    pts = ref_points(n, x, seed=n + x)
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rng = np.random.RandomState(n)
    rep = lockstep(env, ora, REFERENCE_ARM, lambda t: rng.randint(-180, 180, size=(n, 4)), 25)
    assert rep.ok(), rep.notes[:5]


def test_float_actions_and_wide_range(mt):
    """Non-integer targets and targets far outside [-180, 180) (exact half-turn reduction)."""
    n, x = 256, 10
    env = mt.BatchedEnvs(n, x, device=0)
    ora = OracleEnvs(n, x)
    pts = ref_points(n, x, seed=8)
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rng = np.random.RandomState(9)

    def acts(t):
        a = rng.uniform(-720, 720, size=(n, 4))
        return np.float32(a).astype(np.float64)          # the device sees fp32 inputs; give the oracle the same
    rep = lockstep(env, ora, REFERENCE_ARM, acts, 40)
    assert rep.ok(), rep.notes[:5]


def test_terminate_on_ground_option(mt):
    n, x = 128, 10
    env = mt.BatchedEnvs(n, x, device=0, terminate_on_ground=True)
    ora = OracleEnvs(n, x, terminate_on_ground=True)
    pts = ref_points(n, x, seed=5)
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rng = np.random.RandomState(6)
    rep = lockstep(env, ora, REFERENCE_ARM, lambda t: rng.randint(-180, 180, size=(n, 4)), 10)
    assert rep.ok(), rep.notes[:5]


# --------------------------------------------------------------------------
# on-device auto-reset with an uploaded objective stream (no host round trip)
# --------------------------------------------------------------------------
def test_auto_reset_with_objective_stream(mt):
    n, x, sets, steps, horizon = 512, 2, 6, 400, 60
    rs = np.random.RandomState(31)
    stream = np.float32(half_ball_points(rs, (sets, n, x))).astype(np.float64)
    env = mt.BatchedEnvs(n, x, device=0, auto_reset=True, horizon=horizon)
    env.set_objective_stream(stream)
    env.reset()                                           # takes set 0
    ora = OracleEnvs(n, x)
    ora.reset(points=stream[0])
    rng = np.random.RandomState(32)
    rep, stats, slack, forked = lockstep_auto_reset(env, ora, REFERENCE_ARM, stream,
                                                    lambda t: rng.randint(-180, 180, size=(n, 4)), steps, horizon)
    s = env.stats()
    print("auto-reset", rep.summary(), s)
    assert rep.ok(), rep.notes[:5]
    if not forked:
        for k, v in stats.items():
            assert abs(s[k] - v) <= (slack if k == "reward_sum" else 0), (k, s[k], v)
        assert s["live_reward_sum"] == int(ora.total_reward.sum())
        assert stats["episodes"] > n      # every env ended at least once (horizon 60 over 400 steps)


# --------------------------------------------------------------------------
# on-device RNG streams
# --------------------------------------------------------------------------
def test_sample_actions_match_philox_oracle(mt):
    """Joints 0 .. 3 come from one Philox block, joints 4 .. 7 from a second one (draw_actions, mt_step.cuh)."""
    from arms import arm_pair
    n = 1000
    for J, arm in ((4, mt.REFERENCE_ARM), (6, mt.UR5_ARM), *((J, arm_pair(J)[1]) for J in (2, 3, 5, 7, 8))):
        env = mt.BatchedEnvs(n, 3, arm=arm, device=0, seed=0x1234567890ABCDEF, env_id_base=(1 << 33) + 5)
        env.reset()
        a0 = env.sample_actions().cpu().numpy()
        exp0 = device_actions(0x1234567890ABCDEF, (1 << 33) + 5 + np.arange(n), 0, J)
        np.testing.assert_array_equal(a0.astype(np.int64), exp0)
        assert a0.min() >= -180 and a0.max() <= 179
        env.step(a0)                                      # advances the step index
        a1 = env.sample_actions().cpu().numpy()
        np.testing.assert_array_equal(a1.astype(np.int64), device_actions(0x1234567890ABCDEF, (1 << 33) + 5 + np.arange(n), 1, J))


def test_rollout_random_equals_step_of_sampled_actions(mt):
    import torch
    n, x, k = 4096 + 17, 10, 12
    a = mt.BatchedEnvs(n, x, device=0, seed=7, auto_reset=True, horizon=5)
    b = mt.BatchedEnvs(n, x, device=0, seed=7, auto_reset=True, horizon=5)
    a.reset(); b.reset()
    for _ in range(k):
        oa, ra, da = a.rollout_random(1)
        ob, rb, db = b.step(b.sample_actions())
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    sa, sb = a.get_state(), b.get_state()
    for key in sa:
        assert torch.equal(sa[key], sb[key]), key
    assert torch.equal(a.get_points(False), b.get_points(False))
    assert a.stats() == b.stats()
    # without observation write the state evolves identically
    c = mt.BatchedEnvs(n, x, device=0, seed=7, auto_reset=True, horizon=5)
    c.reset()
    c.rollout_random(k, write_obs=False)
    sc = c.get_state()
    for key in sa:
        assert torch.equal(sa[key], sc[key]), key


@pytest.mark.parametrize("n", [150_001, 40_000])
def test_back_to_back_launches_equal_synchronised_steps(mt, n):
    """Consecutive step launches hand their work items over block by block (no grid-wide wait between
    steps, mt_step.cuh): a burst of launches with nothing between them must leave exactly the state,
    outputs and statistics of the same steps run one at a time -- eagerly, as a replayed CUDA graph, and
    with the hand-over replaced by stream order.  150 001 envs = full 28-warp blocks on every SM; 40 000 =
    several smaller blocks per SM."""
    import torch
    x, k = 10, 24
    g = torch.Generator(device="cuda").manual_seed(n)
    acts = [torch.randint(-180, 180, (n, 4), device="cuda", generator=g).float() for _ in range(k)]

    def fresh():
        env = mt.BatchedEnvs(n, x, device=0, seed=21, auto_reset=True, horizon=7)
        env.reset()
        return env

    def snapshot(env, out):
        st = env.get_state()
        return ([v.clone() for v in st.values()], env.get_points(False).clone(), [o.clone() for o in out], env.stats())

    def same(p, q):
        # the statistics include env_steps: it is counted on the device, so graph replays count too
        return (all(torch.equal(u, v) for u, v in zip(p[0], q[0])) and torch.equal(p[1], q[1]) and
                all(torch.equal(u, v) for u, v in zip(p[2], q[2])) and p[3] == q[3])

    ref = fresh()
    for t in range(2 * k):
        out = ref.step(acts[t % k])
        torch.cuda.synchronize()
    want = snapshot(ref, out)

    burst = fresh()
    for t in range(2 * k):
        out = burst.step(acts[t % k])
    assert same(snapshot(burst, out), want)

    env2 = fresh()
    env2._out_buffers(True, False)                                           # output buffers exist before capture
    torch.cuda.synchronize()
    cg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(cg):
        for t in range(k):
            out = env2.step(acts[t])
    cg.replay(); cg.replay()
    torch.cuda.synchronize()
    assert same(snapshot(env2, out), want)
    out = env2.step(acts[0])                                                 # eager launches after a captured graph
    out = env2.step(acts[1])
    out_ref = ref.step(acts[0]); torch.cuda.synchronize()
    out_ref = ref.step(acts[1]); torch.cuda.synchronize()
    assert same(snapshot(env2, out), snapshot(ref, out_ref))


def test_shard_invariance(mt):
    """N envs on one handle == the same envs split over two handles (global env ids key the RNG)."""
    import torch
    n, x, k = 3000, 10, 30
    whole = mt.BatchedEnvs(n, x, device=0, seed=99, auto_reset=True, horizon=7)
    cut = 1234
    parts = [mt.BatchedEnvs(cut, x, device=0, seed=99, auto_reset=True, horizon=7, env_id_base=0),
             mt.BatchedEnvs(n - cut, x, device=0, seed=99, auto_reset=True, horizon=7, env_id_base=cut)]
    whole.reset()
    for p in parts:
        p.reset()
    for _ in range(k):
        ow, rw, dw = whole.rollout_random(1)
        outs = [p.rollout_random(1) for p in parts]
        assert torch.equal(ow, torch.cat([o[0] for o in outs]))
        assert torch.equal(rw, torch.cat([o[1] for o in outs]))
        assert torch.equal(dw, torch.cat([o[2] for o in outs]))
    sw = whole.stats()
    sp = [p.stats() for p in parts]
    for key in sw:
        assert sw[key] == sp[0][key] + sp[1][key], key


def test_objective_sampler_distribution(mt):
    """On-device refresh must follow the reference's law (manytor.py:228-239): uniform in the
    upper half ball -> radius CDF (r/R)^3, z >= 0, azimuth uniform, cos(polar) uniform."""
    from scipy import stats as sst
    n, x, R = 40000, 10, 51.3
    env = mt.BatchedEnvs(n, x, device=0, seed=5)
    env.reset()
    p = env.get_points(zero_dead=False).cpu().numpy().astype(np.float64).reshape(-1, 3)
    r = np.linalg.norm(p, axis=1)
    assert (p[:, 2] >= 0).all() and (r <= R * (1 + 1e-6)).all()
    sub = slice(0, 50000)
    assert sst.kstest((r[sub] / R) ** 3, "uniform").pvalue > 1e-3
    assert sst.kstest((np.arctan2(p[sub, 1], p[sub, 0]) + np.pi) / (2 * np.pi), "uniform").pvalue > 1e-3
    assert sst.kstest(p[sub, 2] / r[sub], "uniform").pvalue > 1e-3
    # same law as the reference's rejection sampler
    ref = np.stack([sample_points_reference_stream(1)[0] for _ in range(4000)])
    assert sst.ks_2samp(np.linalg.norm(ref, axis=1), r[:20000]).pvalue > 1e-3
    assert sst.ks_2samp(ref[:, 0], p[:20000, 0]).pvalue > 1e-3
    assert sst.ks_2samp(ref[:, 2], p[:20000, 2]).pvalue > 1e-3
    # a second reset draws new objectives; another seed draws different ones
    env.reset()
    p2 = env.get_points(zero_dead=False).cpu().numpy().reshape(-1, 3)
    assert np.abs(p2 - p).max() > 1.0


# --------------------------------------------------------------------------
# API behaviour
# --------------------------------------------------------------------------
def test_errors_are_loud(mt):
    import torch
    env = mt.BatchedEnvs(64, 10, device=0)
    with pytest.raises(mt.MantorLibraryError, match="before mt_reset"):
        env.step(np.zeros((64, 4), dtype=np.float32))       # the reference raises IndexError here
    with pytest.raises(mt.MantorLibraryError):
        mt.BatchedEnvs(64, 33, device=0)                     # n_obj > MT_MAX_OBJ
    with pytest.raises(mt.MantorLibraryError):
        mt.BatchedEnvs(0, 10, device=0)
    with pytest.raises(mt.MantorLibraryError):
        mt.BatchedEnvs(8, 10, device=0, fk_mode=2, arm=mt.UR5_ARM)
    with pytest.raises(mt.MantorLibraryError):
        mt.BatchedEnvs(8, 10, device="cpu")


def test_step_host_equals_device_step(mt):
    import torch
    n, x = 5000, 10
    a = mt.BatchedEnvs(n, x, device=0, seed=3)
    b = mt.BatchedEnvs(n, x, device=0, seed=3)
    a.reset(); b.reset()
    rng = np.random.RandomState(1)
    for _ in range(5):
        act = rng.randint(-180, 180, size=(n, 4)).astype(np.float32)
        oa, ra, da = a.step(act)
        ob, rb, db = b.step_host(act)
        np.testing.assert_array_equal(oa.cpu().numpy(), ob)
        np.testing.assert_array_equal(ra.cpu().numpy(), rb)
        np.testing.assert_array_equal(da.cpu().numpy(), db)


@pytest.mark.parametrize("x,horizon,ep_hi", [(10, 0, 65536), (16, 0, 65536), (20, 0, 65536), (20, 1000, 4096), (29, 5, 8),
                                             (32, 1000, 65536)])
def test_state_roundtrip_and_dead_points(mt, x, horizon, ep_hi):
    """set_state / get_state / get_points / observe / fetch_env, for every layout of the state word
    (ep_len above the alive mask at bit 16, bit 20, bit 29; or in its own array)."""
    n = 77
    env = mt.BatchedEnvs(n, x, device=0, seed=3, horizon=horizon)
    env.reset()
    rng = np.random.RandomState(2)
    goals = rng.uniform(-180, 180, size=(n, 4)).astype(np.float32)
    alive = rng.rand(n, x) > 0.4
    tot = rng.randint(-50, 5, size=n).astype(np.float32)
    ep = rng.randint(0, ep_hi, size=n).astype(np.int32)
    env.set_state(goals=goals, alive=alive, total_reward=tot, ep_len=ep)
    st = env.get_state()
    np.testing.assert_array_equal(st["goals"].cpu().numpy(), goals)
    np.testing.assert_array_equal(alive_bits_to_matrix(st["alive"].cpu().numpy(), x), alive)
    np.testing.assert_array_equal(st["total_reward"].cpu().numpy(), tot)
    np.testing.assert_array_equal(st["ep_len"].cpu().numpy(), ep)
    raw = env.get_points(zero_dead=False).cpu().numpy()
    z = env.get_points(zero_dead=True).cpu().numpy()
    assert np.all(z[~alive] == 0) and np.array_equal(z[alive], raw[alive])     # manytor.py:148
    obs = env.observe().cpu().numpy().reshape(n, x, 3)
    assert np.all(obs[~alive] == 0) and np.all(obs[alive][:, 0] > 0)
    f = env.fetch_env(5)
    np.testing.assert_array_equal(f["alives"], alive[5])
    np.testing.assert_array_equal(f["goals"], goals[5])
    from oracle.manytor_oracle import joints_coordinates
    np.testing.assert_allclose(f["joints_coordinates"], joints_coordinates(goals[5].astype(np.float64)), atol=5.6e-4)
    # partial updates leave the other half of the state word alone; ep_len saturates, never wraps into the mask
    env.set_state(ep_len=np.full(n, 10 ** 6, np.int32))
    st = env.get_state()
    np.testing.assert_array_equal(alive_bits_to_matrix(st["alive"].cpu().numpy(), x), alive)
    assert np.all(st["ep_len"].cpu().numpy() == ep_hi - 1)
    env.set_state(alive=~alive)
    st = env.get_state()
    np.testing.assert_array_equal(alive_bits_to_matrix(st["alive"].cpu().numpy(), x), ~alive)
    assert np.all(st["ep_len"].cpu().numpy() == ep_hi - 1)
    act = rng.randint(-180, 180, size=(n, 4)).astype(np.float32)
    env.step(act)                                                   # one step at the saturated counter
    st = env.get_state()
    assert np.all(st["ep_len"].cpu().numpy() == ep_hi - 1)
    assert np.all(alive_bits_to_matrix(st["alive"].cpu().numpy(), x) <= ~alive)


def test_state_layouts_agree(mt):
    """x = 20 with a horizon that fits the 12 spare bits of the alive word (packed layout) and with
    no horizon (episode length in its own array) must produce bit-identical steps."""
    n, x = 1000, 20
    outs = []
    for horizon in (4000, 0):
        env = mt.BatchedEnvs(n, x, device=0, seed=11, horizon=horizon, auto_reset=True)
        env.reset()
        acc = []
        for t in range(120):
            obs, rew, done = env.rollout_random(1)
            acc.append((obs.cpu().numpy().copy(), rew.cpu().numpy().copy(), done.cpu().numpy().copy()))
        st = env.get_state()
        outs.append((acc, {k: v.cpu().numpy() for k, v in st.items()}, env.stats()))
    for (o1, r1, d1), (o2, r2, d2) in zip(outs[0][0], outs[1][0]):
        assert np.array_equal(o1, o2) and np.array_equal(r1, r2) and np.array_equal(d1, d2)
    for k in outs[0][1]:
        np.testing.assert_array_equal(outs[0][1][k], outs[1][1][k])
    assert outs[0][2] == outs[1][2]


# --------------------------------------------------------------------------
# more edge cases of the configuration space
# --------------------------------------------------------------------------
@pytest.mark.parametrize("substeps,fk_mode", [(2, 0), (8, 0), (24, 0), (25, 1), (8, 1), (9, 1), (2, 1)])
def test_other_substep_counts(mt, substeps, fk_mode):
    """`step = 25` is a literal in the reference (manytor.py:178); the kernels take it as a parameter
    (even and odd numbers of interior sub-poses take different pairings in the generic chain)."""
    import dataclasses
    n, x = 300, 10
    spec = dataclasses.replace(REFERENCE_ARM, substeps=substeps)
    env = mt.BatchedEnvs(n, x, device=0, substeps=substeps, fk_mode=fk_mode)
    ora = OracleEnvs(n, x, spec=spec)
    pts = ref_points(n, x, seed=substeps)
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rng = np.random.RandomState(substeps + 100 * fk_mode)
    rep = lockstep(env, ora, spec, lambda t: rng.randint(-180, 180, size=(n, 4)), 30)
    assert rep.ok(), rep.notes[:5]


def test_non_standard_frame_selectors(mt):
    """Run-time frame selectors of the generic chain: observe from frame 2, ground-test frames 2 and 4,
    catch with frame 3 (the reference hard-codes 3 / 3,4 / 4, manytor.py:143,162,191)."""
    import dataclasses
    n, x = 256, 6
    spec = dataclasses.replace(REFERENCE_ARM, obs_frame=2, ground_frames=(2, 4), catch_frame=3)
    arm = mt.ArmSpec(dh=mt.REFERENCE_ARM.dh, obs_frame=2, ground_frames=(2, 4), catch_frame=3)
    env = mt.BatchedEnvs(n, x, arm=arm, device=0)
    ora = OracleEnvs(n, x, spec=spec)
    pts = ref_points(n, x, seed=77)
    ora.reset(points=pts)
    env.reset()
    env.set_points(pts)
    rng = np.random.RandomState(78)
    rep = lockstep(env, ora, spec, lambda t: rng.randint(-180, 180, size=(n, 4)), 30)
    assert rep.ok(), rep.notes[:5]


@pytest.mark.parametrize("n,x,tog", [(77, 32, False), (45, 10, True), (130, 3, False), (70, 20, False), (33, 29, False),
                                     (50, 31, False)])
def test_auto_reset_tail_tiles_and_ground_termination(mt, n, x, tog):
    """In-kernel reset on ragged shards, the maximum objective count, and README-style termination
    on ground contact: every reset must restore the reference's reset() state (manytor.py:219-241).
    The cases cover both state layouts: episode length inside the alive word (x <= 16; x = 20 and
    x = 29, whose spare bits hold the horizon) and in its own array (x = 31, 32)."""
    horizon = 6
    env = mt.BatchedEnvs(n, x, device=0, auto_reset=True, horizon=horizon, terminate_on_ground=tog, seed=n)
    env.reset()
    ora = OracleEnvs(n, x, terminate_on_ground=tog)
    ora.reset(points=env.get_points(zero_dead=False).cpu().numpy().astype(np.float64))
    rng = np.random.RandomState(x)
    episodes = 0
    for t in range(40):
        act = rng.randint(-180, 180, size=(n, 4)).astype(np.float64)
        obs, rew, done = (o.cpu().numpy() for o in env.step(act.astype(np.float32)))
        r = ora.step(act)
        near = (r.ground_margin < 1e-3) | (np.where(ora.alive | r.alive, np.abs(r.catch_margin), np.inf).min(axis=1) < 1e-3)
        trunc = (ora.ep_len >= horizon) & ~r.done
        ok = (rew.astype(np.int64) == r.reward) & ((done & 1).astype(bool) == r.done) & ((done & 2).astype(bool) == trunc)
        assert (ok | near).all()
        ended = (done != 0)
        st = env.get_state()
        if ended.any():
            episodes += int(ended.sum())
            assert np.all(st["goals"].cpu().numpy()[ended] == 0) and np.all(st["ep_len"].cpu().numpy()[ended] == 0)
            assert np.all(alive_bits_to_matrix(st["alive"].cpu().numpy(), x)[ended])
            pts = env.get_points(zero_dead=False).cpu().numpy().astype(np.float64)
            assert (np.linalg.norm(pts[ended], axis=-1) <= 51.3 * (1 + 1e-6)).all() and (pts[ended][..., 2] >= 0).all()
        # follow the device (its sampler drew the fresh objectives; flips near a threshold re-sync too)
        ora.reset(mask=ended, points=env.get_points(zero_dead=False).cpu().numpy().astype(np.float64))
        keep = ~ended
        ora.goals[keep] = st["goals"].cpu().numpy()[keep]
        ora.alive[keep] = alive_bits_to_matrix(st["alive"].cpu().numpy(), x)[keep]
        ora.total_reward[keep] = st["total_reward"].cpu().numpy()[keep]
        ora.ep_len[keep] = st["ep_len"].cpu().numpy()[keep]
        from oracle.manytor_oracle import joints_coordinates
        ora.joints = joints_coordinates(ora.goals)
    assert env.stats()["episodes"] == episodes and episodes >= n * 5


# --------------------------------------------------------------------------
# pluggable FK: a user-supplied DH table, specialised at run time with NVRTC (fk_mode 3 / auto)
# --------------------------------------------------------------------------
_CUSTOM_DH = ((0.0, np.pi / 2, 0.30, 0.0), (0.50, 0.0, 0.0, 0.2), (0.40, 0.3, 0.10, 0.0),
              (0.0, -np.pi / 2, 0.20, -np.pi / 2), (0.10, 0.0, 0.05, 0.0))


@pytest.mark.parametrize("x,fk_mode", [(12, 3), (7, 3), (12, 1), (10, 0), (20, 0)])
def test_custom_arm_runtime_specialisation(mt, x, fk_mode):
    from oracle import ArmSpec as OArm
    n = 700
    oarm = OArm(dh=_CUSTOM_DH, obs_frame=4, ground_frames=(4, 5), catch_frame=5, radius=0.9, catch_tol=0.15)
    arm = mt.ArmSpec(dh=_CUSTOM_DH, obs_frame=4, ground_frames=(4, 5), catch_frame=5, radius=0.9, catch_tol=0.15)
    env = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=fk_mode, seed=x)
    ora = OracleEnvs(n, x, spec=oarm)
    env.reset()
    pts = env.get_points(zero_dead=False).cpu().numpy().astype(np.float64)
    assert (np.linalg.norm(pts, axis=-1) <= 0.9 * (1 + 1e-6)).all() and (pts[..., 2] >= 0).all()
    ora.reset(points=pts)
    rng = np.random.RandomState(x + fk_mode)
    rep = lockstep(env, ora, oarm, lambda t: rng.randint(-180, 180, size=(n, 5)), 40)
    print("custom arm", x, fk_mode, rep.summary())
    assert rep.ok(), rep.notes[:5]


def test_runtime_specialisation_matches_runtime_table_path(mt):
    """Same arm, same seed: the NVRTC-specialised kernels and the run-time-table kernels walk the same
    trajectory (rewards / done / alive identical, observations to fp32 rounding), also through auto-reset."""
    arm = mt.ArmSpec(dh=_CUSTOM_DH, obs_frame=4, ground_frames=(4, 5), catch_frame=5, radius=0.9, catch_tol=0.15)
    _specialised_equals_runtime_table(mt, arm)


@pytest.mark.parametrize("J", [2, 3, 4, 5, 6, 7, 8])
def test_runtime_specialisation_matches_runtime_table_path_at_every_joint_count(mt, J):
    """The same comparison for the table of every joint count in tests/arms.py (Preset<1000 + J> against
    step_kernel<J, 0, ...>), whose inner rows hold every alpha and offset the specialisation folds."""
    from arms import arm_pair
    _specialised_equals_runtime_table(mt, arm_pair(J)[1])


def _specialised_equals_runtime_table(mt, arm):
    import torch
    n, x = 4096 + 5, 12
    a = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=3, seed=5, auto_reset=True, horizon=9)
    b = mt.BatchedEnvs(n, x, arm=arm, device=0, fk_mode=1, seed=5, auto_reset=True, horizon=9)
    a.reset(); b.reset()
    assert torch.equal(a.get_points(False), b.get_points(False))
    same = 0
    for t in range(30):
        oa, ra, da = a.rollout_random(1)
        ob, rb, db = b.rollout_random(1)
        agree = (ra == rb) & (da == db)
        same += int(agree.sum())
        d = (oa - ob).abs()[agree].view(-1, x, 3)
        assert float(d[..., 0].max()) < 1e-4 and float(d[..., 1:].max()) < 0.5      # distances tight; bearings are ill-conditioned near the anchor
        if not bool(agree.all()):      # a threshold flip between the two roundings: put b back on a's track
            st = a.get_state()
            b.set_state(goals=st["goals"], alive=st["alive"], total_reward=st["total_reward"], ep_len=st["ep_len"])
            b.set_points(a.get_points(False))
    assert same >= 30 * n - 20
