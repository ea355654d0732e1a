"""State estimation in the ground-plant loop (wbc_estimator_set_create, wbc_rollout_estimator[_host], wbc_estimator_step[_host];
include/wbc.h, wbc_estimator_desc / wbc_estimator).

CPU half: the numpy restatement oracle/estimator.py against known answers (dead reckoning of a falling robot against the plant,
a standing robot converging, swing feet, dropped rows, the Philox draws, failure and re-prime), its leg kinematics against
oracle/dynamics.py, the kernel of csrc/wbc_estimator.cuh on the host (tests/emu/emu_estimator.cpp) against the oracle, and the
record check of wbc_estimator_set_create.
GPU half: est == NULL is wbc_rollout_motor; one more launch per step; the fused rollout equals a manual loop of existing entries
and wbc_estimator_step; wbc_estimator_step against the oracle; continuation and permutation; the closed loop against the oracle
controller, sensing, estimator and plant; standing on the estimate; a bad index; argument errors."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from oracle import estimator as oe
from oracle import sensing as osn

KIND_NAMES = ["id", "clf", "pc", "mptc", "pd"]
P_ = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
INF = np.inf
Q0 = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4)


def load(robot="mini_cheetah", order="depth_first"):
    from quadruped_drake_b200.model import load_robot
    return load_robot(robot, order)


def rand_quat(rng, n, spread=0.3):
    q = np.concatenate([np.ones((n, 1)), rng.normal(0, spread, (n, 3))], axis=1)
    return q / np.linalg.norm(q, axis=1, keepdims=True)


def standing(model, z_offset=0.0):
    """The nominal posture with every foot at z = 0 (the four feet are at one height)."""
    q = model.nominal_q() if hasattr(model, "nominal_q") else Q0.copy()
    r = [oe.leg_kinematics(model, q, np.zeros(18), k)[0] for k in range(4)]
    q[6] = -r[0][2] + z_offset
    return q


# ------------------------------------------------------------------------------------------------------------------ CPU half
def test_oracle_dead_reckoning_reproduces_the_plant():
    """A robot falling through the air, 500 steps of oracle/rollout.py:plant_step: with a perfect IMU, an exact prime and every
    r_* = +inf, the estimate is the plant's base position and velocity to 1e-9."""
    from oracle import rollout as ro
    from oracle.dynamics import Plant
    model, plant = load(), Plant("mini_cheetah")
    d = oe.desc(r_pos=INF, r_vel=INF, r_height=INF)
    rng = np.random.default_rng(1)
    q = Q0.copy()
    q[0:4] = rand_quat(rng, 1)[0]
    q[6] = 60.0
    v = np.concatenate([rng.normal(0, 1.0, 3), rng.normal(0, 1.0, 3), rng.normal(0, 2.0, 12)])
    dt, st, worst = 5e-3, oe.State(), 0.0
    contact = np.zeros(4, bool)
    for c in range(500):
        qo, vo, st, status = oe.step(d, model, dt, q, v, q, v, contact, st)
        assert status == 0
        worst = max(worst, np.abs(st.x[0:3] - q[4:7]).max(), np.abs(st.x[3:6] - v[3:6]).max())
        q, v, _ = ro.plant_step(plant, q, v, np.zeros(12), dt)
    assert q[6] > 1.0 and v[5] < -20.0                    # it fell freely throughout
    assert worst < 1e-9, worst


def test_oracle_standing_converges():
    """A static standing robot with exact sensing, primed 2 cm too high and 0.1 m/s off vertically: the flat-ground height and
    the zero-velocity rows pull the estimate onto the true state, within 1e-6 m and 1e-6 m/s after 1 s, and it stays there.
    (The horizontal position has no absolute measurement: an error there stays, which is the drift of the real filter.)"""
    model = load()
    d = oe.desc()
    q, v = standing(model), np.zeros(18)
    qo, vo = q.copy(), v.copy()
    qo[6] += 0.02
    vo[5] = 0.1
    st = oe.State()
    _, _, st, _ = oe.step(d, model, 5e-3, q, v, qo, vo, np.ones(4, bool), st)
    errs = []
    for c in range(600):
        out_q, out_v, st, status = oe.step(d, model, 5e-3, q, v, q, v, np.ones(4, bool), st)
        assert status == 0
        errs.append((np.abs(st.x[0:3] - q[4:7]).max(), np.abs(st.x[3:6]).max()))
    errs = np.array(errs)
    assert errs[0, 0] > 1e-3
    assert errs[200:, 0].max() < 1e-6 and errs[200:, 1].max() < 1e-6, errs[200:].max(axis=0)
    assert np.array_equal(out_q[4:7], st.x[0:3]) and np.array_equal(out_v[3:6], st.x[3:6])


def test_oracle_swing_foot_is_ignored():
    """The same innovation on foot LF (its state 1 cm off) moves p by a factor of about 1.6 / swing_scale^2 less when LF is
    planned in swing than in stance: 1.6e-6 at swing_scale = 1e3, 1.6e-8 at 1e4 (both its measurement std and its process std
    scale by swing_scale, so the gain falls with the square)."""
    model = load()
    q, v = standing(model), np.zeros(18)
    for s in (1e3, 1e4):
        d = oe.desc(swing_scale=s)
        st = oe.State()
        for _ in range(51):
            _, _, st, _ = oe.step(d, model, 5e-3, q, v, q, v, np.ones(4, bool), st)
        moves = []
        for lf in (True, False):
            contact = np.array([lf, True, True, True])
            base = oe.step(d, model, 5e-3, q, v, q, v, contact, st)[2].x[0:3]
            off = st.copy()
            off.x[6:9] += [0.01, -0.01, 0.01]
            moves.append(np.linalg.norm(oe.step(d, model, 5e-3, q, v, q, v, contact, off)[2].x[0:3] - base))
        assert moves[0] > 1e-4 and moves[1] < 2.0 / s**2 * moves[0], (s, moves)


def test_oracle_inf_rows_are_dropped():
    """r_* = +inf: the update is the prediction alone (x and P = A P A' + Q); r_vel = +inf alone leaves the velocity rows out."""
    model, rng = load(), np.random.default_rng(2)
    q, v = standing(model), np.zeros(18)
    v[3:6] = [0.1, 0.0, -0.02]
    st = oe.State()
    _, _, st, _ = oe.step(oe.desc(), model, 5e-3, q, v, q, v, np.ones(4, bool), st)
    q2, v2 = q.copy(), v + rng.normal(0, 0.01, 18)
    d = oe.desc(r_pos=INF, r_vel=INF, r_height=INF)
    _, _, a, _ = oe.step(d, model, 5e-3, q2, v2, q2, v2, np.ones(4, bool), st)
    A = np.eye(18)
    A[0:3, 3:6] = 5e-3 * np.eye(3)
    Q = 5e-3 * np.diag([d["q_pos"] ** 2] * 3 + [d["q_vel"] ** 2] * 3 + [d["q_foot"] ** 2] * 12)
    want = A @ st.P @ A.T + Q
    assert np.allclose(a.P, 0.5 * (want + want.T), rtol=1e-15, atol=0)
    vh = st.x[3:6] + 5e-3 * (v2[3:6] - v[3:6]) / 5e-3
    assert np.allclose(a.x[3:6], vh, atol=1e-15) and np.array_equal(a.x[6:], st.x[6:])
    H, y, sd = oe.measurements(oe.desc(r_vel=INF), model, q2, v2, np.ones(4, bool))
    assert np.isinf(sd).sum() == 12 and (np.isinf(sd) == np.tile([0, 0, 0, 1, 1, 1, 0], 4).astype(bool)).all()


def test_philox_draws_18_and_19():
    """The accelerometer normals are Philox draws 18 and 19 of the loop counter, and the loop's 36 normals are draws 0-17 of the
    same counter, unchanged."""
    seed, stream, c = 0x1234_5678_9ABC_DEF0, -7, (3 << 32) + 11
    z = oe.draws(seed, stream, c, range(20))
    assert np.array_equal(z[:18].reshape(-1), osn.normals(seed, stream, c))
    ctr = np.array([[18, stream & 0xFFFFFFFF, c & 0xFFFFFFFF, c >> 32]], np.uint64)
    key = np.array([[seed & 0xFFFFFFFF, seed >> 32]], np.uint64)
    ua, ub = osn.uniforms(osn.philox4x32_10(ctr, key))
    r = np.sqrt(-2.0 * np.log(ua[0]))
    assert oe.accel_normals(seed, stream, c)[0] == r * np.cos(np.pi * (2.0 * ub[0]))
    assert np.array_equal(oe.accel_normals(seed, stream, c), np.array([z[18, 0], z[18, 1], z[19, 0]]))


def test_oracle_failure_and_reprime():
    """A zero innovation variance and a non-finite measurement fail the step: output observed, count 0, x / P unchanged,
    WBC_ST_BADESTIM; the next step primes afresh. A bad index changes nothing."""
    model = load()
    q, v = standing(model), np.zeros(18)
    d0 = oe.desc(r_pos=0.0, q_pos=0.0, q_foot=0.0, p0_pos=0.0, p0_foot=0.0)
    st = oe.State()
    _, _, st, s = oe.step(d0, model, 5e-3, q, v, q, v, np.ones(4, bool), st)
    assert s == 0 and st.count == 1
    qo, vo, st2, s = oe.step(d0, model, 5e-3, q, v, q + 0.001, v, np.ones(4, bool), st)
    assert s == oe.ST_BADESTIM and st2.count == 0 and np.array_equal(st2.x, st.x) and np.array_equal(st2.P, st.P)
    assert np.array_equal(qo, q + 0.001)
    _, _, st3, s = oe.step(d0, model, 5e-3, q, v, q, v, np.ones(4, bool), st2)
    assert s == 0 and st3.count == 1 and np.array_equal(st3.x[0:3], q[4:7])
    d = oe.desc()
    bad = q.copy()
    bad[8] = np.nan
    _, _, st4, s = oe.step(d, model, 5e-3, q, v, bad, v, np.ones(4, bool), st3)
    assert s == oe.ST_BADESTIM and st4.count == 0
    _, _, st5, s = oe.step(None, model, 5e-3, q, v, q, v, np.ones(4, bool), st3)
    assert s == oe.ST_BADESTIM and st5.count == st3.count and np.array_equal(st5.x, st3.x)


ROBOTS = [("mini_cheetah", "depth_first"), ("mini_cheetah", "breadth_first"), ("anymal_b", "depth_first"), ("anymal_b", "breadth_first")]


@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_estimator.so"))
    lib.emu_estimator_step.argtypes = [C.c_void_p, C.c_longlong, C.c_double, C.c_void_p, C.c_int] + [C.c_void_p] * 7 + \
        [C.c_uint64] + [C.c_void_p] * 8
    lib.emu_leg_kinematics.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.emu_estimator_desc_problem.argtypes = [C.c_void_p]
    lib.emu_estimator_desc_problem.restype = C.c_char_p
    return lib


@pytest.mark.parametrize("robot,order", ROBOTS)
def test_leg_kinematics_match_the_plant(emu, robot, order):
    """r_k and J_k thetadot of the oracle (and of the kernel's device function on the host) against
    oracle/dynamics.Plant.frame_position_quantities: foot position p + R r_k and joint-column velocity R J_k thetadot."""
    from oracle.dynamics import Plant
    model, plant = load(robot, order), Plant(robot, order)
    ms = model.as_struct()
    rng = np.random.default_rng(5)
    for _ in range(5):
        q = model.nominal_q()
        q[0:4] = rand_quat(rng, 1)[0]
        q[4:7] = rng.normal(0, 1, 3)
        q[7:] += rng.normal(0, 0.4, 12)
        v = rng.normal(0, 2, 18)
        vj = v.copy()
        vj[0:6] = 0.0
        R = oe.quat_matrix(q[0:4])
        for k, frame in enumerate(plant.foot_frames):
            p, J, _ = plant.frame_position_quantities(q, v, frame)
            r, jv = oe.leg_kinematics(model, q, v, k)
            assert np.abs(q[4:7] + R @ r - p).max() < 1e-12
            assert np.abs(R @ jv - J @ vj).max() < 1e-12
            re, je = np.zeros(3), np.zeros(3)
            emu.emu_leg_kinematics(C.byref(ms), P_(q), P_(v), k, P_(re), P_(je))
            assert np.abs(re - r).max() < 1e-14 and np.abs(je - jv).max() < 1e-13


def desc_array(recs):
    from quadruped_drake_b200.capi import WbcEstimatorDesc
    return (WbcEstimatorDesc * len(recs))(*[WbcEstimatorDesc(**r) for r in recs])


def random_records(rng, k):
    recs = []
    for j in range(k):
        r = oe.desc(**{f: oe.DEFAULTS[f] * rng.uniform(0.3, 3.0) for f in oe.FIELDS if f != "swing_scale"},
                    swing_scale=rng.uniform(1.0, 300.0))
        if j == 1:
            r["r_vel"] = INF
        if j == 2:
            r["r_pos"] = r["r_vel"] = r["r_height"] = INF
        recs.append(r)
    return recs


def random_world(rng, model, n):
    """n robots near standing, moving a little: true q, v; base states at two consecutive steps."""
    q = np.tile(standing(model), (n, 1))
    q[:, 0:4] = rand_quat(rng, n, 0.1)
    q[:, 4:7] += rng.normal(0, 0.05, (n, 3))
    q[:, 7:] += rng.normal(0, 0.1, (n, 12))
    v = rng.normal(0, 0.3, (n, 18))
    return q, v


def noisy(rng, q, v, s=1e-3):
    qo, vo = q + rng.normal(0, s, q.shape), v + rng.normal(0, 10 * s, v.shape)
    qo[:, 0:4] /= np.linalg.norm(qo[:, 0:4], axis=1, keepdims=True)
    return qo, vo


def close(a, b, tol=1e-10):
    """Per robot: |a - b| <= tol max(|b|) (x and P rows of one robot share one scale)."""
    a, b = a.reshape(len(a), -1), b.reshape(len(b), -1)
    scale = np.maximum(np.abs(b).max(axis=1, keepdims=True), 1e-300)
    return (np.abs(a - b) <= tol * scale).all(axis=1)


@pytest.mark.parametrize("robot,order", ROBOTS)
def test_emulated_estimator_matches_oracle(emu, robot, order):
    """6 steps of 24 robots on 4 distinct records (rows dropped by +inf on two), accelerometer noise, swing feet, a bad index
    and robots primed at different steps: x and P within 1e-10 relative per step, counters, status and the primed output exact."""
    model = load(robot, order)
    ms = model.as_struct()
    rng = np.random.default_rng(11)
    n, k, dt, seed = 24, 4, 5e-3, 99
    recs = random_records(rng, k)
    arr = desc_array(recs)
    index = rng.integers(0, k, n).astype(np.int32)
    index[5] = k
    sig = np.where(rng.random(n) < 0.5, 0.0, rng.uniform(0.01, 0.5, n))
    stream = rng.integers(-2**31, 2**31, n).astype(np.int32)
    tick = rng.integers(0, 1 << 40, n).astype(np.int64)
    sts = [oe.State() for _ in range(n)]
    q, v = random_world(rng, model, n)
    for c in range(6):
        qo, vo = noisy(rng, q, v)
        contact = rng.random((n, 4)) < 0.7
        if c == 2:
            for i in range(0, n, 5):
                sts[i].count = 0                             # re-primed mid-run
        x = np.array([s.x for s in sts]); Pm = np.array([s.P for s in sts]); vp = np.array([s.v_prev for s in sts])
        cnt = np.array([s.count for s in sts], np.int64); stats = np.array([s.stats for s in sts])
        status = np.zeros(n, np.int32)
        eq, ev = qo.copy(), vo.copy()
        ct = contact.astype(np.uint8)
        emu.emu_estimator_step(C.byref(ms), n, dt, arr, k, P_(index), P_(sig), P_(x), P_(Pm), P_(vp), P_(cnt), P_(stats), seed,
                               P_(stream), P_(tick), P_(q), P_(v), P_(eq), P_(ev), P_(ct), P_(status))
        for i in range(n):
            d = recs[index[i]] if 0 <= index[i] < k else None
            oq, ov, sts[i], s = oe.step(d, model, dt, q[i], v[i], qo[i], vo[i], contact[i], sts[i], seed=seed, stream=stream[i],
                                        c=tick[i], sigma_acc=sig[i])
            assert s == status[i] and cnt[i] == sts[i].count, (c, i)
            assert close(x[i:i + 1], sts[i].x[None]).all() and close(Pm[i:i + 1], sts[i].P[None]).all(), (c, i)
            assert close(eq[i:i + 1], oq[None]).all() and close(ev[i:i + 1], ov[None]).all(), (c, i)
            assert np.abs(stats[i] - sts[i].stats).max() <= 1e-9 * max(1e-3, np.abs(sts[i].stats).max()), (c, i)
            if c == 0 and d is not None:
                assert np.array_equal(eq[i], qo[i]) and np.array_equal(ev[i], vo[i])
        assert status[5] == oe.ST_BADESTIM
        tick += 1
        v_new = v + rng.normal(0, 0.05, v.shape)
        q = q.copy()
        q[:, 4:7] += dt * v_new[:, 3:6]
        v = v_new
    assert all(s.count == (4 if i % 5 == 0 else 6) for i, s in enumerate(sts) if i != 5)


def test_set_creation_checks(emu):
    from quadruped_drake_b200.capi import WbcEstimatorDesc
    from quadruped_drake_b200.rollout import ESTIMATOR_DEFAULTS, estimator_desc
    assert ESTIMATOR_DEFAULTS == oe.DEFAULTS

    def why(**edit):
        d = estimator_desc(**edit)
        msg = emu.emu_estimator_desc_problem(C.byref(d))
        return None if msg is None else msg.decode()

    assert why() is None and why(r_pos=INF, r_vel=INF, r_height=INF) is None and why(swing_scale=1.0) is None
    assert why(q_pos=0.0, q_vel=0.0, q_foot=0.0, p0_pos=0.0, p0_vel=0.0, p0_foot=0.0, r_pos=0.0, r_vel=0.0, r_height=0.0) is None
    for f in oe.FIELDS:
        assert why(**{f: np.nan}) is not None, f
        assert why(**{f: -1e-300}) is not None, f
        assert (why(**{f: INF}) is None) == (f in ("r_pos", "r_vel", "r_height")), f
        assert (oe.desc_problem(oe.desc(**{f: INF})) is None) == (f in ("r_pos", "r_vel", "r_height")), f
    assert "swing_scale" in why(swing_scale=0.999)
    assert C.sizeof(WbcEstimatorDesc) == 10 * 8


# ------------------------------------------------------------------------------------------------------------------ GPU half
gpu = pytest.mark.gpu
NOISE = np.array([0.01, 0.002, 0.01, 0.05, 0.02, 0.1])
ROLL_KEYS = ("q", "v", "t", "tau", "metrics", "status_or", "err_max", "f_contact")
MON_KEYS = ("stats", "steps", "fail_step", "fail_why")
EST_KEYS = ("x", "P", "v_prev", "count", "stats")


@pytest.fixture(scope="module")
def ctl(built):
    from quadruped_drake_b200.controller import BatchedController
    c = BatchedController("mini_cheetah", device=0)
    yield c
    c.close()


def grounded(ctl, n, rng, jitter):
    q0 = np.tile(Q0, (n, 1))
    q0[:, 7:] += rng.uniform(-jitter, jitter, (n, 12))
    pz = ctl.dynamics(q0, np.zeros((n, 18)))["p_feet"][:, :, 2]
    q0[:, 6] -= pz.min(axis=1)
    return q0


def standing_sampler(ctl, bh):
    from quadruped_drake_b200 import planner as pl
    return pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh))


@pytest.fixture(scope="module")
def world(ctl):
    """Variants, pushes, terrain and parameter sets of a 256-robot trotting rollout, and estimator sets: the defaults, and 16
    distinct records."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.capi import DEFAULT_PARAMS
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import EstimatorSet, PlantSet, Terrain, TerrainSet, estimator_desc
    from quadruped_drake_b200.urdf import load_description
    n = 256
    rng = np.random.default_rng(21)
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    ps = PlantSet(ctl, [flatten(d), flatten(with_payload(d, 1.2, (0.04, -0.02, 0.05)))], [1.0, 0.6])
    ts = TerrainSet(ctl, [Terrain(), Terrain(slope=(np.tan(np.radians(5.0)), 0.0))])
    names = ["id_kp_body_p", "id_kd_body_p", "id_kp_foot", "clf_q_body_p", "pc_kp_body_p", "pc_kd_foot", "pd_kp", "pd_kd"]
    pset = ParamSet(ctl, [{m: DEFAULT_PARAMS[m] * float(rng.uniform(0.7, 1.4)) for m in names} for _ in range(4)])
    push = np.zeros((n, 8))
    push[:, 0:3] = rng.uniform(-40, 40, (n, 3)); push[:, 3:6] = rng.uniform(-0.1, 0.1, (n, 3))
    push[:, 6], push[:, 7] = 0.3, 0.4
    bh = float(grounded(ctl, 1, rng, 0.0)[0, 6])
    s = pl.TrajectorySampler(ctl, pl.make_gait_plan("mini_cheetah", "trot", goal=(1.5, 0.0), base_height=bh))
    default = EstimatorSet(ctl, [estimator_desc()])
    recs = random_records(rng, 16)
    distinct = EstimatorSet(ctl, list(desc_array(recs)))
    w = dict(q0=grounded(ctl, n, rng, 0.02), s=s, n=n, default=default, distinct=distinct, recs=recs,
             est_index=rng.integers(0, 16, n).astype(np.int32), accel=rng.uniform(0.0, 0.3, n),
             kw=dict(plant_set=ps, terrain_set=ts, param_set=pset, variant=(np.arange(n) % 2).astype(np.int32), push=push,
                     terrain=(np.arange(n) // 2 % 2).astype(np.int32), param_index=rng.integers(0, 4, n).astype(np.int32)))
    yield w
    distinct.close(); default.close(); pset.close(); ts.close(); ps.close(); s.close()


def noisy_loop(n, rng, dmax=3, seed=7):
    from quadruped_drake_b200.rollout import Loop
    return Loop(noise=NOISE * rng.uniform(0.5, 2.0, (n, 1)), delay=rng.integers(0, dmax + 1, n).astype(np.int32),
                strength=rng.uniform(0.8, 1.2, n), stream=rng.integers(-2**31, 2**31, n).astype(np.int32), seed=seed)


def to_dev(kw):
    import torch
    return {k: (torch.from_numpy(np.ascontiguousarray(x)).cuda() if isinstance(x, np.ndarray) else x) for k, x in kw.items()}


def dev_loop(loop):
    from quadruped_drake_b200.rollout import Loop
    T = lambda x: None if x is None else __import__("torch").from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    return Loop(noise=T(loop.noise), delay=T(loop.delay), strength=T(loop.strength), stream=T(loop.stream), seed=loop.seed)


def np_of(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else x


@gpu
def test_null_estimator_is_rollout_motor(ctl, world):
    """wbc_rollout_estimator_host with est == NULL: the bits and launch count of wbc_rollout_motor_host, all five kinds, with a
    loop, variants, pushes, terrain and parameter sets, with and without a motor and a monitor."""
    from quadruped_drake_b200.rollout import Monitor, Motor, rollout
    import quadruped_drake_b200.rollout as rmod
    n, steps = 64, 40
    q0, s, kw = world["q0"][:n], world["s"], {k: (x[:n] if isinstance(x, np.ndarray) else x) for k, x in world["kw"].items()}
    loop = noisy_loop(n, np.random.default_rng(5))
    real = ctl.lib.wbc_rollout_estimator_host
    for k, kind in enumerate(KIND_NAMES):
        for extra in (dict(), dict(motor=Motor()), dict(monitor=Monitor()), dict(motor=Motor(), monitor=Monitor())):
            l0 = ctl.launches
            ref = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, plant=True, loop=loop, **extra, **kw)
            l1 = ctl.launches
            from quadruped_drake_b200.capi import WbcRolloutIO, WbcRolloutOpts, WbcPlantOpts
            q, v, t = q0.copy(), np.zeros((n, 18)), np.zeros(n)
            # the same call through wbc_rollout_estimator_host with est == NULL
            r = [np.zeros((n, 12)), np.zeros((n, 4)), np.zeros(n, np.int32), np.zeros(n), np.zeros((steps, n, 4)), np.zeros((n, 12))]
            io = WbcRolloutIO(P_(q), P_(v), P_(t), None, *map(P_, r[:4]), None)
            o = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), P_(r[5]))
            vi, pu = rmod._perturb_arrays(n, kw["variant"], kw["push"])
            ti, ci = rmod._terrain_index(n, kw["terrain"]), rmod._terrain_index(n, kw["param_index"])
            arrays = rmod._loop_arrays(loop, n)
            pt = rmod._perturb(kw["plant_set"], vi, pu, P_)
            tr = rmod._terrain(kw["terrain_set"], ti, P_)
            from quadruped_drake_b200.capi import WbcCtrlParams, WbcMonitor, WbcPlantMotor
            cp = WbcCtrlParams(kw["param_set"]._p, P_(ci))
            lp = rmod._wbc_loop(loop, arrays, P_)
            ms = [np.zeros((n, 11)), np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int32), np.zeros(n, np.int32)]
            mo = C.byref(WbcMonitor(0.05, 0.3, *map(P_, ms))) if "monitor" in extra else None
            mt = C.byref(WbcPlantMotor(None, None, None, None)) if "motor" in extra else None
            l2 = ctl.launches
            ctl._check(real(ctl._h, k, s._p, n, steps, 5e-3, C.byref(io), C.byref(o), C.byref(pt), C.byref(tr), C.byref(cp), C.byref(lp),
                            mo, mt, None), "wbc_rollout_estimator_host")
            assert ctl.launches - l2 == l1 - l0, kind
            for key, x in zip(("q", "v", "t", "tau", "metrics", "status_or", "err_max"), [q, v, t] + r[:4]):
                assert np.array_equal(x, getattr(ref, key)), (kind, key, extra)
            assert np.array_equal(r[5].reshape(n, 4, 3), ref.f_contact)
            if "monitor" in extra:
                for key, x in zip(MON_KEYS, ms):
                    assert np.array_equal(x, getattr(ref.monitor, key)), (kind, key)


@gpu
@pytest.mark.parametrize("graph", [True, False])
def test_one_more_launch_per_step(ctl, world, graph):
    """With an estimator: exactly one more launch per step than the same call without, on the host and the device entries."""
    import torch
    from quadruped_drake_b200.rollout import Estimator, EstimatorState, Monitor, Motor, rollout
    n, steps = 64, 30
    q0, s = world["q0"][:n], world["s"]
    loop = noisy_loop(n, np.random.default_rng(6))
    for extra in (dict(), dict(motor=Motor(), monitor=Monitor())):
        l0 = ctl.launches
        rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, use_graph=graph, loop=loop, **extra)
        l1 = ctl.launches
        r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, use_graph=graph, loop=loop,
                    estimator=Estimator(world["default"], state=EstimatorState(n)), **extra)
        l2 = ctl.launches
        assert l2 - l1 == (l1 - l0) + steps
        assert (r.estimator.count == steps).all()
        q, v, t = (torch.from_numpy(x.copy()).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
        with torch.cuda.stream(torch.cuda.Stream()):
            l3 = ctl.launches
            rollout(ctl, s, "id", q, v, t, steps, plant=True, use_graph=graph, loop=dev_loop(loop),
                    estimator=Estimator(world["default"]), **extra)
        torch.cuda.synchronize()
        assert ctl.launches - l3 == l2 - l1
        assert np.array_equal(q.cpu().numpy(), r.q)


@gpu
@pytest.mark.parametrize("kind", ["id", "pd"])
def test_fused_rollout_equals_a_manual_loop(ctl, world, kind):
    """256 robots x 200 steps with 16 distinct records, accelerometer noise, a noisy delay-0 strength-1 loop, variants, pushes,
    terrain and parameter sets: the fused rollout has the bits of sample -> wbc_loop_observe -> wbc_estimator_step ->
    wbc_step_params -> wbc_plant_step_terrain (tick advanced by hand), and its estimator state equals the manual loop's."""
    import torch
    from quadruped_drake_b200.capi import KINDS, WbcCtrlParams, WbcIO, WbcPlantOpts, WbcPlantPerturb, WbcPlantTerrain
    from quadruped_drake_b200.rollout import Estimator, EstimatorState, Loop, _wbc_estimator, _wbc_loop, _loop_arrays, rollout
    n, steps, dt = world["n"], 200, 2e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    rng = np.random.default_rng(12)
    loop = Loop(noise=NOISE * rng.uniform(0.5, 2.0, (n, 1)), stream=rng.integers(-2**31, 2**31, n).astype(np.int32), seed=31)
    est = Estimator(world["distinct"], world["est_index"], world["accel"], EstimatorState(n))
    r = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop, estimator=est, **kw)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    q, v, t = T(q0), T(np.zeros((n, 18))), T(np.zeros(n))
    variant, push, terrain, pidx = (T(kw[k]) for k in ("variant", "push", "terrain", "param_index"))
    traj = torch.empty((n, 54), dtype=torch.float64, device="cuda"); contact = torch.empty((n, 4), dtype=torch.uint8, device="cuda")
    qo, vo = torch.empty_like(q), torch.empty_like(v)
    tau, met = torch.zeros((n, 12), dtype=torch.float64, device="cuda"), torch.zeros((n, 4), dtype=torch.float64, device="cuda")
    st, st_or = torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")
    f = torch.zeros((n, 12), dtype=torch.float64, device="cuda")
    tick = torch.zeros(n, dtype=torch.int64, device="cuda")
    hist = torch.zeros((n, 16, 12), dtype=torch.float64, device="cuda")     # (observe reads only the tick)
    dst = EstimatorState(n, like=q)
    dl = dev_loop(loop)
    arrays = _loop_arrays(dl, n, q.device)
    lp = _wbc_loop(dl, arrays, p)
    lp.hist, lp.tick = p(hist), p(tick)       # observe and the estimator read the tick; the manual loop advances it
    dest = Estimator(world["distinct"], T(world["est_index"]), T(world["accel"]), dst)
    es = _wbc_estimator(dest, dest.index, dest.accel_noise, dst, p)
    cs = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    io = WbcIO(p(qo), p(vo), p(traj), p(contact), p(tau), p(met), p(st), None, None, None, None)
    cp = WbcCtrlParams(kw["param_set"]._p, p(pidx))
    po = WbcPlantOpts(1.0, 0.2, 30, 0)
    pt, tr = WbcPlantPerturb(kw["plant_set"]._p, p(variant), p(push)), WbcPlantTerrain(kw["terrain_set"]._p, p(terrain))
    for c in range(steps):
        ctl._check(ctl.lib.wbc_sample_trajectory(ctl._h, s._p, n, None, p(t), p(traj), p(contact), None, None, None, cs), "sample")
        ctl._check(ctl.lib.wbc_loop_observe(ctl._h, n, C.byref(lp), p(q), p(v), p(qo), p(vo), cs), "observe")
        ctl._check(ctl.lib.wbc_estimator_step(ctl._h, n, dt, C.byref(es), C.byref(lp), p(q), p(v), p(qo), p(vo), p(contact), p(st_or), cs),
                   "estimate")
        ctl._check(ctl.lib.wbc_step_params(ctl._h, KINDS[kind], n, C.byref(io), C.byref(cp), cs), "step")
        ctl._check(ctl.lib.wbc_plant_step_terrain(ctl._h, n, dt, C.byref(po), C.byref(pt), C.byref(tr), p(q), p(v), p(tau), p(t),
                                                  p(st), p(st_or), p(f), cs), "plant")
        tick += 1
    torch.cuda.synchronize()
    for key, x in (("q", q), ("v", v), ("t", t), ("tau", tau), ("status_or", st_or), ("f_contact", f.reshape(n, 4, 3))):
        assert np.array_equal(getattr(r, key), x.cpu().numpy()), (kind, key)
    for key in EST_KEYS:
        assert np.array_equal(getattr(est.state, key), getattr(dst, key).cpu().numpy()), (kind, key)
    assert (r.status_or == 0).mean() > 0.5 and (est.state.count > 0).mean() > 0.5


@gpu
def test_estimator_step_matches_oracle(ctl):
    """wbc_estimator_step on 10^4 random rows of 4 distinct records, a few bad indices, accelerometer noise, swing feet and primes,
    host and device entries: x and P within 1e-10 relative, counters, status and priming exact."""
    import torch
    from quadruped_drake_b200.rollout import Estimator, EstimatorSet, EstimatorState, Loop, estimator_step
    model = ctl.model
    rng = np.random.default_rng(14)
    n, k, dt = 10000, 4, 5e-3
    recs = random_records(rng, k)
    es = EstimatorSet(ctl, list(desc_array(recs)))
    index = rng.integers(0, k, n).astype(np.int32)
    index[rng.random(n) < 0.01] = k
    sig = np.where(rng.random(n) < 0.5, 0.0, rng.uniform(0.01, 0.5, n))
    loop = Loop(stream=rng.integers(-2**31, 2**31, n).astype(np.int32), seed=1234)
    tick = rng.integers(0, 1 << 40, n).astype(np.int64)
    from quadruped_drake_b200.rollout import LoopState
    loop.state = LoopState(n)
    loop.state.tick[:] = tick
    q, v = random_world(rng, model, n)
    sts = [oe.State() for _ in range(n)]
    for i in range(n):                           # a primed filter, one step in, for most rows; count 0 for the rest
        if rng.random() < 0.85:
            qo, vo = noisy(rng, q[i:i + 1], v[i:i + 1])
            _, _, sts[i], _ = oe.step(recs[index[i] % k], model, dt, q[i], v[i], qo[0], vo[0], rng.random(4) < 0.7, sts[i])
    st = EstimatorState(n)
    for key in EST_KEYS:
        getattr(st, key)[:] = np.array([getattr(s, key) for s in sts])
    init = {key: getattr(st, key).copy() for key in EST_KEYS}
    q2, v2 = q.copy(), v + rng.normal(0, 0.05, v.shape)
    q2[:, 4:7] += dt * v2[:, 3:6]
    qo, vo = noisy(rng, q2, v2)
    contact = (rng.random((n, 4)) < 0.7).astype(np.uint8)
    hq, hv, hs = estimator_step(ctl, q2, v2, qo, vo, contact, Estimator(es, index, sig, st), loop, dt)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    dst = EstimatorState(n, like=T(q2))
    for key in EST_KEYS:
        getattr(dst, key).copy_(T(init[key]))
    dl = dev_loop(loop)
    dl.state = LoopState(n, like=T(q2))
    dl.state.tick.copy_(T(tick))
    dq, dv, ds = estimator_step(ctl, T(q2), T(v2), T(qo), T(vo), T(contact), Estimator(es, T(index), T(sig), dst), dl, dt)
    torch.cuda.synchronize()
    assert np.array_equal(dq.cpu().numpy(), hq) and np.array_equal(ds.cpu().numpy(), hs)
    for key in EST_KEYS:
        assert np.array_equal(getattr(dst, key).cpu().numpy(), getattr(st, key)), key
    for i in range(n):
        d = recs[index[i]] if index[i] < k else None
        oq, ov, o, s = oe.step(d, model, dt, q2[i], v2[i], qo[i], vo[i], contact[i].astype(bool), sts[i], seed=1234, stream=loop.stream[i],
                               c=tick[i], sigma_acc=sig[i])
        assert s == hs[i] and o.count == st.count[i], i
        assert close(st.x[i:i + 1], o.x[None]).all() and close(st.P[i:i + 1], o.P[None]).all(), i
        assert close(hq[i:i + 1], oq[None]).all() and close(hv[i:i + 1], ov[None]).all(), i
        if init["count"][i] == 0 and d is not None:
            assert np.array_equal(hq[i], qo[i]) and np.array_equal(hv[i], vo[i])
    assert (hs != 0).sum() >= (index == k).sum() > 0
    es.close()


@gpu
def test_continuation_and_permutation(ctl, world):
    """Four calls of 100 steps with an EstimatorState equal one call of 400; permuting the robots with their estimator indices,
    accelerometer noise and loop streams permutes every output."""
    from quadruped_drake_b200.rollout import Estimator, EstimatorState, Loop, LoopState, Monitor, MonitorState, rollout
    n, dt = world["n"], 2e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    loop = noisy_loop(n, np.random.default_rng(8))
    ei, ac = world["est_index"], world["accel"]
    loop.state = LoopState(n)
    one = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 400, dt, plant=True, loop=loop, monitor=Monitor(),
                  estimator=Estimator(world["distinct"], ei, ac, EstimatorState(n)), **kw)
    loop.state = LoopState(n)
    mon, est = Monitor(state=MonitorState(n)), Estimator(world["distinct"], ei, ac, EstimatorState(n))
    q, v, t = q0, np.zeros((n, 18)), np.zeros(n)
    status_or = np.zeros(n, np.int32)
    for _ in range(4):
        r = rollout(ctl, s, "id", q, v, t, 100, dt, plant=True, loop=loop, monitor=mon, estimator=est, **kw)
        q, v, t = r.q, r.v, r.t
        status_or |= r.status_or                  # each call ORs its own steps
    assert np.array_equal(status_or, one.status_or)
    for key in ("q", "v", "t", "tau", "f_contact", "why"):
        assert np.array_equal(getattr(r, key), getattr(one, key)), key
    for key in EST_KEYS:
        assert np.array_equal(getattr(est.state, key), getattr(one.estimator, key)), key
    perm = np.random.default_rng(9).permutation(n)
    pl = Loop(noise=loop.noise[perm], delay=loop.delay[perm], strength=loop.strength[perm], stream=loop.stream[perm], seed=loop.seed)
    loop.state = None
    a = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 200, dt, plant=True, loop=loop, monitor=Monitor(),
                estimator=Estimator(world["distinct"], ei, ac, EstimatorState(n)), **kw)
    pkw = {k: (x[perm] if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    b = rollout(ctl, s, "id", q0[perm], np.zeros((n, 18)), 0.0, 200, dt, plant=True, loop=pl, monitor=Monitor(),
                estimator=Estimator(world["distinct"], ei[perm], ac[perm], EstimatorState(n)), **pkw)
    for key in ROLL_KEYS + ("why",):
        assert np.array_equal(getattr(a, key)[perm], getattr(b, key)), key
    for key in EST_KEYS:
        assert np.array_equal(getattr(a.estimator, key)[perm], getattr(b.estimator, key)), key
    # library scratch (no state) primes afresh each call: the bits of a fresh EstimatorState
    c = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 200, dt, plant=True, loop=loop, monitor=Monitor(),
                estimator=Estimator(world["distinct"], ei, ac), **kw)
    assert c.estimator is None and np.array_equal(c.q, a.q) and np.array_equal(c.tau, a.tau)


@gpu
@pytest.mark.parametrize("kind", ["id", "pd"])
def test_closed_loop_matches_oracle(ctl, kind):
    """Standing robots, 24 steps with sensing noise and accelerometer noise: the oracle controller + oracle/sensing.py +
    oracle/estimator.py + oracle/rollout.py:plant_step agree with the GPU rollout to q 1e-6, v and tau 1e-5."""
    from oracle import controllers as oc, rollout as ro
    from oracle.dynamics import Plant
    from quadruped_drake_b200.rollout import Estimator, EstimatorSet, EstimatorState, Loop, estimator_desc, rollout
    n, steps, dt = 4, 24, (5e-3 if kind == "id" else 1e-3)
    rng = np.random.default_rng(41)
    q0 = grounded(ctl, n, rng, 0.01)
    s = standing_sampler(ctl, float(grounded(ctl, 1, rng, 0.0)[0, 6]))
    es = EstimatorSet(ctl, [estimator_desc()])
    noise = np.array([0.002, 0.001, 0.002, 0.01, 0.005, 0.02])
    loop = Loop(noise=noise, stream=np.arange(n, dtype=np.int32) * 3 + 1, seed=17)
    est = Estimator(es, accel_noise=np.full(n, 0.05), state=EstimatorState(n))
    r = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop, estimator=est)
    assert (r.status_or == 0).all()
    plant, model, d = Plant("mini_cheetah"), ctl.model, oe.desc()
    for i in range(n):
        ctrl = oc.IDController("mini_cheetah") if kind == "id" else oc.BasicController("mini_cheetah")
        q, v, t, st = q0[i].copy(), np.zeros(18), 0.0, oe.State()
        for c in range(steps):
            g = s.sample(np.array([t]))
            qo, vo = osn.observe_batch(q[None], v[None], noise, 17, [3 * i + 1], [c])
            qo, vo, st, status = oe.step(d, model, dt, q, v, qo[0], vo[0], g["contact"][0].astype(bool), st, seed=17, stream=3 * i + 1,
                                         c=c, sigma_acc=0.05)
            assert status == 0
            if kind == "id":
                tau = ctrl.control_law(qo, vo, oc.traj_to_dict(g["traj"][0], g["contact"][0])).tau
            else:
                tau = ctrl.control_law(qo, vo)
            q, v, _ = ro.plant_step(plant, q, v, tau, dt)
            t += dt
        assert np.abs(r.q[i] - q).max() < 1e-6, (i, np.abs(r.q[i] - q).max())
        assert np.abs(r.v[i] - v).max() < 1e-5 and np.abs(r.tau[i] - tau).max() < 1e-5
        assert np.abs(est.state.x[i] - st.x).max() < 1e-6
    es.close(); s.close()


@gpu
@pytest.mark.parametrize("kind", ["id", "clf", "pc", "pd"])
def test_standing_on_the_estimate(ctl, kind):
    """Noise-free sensing, 6 s of standing on the default filter: every robot stands (the monitor never fails). After the first
    second the velocity error stays below 1 cm/s and the position error below 2 mm. (In the first steps the jittered robots settle
    onto feet the plan already holds in stance, which costs up to about 0.3 m/s of velocity error and a horizontal drift of
    about 1.4 mm that no measurement can remove.)"""
    from quadruped_drake_b200.rollout import (Estimator, EstimatorSet, EstimatorState, Loop, LoopState, Monitor, MonitorState,
                                              estimator_desc, rollout)
    n, dt = 64, (5e-3 if kind != "pd" else 1e-3)
    first, steps = int(round(1.0 / dt)), int(round(6.0 / dt))
    rng = np.random.default_rng(43)
    q0 = grounded(ctl, n, rng, 0.01)
    s = standing_sampler(ctl, float(grounded(ctl, 1, rng, 0.0)[0, 6]))
    es = EstimatorSet(ctl, [estimator_desc()])
    est, mon, loop = Estimator(es, state=EstimatorState(n)), Monitor(state=MonitorState(n)), Loop(state=LoopState(n))
    r = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, first, dt, plant=True, loop=loop, monitor=mon, estimator=est)
    est.state.stats[:] = 0.0
    r = rollout(ctl, s, kind, r.q, r.v, r.t, steps - first, dt, plant=True, loop=loop, monitor=mon, estimator=est)
    assert (r.status_or == 0).all() and not mon.state.failed.any() and (est.state.count == steps).all()
    assert (est.state.max_vel < 1e-2).all(), est.state.max_vel.max()
    assert (est.state.max_pos < 2e-3).all(), est.state.max_pos.max()
    es.close(); s.close()


@gpu
def test_bad_index(ctl, world):
    """A bad record index: WBC_ST_BADESTIM in status_or with and without a monitor; with one the robot fails at step 1 for
    WBC_MON_STATUS. Its estimator state stays zero and its neighbours keep the bits of a run where it is good."""
    from quadruped_drake_b200.capi import MON_STATUS, ST_BADESTIM
    from quadruped_drake_b200.rollout import Estimator, EstimatorState, Monitor, MonitorState, rollout
    n, steps = 32, 50
    q0, s = world["q0"][:n], world["s"]
    loop = noisy_loop(n, np.random.default_rng(3))
    idx = np.zeros(n, np.int32)
    bad = idx.copy()
    bad[7] = 5
    good = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, loop=loop, estimator=Estimator(world["default"], idx, state=EstimatorState(n)))
    for mon in (None, Monitor(state=MonitorState(n))):
        est = Estimator(world["default"], bad, state=EstimatorState(n))
        r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, loop=loop, monitor=mon, estimator=est)
        assert r.status_or[7] & ST_BADESTIM and not (np.delete(r.status_or, 7) & ST_BADESTIM).any()
        for key in EST_KEYS:
            assert not getattr(est.state, key)[7].any(), key
            assert np.array_equal(np.delete(getattr(est.state, key), 7, 0), np.delete(getattr(good.estimator, key), 7, 0)), key
        assert np.array_equal(np.delete(r.q, 7, 0), np.delete(good.q, 7, 0))
        if mon is not None:
            assert mon.state.fail_step[7] == 1 and mon.state.fail_why[7] & MON_STATUS


@gpu
def test_argument_errors(ctl, world):
    import torch
    from quadruped_drake_b200.capi import WbcEstimator
    from quadruped_drake_b200.rollout import Estimator, EstimatorState, Loop, estimator_step, rollout
    n, s = 8, world["s"]
    q0 = world["q0"][:n]
    est = Estimator(world["default"], state=EstimatorState(n))
    with pytest.raises(ValueError):
        rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 5, plant=True, estimator=est)             # no loop
    with pytest.raises(ValueError):
        rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 5, plant=False, loop=Loop(), estimator=est)
    with pytest.raises(ValueError):
        rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 5, plant=True, loop=Loop(),
                estimator=Estimator(world["default"], state=EstimatorState(n + 1)))
    with pytest.raises(ValueError):
        estimator_step(ctl, q0, np.zeros((n, 18)), q0, np.zeros((n, 18)), np.ones((n, 4), np.uint8), Estimator(world["default"]))
    tq = torch.from_numpy(q0.copy()).cuda()
    with pytest.raises(ValueError):                                   # host state with device arrays
        rollout(ctl, s, "id", tq, torch.zeros((n, 18), dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda"),
                5, plant=True, loop=Loop(), estimator=est)
    with pytest.raises(ValueError):                                   # wrong index dtype on the device
        rollout(ctl, s, "id", tq, torch.zeros((n, 18), dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda"),
                5, plant=True, loop=Loop(), estimator=Estimator(world["default"], torch.zeros(n, dtype=torch.int64, device="cuda")))
    # the C ABI: partial state, no set, no loop
    x = np.zeros((n, 18))
    io_args = (ctl._h, 0, s._p, n, 5, 5e-3)
    for e in (WbcEstimator(world["default"]._p, None, None, P_(x), None, None, None, None), WbcEstimator(None, *([None] * 7))):
        rc = ctl.lib.wbc_estimator_step_host(ctl._h, n, 5e-3, C.byref(e), None, P_(q0), P_(x), P_(q0.copy()), P_(x.copy()),
                                             P_(np.ones((n, 4), np.uint8)), None)
        assert rc != 0
    from quadruped_drake_b200.capi import WbcPlantOpts, WbcRolloutIO, WbcRolloutOpts
    q, v, t = q0.copy(), np.zeros((n, 18)), np.zeros(n)
    io = WbcRolloutIO(P_(q), P_(v), P_(t), *([None] * 6))
    o = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    e = WbcEstimator(world["default"]._p, *([None] * 7))
    assert ctl.lib.wbc_rollout_estimator_host(*io_args, C.byref(io), C.byref(o), None, None, None, None, None, None, C.byref(e)) != 0
    assert np.array_equal(q, q0)
