"""Actuator model of the ground-plant loop (wbc_motor_set_create, wbc_rollout_motor[_host], wbc_motor_apply[_host]; include/wbc.h,
wbc_motor_desc / wbc_plant_motor).

CPU half: the numpy restatement oracle/motor.py against known answers (lag step response, envelope, NaN and signed zeros,
friction, bad index), the motor of csrc/wbc_motor.cuh on the host (tests/emu/emu_motor.cpp) against the oracle, and the record
check of wbc_motor_set_create.
GPU half: motor == NULL is wbc_rollout_monitor; the ideal motor leaves every output alone; the fused rollout equals a manual loop
of existing entries and wbc_motor_apply; wbc_motor_apply against the oracle; continuation and permutation; the closed loop
against the oracle controller, motor and plant; saturation, a torque-starved robot, over-damping and a bad index; argument
errors."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from oracle import motor as om

KIND_NAMES = ["id", "clf", "pc", "mptc", "pd"]
P = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
INF = np.inf


def model_maps(robot="mini_cheetah", order="depth_first"):
    from quadruped_drake_b200.model import load_robot
    m = load_robot(robot, order)
    return np.ascontiguousarray(m.v_index, np.int32), np.ascontiguousarray(m.act_index, np.int32), np.ascontiguousarray(m.effort)


def one_joint(u, w, dt=1e-3, steps=None, **rec):
    """The oracle on one robot whose joints all get u [steps, 12] (or one step) and velocities w [12]: the motor torque and plant
    input of every step (actuator = joint = velocity order)."""
    rec.setdefault("effort", np.full(12, 10.0))
    r = om.record(**rec)
    u = np.atleast_2d(np.asarray(u, float))
    tau_m, count = np.zeros((1, 12)), np.zeros(1, np.int64)
    v = np.zeros((1, 18))
    v[0, 6:] = w
    outs, plants = [], []
    for uk in u:
        plant, _ = om.apply([r], None, tau_m, count, dt, np.arange(6, 18), np.arange(12), v, uk[None])
        outs.append(tau_m[0].copy())
        plants.append(plant[0])
    return np.array(outs), np.array(plants)


# ------------------------------------------------------------------------------------------------------------------ CPU half
def test_oracle_lag_step_response():
    """u = 0 at step 0 (it primes the filter), then U: s_k = U (1 - (1 - alpha)^k), alpha = -expm1(-dt / lag)."""
    dt, lag = 1e-3, np.array([1e-3, 2e-3, 5e-3, 1e-2, 2e-2, 5e-2, 0.1, 0.3, 1.0, 3e-3, 7e-3, 4e-2])
    U = np.linspace(-30.0, 30.0, 12) + 0.1
    k = np.arange(60)
    u = np.where(k[:, None] == 0, 0.0, U)
    out, plant = one_joint(u, np.zeros(12), dt=dt, effort=np.full(12, INF), lag=lag)
    alpha = -np.expm1(-dt / lag)
    want = U * -np.expm1(k[:, None] * np.log1p(-alpha))
    assert (out[0] == 0.0).all()
    assert (np.abs(out[1:] - want[1:]) <= 1e-15 * np.abs(want[1:])).all(), np.abs(out[1:] / want[1:] - 1).max()
    assert np.array_equal(out, plant)
    # lag 0 and the first command pass straight through
    out0, _ = one_joint([[3.0] * 12, [-7.0] * 12], np.zeros(12), effort=np.full(12, INF))
    assert (out0 == [[3.0] * 12, [-7.0] * 12]).all()
    out1, _ = one_joint([[3.0] * 12], np.zeros(12), effort=np.full(12, INF), lag=0.5)
    assert (out1 == 3.0).all()


def test_oracle_envelope():
    """peak 10, knee 4, free 12: |w| = 0, knee, midway, free and beyond, motoring and braking; +inf knee and free."""
    peak, knee, free = 10.0, 4.0, 12.0
    for sign in (1.0, -1.0):
        w = sign * np.array([0.0, 4.0, 8.0, 12.0, 20.0, 4.0 + 1e-9, 11.0, 0.0, 8.0, 12.0, 20.0, 6.0])
        u = np.array([50.0, 50.0, 50.0, 50.0, 50.0, 50.0, 50.0, -50.0, -50.0, -50.0, -50.0, 3.0]) * sign   # last: under the limit
        out, _ = one_joint(u, w, effort=np.full(12, peak), speed_knee=knee, speed_free=free)
        want = sign * np.array([10.0, 10.0, 10.0 * 4.0 / 8.0, 0.0, 0.0, 10.0 * (12.0 - (4.0 + 1e-9)) / 8.0, 10.0 * 1.0 / 8.0,
                                -10.0, -10.0, -10.0, -10.0, 3.0])
        assert np.array_equal(out[0], want), (sign, out[0], want)
    w = np.array([0.0, 1.0, 1e3, 1e300, INF, -INF, 5.0, -5.0, 5.0, 1e300, INF, 0.0])
    out, _ = one_joint(np.full(12, 50.0), w, effort=np.full(12, peak), speed_knee=INF, speed_free=INF)
    assert (out[0] == peak).all()
    out, _ = one_joint(np.full(12, 50.0), w, effort=np.full(12, peak), speed_knee=2.0, speed_free=INF)
    assert np.array_equal(out[0], np.where(w == INF, 0.0, peak))        # free = inf: flat beyond the knee, 0 only at |w| = inf
    out, _ = one_joint(np.full(12, 50.0), w, effort=np.full(12, peak), speed_knee=0.0, speed_free=0.0)
    assert np.array_equal(out[0], np.where(w > 0, 0.0, peak))            # knee = free = 0: no motoring torque at all


def test_oracle_nan_and_the_ideal_motor():
    """A NaN command stays NaN through the clamp; the ideal record returns u bit for bit, signed zeros and infinities included."""
    u = np.array([np.nan, -np.nan, 1e300, -1e300, 0.0, -0.0, 5e-324, -5e-324, INF, -INF, 3.5, -2.25])
    out, plant = one_joint(u, np.linspace(-30, 30, 12), effort=np.full(12, 10.0), speed_knee=1.0, speed_free=2.0)
    assert np.isnan(out[0, :2]).all() and np.isnan(plant[0, :2]).all()
    out, plant = one_joint(u, np.linspace(-30, 30, 12), effort=np.full(12, 10.0), peak_scale=INF)
    assert np.array_equal(out.view(np.int64), u[None].view(np.int64)) and np.array_equal(plant.view(np.int64), u[None].view(np.int64))
    out, plant = one_joint([u, u[::-1]], np.full(12, np.nan), effort=np.full(12, 10.0), peak_scale=INF)
    assert np.array_equal(plant.view(np.int64), np.array([u, u[::-1]]).view(np.int64))      # a NaN w passes no zero coefficient


def test_oracle_friction():
    """f = -damping w - coulomb clamp(w / coulomb_speed, -1, 1), on top of the motor torque."""
    w = np.array([-3.0, -0.05, 0.0, 0.02, 0.1, 2.0, -0.1, 0.3, -1e-3, 7.0, -7.0, 0.06])
    u = np.linspace(-4.0, 4.0, 12)
    d, c, cs = 0.05, 0.4, 0.1
    out, plant = one_joint(u, w, effort=np.full(12, INF), damping=d, coulomb=c, coulomb_speed=cs)
    assert np.array_equal(out[0], u)
    assert np.allclose(plant[0], u - d * w - c * np.clip(w / cs, -1, 1), rtol=0, atol=1e-15)
    _, pd_ = one_joint(u, w, effort=np.full(12, INF), damping=d)
    _, pc_ = one_joint(u, w, effort=np.full(12, INF), coulomb=c, coulomb_speed=cs)
    assert np.array_equal(pd_[0], u + -(d * w)) and np.array_equal(pc_[0], u + -(c * np.clip(w / cs, -1, 1)))
    _, p0 = one_joint(-np.zeros(12), w, effort=np.full(12, INF), damping=0.0, coulomb=0.0, coulomb_speed=0.0)
    assert np.array_equal(p0.view(np.int64), (-np.zeros((1, 12))).view(np.int64))          # nothing added: -0 stays -0


def test_oracle_bad_index():
    vi, ai, eff = model_maps()
    n = 5
    recs = [om.record(eff), om.record(eff, lag=0.01)]
    tau_m, count = np.full((n, 12), 0.5), np.array([0, 3, 7, 1, 2], np.int64)
    v, u = np.ones((n, 18)), np.full((n, 12), 2.0)
    plant, st = om.apply(recs, np.array([0, 2, -1, 1, 0]), tau_m, count, 1e-3, vi, ai, v, u)
    bad = np.array([False, True, True, False, False])
    assert list(st) == [0, om.ST_BADMOTOR, om.ST_BADMOTOR, 0, 0]
    assert (plant[bad] == 0).all() and (tau_m[bad] == 0.5).all() and list(count) == [1, 3, 7, 2, 3]
    assert (plant[~bad] != 0).all()


@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_motor.so"))
    lib.emu_motor_apply.argtypes = [C.c_longlong, C.c_double, C.c_void_p, C.c_int] + [C.c_void_p] * 10
    lib.emu_motor_desc_problem.argtypes = [C.c_void_p]
    lib.emu_motor_desc_problem.restype = C.c_char_p
    return lib


def desc_array(recs):
    from quadruped_drake_b200.capi import WbcMotorDesc
    arr = (WbcMotorDesc * len(recs))()
    for d, r in zip(arr, recs):
        for f in om.FIELDS:
            getattr(d, f)[:] = [float(x) for x in r[f]]
    return arr


def random_records(rng, eff, k):
    """k distinct records: lag 0-20 ms (some 0), peak 0.3-1.5 x effort (one +inf), knee / free in 0-30 rad/s (some +inf),
    damping and Coulomb friction (some 0)."""
    recs = []
    for j in range(k):
        knee = rng.uniform(0, 15, 12)
        free = knee + rng.uniform(0, 15, 12)
        knee[rng.random(12) < 0.2] = INF
        free[np.isinf(knee)] = INF
        free[rng.random(12) < 0.1] = INF
        r = om.record(eff, rng.uniform(0.3, 1.5), speed_knee=knee, speed_free=free,
                      lag=np.where(rng.random(12) < 0.3, 0.0, rng.uniform(1e-3, 2e-2, 12)),
                      damping=np.where(rng.random(12) < 0.4, 0.0, rng.uniform(0, 0.2, 12)),
                      coulomb=np.where(rng.random(12) < 0.4, 0.0, rng.uniform(0, 0.5, 12)), coulomb_speed=rng.uniform(0.01, 0.5, 12))
        if j == 0:
            r["peak"][:] = INF
        recs.append(r)
    return recs


def random_batch(rng, n, eff, k):
    """A motor step of n robots: indices (a few out of range), states mid-run, velocities near the knees, torques near the limits,
    a few NaN."""
    index = rng.integers(0, k, n).astype(np.int32)
    index[rng.random(n) < 0.03] = rng.choice([-1, k, 1 << 30])
    tau_m = rng.normal(0, 1, (n, 12)) * eff.max() * 0.5
    count = np.where(rng.random(n) < 0.2, 0, rng.integers(1, 1000, n)).astype(np.int64)
    v = rng.normal(0, 10, (n, 18))
    u = rng.normal(0, 1, (n, 12)) * eff.max()
    u[rng.random((n, 12)) < 0.01] = np.nan
    u[rng.random((n, 12)) < 0.01] = -0.0
    return index, tau_m, count, v, u


def lagged(recs, index, count, ai):
    """Where the lag filter ran: [n, 12] in actuator order (the only entries whose expm1 may differ by an ulp)."""
    k = len(recs)
    ok = (index >= 0) & (index < k)
    lag = np.stack([r["lag"] for r in recs])[np.where(ok, index, 0)]
    m = np.zeros((len(index), 12), bool)
    m[:, ai] = ok[:, None] & (count[:, None] != 0) & (lag != 0)
    return m


def compare(a, b, lag_mask, scale):
    """Exact equality (NaN = NaN) except entries under lag_mask, which agree to 1e-15 relative to `scale`: the magnitude of the
    filter's operands u and m, since an ulp of alpha = -expm1(-dt / lag) (the host's and CUDA's expm1 may differ by one) moves
    m + alpha (u - m) by alpha |u - m| ulp, and the motor torque and friction may cancel in the plant input."""
    same = (a == b) | (np.isnan(a) & np.isnan(b))
    rel = np.abs(a - b) <= 1e-15 * np.maximum(scale, 1e-300)
    assert (same | (lag_mask & rel)).all(), np.argwhere(~(same | (lag_mask & rel)))[:5]


@pytest.mark.parametrize("robot,order", [("mini_cheetah", "depth_first"), ("mini_cheetah", "breadth_first"),
                                         ("anymal_b", "depth_first"), ("anymal_b", "breadth_first")])
def test_emulated_motor_matches_oracle(emu, robot, order):
    """20 steps of 500 robots on 6 distinct records and the NULL set: states, counters and status exact; lag within 1e-15."""
    vi, ai, eff = model_maps(robot, order)
    rng = np.random.default_rng(3)
    n, k, dt = 500, 6, 2e-3
    recs = random_records(rng, eff, k)
    arr = desc_array(recs)
    for use_set in (True, False):
        index, tau_m, count, v, u = random_batch(rng, n, eff, k)
        if not use_set:
            index = None
        a_m, a_c = tau_m.copy(), count.copy()
        b_m, b_c = tau_m.copy(), count.copy()
        st = np.zeros(n, np.int32)
        rr = recs if use_set else [om.record(eff)]
        for _ in range(20):
            v = v + rng.normal(0, 0.5, v.shape)
            mask = lagged(rr, np.zeros(n, np.int32) if index is None else index, a_c, ai)
            prev = a_m.copy()
            pa, sa = om.apply(rr, index, a_m, a_c, dt, vi, ai, v, u)
            pb = np.zeros((n, 12))
            emu.emu_motor_apply(n, dt, arr if use_set else None, k, P(index), P(b_m), P(b_c), P(vi), P(ai), P(eff), P(v), P(u), P(pb), P(st))
            scale = np.maximum(np.maximum(np.abs(u), np.abs(prev)), np.abs(a_m))
            compare(a_m, b_m, mask, scale)
            compare(pa, pb, mask, scale)
            assert np.array_equal(a_c, b_c) and np.array_equal(st, sa)
            b_m[:] = a_m                                  # restart each step from the oracle's state
            u = u + rng.normal(0, 1, u.shape)
        assert (sa != 0).any() == use_set


def test_set_creation_checks(emu):
    from quadruped_drake_b200.capi import WbcMotorDesc
    eff = model_maps()[2]
    good = om.record(eff, speed_knee=5.0, speed_free=20.0, lag=0.01, damping=0.1, coulomb=0.2, coulomb_speed=0.1)

    def why(**edit):
        r = {f: x.copy() for f, x in good.items()}
        for f, (j, x) in edit.items():
            r[f][j] = x
        msg = emu.emu_motor_desc_problem(C.byref(desc_array([r])[0]))
        return None if msg is None else msg.decode()

    assert why() is None and why(peak=(3, INF)) is None and why(speed_knee=(0, INF), speed_free=(0, INF)) is None
    assert why(speed_free=(2, INF)) is None and why(coulomb=(1, 0.0), coulomb_speed=(1, 0.0)) is None
    for f in ("peak", "speed_knee", "speed_free", "lag", "damping", "coulomb", "coulomb_speed"):
        assert why(**{f: (5, np.nan)}) is not None, f
        assert why(**{f: (5, -1e-300)}) is not None, f
    for f in ("lag", "damping", "coulomb", "coulomb_speed"):
        assert "finite" in why(**{f: (11, INF)}), f
    assert "speed_knee must be <= speed_free" in why(speed_knee=(4, 21.0))
    assert "speed_knee must be <= speed_free" in why(speed_knee=(4, INF))
    assert "coulomb_speed > 0" in why(coulomb_speed=(7, 0.0))
    assert C.sizeof(WbcMotorDesc) == 7 * 12 * 8


# ------------------------------------------------------------------------------------------------------------------ GPU half
gpu = pytest.mark.gpu
Q0 = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4)
NOISE = np.array([0.01, 0.002, 0.01, 0.05, 0.02, 0.1])
ROLL_KEYS = ("q", "v", "t", "tau", "metrics", "status_or", "err_max", "f_contact")
MON_KEYS = ("stats", "steps", "fail_step", "fail_why")


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
    """Variants, pushes, terrain and parameter sets of a 256-robot trotting robustness rollout, and two motor sets: the ideal
    motor, and 8 distinct records (lag, friction, and an envelope of 0.1-0.3 x effort with knees at 1-4 rad/s, below what
    the trot commands)."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.capi import DEFAULT_PARAMS
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import MotorSet, PlantSet, Terrain, TerrainSet, motor_desc
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
    ideal = MotorSet(ctl, [motor_desc(ctl.model, INF)])
    peaks = rng.uniform(0.1, 0.3, 8)
    distinct = MotorSet(ctl, [motor_desc(ctl.model, float(p), speed_knee=rng.uniform(1, 4, 12), speed_free=rng.uniform(8, 15, 12),
                                         lag=rng.uniform(0, 4e-3, 12), damping=rng.uniform(0, 0.02, 12), coulomb=rng.uniform(0, 0.2, 12),
                                         coulomb_speed=0.1) for p in peaks])
    w = dict(q0=grounded(ctl, n, rng, 0.02), s=s, n=n, ideal=ideal, distinct=distinct, peaks=peaks, motor_index=rng.integers(0, 8, n).astype(np.int32),
             kw=dict(plant_set=ps, terrain_set=ts, param_set=pset, variant=(np.arange(n) % 2).astype(np.int32), push=push,
                     terrain=(np.arange(n) // 2 % 2).astype(np.int32), param_index=rng.integers(0, 4, n).astype(np.int32)))
    yield w
    distinct.close(); ideal.close(); pset.close(); ts.close(); ps.close(); s.close()


def noisy_loop(n, rng, dmax=3):
    from quadruped_drake_b200.rollout import Loop
    return Loop(noise=NOISE * rng.uniform(0.5, 2.0, (n, 1)), delay=rng.integers(0, dmax + 1, n).astype(np.int32),
                strength=rng.uniform(0.8, 1.2, n), stream=rng.integers(-2**31, 2**31, n).astype(np.int32), seed=7)


def to_dev(kw):
    import torch
    return {k: (torch.from_numpy(np.ascontiguousarray(x)).cuda() if isinstance(x, np.ndarray) else x) for k, x in kw.items()}


def dev_loop(loop):
    from quadruped_drake_b200.rollout import Loop
    T = lambda x: None if x is None else __import__("torch").from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    return Loop(noise=T(loop.noise), delay=T(loop.delay), strength=T(loop.strength), stream=T(loop.stream), seed=loop.seed)


def np_of(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else x


def c_structs(kw, loop, rows):
    """Host ctypes structs of the world's perturbations, terrain, parameters and loop for the rows `rows` (arrays kept alive in
    the returned list)."""
    from quadruped_drake_b200.capi import WbcCtrlParams, WbcLoop, WbcPlantPerturb, WbcPlantTerrain
    keep = [np.ascontiguousarray(kw[k][rows]) for k in ("variant", "push", "terrain", "param_index")]
    keep += [np.ascontiguousarray(x[rows]) for x in (loop.noise, loop.delay, loop.strength, loop.stream)]
    pt = WbcPlantPerturb(kw["plant_set"]._p, P(keep[0]), P(keep[1]))
    tr = WbcPlantTerrain(kw["terrain_set"]._p, P(keep[2]))
    cp = WbcCtrlParams(kw["param_set"]._p, P(keep[3]))
    lp = WbcLoop(P(keep[4]), P(keep[5]), P(keep[6]), P(keep[7]), loop.seed, None, None)
    return pt, tr, cp, lp, keep


@gpu
def test_null_motor_is_rollout_monitor(ctl, world):
    """wbc_rollout_motor_host with motor == NULL: the bits and launch count of wbc_rollout_monitor_host, all five kinds, with
    variants, pushes, terrain and parameter sets, with and without a loop and a monitor."""
    from quadruped_drake_b200.capi import WbcMonitor, WbcPlantOpts, WbcRolloutIO, WbcRolloutOpts
    n, steps = 64, 40
    q0, s, kw = world["q0"][:n], world["s"], world["kw"]
    pt, tr, cp, lp, keep = c_structs(kw, noisy_loop(world["n"], np.random.default_rng(5)), np.arange(n))
    for k, kind in enumerate(KIND_NAMES):
        for with_lm in (True, False):
            outs, counts = [], []
            for fn, extra in (("wbc_rollout_monitor_host", ()), ("wbc_rollout_motor_host", (None,))):
                q, v, t = q0.copy(), np.zeros((n, 18)), np.zeros(n)
                r = [np.zeros((n, 12)), np.zeros((n, 4)), np.zeros(n, np.int32), np.zeros(n), np.zeros((steps, n, 4)), np.zeros((n, 12))]
                ms = [np.zeros((n, 11)), np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int32), np.zeros(n, np.int32)]
                io = WbcRolloutIO(P(q), P(v), P(t), None, *map(P, r[:5]))
                o = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), P(r[5]))
                mo = C.byref(WbcMonitor(0.05, 0.3, *map(P, ms))) if with_lm else None
                l0 = ctl.launches
                ctl._check(getattr(ctl.lib, fn)(ctl._h, k, s._p, n, steps, 5e-3, C.byref(io), C.byref(o), C.byref(pt), C.byref(tr),
                                                C.byref(cp), C.byref(lp) if with_lm else None, mo, *extra), fn)
                counts.append(ctl.launches - l0)
                outs.append([q, v, t] + r + ms)
            assert counts[0] == counts[1], kind
            for a, b in zip(*outs):
                assert np.array_equal(a, b), (kind, with_lm)


@gpu
@pytest.mark.parametrize("kind", KIND_NAMES)
def test_ideal_motor_leaves_every_output_alone(ctl, world, kind):
    """An ideal-motor set: every output of wbc_rollout_monitor (rollout and monitor) keeps its bits, with variants, pushes,
    terrain, parameter sets and a loop, with one more launch per step; the device entry, with and without the graph, too."""
    import torch
    from quadruped_drake_b200.rollout import Monitor, Motor, MotorState, rollout
    n, steps, dt = world["n"], 150, 5e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    loop = noisy_loop(n, np.random.default_rng(6))
    l0 = ctl.launches
    ref = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, log_metrics=True, loop=loop, monitor=Monitor(), **kw)
    l1 = ctl.launches
    motor = Motor(world["ideal"], state=MotorState(n))
    got = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, log_metrics=True, loop=loop, monitor=Monitor(),
                  motor=motor, **kw)
    l2 = ctl.launches
    assert l2 - l1 == (l1 - l0) + steps
    for key in ROLL_KEYS + ("metrics_log", "why"):
        assert np.array_equal(getattr(got, key), getattr(ref, key)), (kind, key)
    for key in MON_KEYS:
        assert np.array_equal(getattr(got.monitor, key), getattr(ref.monitor, key)), (kind, key)
    assert (motor.state.count == steps).all()
    for graph in (True, False):
        q, v, t = (torch.from_numpy(x.copy()).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
        with torch.cuda.stream(torch.cuda.Stream()):
            r = rollout(ctl, s, kind, q, v, t, steps, dt, plant=True, use_graph=graph, loop=dev_loop(loop), monitor=Monitor(),
                        motor=Motor(world["ideal"], index=torch.zeros(n, dtype=torch.int32, device="cuda")), **to_dev(kw))
        torch.cuda.synchronize()
        for key in ROLL_KEYS + ("why",):
            assert np.array_equal(np_of(getattr(r, key)), getattr(ref, key)), (kind, graph, key)
        for key in MON_KEYS:
            assert np.array_equal(np_of(getattr(r.monitor, key)), getattr(ref.monitor, key)), (kind, graph, key)


@gpu
@pytest.mark.parametrize("kind", ["id", "pd"])
def test_fused_rollout_equals_a_manual_loop(ctl, world, kind):
    """256 robots x 200 steps at dt = 1e-3 with distinct records (lag, envelope, friction), variants, pushes, terrain and
    parameter sets: the fused rollout has the bits of sample -> wbc_step_params -> wbc_motor_apply -> wbc_plant_step_terrain, and
    its motor state equals the manual loop's."""
    import torch
    from quadruped_drake_b200.capi import KINDS, WbcCtrlParams, WbcIO, WbcPlantMotor, WbcPlantOpts, WbcPlantPerturb, WbcPlantTerrain
    from quadruped_drake_b200.rollout import Motor, MotorState, rollout
    n, steps, dt = world["n"], 200, 1e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    motor = Motor(world["distinct"], world["motor_index"], MotorState(n))
    r = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, motor=motor, **kw)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    q, v, t = T(q0), T(np.zeros((n, 18))), T(np.zeros(n))
    variant, push, terrain, pidx = (T(kw[k]) for k in ("variant", "push", "terrain", "param_index"))
    midx = T(world["motor_index"])
    traj = torch.empty((n, 54), dtype=torch.float64, device="cuda"); contact = torch.empty((n, 4), dtype=torch.uint8, device="cuda")
    tau, met = torch.zeros((n, 12), dtype=torch.float64, device="cuda"), torch.zeros((n, 4), dtype=torch.float64, device="cuda")
    st, st_or = torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")
    f, plant_tau = torch.zeros((n, 12), dtype=torch.float64, device="cuda"), torch.zeros((n, 12), dtype=torch.float64, device="cuda")
    tau_m, count = torch.zeros((n, 12), dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.int64, device="cuda")
    cs = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    io = WbcIO(p(q), p(v), p(traj), p(contact), p(tau), p(met), p(st), None, None, None, None)
    cp = WbcCtrlParams(kw["param_set"]._p, p(pidx))
    mt = WbcPlantMotor(world["distinct"]._p, p(midx), p(tau_m), p(count))
    po = WbcPlantOpts(1.0, 0.2, 30, 0)
    pt, tr = WbcPlantPerturb(kw["plant_set"]._p, p(variant), p(push)), WbcPlantTerrain(kw["terrain_set"]._p, p(terrain))
    limit = T(world["peaks"][world["motor_index"]][:, None] * np.asarray(ctl.model.effort)[np.argsort(ctl.model.act_index)])
    beyond = torch.zeros(n, dtype=torch.bool, device="cuda")
    for c in range(steps):
        ctl._check(ctl.lib.wbc_sample_trajectory(ctl._h, s._p, n, None, p(t), p(traj), p(contact), None, None, None, cs), "sample")
        ctl._check(ctl.lib.wbc_step_params(ctl._h, KINDS[kind], n, C.byref(io), C.byref(cp), cs), "step")
        beyond |= (tau.abs() > limit).any(dim=1)
        ctl._check(ctl.lib.wbc_motor_apply(ctl._h, n, dt, C.byref(mt), p(v), p(tau), p(plant_tau), p(st), cs), "motor")
        ctl._check(ctl.lib.wbc_plant_step_terrain(ctl._h, n, dt, C.byref(po), C.byref(pt), C.byref(tr), p(q), p(v), p(plant_tau), p(t),
                                                  p(st), p(st_or), p(f), cs), "plant")
    torch.cuda.synchronize()
    for key, x in (("q", q), ("v", v), ("t", t), ("tau", tau), ("status_or", st_or), ("f_contact", f.reshape(n, 4, 3))):
        assert np.array_equal(getattr(r, key), x.cpu().numpy()), (kind, key)
    assert np.array_equal(motor.state.tau_m, tau_m.cpu().numpy()) and np.array_equal(motor.state.count, count.cpu().numpy())
    assert (r.status_or == 0).mean() > 0.5
    assert beyond.float().mean().item() > 0.1                  # commands beyond the motors' peak torque: the envelope binds


@gpu
def test_motor_apply_matches_oracle(ctl):
    """wbc_motor_apply on 10^4 random rows of 6 distinct records and a few bad indices, and on the NULL set, host and device
    entries: states, counters and status exact, lag within 1e-15 relative, as the emulated kernel."""
    import torch
    from quadruped_drake_b200.rollout import Motor, MotorSet, MotorState, motor_apply
    vi, ai, eff = (np.asarray(x) for x in (ctl.model.v_index, ctl.model.act_index, ctl.model.effort))
    rng = np.random.default_rng(4)
    n, k, dt = 10000, 6, 2e-3
    recs = random_records(rng, eff, k)
    ms = MotorSet(ctl, list(desc_array(recs)))
    for use_set in (True, False):
        index, tau_m, count, v, u = random_batch(rng, n, eff, k)
        rr = recs if use_set else [om.record(eff)]
        idx = index if use_set else None
        mask = lagged(rr, index if use_set else np.zeros(n, np.int32), count, ai)
        a_m, a_c = tau_m.copy(), count.copy()
        pa, sa = om.apply(rr, idx, a_m, a_c, dt, vi, ai, v, u)
        st = MotorState(n)
        st.tau_m[:], st.count[:] = tau_m, count
        pb, sb = motor_apply(ctl, v, u, Motor(ms if use_set else None, idx, st), dt)
        scale = np.maximum(np.maximum(np.abs(u), np.abs(tau_m)), np.abs(a_m))
        compare(a_m, st.tau_m, mask, scale); compare(pa, pb, mask, scale)
        assert np.array_equal(a_c, st.count) and np.array_equal(sa, sb)
        T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
        dst = MotorState(n, like=T(v))
        dst.tau_m.copy_(T(tau_m)); dst.count.copy_(T(count))
        pc, sc = motor_apply(ctl, T(v), T(u), Motor(ms if use_set else None, None if idx is None else T(idx), dst), dt)
        torch.cuda.synchronize()
        assert np.array_equal(pc.cpu().numpy().view(np.int64), pb.view(np.int64)) and np.array_equal(sc.cpu().numpy(), sb)
        assert np.array_equal(dst.tau_m.cpu().numpy().view(np.int64), st.tau_m.view(np.int64))
        assert (sa != 0).any() == use_set and mask.any() == use_set
    ms.close()


@gpu
def test_continuation_and_permutation(ctl, world):
    """Four calls of 100 steps with a MotorState equal one call of 400 (host and device state); permuting the robots with their
    motor indices and loop streams permutes every output."""
    import torch
    from quadruped_drake_b200.rollout import Loop, LoopState, Monitor, MonitorState, Motor, MotorState, rollout
    n, dt = world["n"], 1e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    loop = noisy_loop(n, np.random.default_rng(8))
    mi = world["motor_index"]
    loop.state = LoopState(n)
    one = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 400, dt, plant=True, loop=loop, monitor=Monitor(),
                  motor=Motor(world["distinct"], mi, MotorState(n)), **kw)
    loop.state = LoopState(n)
    mon, motor = Monitor(state=MonitorState(n)), Motor(world["distinct"], mi, MotorState(n))
    q, v, t = q0, np.zeros((n, 18)), np.zeros(n)
    for _ in range(4):
        r = rollout(ctl, s, "id", q, v, t, 100, dt, plant=True, loop=loop, monitor=mon, motor=motor, **kw)
        q, v, t = r.q, r.v, r.t
    for key in ("q", "v", "t", "tau", "status_or", "f_contact", "why"):
        assert np.array_equal(getattr(r, key), getattr(one, key)), key
    for key in MON_KEYS:
        assert np.array_equal(getattr(mon.state, key), getattr(one.monitor, key)), key
    assert (motor.state.count == 400).all()
    host_m = motor.state.tau_m.copy()
    tq, tv, tt = (torch.from_numpy(x.copy()).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
    loop.state = LoopState(n, like=tq)
    dl = dev_loop(loop)
    dl.state = loop.state
    dmotor = Motor(world["distinct"], torch.from_numpy(mi).cuda(), MotorState(n, like=tq))
    dkw = to_dev(kw)
    for _ in range(4):
        rollout(ctl, s, "id", tq, tv, tt, 100, dt, plant=True, loop=dl, motor=dmotor, **dkw)
    torch.cuda.synchronize()
    assert np.array_equal(tq.cpu().numpy(), one.q) and np.array_equal(dmotor.state.tau_m.cpu().numpy(), host_m)
    perm = np.random.default_rng(9).permutation(n)
    pl = Loop(noise=loop.noise[perm], delay=loop.delay[perm], strength=loop.strength[perm], stream=loop.stream[perm], seed=loop.seed)
    loop.state = None
    a = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 200, dt, plant=True, loop=loop, monitor=Monitor(),
                motor=Motor(world["distinct"], mi), **kw)
    pkw = {k: (x[perm] if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    b = rollout(ctl, s, "id", q0[perm], np.zeros((n, 18)), 0.0, 200, dt, plant=True, loop=pl, monitor=Monitor(),
                motor=Motor(world["distinct"], mi[perm]), **pkw)
    for key in ROLL_KEYS + ("why",):
        assert np.array_equal(getattr(a, key)[perm], getattr(b, key)), key
    for key in MON_KEYS:
        assert np.array_equal(getattr(a.monitor, key)[perm], getattr(b.monitor, key)), key


@gpu
@pytest.mark.parametrize("kind", ["id", "pd"])
def test_closed_loop_matches_oracle(ctl, kind):
    """Standing robots, 24 steps, a record with lag, a torque-speed envelope and friction: the oracle controller + oracle/motor.py
    + oracle/rollout.py:plant_step agree with the GPU rollout to q 1e-6, v and tau 1e-5. ID at dt = 5e-3, PD at 1e-3 (at 5e-3
    its reference gains are unstable on the ground plant, DESIGN section 10)."""
    from oracle import controllers as oc, rollout as ro
    from oracle.dynamics import Plant
    from quadruped_drake_b200.rollout import Motor, MotorSet, motor_desc, rollout
    n, steps, dt = 4, 24, (5e-3 if kind == "id" else 1e-3)
    rng = np.random.default_rng(41)
    q0 = grounded(ctl, n, rng, 0.01)
    s = standing_sampler(ctl, float(grounded(ctl, 1, rng, 0.0)[0, 6]))
    kw = dict(peak_scale=0.8, speed_knee=0.5, speed_free=3.0, lag=4e-3, damping=0.02, coulomb=0.1, coulomb_speed=0.2)
    ms = MotorSet(ctl, [motor_desc(ctl.model, **kw)])
    r = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, motor=Motor(ms))
    assert (r.status_or == 0).all()
    plant = Plant("mini_cheetah")
    vi, ai, eff = (np.asarray(x) for x in (ctl.model.v_index, ctl.model.act_index, ctl.model.effort))
    rec = om.record(eff, **kw)
    for i in range(n):
        ctrl = oc.IDController("mini_cheetah") if kind == "id" else oc.BasicController("mini_cheetah")
        q, v, t = q0[i].copy(), np.zeros(18), 0.0
        tau_m, count = np.zeros((1, 12)), np.zeros(1, np.int64)
        for c in range(steps):
            if kind == "id":
                g = s.sample(np.array([t]))
                tau = ctrl.control_law(q, v, oc.traj_to_dict(g["traj"][0], g["contact"][0])).tau
            else:
                tau = ctrl.control_law(q, v)
            plant_tau, _ = om.apply([rec], None, tau_m, count, dt, vi, ai, v[None], np.asarray(tau)[None])
            q, v, _ = ro.plant_step(plant, q, v, plant_tau[0], dt)
            t += dt
        assert np.abs(r.q[i] - q).max() < 1e-6, (i, np.abs(r.q[i] - q).max())
        assert np.abs(r.v[i] - v).max() < 1e-5 and np.abs(r.tau[i] - tau).max() < 1e-5
    ms.close(); s.close()


@gpu
@pytest.mark.parametrize("kind", ["id", "pc", "pd"])
def test_null_set_saturates_at_the_effort(ctl, world, kind):
    """With the NULL set (peak = the URDF effort) the monitor's SAT_MAX is at most 1 for every robot, with pushes, variants,
    terrain, parameter sets and a loop whose strength reaches 1.2; without the motor the same runs exceed it."""
    from quadruped_drake_b200.rollout import Monitor, Motor, rollout
    n, steps, dt = world["n"], 300, 5e-3 if kind != "pd" else 1e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    loop = noisy_loop(n, np.random.default_rng(12))
    a = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop, monitor=Monitor(), **kw)
    b = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop, monitor=Monitor(), motor=Motor(), **kw)
    assert (a.monitor.sat_max > 1.0).any()
    assert (b.monitor.sat_max <= 1.0).all(), b.monitor.sat_max.max()


@gpu
def test_standing_with_weak_motors(ctl):
    """Jittered standing ID robots at dt = 5e-3 over 3 s, reading their state through the loop's noise profile: with peak =
    effort none fails in the monitor, and the peak torque exceeds 0.3 x effort. With peak = 0.3 x effort none fails either,
    although the motors saturate (SAT_MAX exactly 0.3): SAT_MAX is the PEAK torque over the effort, and the median of 0.52 that
    DESIGN section 10 reports for standing ID comes from torque spikes that the sensing noise drives; holding the stance takes
    about 0.12 x effort (the SAT_MAX of a noise-free standing robot), so clamping the spikes does not bring a robot down. With
    peak = 0.05 x effort the legs cannot carry the body and every robot fails."""
    from quadruped_drake_b200.rollout import Loop, Monitor, Motor, MotorSet, motor_desc, rollout
    per, dt, steps = 32, 5e-3, 600
    rng = np.random.default_rng(13)
    q = grounded(ctl, 1, rng, 0.0)
    s = standing_sampler(ctl, float(q[0, 6]))
    q0 = np.tile(q, (3 * per, 1))
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (3 * per, 12))
    ms = MotorSet(ctl, [motor_desc(ctl.model, 1.0), motor_desc(ctl.model, 0.3), motor_desc(ctl.model, 0.05)])
    idx = np.repeat([0, 1, 2], per).astype(np.int32)
    r = rollout(ctl, s, "id", q0, np.zeros((3 * per, 18)), 0.0, steps, dt, plant=True, loop=Loop(noise=NOISE, seed=13), monitor=Monitor(),
                motor=Motor(ms, idx))
    m, cell = r.monitor, idx
    assert (m.fail_step[cell < 2] == 0).all() and (r.status_or[cell < 2] == 0).all()
    assert np.median(m.sat_max[cell == 0]) > 0.3 and (m.sat_max[cell == 0] <= 1.0).all()
    assert abs(np.median(m.sat_max[cell == 1]) - 0.3) < 1e-12
    assert (m.fail_step[cell == 2] > 0).all(), m.fail_step[cell == 2]
    ms.close(); s.close()


@gpu
def test_over_damping_diverges_and_freezes(ctl):
    """Damping of 50 N m s/rad at dt = 5e-3 (Kd dt / I far past 2 on the 1e-3 kg m^2 knee links): the plant flags
    WBC_ST_DIVERGED and freezes every robot; no NaN reaches q or v. A damping of 0.05 keeps them standing."""
    from quadruped_drake_b200.capi import ST_DIVERGED
    from quadruped_drake_b200.rollout import Motor, MotorSet, motor_desc, rollout
    n, dt = 16, 5e-3
    rng = np.random.default_rng(14)
    q0 = grounded(ctl, n, rng, 0.02)
    s = standing_sampler(ctl, float(grounded(ctl, 1, rng, 0.0)[0, 6]))
    ms = MotorSet(ctl, [motor_desc(ctl.model, damping=50.0), motor_desc(ctl.model, damping=0.05)])
    idx = np.repeat([0, 1], n // 2).astype(np.int32)
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 200, dt, plant=True, motor=Motor(ms, idx))
    assert ((r.status_or[: n // 2] & ST_DIVERGED) != 0).all() and (r.status_or[n // 2:] == 0).all()
    assert np.isfinite(r.q).all() and np.isfinite(r.v).all()
    ms.close(); s.close()


@gpu
def test_bad_index(ctl, world):
    """Robots with an out-of-range motor index: WBC_ST_BADMOTOR and a monitor failure at step 1, their state left alone; the
    neighbours have the bits of the batch without them."""
    from quadruped_drake_b200.capi import ST_BADMOTOR
    from quadruped_drake_b200.rollout import Monitor, Motor, MotorState, rollout
    n, steps, dt = 64, 80, 1e-3
    q0, s = world["q0"][:n], world["s"]
    kw = {k: (x[:n] if isinstance(x, np.ndarray) else x) for k, x in world["kw"].items()}
    idx = world["motor_index"][:n].copy()
    bad = [5, 40]
    idx[bad] = [8, -1]
    st = MotorState(n)
    st.tau_m[:], st.count[:] = 0.25, 3
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, monitor=Monitor(), motor=Motor(world["distinct"], idx, st),
                **kw)
    assert ((r.status_or[bad] & ST_BADMOTOR) != 0).all() and (r.monitor.fail_step[bad] == 1).all() and (r.monitor.fail_why[bad] & 4).all()
    assert (st.tau_m[bad] == 0.25).all() and (st.count[bad] == 3).all()
    rest = np.setdiff1d(np.arange(n), bad)
    assert (st.count[rest] == 3 + steps).all() and ((r.status_or[rest] & ST_BADMOTOR) == 0).all()
    rkw = {k: (x[rest] if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    rst = MotorState(len(rest))
    rst.tau_m[:], rst.count[:] = 0.25, 3
    ref = rollout(ctl, s, "id", q0[rest], np.zeros((len(rest), 18)), 0.0, steps, dt, plant=True, monitor=Monitor(),
                  motor=Motor(world["distinct"], idx[rest], rst), **rkw)
    for key in ROLL_KEYS + ("why",):
        assert np.array_equal(getattr(r, key)[rest], getattr(ref, key)), key
    for key in MON_KEYS:
        assert np.array_equal(getattr(r.monitor, key)[rest], getattr(ref.monitor, key)), key
    assert np.array_equal(st.tau_m[rest], rst.tau_m)


@gpu
def test_argument_errors(ctl, world):
    import torch
    from quadruped_drake_b200.capi import WbcMotorDesc, WbcPlantMotor, WbcPlantOpts, WbcRolloutIO, WbcRolloutOpts
    from quadruped_drake_b200.rollout import Motor, MotorSet, MotorState, motor_apply, motor_desc, rollout
    n = 4
    s = world["s"]
    q, v, t = world["q0"][:n].copy(), np.zeros((n, 18)), np.zeros(n)
    io = WbcRolloutIO(P(q), P(v), P(t), None, None, None, None, None, None)
    st = MotorState(n)
    integ = WbcRolloutOpts(1, 0, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    ground = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    call = lambda o, m: ctl.lib.wbc_rollout_motor_host(ctl._h, 0, s._p, n, 2, 5e-3, C.byref(io), C.byref(o), None, None, None, None,  # noqa: E731
                                                       None, C.byref(m))
    assert call(integ, WbcPlantMotor(None, None, None, None)) == 1 and b"ground plant" in ctl.lib.wbc_last_error(ctl._h)
    assert call(ground, WbcPlantMotor(None, None, P(st.tau_m), None)) == 1 and b"together" in ctl.lib.wbc_last_error(ctl._h)
    assert call(ground, WbcPlantMotor(None, None, None, P(st.count))) == 1
    u = np.zeros((n, 12))
    assert ctl.lib.wbc_motor_apply_host(ctl._h, n, 1e-3, C.byref(WbcPlantMotor(None, None, None, None)), P(v), P(u), P(u), None) == 1
    assert ctl.lib.wbc_motor_apply_host(ctl._h, n, 0.0, C.byref(WbcPlantMotor(None, None, P(st.tau_m), P(st.count))), P(v), P(u), P(u),
                                        None) == 1
    assert np.array_equal(q, world["q0"][:n]) and (st.count == 0).all()          # nothing ran
    h = C.c_void_p()
    bad = motor_desc(ctl.model, speed_knee=5.0, speed_free=4.0)
    assert ctl.lib.wbc_motor_set_create(ctl._h, 1, C.byref(bad), C.byref(h)) == 1 and b"speed_knee" in ctl.lib.wbc_last_error(ctl._h)
    assert ctl.lib.wbc_motor_set_create(ctl._h, 0, C.byref(motor_desc(ctl.model)), C.byref(h)) == 1 and not h
    with pytest.raises(RuntimeError):
        MotorSet(ctl, [motor_desc(ctl.model), motor_desc(ctl.model, coulomb=0.1)])
    assert C.sizeof(WbcMotorDesc) == 672 and C.sizeof(WbcPlantMotor) == 32
    tq, tv, tt = (torch.from_numpy(x.copy()).cuda() for x in (q, v, t))
    l0 = ctl.launches
    for field, fix in (("tau_m", lambda x: x.float()), ("tau_m", lambda x: x[:, :11].contiguous()), ("count", lambda x: x.int()),
                       ("count", lambda x: x.cpu()), ("tau_m", lambda x: x.t().contiguous().t())):
        ms = MotorState(n, like=tq)
        setattr(ms, field, fix(getattr(ms, field)))
        with pytest.raises(ValueError, match="motor.state." + field):
            rollout(ctl, s, "id", tq, tv, tt, 2, 5e-3, plant=True, motor=Motor(state=ms))
    with pytest.raises(ValueError, match="motor.index"):
        rollout(ctl, s, "id", tq, tv, tt, 2, 5e-3, plant=True, motor=Motor(index=torch.zeros(n, dtype=torch.int64, device="cuda")))
    with pytest.raises(ValueError, match="motor.state"):
        rollout(ctl, s, "id", q, v, t, 2, 5e-3, plant=True, motor=Motor(state=MotorState(n + 1)))
    with pytest.raises(ValueError, match="motor.state is required"):
        motor_apply(ctl, v, u, Motor())
    with pytest.raises(ValueError, match="tau"):
        motor_apply(ctl, tv, torch.zeros((n, 12), dtype=torch.float32, device="cuda"), Motor(state=MotorState(n, like=tq)))
    assert ctl.launches == l0
