"""Contact detection in the ground-plant loop (wbc_contact_set_create, wbc_rollout_contact[_host], wbc_contact_step[_host];
include/wbc.h, wbc_contact_desc / wbc_contact).

CPU half: the numpy restatement oracle/contact.py against the known answer of the plant's time-stepping scheme (one
oracle/rollout.py:plant_step: the force estimate is the plant's ground force), its prime / filter / hysteresis / singular-leg /
failure rules, the kernel of csrc/wbc_contact.cuh on the host (tests/emu/emu_contact.cpp) against the oracle, and the record check
of wbc_contact_set_create.
GPU half: det == NULL is wbc_rollout_estimator; two more launches per step; feed = 0 changes no output; the controller feed with a
detector that never releases equals feed = 0; rounding-level force errors without a loop; wbc_contact_step against the oracle;
the fused rollout equals a manual loop; continuation, permutation, graph replay; a bad index; argument errors."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from oracle import contact as ocn

P_ = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
INF = np.inf
ROBOTS = [("mini_cheetah", "depth_first"), ("mini_cheetah", "breadth_first"), ("anymal_b", "depth_first"), ("anymal_b", "breadth_first")]


def load(robot="mini_cheetah", order="depth_first"):
    from quadruped_drake_b200.model import load_robot
    return load_robot(robot, order)


def plant_of(robot="mini_cheetah", order="depth_first"):
    from oracle.dynamics import Plant
    return Plant(robot, order)


def rand_quat(rng, spread=0.1):
    q = np.concatenate([[1.0], rng.normal(0, spread, 3)])
    return q / np.linalg.norm(q)


def standing(plant, model, dz=0.0):
    """The nominal posture with the lowest foot at z = dz."""
    q = model.nominal_q()
    pz = [plant.frame_position_quantities(q, np.zeros(18), f)[0][2] for f in plant.foot_frames]
    q[6] -= min(pz) - dz
    return q


def weight(plant):
    return plant.total_mass() * 9.81


class _Pushed:
    """A plant with a point force F (world) at base point r (base axes) on its base: the generalized force [(R r) x F; F], which
    enters the dynamics as a negative bias."""

    def __init__(self, plant, F, r):
        self.plant, self.F, self.r = plant, np.asarray(F, float), np.asarray(r, float)

    def __getattr__(self, name):
        return getattr(self.plant, name)

    def calc_dynamics(self, q, v):
        from oracle.dynamics import quat_to_matrix
        M, Cv, tg, S = self.plant.calc_dynamics(q, v)
        g = np.zeros(len(v))
        g[0:3], g[3:6] = np.cross(quat_to_matrix(*q[0:4]) @ self.r, self.F), self.F
        return M, Cv - g, tg, S


def cases(plant, model, rng):
    """(name, q, v, tau, plant to step, terrain) of the known-answer cases."""
    from oracle import terrain as otr
    q0, n = standing(plant, model), plant.nv
    tau = rng.normal(0, 3.0, 12)
    out = [("standing", q0, np.zeros(n), tau, plant, None)]
    v = np.zeros(n)
    v[3:6] = [0.6, -0.3, 0.0]
    out.append(("sliding", q0, v, tau, plant, None))
    qa = q0.copy()
    qa[6] += 0.2
    out.append(("airborne", qa, rng.normal(0, 0.5, n), tau, plant, None))
    qp = q0.copy()
    qp[6] -= 0.01
    out.append(("penetrating", qp, np.zeros(n), tau, plant, None))
    for j in range(3):
        qr = q0.copy()
        qr[0:4] = rand_quat(rng, 0.05)
        qr[7:] += rng.normal(0, 0.15, 12)
        qr = standing(plant, model, rng.uniform(-0.005, 0.003)) if j == 0 else qr
        qr[6] += rng.uniform(-0.01, 0.01)
        out.append((f"random{j}", qr, rng.normal(0, 0.4, n), rng.normal(0, 6.0, 12), plant, None))
    qt = q0.copy()
    out.append(("incline", qt, rng.normal(0, 0.1, n), tau, plant, otr.incline(8.0, (1.0, 0.4), z0=-0.003)))
    out.append(("push", q0, rng.normal(0, 0.1, n), tau, _Pushed(plant, [30.0, -20.0, 10.0], [0.05, 0.02, 0.01]), None))
    return out


# ------------------------------------------------------------------------------------------------------------------ CPU half
@pytest.mark.parametrize("robot,order", ROBOTS)
def test_oracle_force_is_the_plants(robot, order):
    """After one plant step, the momentum residual of each leg's joint rows gives the plant's ground force within 1e-8 of the
    larger of the robot's weight and the largest force: standing, sliding, airborne (zero force), penetrating and random states,
    on a plane terrain (forces in world axes) and under a push (base rows only)."""
    from oracle import terrain as otr
    plant, model = plant_of(robot, order), load(robot, order)
    rng = np.random.default_rng(3)
    dt = 5e-3
    loaded = 0
    for name, q, v, tau, stepper, ter in cases(plant, model, rng):
        q1, v1, f = otr.plant_step(stepper, q, v, tau, dt, terrain=ter)
        f_raw, singular = ocn.raw_forces(plant, q, v, v1, tau, dt)
        assert not singular.any(), name
        scale = max(weight(plant), np.abs(f).max())
        assert np.abs(f_raw - f).max() <= 1e-8 * scale, (name, np.abs(f_raw - f).max(), scale)
        if name == "airborne":
            assert not f.any()
        loaded += int((f[:, 2] > 0).sum())
    assert loaded >= 12                                  # the grounded cases have feet carrying load


def test_oracle_rules():
    """Prime (plan flags, zero force), the raw first estimate, the low-pass filter, the hysteresis in both directions, tau_f = 0,
    the statistics, failure and re-prime, and a bad index."""
    plant, model = plant_of(), load()
    dt, q, v = 5e-3, standing(plant, model), np.zeros(18)
    tau = np.zeros(12)
    from oracle import rollout as ro
    q1, v1, f = ro.plant_step(plant, q, v, tau, dt)
    d = ocn.desc(tau_f=0.02, f_on=15.0, f_off=5.0)
    plan = np.array([1, 0, 1, 0], np.uint8)
    det, st, s = ocn.step(d, plant, dt, q, v, plan, ocn.State())
    assert s == 0 and st.count == 1 and (det == plan).all() and (st.flag == plan).all() and not st.f_hat.any()
    st = ocn.record(st, tau, f)
    det, st2, s = ocn.step(d, plant, dt, q1, v1, plan, st)
    raw, _ = ocn.raw_forces(plant, q, v, v1, tau, dt)
    assert s == 0 and st2.count == 2 and np.array_equal(st2.f_hat, raw)        # first estimate: raw, no filter
    assert (det == (raw[:, 2] >= 15.0) | (plan.astype(bool) & ~(raw[:, 2] <= 5.0))).all()
    assert np.isclose(st2.stats[0], ((raw - f) ** 2).sum(), rtol=0, atol=1e-12 * weight(plant) ** 2)
    assert st2.stats[2:6].sum() == 4
    # the filter on later steps, the hysteresis band
    st3 = st2.copy()
    st3.f_hat[:, 2] = [10.0, 10.0, 0.0, 20.0]
    st3.flag[:] = [1, 0, 1, 0]
    st3.q_prev, st3.v_prev, st3.tau_prev = q, v, tau
    det, st4, _ = ocn.step(d, plant, dt, q1, v1, plan, st3)
    a = -np.expm1(-dt / 0.02)
    assert np.allclose(st4.f_hat, st3.f_hat + a * (raw - st3.f_hat), rtol=1e-15, atol=1e-13)
    for k in range(4):
        z = st4.f_hat[k, 2]
        assert det[k] == (int(z > 5.0) if st3.flag[k] else int(z >= 15.0)), k
    det, st5, _ = ocn.step(ocn.desc(tau_f=0.0, f_on=15.0, f_off=5.0), plant, dt, q1, v1, plan, st3)
    assert np.array_equal(st5.f_hat, raw)
    # failure: non-finite torque -> count 0, everything else kept, plan out; then a prime
    bad = st3.copy()
    bad.tau_prev[4] = np.nan
    det, st6, s = ocn.step(d, plant, dt, q1, v1, plan, bad)
    assert s == ocn.ST_BADCONTACT and st6.count == 0 and (det == plan).all() and np.array_equal(st6.f_hat, bad.f_hat)
    assert np.array_equal(st6.q_prev, bad.q_prev) and np.array_equal(st6.stats, bad.stats)
    det, st7, s = ocn.step(d, plant, dt, q1, v1, 1 - plan, st6)
    assert s == 0 and st7.count == 1 and (st7.flag == 1 - plan).all()
    det, st8, s = ocn.step(None, plant, dt, q1, v1, plan, st3)
    assert s == ocn.ST_BADCONTACT and (det == plan).all() and st8.count == st3.count and np.array_equal(st8.f_hat, st3.f_hat)


def straight_knee(plant, model):
    """Standing with leg RF's knee straight (its foot in the air): a singular leg block."""
    q = standing(plant, model)
    knee = model.v_index[5] + 1
    q[knee] = 0.0
    return q


def test_oracle_singular_leg_is_held():
    """A straight knee makes leg RF singular: its f_hat and flag are held and it adds nothing to the statistics; the other legs
    are estimated."""
    from oracle import rollout as ro
    plant, model = plant_of(), load()
    dt = 5e-3
    q = straight_knee(plant, model)
    q1, v1, f = ro.plant_step(plant, q, np.zeros(18), np.zeros(12), dt)
    _, sing = ocn.raw_forces(plant, q, np.zeros(18), v1, np.zeros(12), dt)
    assert sing.tolist() == [False, True, False, False]
    st = ocn.State(q_prev=q, v_prev=np.zeros(18), tau_prev=np.zeros(12), f_true=f, f_hat=np.full((4, 3), 7.0), flag=[0, 1, 0, 1],
                   count=5)
    det, st2, s = ocn.step(ocn.desc(tau_f=0.0, f_on=1.0, f_off=0.5), plant, dt, q1, v1, np.ones(4), st)
    assert s == 0 and det[1] == 1 and np.array_equal(st2.f_hat[1], [7.0, 7.0, 7.0]) and st2.stats[2:6].sum() == 3


@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_contact.so"))
    lib.emu_contact_step.argtypes = [C.c_void_p, C.c_longlong, C.c_double, C.c_void_p, C.c_int] + [C.c_void_p] * 15
    lib.emu_contact_record.argtypes = [C.c_longlong, C.c_int] + [C.c_void_p] * 5
    lib.emu_contact_desc_problem.argtypes = [C.c_void_p]
    lib.emu_contact_desc_problem.restype = C.c_char_p
    return lib


def desc_array(recs):
    from quadruped_drake_b200.capi import WbcContactDesc
    return (WbcContactDesc * len(recs))(*[WbcContactDesc(**r) for r in recs])


RECS = [ocn.desc(), ocn.desc(tau_f=0.0, f_on=1.0, f_off=1.0), ocn.desc(tau_f=0.05, f_on=20.0, f_off=-INF),
        ocn.desc(tau_f=1.0, f_on=INF, f_off=0.5)]


def world(plant, model, rng, n):
    """n robots near standing (one with a straight knee), one plant step each: (q, v, tau, q1, v1, f)."""
    from oracle import rollout as ro
    out = []
    for i in range(n):
        q = standing(plant, model, rng.uniform(-0.006, 0.004))
        q[0:4] = rand_quat(rng, 0.04)
        q[7:] += rng.normal(0, 0.08, 12)
        if i == 3:
            q = straight_knee(plant, model)
        v = rng.normal(0, 0.3, 18)
        tau = rng.normal(0, 4.0, 12)
        q1, v1, f = ro.plant_step(plant, q, v, tau, 5e-3)
        out.append((q, v, tau, q1, v1, f.reshape(12)))
    return [np.array(x) for x in zip(*out)]


def pack(sts):
    keys = ("q_prev", "v_prev", "tau_prev", "f_true", "f_hat", "flag", "count", "stats")
    arrs = {k: np.ascontiguousarray(np.array([getattr(s, k) for s in sts])) for k in keys}
    arrs["f_true"] = arrs["f_true"].reshape(len(sts), 12).copy()
    arrs["f_hat"] = arrs["f_hat"].reshape(len(sts), 12).copy()
    arrs["flag"] = arrs["flag"].astype(np.uint8)
    arrs["count"] = arrs["count"].astype(np.int64)
    return arrs


def close(a, b, scale, tol=1e-9):
    return np.abs(np.asarray(a, float) - np.asarray(b, float)).max(initial=0.0) <= tol * scale


def check_against_oracle(recs, plant, index, sts, arrs, q, v, plan, detected, status, ctrl=None):
    """Each robot's outputs and state (arrs, after the step) against one oracle step from `sts` (before it)."""
    w = weight(plant)
    for i in range(len(sts)):
        d = recs[index[i]] if 0 <= index[i] < len(recs) else None
        det, o, s = ocn.step(d, plant, 5e-3, q[i], v[i], plan[i], sts[i])
        assert s == status[i] and o.count == arrs["count"][i], i
        assert np.array_equal(det, detected[i]) and np.array_equal(o.flag, arrs["flag"][i]), i
        if ctrl is not None:
            assert np.array_equal(ctrl[i], det & (plan[i] != 0)), i
        assert close(arrs["f_hat"][i], o.f_hat.reshape(12), w), (i, arrs["f_hat"][i], o.f_hat)
        assert np.array_equal(arrs["q_prev"][i], o.q_prev) and np.array_equal(arrs["v_prev"][i], o.v_prev), i
        assert close(arrs["stats"][i, :2], o.stats[:2], w * w) and np.array_equal(arrs["stats"][i, 2:], o.stats[2:]), i


@pytest.mark.parametrize("robot,order", ROBOTS)
def test_emulated_detector_matches_oracle(emu, robot, order):
    """16 robots on 4 records (raw, filtered, never released, never detected), a bad index, a straight knee, a non-finite torque,
    primes and estimates: flags, counts and status exact, f_hat and stats within 1e-9 of the weight; the record step copies."""
    plant, model = plant_of(robot, order), load(robot, order)
    ms = model.as_struct()
    rng = np.random.default_rng(17)
    n, k = 16, len(RECS)
    arr = desc_array(RECS)
    index = rng.integers(0, k, n).astype(np.int32)
    index[5] = -1
    q, v, tau, q1, v1, f = world(plant, model, rng, n)
    plan = (rng.random((n, 4)) < 0.7).astype(np.uint8)
    sts = [ocn.State() for _ in range(n)]
    for c in range(3):                            # prime, first estimate, filtered estimate
        qs, vs = (q, v) if c == 0 else (q1, v1)
        if c == 2:
            for i in range(n):
                sts[i].q_prev, sts[i].v_prev = q[i].copy(), v[i].copy()
            sts[9].count = 0                      # re-primed
            sts[11].tau_prev[2] = np.nan          # fails
        arrs = pack(sts)
        detected, ctrl, status = np.zeros((n, 4), np.uint8), np.zeros((n, 4), np.uint8), np.zeros(n, np.int32)
        emu.emu_contact_step(C.byref(ms), n, 5e-3, arr, k, P_(index), *(P_(arrs[x]) for x in ("q_prev", "v_prev", "tau_prev", "f_true",
                             "f_hat", "flag", "count", "stats")), P_(qs), P_(vs), P_(plan), P_(detected), P_(ctrl), P_(status))
        check_against_oracle(RECS, plant, index, sts, arrs, qs, vs, plan, detected, status, ctrl)
        sts = [ocn.step(RECS[index[i]] if index[i] >= 0 else None, plant, 5e-3, qs[i], vs[i], plan[i], sts[i])[1] for i in range(n)]
        tp, ft = arrs["tau_prev"].copy(), arrs["f_true"].copy()
        emu.emu_contact_record(n, k, P_(index), P_(tp), P_(ft), P_(tau), P_(f))
        assert np.array_equal(tp[5], arrs["tau_prev"][5]) and np.array_equal(np.delete(tp, 5, 0), np.delete(tau, 5, 0))
        assert np.array_equal(np.delete(ft, 5, 0), np.delete(f, 5, 0))
        sts = [ocn.record(s, tau[i], f[i]) if index[i] >= 0 else s for i, s in enumerate(sts)]
    assert status[5] == ocn.ST_BADCONTACT and status[11] == ocn.ST_BADCONTACT and sts[11].count == 0
    assert sts[3].count == 3 and sts[0].count == 3


def test_set_creation_checks(emu):
    from quadruped_drake_b200.capi import WbcContactDesc
    from quadruped_drake_b200.rollout import CONTACT_DEFAULTS, contact_desc
    assert CONTACT_DEFAULTS == ocn.DEFAULTS

    def why(**edit):
        msg = emu.emu_contact_desc_problem(C.byref(contact_desc(**edit)))
        assert (msg is None) == (ocn.desc_problem(ocn.desc(**edit)) is None), edit
        return None if msg is None else msg.decode()

    assert why() is None and why(tau_f=0.0) is None and why(f_on=INF, f_off=-INF) is None and why(f_on=3.0, f_off=3.0) is None
    assert why(f_on=-INF, f_off=-INF) is None and why(f_on=INF, f_off=INF) is None
    for edit in (dict(tau_f=INF), dict(tau_f=-1e-300), dict(tau_f=np.nan), dict(f_on=np.nan), dict(f_off=np.nan),
                 dict(f_on=1.0, f_off=2.0), dict(f_on=-INF, f_off=0.0)):
        assert why(**edit) is not None, edit
    assert C.sizeof(WbcContactDesc) == 3 * 8


# ------------------------------------------------------------------------------------------------------------------ GPU half
gpu = pytest.mark.gpu
STATE_KEYS = ("q_prev", "v_prev", "tau_prev", "f_true", "f_hat", "flag", "count", "stats")
ROLL_KEYS = ("q", "v", "t", "tau", "metrics", "status_or", "err_max", "f_contact")
MON_KEYS = ("stats", "steps", "fail_step", "fail_why")
EST_KEYS = ("x", "P", "v_prev", "count", "stats")
NOISE = np.array([0.01, 0.002, 0.01, 0.05, 0.02, 0.1])


@pytest.fixture(scope="module")
def ctl(built):
    from quadruped_drake_b200.controller import BatchedController
    c = BatchedController("mini_cheetah", device=0)
    yield c
    c.close()


def grounded(ctl, n, rng, jitter):
    q0 = np.tile(np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4), (n, 1))
    q0[:, 7:] += rng.uniform(-jitter, jitter, (n, 12))
    pz = ctl.dynamics(q0, np.zeros((n, 18)))["p_feet"][:, :, 2]
    q0[:, 6] -= pz.min(axis=1)
    return q0


@pytest.fixture(scope="module")
def gw(ctl):
    """A 128-robot trot with variants, pushes, terrain and parameter sets; the default estimator and detector sets, and a set of
    the four test records."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.capi import DEFAULT_PARAMS
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import ContactSet, EstimatorSet, PlantSet, Terrain, TerrainSet, contact_desc, estimator_desc
    from quadruped_drake_b200.urdf import load_description
    n = 128
    rng = np.random.default_rng(31)
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    ps = PlantSet(ctl, [flatten(d), flatten(with_payload(d, 1.2, (0.04, -0.02, 0.05)))], [1.0, 0.6])
    ts = TerrainSet(ctl, [Terrain(), Terrain(slope=(np.tan(np.radians(5.0)), 0.0))])
    pset = ParamSet(ctl, [{m: DEFAULT_PARAMS[m] * float(rng.uniform(0.8, 1.25)) for m in ("id_kp_body_p", "id_kd_body_p", "pd_kp")}
                          for _ in range(3)])
    push = np.zeros((n, 8))
    push[:, 0:3] = rng.uniform(-40, 40, (n, 3)); push[:, 3:6] = rng.uniform(-0.1, 0.1, (n, 3))
    push[:, 6], push[:, 7] = 0.2, 0.3
    bh = float(grounded(ctl, 1, rng, 0.0)[0, 6])
    s = pl.TrajectorySampler(ctl, pl.make_gait_plan("mini_cheetah", "trot", goal=(1.5, 0.0), base_height=bh))
    es = EstimatorSet(ctl, [estimator_desc()])
    cs = ContactSet(ctl, [contact_desc()])
    recs = ContactSet(ctl, list(desc_array(RECS)))
    w = dict(q0=grounded(ctl, n, rng, 0.02), s=s, n=n, es=es, cs=cs, recs=recs, bh=bh,
             cidx=rng.integers(0, len(RECS), n).astype(np.int32),
             kw=dict(plant_set=ps, terrain_set=ts, param_set=pset, variant=(np.arange(n) % 2).astype(np.int32), push=push,
                     terrain=(np.arange(n) // 2 % 2).astype(np.int32), param_index=rng.integers(0, 3, n).astype(np.int32)))
    yield w
    recs.close(); cs.close(); es.close(); pset.close(); ts.close(); ps.close(); s.close()


def noisy_loop(n, rng, dmax=2, seed=7):
    from quadruped_drake_b200.rollout import Loop
    return Loop(noise=NOISE * rng.uniform(0.5, 2.0, (n, 1)), delay=rng.integers(0, dmax + 1, n).astype(np.int32),
                strength=rng.uniform(0.8, 1.2, n), stream=rng.integers(-2**31, 2**31, n).astype(np.int32), seed=seed)


def same_outputs(a, b, what):
    for key in ROLL_KEYS:
        assert np.array_equal(getattr(a, key), getattr(b, key)), (what, key)
    if a.monitor is not None:
        for key in MON_KEYS:
            assert np.array_equal(getattr(a.monitor, key), getattr(b.monitor, key)), (what, key)
    if a.estimator is not None:
        for key in EST_KEYS:
            assert np.array_equal(getattr(a.estimator, key), getattr(b.estimator, key)), (what, key)


@gpu
def test_null_detector_is_rollout_estimator(ctl, gw):
    """wbc_rollout_contact_host with det == NULL: the bits and launch count of wbc_rollout_estimator_host."""
    from quadruped_drake_b200.capi import WbcEstimator, WbcPlantOpts, WbcRolloutIO, WbcRolloutOpts
    from quadruped_drake_b200.rollout import Estimator, EstimatorState, rollout
    import quadruped_drake_b200.rollout as rmod
    n, steps = 32, 40
    q0, s = gw["q0"][:n], gw["s"]
    loop = noisy_loop(n, np.random.default_rng(5))
    for kind in ("id", "pd"):
        l0 = ctl.launches
        ref = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, plant=True, loop=loop,
                      estimator=Estimator(gw["es"], state=EstimatorState(n)))
        l1 = ctl.launches
        q, v, t = q0.copy(), np.zeros((n, 18)), np.zeros(n)
        r = [np.zeros((n, 12)), np.zeros((n, 4)), np.zeros(n, np.int32), np.zeros(n), np.zeros((n, 12))]
        io = WbcRolloutIO(P_(q), P_(v), P_(t), None, *map(P_, r[:4]), None)
        o = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), P_(r[4]))
        lp = rmod._wbc_loop(loop, rmod._loop_arrays(loop, n), P_)
        est = EstimatorState(n)
        es = WbcEstimator(gw["es"]._p, None, None, *(P_(getattr(est, k)) for k in ("x", "P", "v_prev", "count", "stats")))
        l2 = ctl.launches
        ctl._check(ctl.lib.wbc_rollout_contact_host(ctl._h, 0 if kind == "id" else 4, s._p, n, steps, 5e-3, C.byref(io), C.byref(o), None,
                                                    None, None, C.byref(lp), None, None, C.byref(es), None), "wbc_rollout_contact_host")
        assert ctl.launches - l2 == l1 - l0
        for key, x in zip(("q", "v", "t", "tau", "metrics", "status_or", "err_max"), [q, v, t] + r[:4]):
            assert np.array_equal(x, getattr(ref, key)), (kind, key)
        assert np.array_equal(r[4].reshape(n, 4, 3), ref.f_contact)
        for key in EST_KEYS:
            assert np.array_equal(getattr(est, key), getattr(ref.estimator, key)), key


@gpu
@pytest.mark.parametrize("graph", [True, False])
def test_two_more_launches_per_step(ctl, gw, graph):
    """A detector adds exactly two launches per step, on the host and the device entries, with and without graph capture; without
    a state it primes afresh each call (the bits of a fresh ContactState)."""
    import torch
    from quadruped_drake_b200.rollout import ContactDetector, ContactState, Monitor, Motor, rollout
    n, steps = 32, 25
    q0, s = gw["q0"][:n], gw["s"]
    for extra in (dict(), dict(motor=Motor(), monitor=Monitor())):
        l0 = ctl.launches
        a = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, use_graph=graph, **extra)
        l1 = ctl.launches
        b = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, use_graph=graph, **extra,
                    contact=ContactDetector(gw["cs"], state=ContactState(n)))
        l2 = ctl.launches
        assert l2 - l1 == (l1 - l0) + 2 * steps
        same_outputs(a, b, extra)
        assert (b.contact.count == steps).all()
        c = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, use_graph=graph, **extra,
                    contact=ContactDetector(gw["cs"]))
        assert c.contact is None
        same_outputs(a, c, extra)
        q, v, t = (torch.from_numpy(x.copy()).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
        st = ContactState(n, like=q)
        with torch.cuda.stream(torch.cuda.Stream()):
            l3 = ctl.launches
            rollout(ctl, s, "id", q, v, t, steps, plant=True, use_graph=graph, **extra, contact=ContactDetector(gw["cs"], state=st))
        torch.cuda.synchronize()
        assert ctl.launches - l3 == l2 - l1
        assert np.array_equal(q.cpu().numpy(), b.q)
        for key in STATE_KEYS:
            assert np.array_equal(getattr(st, key).cpu().numpy(), getattr(b.contact, key)), key


@gpu
def test_feed_zero_changes_no_output(ctl, gw):
    """feed = 0 with a loop, an estimator, a motor, a monitor, variants, pushes, terrain and parameter sets: q, v, t, tau, metrics,
    status_or, err_max, metrics_log, f_contact, the monitor state and the estimator state have the bits of the call without a
    detector, for all five kinds."""
    from quadruped_drake_b200.rollout import ContactDetector, ContactState, Estimator, EstimatorState, Monitor, MonitorState, Motor, rollout
    n, steps = gw["n"], 60
    loop = noisy_loop(n, np.random.default_rng(8))
    for kind in ("id", "clf", "pc", "mptc", "pd"):
        runs = []
        for det in (None, ContactDetector(gw["recs"], gw["cidx"], 0, ContactState(n))):
            loop.state = None
            runs.append(rollout(ctl, gw["s"], kind, gw["q0"], np.zeros((n, 18)), 0.0, steps, plant=True, log_metrics=True, loop=loop,
                                monitor=Monitor(state=MonitorState(n)), motor=Motor(), contact=det,
                                estimator=Estimator(gw["es"], state=EstimatorState(n)), **gw["kw"]))
        same_outputs(runs[0], runs[1], kind)
        assert np.array_equal(runs[0].metrics_log, runs[1].metrics_log) and np.array_equal(runs[0].why, runs[1].why)
        assert (runs[1].contact.count > 0).mean() > 0.9


@gpu
def test_controller_feed_with_a_detector_that_never_releases(ctl, gw):
    """FEED_CONTROLLER with f_off = -inf on an all-stance plan: the controller reads plan AND detected = the plan, so every output
    has the bits of feed = 0."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.capi import CONTACT_FEED_CONTROLLER
    from quadruped_drake_b200.rollout import ContactDetector, ContactSet, ContactState, Loop, contact_desc, rollout
    n = 64
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=gw["bh"]))
    cs = ContactSet(ctl, [contact_desc(f_on=1e9, f_off=-INF)])
    runs = []
    for feed in (0, CONTACT_FEED_CONTROLLER):
        st = ContactState(n)
        runs.append(rollout(ctl, s, "id", gw["q0"][:n], np.zeros((n, 18)), 0.0, 150, plant=True, loop=noisy_loop(n, np.random.default_rng(2)),
                            contact=ContactDetector(cs, feed=feed, state=st)))
    same_outputs(runs[0], runs[1], "feed")
    for key in STATE_KEYS:
        assert np.array_equal(getattr(runs[0].contact, key), getattr(runs[1].contact, key)), key
    assert runs[1].contact.flag.all()
    cs.close(); s.close()


@gpu
@pytest.mark.parametrize("motion", ["standing", "raise_foot"])
def test_force_error_at_rounding_level(ctl, gw, motion):
    """No loop and no motor: the detector reads the true state and the plant receives the command, the measured torque. The force
    estimate then matches the plant's forces to rounding (1e-6 of the weight, the plant's own bar), and once the feet have settled
    no foot is falsely in stance or in swing."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.rollout import ContactDetector, ContactSet, ContactState, contact_desc, rollout
    n = 64
    rng = np.random.default_rng(4)
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", motion, 6.0, base_height=gw["bh"]))
    cs = ContactSet(ctl, [contact_desc(tau_f=0.0, f_on=0.5, f_off=0.5)])
    det = ContactDetector(cs, state=ContactState(n))
    r = rollout(ctl, s, "id", grounded(ctl, n, rng, 0.01), np.zeros((n, 18)), 0.0, 500, plant=True, contact=det)
    st = det.state
    w = weight(plant_of())
    assert (r.status_or == 0).all()
    assert (st.max_force < 1e-6 * w).all(), st.max_force.max()
    st.stats[:] = 0.0
    r = rollout(ctl, s, "id", r.q, r.v, r.t, 400, plant=True, contact=det)
    assert (st.max_force < 1e-6 * w).all() and (st.rms_force < 1e-7 * w).all(), (st.max_force.max(), st.rms_force.max())
    assert not st.false_stance.any() and not st.false_swing.any()
    assert (st.true_stance + st.true_swing == 4 * 400).all()
    if motion == "raise_foot":
        assert (st.true_swing == 400).all() and not st.flag[:, 1].any()
    else:
        assert (st.true_stance == 4 * 400).all()
    cs.close(); s.close()


def random_rows(ctl, rng, n):
    """n robots one plant step into a random state: (q, v, tau, q1, v1, f) from the oracle's model-free GPU plant step."""
    from quadruped_drake_b200.rollout import plant_step
    q = grounded(ctl, n, rng, 0.1)
    q[:, 6] += rng.uniform(-0.006, 0.004, n)
    v = rng.normal(0, 0.3, (n, 18))
    tau = rng.normal(0, 4.0, (n, 12))
    out = plant_step(ctl, q, v, tau, 5e-3)
    q1, v1, f = out[0], out[1], out[2]
    return q, v, tau, q1, v1, np.ascontiguousarray(np.asarray(f).reshape(n, 12))


@gpu
def test_contact_step_matches_oracle(ctl, gw):
    """wbc_contact_step on 600 rows of 4 records with bad indices, primes and non-finite torques, host and device entries: the
    same bits, and flags, counts and status exact against the oracle, f_hat and stats within 1e-9 of the weight."""
    import torch
    from quadruped_drake_b200.rollout import ContactDetector, ContactState, contact_step
    rng = np.random.default_rng(6)
    n = 600
    plant = plant_of()
    q, v, tau, q1, v1, f = random_rows(ctl, rng, n)
    index = rng.integers(0, len(RECS), n).astype(np.int32)
    index[rng.random(n) < 0.02] = len(RECS)
    plan = (rng.random((n, 4)) < 0.7).astype(np.uint8)
    sts = []
    for i in range(n):
        st = ocn.State(q_prev=q[i], v_prev=v[i], tau_prev=tau[i], f_true=f[i], f_hat=rng.normal(0, 10, 12),
                       flag=rng.integers(0, 2, 4), count=int(rng.choice([0, 1, 2, 7])))
        if i % 97 == 5:
            st.tau_prev[0] = np.inf
        sts.append(st)
    host = ContactState(n)
    for key, x in pack(sts).items():
        getattr(host, key)[:] = x
    init = {key: getattr(host, key).copy() for key in STATE_KEYS}
    hd, hs = contact_step(ctl, q1, v1, plan, ContactDetector(gw["recs"], index, state=host))
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    dev = ContactState(n, like=T(q1))
    for key in STATE_KEYS:
        getattr(dev, key).copy_(T(init[key]))
    dd, ds = contact_step(ctl, T(q1), T(v1), T(plan), ContactDetector(gw["recs"], T(index), state=dev))
    torch.cuda.synchronize()
    assert np.array_equal(dd.cpu().numpy(), hd) and np.array_equal(ds.cpu().numpy(), hs)
    for key in STATE_KEYS:
        assert np.array_equal(getattr(dev, key).cpu().numpy(), getattr(host, key)), key
    arrs = {key: getattr(host, key) for key in STATE_KEYS}
    check_against_oracle(RECS, plant, index, sts, arrs, q1, v1, plan, hd, hs)
    assert (hs != 0).sum() >= (index == len(RECS)).sum() > 0


@gpu
def test_fused_rollout_equals_a_manual_loop(ctl, gw):
    """128 robots x 150 steps, feed = estimator + controller, a noisy delay-0 strength-1 loop, an estimator, variants, pushes,
    terrain and parameter sets: the fused rollout has the bits of sample -> observe -> wbc_contact_step -> estimator step (on the
    detected flags) -> step (on plan AND detected) -> plant, with the state's tau_prev and f_true written by the test."""
    import torch
    from quadruped_drake_b200.capi import (CONTACT_FEED_CONTROLLER, CONTACT_FEED_ESTIMATOR, KINDS, WbcCtrlParams, WbcIO, WbcPlantOpts,
                                           WbcPlantPerturb, WbcPlantTerrain)
    from quadruped_drake_b200.rollout import (ContactDetector, ContactState, Estimator, EstimatorState, Loop, _contact_arrays, _loop_arrays,
                                              _wbc_contact, _wbc_estimator, _wbc_loop, rollout)
    n, steps, dt = gw["n"], 150, 2e-3
    q0, s, kw = gw["q0"], gw["s"], gw["kw"]
    rng = np.random.default_rng(12)
    loop = Loop(noise=NOISE * rng.uniform(0.5, 2.0, (n, 1)), stream=rng.integers(-2**31, 2**31, n).astype(np.int32), seed=31)
    feed = CONTACT_FEED_ESTIMATOR | CONTACT_FEED_CONTROLLER
    det = ContactDetector(gw["recs"], gw["cidx"], feed, ContactState(n))
    est = Estimator(gw["es"], state=EstimatorState(n))
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop, estimator=est, contact=det, **kw)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    q, v, t = T(q0), T(np.zeros((n, 18))), T(np.zeros(n))
    variant, push, terrain, pidx = (T(kw[k]) for k in ("variant", "push", "terrain", "param_index"))
    traj = torch.empty((n, 54), dtype=torch.float64, device="cuda"); plan = torch.empty((n, 4), dtype=torch.uint8, device="cuda")
    detected, ctrl = torch.empty_like(plan), torch.empty_like(plan)
    qo, vo = torch.empty_like(q), torch.empty_like(v)
    tau, met = torch.zeros((n, 12), dtype=torch.float64, device="cuda"), torch.zeros((n, 4), dtype=torch.float64, device="cuda")
    st, st_or = torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")
    f = torch.zeros((n, 12), dtype=torch.float64, device="cuda")
    tick = torch.zeros(n, dtype=torch.int64, device="cuda")
    hist = torch.zeros((n, 16, 12), dtype=torch.float64, device="cuda")
    dl = Loop(noise=T(loop.noise), stream=T(loop.stream), seed=loop.seed)
    arrays = _loop_arrays(dl, n, q.device)
    lp = _wbc_loop(dl, arrays, p)
    lp.hist, lp.tick = p(hist), p(tick)
    dst = EstimatorState(n, like=q)
    es = _wbc_estimator(Estimator(gw["es"]), None, None, dst, p)
    cst = ContactState(n, like=q)
    dd = ContactDetector(gw["recs"], T(gw["cidx"]), 0, cst)
    cd = _wbc_contact(dd, *_contact_arrays(dd, n, q.device), p)
    cs = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    io = WbcIO(p(qo), p(vo), p(traj), p(ctrl), p(tau), p(met), p(st), None, None, None, None)
    cp = WbcCtrlParams(kw["param_set"]._p, p(pidx))
    po = WbcPlantOpts(1.0, 0.2, 30, 0)
    pt, tr = WbcPlantPerturb(kw["plant_set"]._p, p(variant), p(push)), WbcPlantTerrain(kw["terrain_set"]._p, p(terrain))
    good = (T(gw["cidx"]) >= 0) & (T(gw["cidx"]) < len(RECS))
    for c in range(steps):
        ctl._check(ctl.lib.wbc_sample_trajectory(ctl._h, s._p, n, None, p(t), p(traj), p(plan), None, None, None, cs), "sample")
        ctl._check(ctl.lib.wbc_loop_observe(ctl._h, n, C.byref(lp), p(q), p(v), p(qo), p(vo), cs), "observe")
        ctl._check(ctl.lib.wbc_contact_step(ctl._h, n, dt, C.byref(cd), p(qo), p(vo), p(plan), p(detected), p(st_or), cs), "detect")
        ctl._check(ctl.lib.wbc_estimator_step(ctl._h, n, dt, C.byref(es), C.byref(lp), p(q), p(v), p(qo), p(vo), p(detected), p(st_or), cs),
                   "estimate")
        torch.bitwise_and(plan != 0, detected != 0, out=ctrl)
        ctl._check(ctl.lib.wbc_step_params(ctl._h, KINDS["id"], n, C.byref(io), C.byref(cp), cs), "step")
        ctl._check(ctl.lib.wbc_plant_step_terrain(ctl._h, n, dt, C.byref(po), C.byref(pt), C.byref(tr), p(q), p(v), p(tau), p(t),
                                                  p(st), p(st_or), p(f), cs), "plant")
        cst.tau_prev.copy_(torch.where(good[:, None], tau, cst.tau_prev))
        cst.f_true.copy_(torch.where(good[:, None], f, cst.f_true))
        tick += 1
    torch.cuda.synchronize()
    for key, x in (("q", q), ("v", v), ("t", t), ("tau", tau), ("status_or", st_or), ("f_contact", f.reshape(n, 4, 3))):
        assert np.array_equal(getattr(r, key), x.cpu().numpy()), key
    for key in STATE_KEYS:
        assert np.array_equal(getattr(det.state, key), getattr(cst, key).cpu().numpy()), key
    for key in EST_KEYS:
        assert np.array_equal(getattr(est.state, key), getattr(dst, key).cpu().numpy()), key
    assert (det.state.count > 0).mean() > 0.9


@gpu
def test_continuation_permutation_and_graph(ctl, gw):
    """Two calls of 100 steps with a ContactState equal one call of 200 (graph and plain launches alike); permuting the robots with
    their detector indices and loop streams permutes every output."""
    from quadruped_drake_b200.capi import CONTACT_FEED_CONTROLLER
    from quadruped_drake_b200.rollout import ContactDetector, ContactState, Loop, LoopState, Monitor, MonitorState, rollout
    n, dt = gw["n"], 2e-3
    q0, s, kw, ci = gw["q0"], gw["s"], gw["kw"], gw["cidx"]
    loop = noisy_loop(n, np.random.default_rng(9))
    ref = None
    for graph in (True, False):
        loop.state = LoopState(n)
        one = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 200, dt, plant=True, use_graph=graph, loop=loop, monitor=Monitor(),
                      contact=ContactDetector(gw["recs"], ci, CONTACT_FEED_CONTROLLER, ContactState(n)), **kw)
        loop.state = LoopState(n)
        mon, det = Monitor(state=MonitorState(n)), ContactDetector(gw["recs"], ci, CONTACT_FEED_CONTROLLER, ContactState(n))
        q, v, t, status_or = q0, np.zeros((n, 18)), np.zeros(n), np.zeros(n, np.int32)
        for _ in range(2):
            r = rollout(ctl, s, "id", q, v, t, 100, dt, plant=True, use_graph=graph, loop=loop, monitor=mon, contact=det, **kw)
            q, v, t = r.q, r.v, r.t
            status_or |= r.status_or
        assert np.array_equal(status_or, one.status_or)
        for key in ("q", "v", "t", "tau", "f_contact", "why"):
            assert np.array_equal(getattr(r, key), getattr(one, key)), key
        for key in STATE_KEYS:
            assert np.array_equal(getattr(det.state, key), getattr(one.contact, key)), key
        if ref is None:
            ref = one
        else:                                     # graph replay equals plain launches
            for key in ROLL_KEYS:
                assert np.array_equal(getattr(ref, key), getattr(one, key)), key
            for key in STATE_KEYS:
                assert np.array_equal(getattr(ref.contact, key), getattr(one.contact, key)), key
    perm = np.random.default_rng(10).permutation(n)
    pl = Loop(noise=loop.noise[perm], delay=loop.delay[perm], strength=loop.strength[perm], stream=loop.stream[perm], seed=loop.seed)
    loop.state = None
    pkw = {k: (x[perm] if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    a = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 120, dt, plant=True, loop=loop,
                contact=ContactDetector(gw["recs"], ci, CONTACT_FEED_CONTROLLER, ContactState(n)), **kw)
    b = rollout(ctl, s, "id", q0[perm], np.zeros((n, 18)), 0.0, 120, dt, plant=True, loop=pl,
                contact=ContactDetector(gw["recs"], ci[perm], CONTACT_FEED_CONTROLLER, ContactState(n)), **pkw)
    for key in ROLL_KEYS:
        assert np.array_equal(getattr(a, key)[perm], getattr(b, key)), key
    for key in STATE_KEYS:
        assert np.array_equal(getattr(a.contact, key)[perm], getattr(b.contact, key)), key


@gpu
def test_bad_index(ctl, gw):
    """A bad record index: WBC_ST_BADCONTACT in status_or with and without a monitor (with one the robot fails at step 1 for
    WBC_MON_STATUS); its detector state stays zero and its neighbours keep the bits of a run where it is good."""
    from quadruped_drake_b200.capi import CONTACT_FEED_CONTROLLER, MON_STATUS, ST_BADCONTACT
    from quadruped_drake_b200.rollout import ContactDetector, ContactState, Monitor, MonitorState, rollout
    n, steps = 32, 50
    q0, s = gw["q0"][:n], gw["s"]
    loop = noisy_loop(n, np.random.default_rng(3))
    idx = np.zeros(n, np.int32)
    bad = idx.copy()
    bad[7] = 1
    good = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, loop=loop,
                   contact=ContactDetector(gw["cs"], idx, CONTACT_FEED_CONTROLLER, ContactState(n)))
    for mon in (None, Monitor(state=MonitorState(n))):
        det = ContactDetector(gw["cs"], bad, CONTACT_FEED_CONTROLLER, ContactState(n))
        r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, plant=True, loop=loop, monitor=mon, contact=det)
        assert r.status_or[7] & ST_BADCONTACT and not (np.delete(r.status_or, 7) & ST_BADCONTACT).any()
        for key in STATE_KEYS:
            assert not getattr(det.state, key)[7].any(), key
            assert np.array_equal(np.delete(getattr(det.state, key), 7, 0), np.delete(getattr(good.contact, key), 7, 0)), key
        assert np.array_equal(np.delete(r.q, 7, 0), np.delete(good.q, 7, 0))
        if mon is not None:
            assert mon.state.fail_step[7] == 1 and mon.state.fail_why[7] & MON_STATUS


@gpu
def test_argument_errors(ctl, gw):
    import torch
    from quadruped_drake_b200.capi import CONTACT_FEED_ESTIMATOR, WbcContact, WbcPlantOpts, WbcRolloutIO, WbcRolloutOpts
    from quadruped_drake_b200.rollout import ContactDetector, ContactState, Loop, contact_step, rollout
    n, s = 8, gw["s"]
    q0 = gw["q0"][:n]
    det = ContactDetector(gw["cs"], state=ContactState(n))
    with pytest.raises(ValueError):
        rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 5, plant=False, contact=det)
    with pytest.raises(ValueError):                                   # FEED_ESTIMATOR without an estimator
        rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 5, plant=True, loop=Loop(),
                contact=ContactDetector(gw["cs"], feed=CONTACT_FEED_ESTIMATOR))
    with pytest.raises(ValueError):
        rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 5, plant=True, contact=ContactDetector(gw["cs"], state=ContactState(n + 1)))
    with pytest.raises(ValueError):
        contact_step(ctl, q0, np.zeros((n, 18)), np.ones((n, 4), np.uint8), ContactDetector(gw["cs"]))
    tq = torch.from_numpy(q0.copy()).cuda()
    tv, tt = torch.zeros((n, 18), dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):                                   # host state with device arrays
        rollout(ctl, s, "id", tq, tv, tt, 5, plant=True, contact=det)
    with pytest.raises(ValueError):                                   # wrong index dtype on the device
        rollout(ctl, s, "id", tq, tv, tt, 5, plant=True, contact=ContactDetector(gw["cs"], torch.zeros(n, dtype=torch.int64, device="cuda")))
    # the C ABI: a mixed-NULL state, no set, FEED_ESTIMATOR without an estimator, unknown feed bits; nothing moves
    x = np.zeros((n, 19))
    for c in (WbcContact(gw["cs"]._p, None, 0, P_(x), *([None] * 7)), WbcContact(None, None, 0, *([None] * 8))):
        rc = ctl.lib.wbc_contact_step_host(ctl._h, n, 5e-3, C.byref(c), P_(q0), P_(np.zeros((n, 18))), P_(np.ones((n, 4), np.uint8)),
                                           P_(np.zeros((n, 4), np.uint8)), None)
        assert rc != 0
    q, v, t = q0.copy(), np.zeros((n, 18)), np.zeros(n)
    io = WbcRolloutIO(P_(q), P_(v), P_(t), *([None] * 6))
    o = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    for c in (WbcContact(gw["cs"]._p, None, CONTACT_FEED_ESTIMATOR, *([None] * 8)), WbcContact(gw["cs"]._p, None, 4, *([None] * 8)),
              WbcContact(gw["cs"]._p, None, 0, P_(x), *([None] * 7))):
        assert ctl.lib.wbc_rollout_contact_host(ctl._h, 0, s._p, n, 5, 5e-3, C.byref(io), C.byref(o), None, None, None, None, None, None,
                                                None, C.byref(c)) != 0
    o0 = WbcRolloutOpts(1, 0, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    c = WbcContact(gw["cs"]._p, None, 0, *([None] * 8))
    assert ctl.lib.wbc_rollout_contact_host(ctl._h, 0, s._p, n, 5, 5e-3, C.byref(io), C.byref(o0), None, None, None, None, None, None,
                                            None, C.byref(c)) != 0
    assert np.array_equal(q, q0)
