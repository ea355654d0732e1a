"""Perturbed robots for the ground plant: plant variants (another model, its own ground friction) and base pushes.

CPU half: the device code of the perturbed plant step through the host warp emulator (tests/emu) against the numpy plant of
oracle/rollout.py on the variant's own description (the push enters through `PushedPlant`), the payload helper against the oracle's unwelded tree, and a push from
rest against the momentum balance. GPU half: the same cases through the C ABI, the unperturbed rows of a perturbed rollout
against wbc_rollout_ex, and closed loops with payloads, pushes and mixed friction."""
import copy
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

GOLD = Path(__file__).parent / "golden"
Q0 = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4)      # simulate.py:171-176
DT = 5e-3
PAYLOAD = dict(mass=1.2, com=(0.04, -0.02, 0.05), inertia=(2e-3, 3e-3, 4e-3, 1e-4, -2e-4, 3e-4))


def desc_of(robot):
    from quadruped_drake_b200.model import ROBOT_DIR
    from quadruped_drake_b200.urdf import load_description
    return load_description(ROBOT_DIR / f"{robot}.json")


def scaled(desc, s):
    """Every link mass and inertia scaled by s (the same robot made of a denser material)."""
    d = copy.deepcopy(desc)
    for l in d["links"]:
        l["mass"] *= s
        l["inertia_com"] = [s * x for x in l["inertia_com"]]
    return d


def variants(robot):
    """(name, description, mu) of the variants the parity cases use."""
    from quadruped_drake_b200.model import with_payload
    d = desc_of(robot)
    return [("nominal", d, 1.0), ("payload", with_payload(d, **PAYLOAD), 0.2), ("scaled", scaled(d, 1.15), 1.0),
            ("payload_mu1", with_payload(d, **PAYLOAD), 1.0)]


@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu.so"))
    lib.emu_plant_step.argtypes = [C.c_void_p, C.c_longlong, C.c_double, C.c_double, C.c_double, C.c_int] + [C.c_void_p] * 5
    lib.emu_dynamics.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 8
    return lib


@pytest.fixture(scope="module")
def emu_pt(built):
    """The perturbed plant step (tests/emu/emu_plant_perturbed.cpp)."""
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_perturbed.so"))
    lib.emu_plant_step_perturbed.argtypes = ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_double,
                                              C.c_double, C.c_double, C.c_int] + [C.c_void_p] * 5)
    return lib


def ptr(a):
    from quadruped_drake_b200.capi import np_ptr
    return None if a is None else np_ptr(a)


def model_table(descs):
    from quadruped_drake_b200.model import WbcModelStruct, flatten
    return (WbcModelStruct * len(descs))(*[flatten(d).as_struct() for d in descs])


def emu_perturbed(emu, descs, mu, variant, push, t, q, v, tau, call_mu=1.0):
    """One emulated perturbed step; q, v, t updated in place -> f[N,4,3], status[N]."""
    n = len(q)
    f, st = np.zeros((n, 4, 3)), np.zeros(n, np.int32)
    mu_a = None if mu is None else np.ascontiguousarray(mu, np.float64)
    assert emu.emu_plant_step_perturbed(model_table(descs), ptr(mu_a), len(descs), ptr(variant), ptr(push), ptr(t), n, DT, call_mu, 0.2, 30,
                                        ptr(q), ptr(v), ptr(tau), ptr(f), ptr(st)) == 0
    return f, st


def grounded_q(P, robot, n):
    """n copies of the robot's standing posture with the feet exactly on the ground of plant P."""
    from quadruped_drake_b200 import load_robot
    q = load_robot(robot).nominal_q()
    pz = np.array([P.frame_position_quantities(q, np.zeros(18), fr)[0][2] for fr in P.foot_frames])
    q[6] -= pz.mean()
    return np.tile(q, (n, 1))


def parity_cases(robot):
    """Standing, airborne, sliding, penetrating and random states; variant, push (inside / outside its window) per robot."""
    from oracle.dynamics import Plant
    P = Plant(desc_of(robot))
    rng = np.random.default_rng(17)
    n = 8
    q = grounded_q(P, robot, n)
    v = np.zeros((n, 18))
    tau = rng.uniform(-3, 3, (n, 12))
    q[1, 6] += 0.1                                             # airborne
    v[2, 3:5] = [0.8, -0.4]                                    # sliding
    q[3, 6] -= 0.004                                           # penetrating
    q[4:, 7:] += rng.uniform(-0.2, 0.2, (n - 4, 12)); v[4:] = rng.uniform(-1, 1, (n - 4, 18))
    variant = np.array([1, 1, 1, 2, 0, 3, 1, 2], np.int32)
    t = np.linspace(0.0, 0.35, n)
    push = np.zeros((n, 8))
    push[:, 0:3] = rng.uniform(-40, 40, (n, 3))
    push[:, 3:6] = rng.uniform(-0.15, 0.15, (n, 3))
    push[:, 6], push[:, 7] = 0.0, 1.0                          # active ...
    push[[3, 6], 6] = 0.5                                      # ... except two robots before their window
    push[5, 7] = t[5]                                          # and one at the end of its window (t_off is exclusive)
    return q, v, tau, variant, push, t


class PushedPlant:
    """oracle.dynamics.Plant of a variant with a push: calc_dynamics returns tau_g - J_p' F, J_p the oracle's own Jacobian of the
    point of application (Plant._jac_v on the base), while the push window holds the step's start time t. Through it,
    oracle/rollout.py:plant_step adds the generalized force J_p' F to the right-hand side of the free acceleration."""

    def __init__(self, plant, push, t):
        self.plant, self.push = plant, (push if push is not None and push[6] <= t < push[7] else None)

    def __getattr__(self, name):
        return getattr(self.plant, name)

    def calc_dynamics(self, q, v):
        M, Cv, tau_g, S = self.plant.calc_dynamics(q, v)
        if self.push is not None:
            kin = self.plant.kinematics(q, v)
            pt = kin["p"][0] + kin["R"][0] @ self.push[3:6]
            tau_g = tau_g - self.plant._jac_v(kin, 0, pt).T @ self.push[0:3]
        return M, Cv, tau_g, S


def oracle_step(vs, variant, q, v, tau, push, t):
    from oracle import rollout as ro
    from oracle.dynamics import Plant
    plants = [Plant(d) for _, d, _ in vs]
    return [ro.plant_step(PushedPlant(plants[variant[i]], push[i], t[i]), q[i], v[i], tau[i], DT, vs[variant[i]][2], 0.2, 30)
            for i in range(len(q))]


def assert_matches_oracle(qn, vn, f, ref, what):
    for i, (qo, vo, fo) in enumerate(ref):
        assert np.abs(qn[i] - qo).max() < 1e-9 and np.abs(vn[i] - vo).max() < 1e-8, (what, i, np.abs(vn[i] - vo).max())
        assert np.abs(f[i] - fo).max() < 1e-6 * max(1.0, np.abs(fo).max()), (what, i)


# ------------------------------------------------------------------------------------------------------------------ CPU half
def test_with_payload_keeps_mass_and_first_moment():
    from quadruped_drake_b200.model import flatten, with_payload
    for robot in ("mini_cheetah", "anymal_b"):
        d = desc_of(robot)
        nom, pay = flatten(d), flatten(with_payload(d, **PAYLOAD))
        assert abs(pay.total_mass - nom.total_mass - PAYLOAD["mass"]) < 1e-12
        first = nom.mass[0] * nom.com[0] + PAYLOAD["mass"] * np.array(PAYLOAD["com"])
        assert np.abs(pay.mass[0] * pay.com[0] - first).max() < 1e-14
        assert np.array_equal(pay.mass[1:], nom.mass[1:]) and np.array_equal(pay.v_index, nom.v_index)
        assert len(d["links"]) == len(desc_of(robot)["links"])            # the input description is left as it was
    with pytest.raises(ValueError):
        with_payload(with_payload(d, 1.0, (0, 0, 0)), 1.0, (0, 0, 0))


@pytest.mark.parametrize("case", ["mixed_mini_cheetah", "cfg3_anymal_trot"])
def test_emulated_dynamics_of_payload_variant_match_unwelded_oracle(emu, case):
    """The flattened payload variant (payload merged into body 0) through the device dynamics against oracle.dynamics.Plant on
    the description with the payload as a separate welded body."""
    from oracle.dynamics import Plant
    from quadruped_drake_b200.model import flatten, with_payload
    robot = "anymal_b" if "anymal" in case else "mini_cheetah"
    d = with_payload(desc_of(robot), **PAYLOAD)
    P, ms = Plant(d), flatten(d).as_struct()
    g = np.load(GOLD / f"{case}.npz")
    n = 4
    q, v = np.ascontiguousarray(g["q"][:n]), np.ascontiguousarray(g["v"][:n])
    M, Cv, tg = np.zeros((n, 18, 18)), np.zeros((n, 18)), np.zeros((n, 18))
    J, Jdv, pf = np.zeros((n, 4, 3, 18)), np.zeros((n, 4, 3)), np.zeros((n, 4, 3))
    emu.emu_dynamics(C.byref(ms), n, ptr(q), ptr(v), ptr(M), ptr(Cv), ptr(tg), ptr(J), ptr(Jdv), ptr(pf))
    for i in range(n):
        Mo, Cvo, tgo, _ = P.calc_dynamics(q[i], v[i])
        quant = [P.frame_position_quantities(q[i], v[i], fr) for fr in P.foot_frames]
        ref = {"M": Mo, "Cv": Cvo, "tau_g": tgo, "J": np.stack([x[1] for x in quant]), "Jdv": np.stack([x[2] for x in quant]),
               "p_feet": np.stack([x[0] for x in quant])}
        for name, got in (("M", M[i]), ("Cv", Cv[i]), ("tau_g", tg[i]), ("J", J[i]), ("Jdv", Jdv[i]), ("p_feet", pf[i])):
            assert np.abs(got - ref[name]).max() < 1e-9 * max(np.abs(ref[name]).max(), 1e-3), (name, i)


@pytest.mark.parametrize("robot", ["mini_cheetah", "anymal_b"])
def test_emulated_perturbed_step_matches_oracle(emu_pt, robot):
    """Payload, scaled-mass and nominal variants, friction 0.2 and 1.0, pushes inside and outside their windows; standing,
    airborne, sliding, penetrating and random states; two steps."""
    vs = variants(robot)
    q, v, tau, variant, push, t = parity_cases(robot)
    qe, ve, te = q.copy(), v.copy(), t.copy()
    for step in range(2):
        ref = oracle_step(vs, variant, qe, ve, tau, push, te)
        f, st = emu_perturbed(emu_pt, [d for _, d, _ in vs], [m for _, _, m in vs], variant, push, te, qe, ve, tau)
        assert (st == 0).all()
        assert_matches_oracle(qe, ve, f, ref, (robot, step))
    assert np.allclose(te, t + 2 * DT)
    for k in range(4):                                           # every loaded foot inside its own variant's cone
        mu = np.array([vs[j][2] for j in variant])
        assert (np.abs(f[:, k, :2]) <= mu[:, None] * f[:, k, 2:3] + 1e-9).all()


def test_emulated_unperturbed_variant_keeps_the_bits(emu, emu_pt):
    """Variant = the handle's model, its friction = the call's mu (given or left to the call), push outside its window: the same
    bits as the unperturbed step."""
    from quadruped_drake_b200 import load_robot
    d = desc_of("mini_cheetah")
    ms = load_robot("mini_cheetah").as_struct()
    q, v, tau, _, push, t = parity_cases("mini_cheetah")
    push[:, 6] = 10.0
    qa, va = q.copy(), v.copy()
    fa, sa = np.zeros((len(q), 4, 3)), np.zeros(len(q), np.int32)
    assert emu.emu_plant_step(C.byref(ms), len(q), DT, 1.0, 0.2, 30, ptr(qa), ptr(va), ptr(tau), ptr(fa), ptr(sa)) == 0
    for mu, pu in ((None, push), ([1.0], push), (None, None)):
        qb, vb, tb = q.copy(), v.copy(), t.copy()
        fb, sb = emu_perturbed(emu_pt, [d], mu, None, pu, tb, qb, vb, tau)
        assert np.array_equal(qa, qb) and np.array_equal(va, vb) and np.array_equal(fa, fb) and np.array_equal(sa, sb)


def _com_offset(P, q):
    """World-frame offset of the robot's centre of mass from the base origin, and the total mass."""
    kin = P.kinematics(q, np.zeros(18))
    m = P.mass.sum()
    c = sum(P.mass[i] * (kin["p"][i] + kin["R"][i] @ P.com[i]) for i in range(len(P.mass))) / m
    return c - kin["p"][0], m


@pytest.mark.parametrize("robot", ["mini_cheetah", "anymal_b"])
def test_emulated_push_from_rest_matches_momentum_balance(emu_pt, robot):
    """A robot at rest 0.5 m above the ground, zero torques, pushed with F at r: M(q) v+ = dt (J_p' F - tau_g), whose base rows
    are dt (F + m g) (linear) and dt ((R r) x F + c x m g) (angular about the base origin) - independent of the plant step."""
    from oracle.dynamics import Plant
    from quadruped_drake_b200.model import with_payload
    d = with_payload(desc_of(robot), **PAYLOAD)
    P = Plant(d)
    q = grounded_q(P, robot, 1)
    q[0, 6] += 0.5
    qt = np.array([np.cos(0.2), 0.3 * np.sin(0.2), -0.2 * np.sin(0.2), 0.93 * np.sin(0.2)])      # a tilted, yawed base
    q[0, :4] = qt / np.linalg.norm(qt)
    F, r = np.array([35.0, -20.0, 60.0]), np.array([0.1, -0.05, 0.08])
    push = np.r_[F, r, 0.0, 1.0][None]
    q0 = q.copy()
    v = np.zeros((1, 18))
    f, st = emu_perturbed(emu_pt, [d], None, None, push, np.zeros(1), q, v, np.zeros((1, 12)))
    assert (st == 0).all() and np.abs(f).max() == 0.0
    M = P.mass_matrix(q0[0])
    mv = M @ v[0]
    c, m = _com_offset(P, q0[0])
    g = np.array([0.0, 0.0, -9.81])
    R = P.kinematics(q0[0], np.zeros(18))["R"][0]
    lin, ang = DT * (F + m * g), DT * (np.cross(R @ r, F) + np.cross(c, m * g))
    assert np.abs(mv[3:6] - lin).max() < 1e-9 * np.abs(lin).max()
    assert np.abs(mv[0:3] - ang).max() < 1e-9 * np.abs(ang).max()


# ------------------------------------------------------------------------------------------------------------------ GPU half
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctl(built):
    from quadruped_drake_b200.controller import BatchedController
    c = BatchedController("mini_cheetah", device=0)
    yield c
    c.close()


def plant_set(ctl, descs, mu=None):
    from quadruped_drake_b200.model import flatten
    from quadruped_drake_b200.rollout import PlantSet
    return PlantSet(ctl, [flatten(d) for d in descs], mu)


@gpu
def test_perturbed_plant_step_matches_oracle_on_gpu(ctl):
    """The emulator's parity cases through wbc_plant_step_perturbed_host and through the device entry (torch tensors)."""
    import torch
    from quadruped_drake_b200.rollout import plant_step
    vs = variants("mini_cheetah")
    q, v, tau, variant, push, t = parity_cases("mini_cheetah")
    ps = plant_set(ctl, [d for _, d, _ in vs], [m for _, _, m in vs])
    ref = oracle_step(vs, variant, q, v, tau, push, t)
    qn, vn, f, st = plant_step(ctl, q, v, tau, DT, plant_set=ps, variant=variant, push=push, t=t)
    assert (st == 0).all()
    assert_matches_oracle(qn, vn, f, ref, "host")
    tq, tv, ttau, tt, tvar, tpush = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (q, v, tau, t, variant, push))
    _, _, tf, tst = plant_step(ctl, tq, tv, ttau, DT, plant_set=ps, variant=tvar, push=tpush, t=tt)
    torch.cuda.synchronize()
    assert (tst.cpu().numpy() == 0).all() and np.allclose(tt.cpu().numpy(), t + DT, rtol=0, atol=1e-15)
    assert np.array_equal(tq.cpu().numpy(), qn) and np.array_equal(tv.cpu().numpy(), vn) and np.array_equal(tf.cpu().numpy(), f)
    ps.close()


def grounded(ctl, n, rng=None, jitter=0.0):
    """n copies of simulate.py's q0 with the feet exactly on the ground (+ optional joint jitter)."""
    q0 = np.tile(Q0, (n, 1))
    if rng is not None and jitter > 0:
        q0[:, 7:] += rng.uniform(-jitter, jitter, (n, 12))
    pz = ctl.dynamics(q0, np.zeros((n, 18)))["p_feet"][:, :, 2]
    q0[:, 6] -= pz.min(axis=1)
    return q0


def run_torch(ctl, s, q0, steps, **kw):
    import torch
    from quadruped_drake_b200.rollout import rollout
    n = len(q0)
    q, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    kw = {k: (torch.from_numpy(np.ascontiguousarray(x)).cuda() if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    with torch.cuda.stream(torch.cuda.Stream()):
        before = ctl.launches
        r = rollout(ctl, s, "id", q, v, t, steps, DT, plant=True, **kw)
    torch.cuda.synchronize()
    out = {k: x.cpu().numpy() for k, x in (("q", q), ("v", v), ("t", t), ("tau", r.tau), ("err_max", r.err_max), ("status", r.status_or),
                                             ("f", r.f_contact))}
    out["launches"] = ctl.launches - before
    return out


@gpu
def test_unperturbed_rows_keep_their_bits(ctl):
    """512 robots, ID, 300 steps of the trot plan: the rows with variant 0 = the nominal model, the call's mu and no active push
    are bit-identical to wbc_rollout_ex over the same rows, with and without the graph; graph replay equals plain launches and
    the launches per step are those of the unperturbed rollout."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.model import with_payload
    n, steps = 512, 300
    rng = np.random.default_rng(13)
    q0 = grounded(ctl, n, rng, 0.02)
    bh = float(grounded(ctl, 1)[0, 6])
    s = pl.TrajectorySampler(ctl, pl.make_gait_plan("mini_cheetah", "trot", goal=(1.5, 0.0), base_height=bh))
    d = desc_of("mini_cheetah")
    ps = plant_set(ctl, [d, with_payload(d, **PAYLOAD), scaled(d, 0.9)], [1.0, 0.4, 0.8])
    variant = (np.arange(n) % 3).astype(np.int32)
    push = np.zeros((n, 8))
    push[:, 0:3] = rng.uniform(-30, 30, (n, 3)); push[:, 3:6] = rng.uniform(-0.1, 0.1, (n, 3))
    push[:, 6], push[:, 7] = 0.3, 0.8
    nom = variant == 0
    push[nom & (np.arange(n) % 2 == 0), 6:8] = [2.0, 3.0]       # variant-0 rows: pushes outside the run or no push at all
    push[nom & (np.arange(n) % 2 == 1), 0:3] = 0.0
    push[nom & (np.arange(n) % 2 == 1), 6:8] = [5.0, 6.0]
    outs = {}
    for graph in (False, True):
        outs[("ex", graph)] = run_torch(ctl, s, q0, steps, use_graph=graph)
        outs[("pt", graph)] = run_torch(ctl, s, q0, steps, use_graph=graph, plant_set=ps, variant=variant, push=push)
    for graph in (False, True):
        a, b = outs[("ex", graph)], outs[("pt", graph)]
        for k in ("q", "v", "t", "tau", "err_max", "status", "f"):
            assert np.array_equal(a[k][nom], b[k][nom]), (graph, k)
        assert not np.array_equal(a["q"][~nom], b["q"][~nom])       # the perturbed rows did move differently
        assert a["launches"] == b["launches"]
    for k in ("q", "v", "t", "tau", "err_max", "status", "f"):
        assert np.array_equal(outs[("pt", False)][k], outs[("pt", True)][k]), k
    ps.close(); s.close()


def standing_payload_batch(ctl, n):
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.model import with_payload
    bh = float(grounded(ctl, 1)[0, 6])
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh))
    masses = np.linspace(0.3, 1.5, 5)
    coms = [(0.03, 0.0, 0.04), (-0.02, 0.02, 0.05), (0.0, -0.03, 0.03), (0.04, 0.01, 0.06), (0.0, 0.0, 0.05)]
    d = desc_of("mini_cheetah")
    ps = plant_set(ctl, [with_payload(d, m, c) for m, c in zip(masses, coms)])
    variant = (np.arange(n) % len(masses)).astype(np.int32)
    q0 = grounded(ctl, n, np.random.default_rng(3), 0.02)
    return s, ps, variant, masses[variant], np.array(coms)[variant], q0


@gpu
def test_payload_robots_stand_and_the_ground_carries_the_payload(ctl):
    """Standing ID robots carrying 0.3 - 1.5 kg (mini_cheetah: 8.25 kg) that the controller does not know of: after 1200 steps
    they stand, and the ground carries (m + m_p) g - the plant simulates the variant. An upward push of m_p g at the payload's
    centre of mass for the whole run cancels the payload: the ground carries m g."""
    n = 256
    s, ps, variant, mp, cp, q0 = standing_payload_batch(ctl, n)
    m = ctl.model.total_mass
    push = np.zeros((n, 8))
    push[:, 2] = mp * 9.81
    push[:, 3:6] = cp
    push[:, 6], push[:, 7] = -1.0, 100.0
    for pu, carried in ((None, m + mp), (push, np.full(n, m))):
        kw = dict(plant_set=ps, variant=variant) if pu is None else dict(plant_set=ps, variant=variant, push=pu)
        o = run_torch(ctl, s, q0, 1200, **kw)
        assert (o["status"] == 0).all(), np.unique(o["status"], return_counts=True)
        assert np.abs(o["v"]).max() < 0.05
        fz = o["f"][:, :, 2].sum(axis=1)
        assert (np.abs(fz - carried * 9.81) < 0.02 * carried * 9.81).all(), np.abs(fz / (carried * 9.81) - 1).max()
    ps.close(); s.close()


@gpu
def test_friction_cone_of_each_variant_in_every_step(ctl):
    """Mixed batch, mu in {0.2, 1.0}, a horizontal push of 0.5 m g: every robot's ground forces lie in its own variant's cone in
    every step, and the mu = 0.2 robots reach their cone (they slide)."""
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.rollout import rollout
    n, steps = 128, 120
    d = desc_of("mini_cheetah")
    ps = plant_set(ctl, [d, d], [0.2, 1.0])
    variant = (np.arange(n) % 2).astype(np.int32)
    mu = np.array([0.2, 1.0])[variant]
    bh = float(grounded(ctl, 1)[0, 6])
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh))
    m = ctl.model.total_mass
    push = np.zeros((n, 8))
    push[:, 0] = 0.5 * m * 9.81
    push[:, 6], push[:, 7] = 0.1, 0.4
    q, v, t = (torch.from_numpy(x).cuda() for x in (grounded(ctl, n), np.zeros((n, 18)), np.zeros(n)))
    tvar, tpush = torch.from_numpy(variant).cuda(), torch.from_numpy(push).cuda()
    on_cone = np.zeros(n, bool)
    for _ in range(steps):
        r = rollout(ctl, s, "id", q, v, t, 1, DT, plant=True, plant_set=ps, variant=tvar, push=tpush)
        f = r.f_contact.cpu().numpy()
        assert (f[:, :, 2] >= 0).all()
        lim = mu[:, None] * f[:, :, 2]
        assert (np.abs(f[:, :, 0]) <= lim + 1e-9).all() and (np.abs(f[:, :, 1]) <= lim + 1e-9).all()
        loaded = f[:, :, 2] > 1.0
        on_cone |= (loaded & (np.abs(f[:, :, 0]) > lim - 1e-6 * np.maximum(lim, 1.0))).any(axis=1)
    assert on_cone[variant == 0].all()
    ps.close(); s.close()


@gpu
def test_bad_variant_index_freezes_only_that_robot(ctl):
    """Indices -1 and K: WBC_ST_BADVARIANT, state kept, zero ground forces; the rest of the batch is bit-identical to a batch
    without those robots."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.capi import ST_BADVARIANT
    from quadruped_drake_b200.model import with_payload
    n = 64
    d = desc_of("mini_cheetah")
    ps = plant_set(ctl, [d, with_payload(d, **PAYLOAD)])
    bh = float(grounded(ctl, 1)[0, 6])
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "raise_foot", 6.0, base_height=bh))
    q0 = grounded(ctl, n, np.random.default_rng(4), 0.03)
    variant = (np.arange(n) % 2).astype(np.int32)
    bad = np.zeros(n, bool); bad[[5, 30, 63]] = True
    variant[5], variant[30], variant[63] = -1, 2, 1 << 30
    push = np.zeros((n, 8)); push[:, 1] = 15.0; push[:, 6:8] = [0.05, 0.2]
    a = run_torch(ctl, s, q0, 60, plant_set=ps, variant=variant, push=push)
    b = run_torch(ctl, s, q0[~bad], 60, plant_set=ps, variant=variant[~bad], push=push[~bad])
    assert (a["status"][bad] & ST_BADVARIANT).all() and not (a["status"][~bad] & ST_BADVARIANT).any()
    assert np.array_equal(a["q"][bad], q0[bad]) and (a["v"][bad] == 0).all() and (a["f"][bad] == 0).all()
    assert np.allclose(a["t"], 60 * DT)
    for k in ("q", "v", "t", "tau", "err_max", "status", "f"):
        assert np.array_equal(a[k][~bad], b[k]), k
    ps.close(); s.close()


@gpu
def test_argument_errors_and_set_lifetime(built):
    """Each argument error returns WBC_ERR_ARG with a message; a set destroyed after its handle is safe."""
    import torch
    from quadruped_drake_b200 import load_robot, planner as pl
    from quadruped_drake_b200.capi import WbcPlantOpts, WbcPlantPerturb, WbcRolloutIO, WbcRolloutOpts
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.rollout import PlantSet, plant_step
    ctl = BatchedController("mini_cheetah", device=0)
    lib = ctl.lib
    nominal = load_robot("mini_cheetah")

    def create(models, mu=None):
        arr = (type(models[0]) * len(models))(*models)
        mu_a = None if mu is None else np.ascontiguousarray(mu, np.float64)
        out = C.c_void_p()
        rc = lib.wbc_plant_set_create(ctl._h, len(models), arr, None if mu_a is None else ptr(mu_a), C.byref(out))
        return rc, lib.wbc_last_error(ctl._h).decode(), out

    def broken(edit):
        ms = nominal.as_struct()
        edit(ms)
        return ms
    cases = [
        ([load_robot("mini_cheetah", "breadth_first").as_struct()], None, "v_index"),
        ([broken(lambda m: m.mass.__setitem__(4, 0.0))], None, "mass"),
        ([broken(lambda m: m.inertia_com[0].__setitem__(3, 1.0))], None, "positive definite"),
        ([broken(lambda m: m.com[2].__setitem__(1, float("nan")))], None, "finite"),
        ([broken(lambda m: m.gravity.__setitem__(2, float("inf")))], None, "finite"),
        ([nominal.as_struct()], [-0.1], "mu"),
        ([nominal.as_struct()], [float("nan")], "mu"),
    ]
    for models, mu, word in cases:
        rc, msg, out = create(models, mu)
        assert rc == 1 and word in msg and not out, (word, msg)
    ps = PlantSet(ctl, [nominal])
    n = 4
    q = np.tile(Q0, (n, 1)); v = np.zeros((n, 18)); tau = np.zeros((n, 12)); push = np.zeros((n, 8))
    with pytest.raises(RuntimeError, match="times t"):
        plant_step(ctl, q, v, tau, DT, plant_set=ps, push=push)              # a push without t
    tq, tv, ttau, tpush = (torch.from_numpy(x).cuda() for x in (q, v, tau, push))
    with pytest.raises(RuntimeError, match="times t"):
        plant_step(ctl, tq, tv, ttau, DT, plant_set=ps, push=tpush)
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 1.0, base_height=0.3))
    tt = torch.zeros(n, dtype=torch.float64, device="cuda")
    io = WbcRolloutIO(tq.data_ptr(), tv.data_ptr(), tt.data_ptr(), None, None, None, None, None, None)
    pt = WbcPlantPerturb(ps._p, None, None)
    o = WbcRolloutOpts(1, 0, WbcPlantOpts(1.0, 0.2, 30, 0), None)               # plant = 0: nothing to perturb
    assert lib.wbc_rollout_perturbed(ctl._h, 0, s._p, n, 2, DT, C.byref(io), C.byref(o), C.byref(pt), None) == 1
    assert b"plant" in lib.wbc_last_error(ctl._h)
    assert lib.wbc_rollout_perturbed(ctl._h, 0, s._p, n, 2, DT, C.byref(io), None, C.byref(pt), None) == 1     # opts are required
    if torch.cuda.device_count() > 1:                                          # a set from another device
        other = BatchedController("mini_cheetah", device=1)
        po = PlantSet(other, [nominal])
        with pytest.raises(RuntimeError, match="another device"):
            plant_step(ctl, q, v, tau, DT, plant_set=po)
        other.close(); po.close()
    s.close()
    ctl.close()                                                                # the set outlives its handle
    ps.close()
    c2 = BatchedController("mini_cheetah", device=0)
    ps2 = PlantSet(c2, [nominal], [0.5])
    qn, vn, f, st = plant_step(c2, grounded(c2, 2), np.zeros((2, 18)), np.zeros((2, 12)), DT, plant_set=ps2, variant=np.zeros(2, np.int32))
    assert (st == 0).all() and np.isfinite(qn).all()
    ps2.close(); c2.close()
