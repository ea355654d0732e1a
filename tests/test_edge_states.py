"""The control step at the edges of its input domain, against the float64 oracle: NaN / inf inputs in every block, a stance
knee swept toward its stretched (singular) pose, the approach to gimbal lock, quaternion sign and scale, and a NaN sampler
time. Every instance either agrees with the oracle at the golden bars (tau 1e-5, vd 1e-6) or carries a status bit and
returns zero torques (include/wbc.h). The first half runs the exact device source through the host warp emulator
(tests/emu), the `gpu` half the same cases through the C ABI, on every data path."""
import ctypes as C
import math
from pathlib import Path

import numpy as np
import pytest

from oracle import controllers as oc

GOLD = Path(__file__).parent / "golden"
ST_RANKDEF, ST_GIMBAL, ST_BADQUAT, ST_DIVERGED, ST_NONFINITE = 4, 8, 32, 128, 256
KINDS4 = ("id", "clf", "pc", "mptc")
ORACLE = {"id": oc.IDController, "clf": oc.CLFController, "pc": oc.PCController, "mptc": oc.MPTCController}
CASE = {"mini_cheetah": "mixed_mini_cheetah", "anymal_b": "cfg3_anymal_trot"}
# input blocks (array, slice) that may carry a NaN / inf: q quaternion, base position, joint angle; v angular, linear, joint;
# traj base position, rpy, foot position
BLOCKS = [("q", 0, 4), ("q", 4, 7), ("q", 7, 19), ("v", 0, 3), ("v", 3, 6), ("v", 6, 18),
          ("traj", 0, 3), ("traj", 9, 12), ("traj", 18, 30)]


# ------------------------------------------------------------------------------------------------------------- states
def golden_rows(robot, rows, dof_order="depth_first"):
    """q, v, traj of golden rows (all four feet in stance), joints permuted into `dof_order`."""
    from quadruped_drake_b200 import load_robot
    g = np.load(GOLD / f"{CASE[robot]}.npz")
    q, v, traj = (np.array(g[k][rows], dtype=np.float64) for k in ("q", "v", "traj"))
    if dof_order != "depth_first":
        src, dst = load_robot(robot).v_index, load_robot(robot, dof_order=dof_order).v_index
        q2, v2 = q.copy(), v.copy()
        q2[:, 1 + dst], v2[:, dst] = q[:, 1 + src], v[:, src]
        q, v = q2, v2
    return q, v, traj, np.ones((len(q), 4), np.uint8)


def poison(q, v, traj, block, which, value):
    """Copy of (q, v, traj) with one entry of `block` set to `value`."""
    q, v, traj = q.copy(), v.copy(), traj.copy()
    name, lo, hi = BLOCKS[block]
    {"q": q, "v": v, "traj": traj}[name][:, lo + which % (hi - lo)] = value
    return q, v, traj


def nonfinite_batch(robot, kinds_index, values):
    """Clean golden rows with one bad row between each pair: [c0, b0, c1, b1, ..., c_m]. Returns the batch, the bad rows'
    positions and the clean rows' positions."""
    nb = len(BLOCKS) * len(values)
    cq, cv, ct, cc = golden_rows(robot, np.arange(nb + 1) % 4)
    rows_q, rows_v, rows_t = [cq[0]], [cv[0]], [ct[0]]
    for b in range(len(BLOCKS)):
        for j, val in enumerate(values[(b + kinds_index) % len(values):] + values[:(b + kinds_index) % len(values)]):
            i = len(rows_q) // 2
            bq, bv, bt = poison(cq[i:i + 1], cv[i:i + 1], ct[i:i + 1], b, 3 * j + b, val)
            rows_q += [bq[0], cq[i + 1]]; rows_v += [bv[0], cv[i + 1]]; rows_t += [bt[0], ct[i + 1]]
    q, v, traj = np.array(rows_q), np.array(rows_v), np.array(rows_t)
    n = len(q)
    bad, good = np.arange(1, n, 2), np.arange(0, n, 2)
    return q, v, traj, np.ones((n, 4), np.uint8), bad, good


def singular_knee(robot, dof_order, q0):
    """Knee angle of leg LF at which |det| of the leg's 3x3 block of the oracle's foot Jacobian is minimal (a root of det)."""
    from scipy.optimize import brentq, minimize_scalar
    from oracle.dynamics import Plant
    from quadruped_drake_b200 import load_robot
    P, vi = Plant(robot, dof_order), load_robot(robot, dof_order=dof_order).v_index
    kq = 1 + vi[2]

    def det(th):
        q = q0.copy(); q[kq] = th
        _, J, _ = P.frame_position_quantities(q, np.zeros(18), P.foot_frames[0])
        return np.linalg.det(J[:, vi[:3]])
    th = minimize_scalar(lambda t: abs(det(t)), bounds=(-0.6, 0.6), method="bounded", options={"xatol": 1e-12}).x
    if det(th - 1e-3) * det(th + 1e-3) < 0:
        th = brentq(det, th - 1e-3, th + 1e-3, xtol=1e-300, rtol=1e-15)
    assert abs(det(th)) < 1e-15
    return kq, th


def knee_sweep(robot, dof_order, offsets):
    q0, v0, t0, c0 = golden_rows(robot, [0], dof_order)
    kq, th = singular_knee(robot, dof_order, q0[0])
    side = 1.0 if q0[0, kq] >= th else -1.0                      # approach from the side of the golden posture
    n = len(offsets)
    q, v, traj, contact = np.repeat(q0, n, 0), np.repeat(v0, n, 0), np.repeat(t0, n, 0), np.repeat(c0, n, 0)
    q[:, kq] = th + side * np.asarray(offsets)
    return q, v, traj, contact


def gimbal_states(cps):
    q0, v0, t0, c0 = golden_rows("mini_cheetah", [0])
    n = len(cps)
    q, v, traj, contact = np.repeat(q0, n, 0), np.repeat(v0, n, 0), np.repeat(t0, n, 0), np.repeat(c0, n, 0)
    for i, cp in enumerate(cps):
        p = math.acos(cp)
        q[i, 0:4] = [math.cos(p / 2), 0.0, math.sin(p / 2), 0.0]
    v[:, 0:3] = [2e-4, 0.3, -0.2]                                # roll rate: rpyd[0] = (cy wx + sy wy) / cos(pitch)
    return q, v, traj, contact


QUAT_SCALES = (1e-140, 1e-3, 3.0, 1e140)
QUAT_BAD = (1e-151, 1e151)                                        # |q|^2 outside (1e-300, 1e300)


def quat_states():
    q0, v0, t0, c0 = golden_rows("mini_cheetah", [5])
    q0[0, 0:4] /= np.linalg.norm(q0[0, 0:4])
    scales = (1.0, -1.0) + QUAT_SCALES + QUAT_BAD
    n = len(scales)
    q = np.repeat(q0, n, 0)
    q[:, 0:4] *= np.asarray(scales)[:, None]
    return q, np.repeat(v0, n, 0), np.repeat(t0, n, 0), np.repeat(c0, n, 0)


# ---------------------------------------------------------------------------------------------------------- checks
def oracle_out(robot, dof_order, kind, q, v, traj, contact):
    ref = ORACLE[kind](robot, dof_order)
    return [ref.control_law(q[i], v[i], oc.traj_to_dict(traj[i], contact[i])) for i in range(len(q))]


def check_nonfinite(out, ref, bad, good):
    """Bad rows: NONFINITE and zero outputs; clean rows: the bits of the batch without the bad rows."""
    st = np.asarray(out.status)
    assert (st[bad] & ST_NONFINITE).all(), st[bad]
    for name in ("tau", "f", "vd", "lam"):
        arr = np.asarray(getattr(out, name))
        assert (arr[bad] == 0).all(), name
    assert (st[good] == np.asarray(ref.status)).all()
    for name in ("tau", "metrics", "status", "f", "vd", "lam", "qp_info"):
        assert np.array_equal(np.asarray(getattr(out, name))[good], np.asarray(getattr(ref, name))), name


def check_against_oracle(out, oracle, must_solve=None, flag=ST_RANKDEF, tau_bar=1e-5, vd_bar=1e-6):
    """Each instance passes the golden bars or is flagged `flag` with zero torques; returns the solved mask."""
    st, tau, vd = np.asarray(out.status), np.asarray(out.tau), np.asarray(out.vd)
    solved = st == 0
    for i, o in enumerate(oracle):
        if solved[i]:
            assert o.status == "optimal", (i, o.status)
            assert np.abs(tau[i] - o.tau).max() < tau_bar, (i, np.abs(tau[i] - o.tau).max())
            assert np.abs(vd[i] - o.vd).max() < vd_bar, (i, np.abs(vd[i] - o.vd).max())
        else:
            assert st[i] & flag and (tau[i] == 0).all() and (vd[i] == 0).all(), (i, st[i])
    if must_solve is not None:
        assert solved[must_solve].all(), st
    return solved


# ------------------------------------------------------------------------------------------------------ CPU: emulator
class EmuOut:
    def __init__(self, **kw):
        self.__dict__.update(kw)


@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu.so"))
    lib.emu_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
    lib.emu_plant_step.argtypes = [C.c_void_p, C.c_longlong, C.c_double, C.c_double, C.c_double, C.c_int] + [C.c_void_p] * 5
    return lib


def emu_step(emu, robot, kind, q, v, traj, contact, dof_order="depth_first"):
    from quadruped_drake_b200 import load_robot
    from quadruped_drake_b200.capi import KINDS, WbcIO, make_params, np_ptr
    ms, pr = load_robot(robot, dof_order=dof_order).as_struct(), make_params()
    q, v, traj, contact = (np.ascontiguousarray(x) for x in (q, v, traj, contact))
    n = len(q)
    o = EmuOut(tau=np.zeros((n, 12)), metrics=np.zeros((n, 4)), status=np.zeros(n, np.int32), vd=np.zeros((n, 18)),
               f=np.zeros((n, 4, 3)), qp_info=np.zeros((n, 4)), lam=np.zeros((n, 42)))
    io = WbcIO(*(np_ptr(x) for x in (q, v, traj, contact, o.tau, o.metrics, o.status, o.vd, o.f, o.qp_info, o.lam)))
    assert emu.emu_step(C.byref(ms), C.byref(pr), KINDS[kind], n, C.byref(io)) == 0
    return o


@pytest.mark.parametrize("ki,kind", list(enumerate(KINDS4)))
def test_emulated_nonfinite_inputs_are_flagged_and_zeroed(emu, ki, kind):
    """One bad value per input block (NaN or +-inf, rotating over the kinds) between clean neighbours."""
    q, v, traj, contact, bad, good = nonfinite_batch("mini_cheetah", ki, [np.nan] if ki % 2 == 0 else [np.inf if ki == 1 else -np.inf])
    out = emu_step(emu, "mini_cheetah", kind, q, v, traj, contact)
    ref = emu_step(emu, "mini_cheetah", kind, q[good[:4]], v[good[:4]], traj[good[:4]], contact[good[:4]])   # golden rows 0-3
    reps = EmuOut(**{k: np.asarray(getattr(ref, k))[np.arange(len(good)) % 4] for k in ("tau", "metrics", "status", "f", "vd", "lam", "qp_info")})
    check_nonfinite(out, reps, bad, good)


@pytest.mark.parametrize("robot,dof_order", [("mini_cheetah", "depth_first"), ("anymal_b", "breadth_first")])
def test_emulated_stretched_stance_knee(emu, robot, dof_order):
    """LF knee swept toward its singular angle in stance: golden bars or RANKDEF with zero torques; the exact angle is flagged."""
    offsets = [1e-1, 1e-2, 5e-3, 1e-3, 1e-4, 1e-6, 1e-9, 1e-12, 0.0]
    q, v, traj, contact = knee_sweep(robot, dof_order, offsets)
    for kind in ("id", "clf", "pc"):
        out = emu_step(emu, robot, kind, q, v, traj, contact, dof_order)
        check_against_oracle(out, oracle_out(robot, dof_order, kind, q, v, traj, contact), must_solve=[0, 1, 2])
        assert out.status[-1] & ST_RANKDEF and out.status[-2] & ST_RANKDEF, out.status


def test_emulated_gimbal_approach(emu):
    cps = [1e-2, 1e-4, 1e-5, 3e-6, 1.5e-6, 1.01e-6, 0.99e-6]
    q, v, traj, contact = gimbal_states(cps)
    out = emu_step(emu, "mini_cheetah", "id", q, v, traj, contact)
    ora = oracle_out("mini_cheetah", "depth_first", "id", q[:-1], v[:-1], traj[:-1], contact[:-1])
    sub = EmuOut(status=out.status[:-1], tau=out.tau[:-1], vd=out.vd[:-1])
    check_against_oracle(sub, ora, must_solve=list(range(len(cps) - 1)))
    assert out.status[-1] == ST_GIMBAL and (out.tau[-1] == 0).all()


def test_emulated_quaternion_sign_and_scale(emu):
    q, v, traj, contact = quat_states()
    check_quaternion(emu_step(emu, "mini_cheetah", "id", q, v, traj, contact))


def check_quaternion(out):
    for name in ("tau", "metrics", "status", "f", "vd", "lam", "qp_info"):
        a = np.asarray(getattr(out, name))
        assert np.array_equal(a[1], a[0]), name                 # -q: the same rotation, the same bits
    st, tau, vd = (np.asarray(x) for x in (out.status, out.tau, out.vd))
    assert st[0] == 0
    for i in range(2, 2 + len(QUAT_SCALES)):
        assert st[i] == 0, (i, st[i])
        assert np.abs(tau[i] - tau[0]).max() < 1e-8 * np.abs(tau[0]).max(), i
        assert np.abs(vd[i] - vd[0]).max() < 1e-8 * np.abs(vd[0]).max(), i
    for i in range(2 + len(QUAT_SCALES), len(st)):
        assert st[i] & ST_BADQUAT and (tau[i] == 0).all(), (i, st[i])


def test_emulated_plant_freezes_nan_torque(emu):
    """A NaN torque (what the PD law returns for a NaN state) reaching the ground plant freezes the robot as DIVERGED."""
    from quadruped_drake_b200 import load_robot
    from quadruped_drake_b200.capi import np_ptr
    q, v, _, _ = golden_rows("mini_cheetah", [0, 1])
    tau = np.zeros((2, 12)); tau[1, 4] = np.nan
    f, st = np.zeros((2, 4, 3)), np.zeros(2, np.int32)
    q0, v0 = q.copy(), v.copy()
    assert emu.emu_plant_step(C.byref(load_robot("mini_cheetah").as_struct()), 2, 5e-3, 1.0, 0.2, 30,
                              np_ptr(q), np_ptr(v), np_ptr(tau), np_ptr(f), np_ptr(st)) == 0
    assert st[0] == 0 and st[1] & ST_DIVERGED
    assert np.isfinite(q).all() and np.isfinite(v).all() and np.array_equal(q[1], q0[1]) and np.array_equal(v[1], v0[1])


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctl_cache(built):
    from quadruped_drake_b200.controller import BatchedController
    cache = {}

    def get(robot="mini_cheetah", dof_order="depth_first"):
        if (robot, dof_order) not in cache:
            cache[(robot, dof_order)] = BatchedController(robot, device=0, dof_order=dof_order)
        return cache[(robot, dof_order)]
    yield get
    for c in cache.values():
        c.close()


def pinned_io(capi, q, v, traj, contact):
    n = len(q)
    h = {k: capi.pinned_empty(s) for k, s in (("q", (n, 19)), ("v", (n, 18)), ("traj", (n, 54)), ("tau", (n, 12)),
                                                ("metrics", (n, 4)), ("vd", (n, 18)), ("f", (n, 4, 3)), ("qp_info", (n, 4)),
                                                ("lam", (n, 42)))}
    h["contact"], h["status"] = capi.pinned_empty((n, 4), np.uint8), capi.pinned_empty((n,), np.int32)
    h["q"][:], h["v"][:], h["traj"][:], h["contact"][:] = q, v, traj, contact
    io = capi.WbcIO(*(capi.np_ptr(h[k]) for k in ("q", "v", "traj", "contact", "tau", "metrics", "status", "vd", "f", "qp_info", "lam")))
    return io, EmuOut(**h)                                       # keeps the page-locked inputs alive too


def to_np(out):
    return EmuOut(**{k: (getattr(out, k).cpu().numpy() if hasattr(getattr(out, k), "cpu") else np.asarray(getattr(out, k)))
                     for k in ("tau", "metrics", "status", "vd", "f", "qp_info", "lam")})


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS4)
def test_nonfinite_inputs_every_data_path(ctl_cache, kind):
    """A NaN and a +-inf in every input block: NONFINITE and zero outputs, clean neighbours unchanged, through wbc_step on
    device pointers (small, and 65536 instances with the bad rows in the last chunk), wbc_step_host on pageable buffers and
    on page-locked buffers below and above 24576 instances."""
    import torch
    from quadruped_drake_b200 import capi
    ctl = ctl_cache()
    k = capi.KINDS[kind]
    q, v, traj, contact, bad, good = nonfinite_batch("mini_cheetah", 0, [np.nan, np.inf, -np.inf])
    ref = ctl.step(kind, q[good], v[good], traj[good], contact[good], debug=True)
    check_nonfinite(ctl.step(kind, q, v, traj, contact, debug=True), ref, bad, good)     # pageable host buffers
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    out = to_np(ctl.step(kind, t(q), t(v), t(traj), t(contact), debug=True))
    torch.cuda.synchronize()
    check_nonfinite(out, ref, bad, good)
    for n in (65536, 24581, 1024):
        cq, cv, ct, cc = golden_rows("mini_cheetah", np.arange(n) % 256)
        m = len(q)
        cq[n - m:], cv[n - m:], ct[n - m:] = q, v, traj              # the bad rows sit in the last chunk
        sel_bad, sel_good = n - m + bad, np.r_[np.arange(n - m), n - m + good]
        cref = ctl.step(kind, cq[sel_good], cv[sel_good], ct[sel_good], cc[sel_good], debug=True)
        if n == 65536:
            got = to_np(ctl.step(kind, t(cq), t(cv), t(ct), t(cc), debug=True))
            torch.cuda.synchronize()
        else:
            io, got = pinned_io(capi, cq, cv, ct, cc)
            assert ctl.lib.wbc_step_host(ctl._h, k, n, C.byref(io)) == 0
        check_nonfinite(got, cref, sel_bad, sel_good)


@pytest.mark.gpu
def test_nonfinite_plan_multi_and_mirror(ctl_cache):
    """wbc_step_plan_host, wbc_multi_step_host on [0, 0] and the LeafSystem mirror (which raises on any status)."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import IDController
    from quadruped_drake_b200.sharding import MultiGpuController
    ctl = ctl_cache()
    q, v, traj, contact, bad, good = nonfinite_batch("mini_cheetah", 0, [np.nan, np.inf])
    bh = float(ctl.model.nominal_q()[6])
    s = pl.TrajectorySampler(ctl, [pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh)])
    n = len(q)
    tt = np.linspace(0.5, 5.5, n)
    qp, vp = q.copy(), v.copy()
    tb = bad[len(bad) // 2]
    qp[bad], vp[bad] = np.where(np.isfinite(q[bad]), q[bad], np.nan), v[bad]      # state blocks only: traj comes from the plan
    for i in bad:
        if np.isfinite(qp[i]).all() and np.isfinite(vp[i]).all():
            qp[i, 9] = np.nan
    tt[tb] = np.nan                                                              # a NaN time alone is clamped, not failed
    qp[tb], vp[tb] = q[good[0]], v[good[0]]
    fail = np.setdiff1d(bad, [tb])
    a = ctl.step_plan("clf", s, qp, vp, tt)
    o = s.sample(np.where(np.isnan(tt), 0.0, tt))
    r = ctl.step("clf", qp, vp, o["traj"], o["contact"])
    assert (a.status[fail] & ST_NONFINITE).all() and (a.tau[fail] == 0).all()
    assert np.array_equal(a.tau[good], r.tau[good]) and np.array_equal(a.status[good], r.status[good])
    assert np.array_equal(a.tau[tb], r.tau[tb])
    multi = MultiGpuController("mini_cheetah", devices=[0, 0])
    try:
        buf = multi.pinned(n)
        buf["q"][:], buf["v"][:], buf["traj"][:], buf["contact"][:] = q, v, traj, contact
        m = multi.step("pc", buf["q"], buf["v"], buf["traj"], buf["contact"], buf["tau"], buf["metrics"], buf["status"])
        ref = ctl.step("pc", q[good], v[good], traj[good], contact[good])
        st, tau = np.asarray(m.status), np.asarray(m.tau)
        assert (st[bad] & ST_NONFINITE).all() and (tau[bad] == 0).all()
        assert np.array_equal(tau[good], ref.tau) and np.array_equal(st[good], ref.status)
    finally:
        multi.close()
    mirror = IDController("mini_cheetah", 5e-3)
    ctx = mirror.CreateDefaultContext()
    x = np.hstack([q[0], v[0]]); x[19 + 10] = np.nan                           # a NaN joint velocity
    ctx.FixValue(0, x)
    ctx.FixValue(1, oc.standing_dict())
    with pytest.raises(AssertionError):
        mirror.EvalOutput(ctx, 0)


@pytest.mark.gpu
def test_pd_law_keeps_nan_and_plant_freezes(ctl_cache):
    """The PD law has no status: a NaN input gives a NaN torque, as np.clip does in the reference, and the ground plant then
    freezes the robot as DIVERGED."""
    from quadruped_drake_b200 import capi
    ctl = ctl_cache()
    q, v, _, _ = golden_rows("mini_cheetah", np.arange(4))
    q[1, 7:] += 10.0                                                          # clipped at +-150
    v[2, 8] = np.nan
    q[3, 12] = -np.inf
    tau = ctl.step_pd(q, v)
    ref = oc.BasicController("mini_cheetah")
    for i in range(4):
        r = ref.control_law(q[i], v[i])
        # the reference's S.T product spreads a NaN / inf input over all twelve outputs (0 * NaN, 0 * inf); the kernel keeps
        # it on its own joint: every NaN of the kernel is one of the reference, every finite reference value is matched
        assert not (np.isnan(tau[i]) & ~np.isnan(r)).any(), i
        fin = np.isfinite(r)
        assert not fin.any() or np.abs(tau[i][fin] - r[fin]).max() < 1e-12, i
    assert np.isnan(tau[2]).sum() == 1 and np.abs(tau[1]).max() == 150.0
    n = 4
    po = capi.WbcPlantOpts()
    assert ctl.lib.wbc_default_plant_opts(C.byref(po)) == 0
    qq, vv, st = np.ascontiguousarray(q.copy()), np.ascontiguousarray(v.copy()), np.zeros(n, np.int32)
    vv[2, 8] = 0.0; qq[3, 12] = 0.0                                           # a finite state driven by the NaN torques
    tt = np.ascontiguousarray(tau)
    rc = ctl.lib.wbc_plant_step_host(ctl._h, n, 5e-3, C.byref(po), capi.np_ptr(qq), capi.np_ptr(vv),
                                     capi.np_ptr(tt), None, None, capi.np_ptr(st), None)
    assert rc == 0
    assert st[2] & ST_DIVERGED and not st[0] & ST_DIVERGED, st                  # row 3's -inf angle is clipped to +-150
    assert np.isfinite(qq).all() and np.isfinite(vv).all()


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["mini_cheetah", "anymal_b"])
@pytest.mark.parametrize("dof_order", ["depth_first", "breadth_first"])
def test_stretched_stance_knee(ctl_cache, robot, dof_order):
    """12 decades toward the singular knee angle (plus the exact angle), ID / CLF / PC: golden bars for every unflagged
    instance (and, for ID / CLF, which tests/kkt.py certifies, a KKT point of the reference QP), RANKDEF with zero torques
    otherwise."""
    from test_gpu_parity import assert_optimal
    offsets = [10.0 ** -e for e in range(1, 13)] + [5e-3, 3e-3, 2e-3, 0.0]
    q, v, traj, contact = knee_sweep(robot, dof_order, offsets)
    ctl = ctl_cache(robot, dof_order)
    for kind in ("id", "clf", "pc"):
        out = ctl.step(kind, q, v, traj, contact, debug=True)
        solved = check_against_oracle(out, oracle_out(robot, dof_order, kind, q, v, traj, contact), must_solve=[0, 1, 12])
        assert out.status[-1] & ST_RANKDEF
        if kind != "pc":
            assert_optimal(kind, ctl, q, v, traj, contact, out, sel=solved)


@pytest.mark.gpu
def test_gimbal_and_quaternion_edges(ctl_cache):
    ctl = ctl_cache()
    cps = [1e-2, 1e-3, 1e-4, 1e-5, 3e-6, 1.5e-6, 1.01e-6, 0.99e-6]
    q, v, traj, contact = gimbal_states(cps)
    for kind in ("id", "clf", "pc"):
        out = ctl.step(kind, q, v, traj, contact, debug=True)
        sub = EmuOut(status=out.status[:-1], tau=out.tau[:-1], vd=out.vd[:-1])
        check_against_oracle(sub, oracle_out("mini_cheetah", "depth_first", kind, q[:-1], v[:-1], traj[:-1], contact[:-1]),
                             must_solve=list(range(len(cps) - 1)))
        assert out.status[-1] & ST_GIMBAL and (out.tau[-1] == 0).all()
    q, v, traj, contact = quat_states()
    for kind in KINDS4:
        check_quaternion(ctl.step(kind, q, v, traj, contact, debug=True))


@pytest.mark.gpu
def test_sampler_nan_time_is_clamped(ctl_cache):
    """A NaN plan time is flagged WBC_TRAJ_CLAMPED and evaluated at t = 0, in continuous mode and in grid mode."""
    from quadruped_drake_b200 import planner as pl
    ctl = ctl_cache()
    cont = pl.TrajectorySampler(ctl, [pl.make_gait_plan("mini_cheetah", 1)])
    grid = pl.TowrTrunkPlanner(ctl, robot="mini_cheetah", gait="trot")
    for s in (cont, grid):
        t = np.array([0.7, np.nan, 0.0, 1.3])
        a = s.sample(t)
        st = np.asarray(a["status"]) if "status" in a else None
        assert st is not None and st[1] & 1 and not st[0] & 1
        for key in ("traj", "contact", "t_eval"):
            arr = np.asarray(a[key])
            assert np.array_equal(arr[1], arr[2]), key
