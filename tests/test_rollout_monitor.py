"""Rollout monitor of the ground-plant loop (wbc_rollout_monitor[_host], wbc_monitor_step[_host]; include/wbc.h, wbc_monitor).

CPU half: the numpy restatement oracle/monitor.py against known answers, and the monitor of csrc/wbc_monitor.cuh on the host
(tests/emu/emu_monitor.cpp) against the oracle.
GPU half: mon == NULL is wbc_rollout_loop; a monitor leaves every existing output alone; the fused rollout equals a manual loop
of 1-step rollouts and wbc_monitor_step, and the oracle on that loop's records; continuation and permutation; free fall, pushes
and a bad parameter index; the end-state verdict of the tools; argument errors."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from oracle import monitor as om
from oracle.dynamics import rpy_matrix

GOLD = Path(__file__).parent / "golden"
KIND_NAMES = ["id", "clf", "pc", "mptc", "pd"]
P = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731


# ------------------------------------------------------------------------------------------------------------------ CPU half
def test_oracle_reference_quaternion_matches_rpy_matrix():
    rng = np.random.default_rng(0)
    rpy = np.concatenate([rng.uniform(-np.pi, np.pi, (200, 3)), [[0.0, 0.0, 0.0], [0.0, np.pi / 2 - 1e-9, 0.0], [np.pi, 0.0, -np.pi]]])
    for r, q in zip(rpy, om.rpy_quat(rpy)):
        assert abs(np.linalg.norm(q) - 1.0) < 1e-15
        assert np.abs(om.quat_matrix(q) - rpy_matrix(r)).max() < 1e-14


def axis_angle(axis, angle):
    return np.concatenate([[np.cos(0.5 * angle)], np.sin(0.5 * angle) * axis / np.linalg.norm(axis)])


def test_oracle_orientation_error_of_known_rotations():
    """q = q_ref (x) rot(axis, angle) about random axes, at scaled quaternions of either sign: e_theta is the angle."""
    rng = np.random.default_rng(1)
    for angle in [0.0, 1e-8, 1e-3, 0.3, 1.0, 2.5, np.pi - 1e-6]:
        for _ in range(20):
            rpy = rng.uniform(-1.2, 1.2, 3)
            q = np.zeros(19)
            q[:4] = om.quat_mul(om.rpy_quat(rpy), axis_angle(rng.normal(size=3), angle)) * rng.choice([-1.0, 1.0]) * rng.uniform(0.5, 2)
            traj = np.zeros(54)
            traj[9:12] = rpy
            ep, eth = om.errors(q, traj)
            assert ep[0] == 0.0
            assert abs(eth[0] - angle) < 1e-14 and abs(eth[0] - angle) <= 1e-6 * angle + 1e-15, (angle, eth[0])


def model_maps(robot="mini_cheetah", order="depth_first"):
    from quadruped_drake_b200.model import load_robot
    m = load_robot(robot, order)
    return np.ascontiguousarray(m.v_index, np.int32), np.ascontiguousarray(m.act_index, np.int32), np.ascontiguousarray(m.effort)


def standing_traj(n, z=0.3):
    traj = np.zeros((n, 54))
    traj[:, 2] = z
    return traj


def standing_q(n, z=0.3):
    q = np.zeros((n, 19))
    q[:, 0], q[:, 6] = 1.0, z
    return q


def test_oracle_constant_torque_and_velocity_give_the_closed_forms():
    vi, ai, eff = model_maps("anymal_b", "breadth_first")
    rng = np.random.default_rng(2)
    n, k, dt = 5, 37, 2e-3
    tau, v = rng.normal(0, 20, (n, 12)), rng.normal(0, 1, (n, 18))
    st = om.State(n)
    for _ in range(k):
        om.step(st, dt, 0.05, 0.3, vi, ai, eff, standing_q(n), v, standing_traj(n), np.ones((n, 4)), tau, np.zeros((n, 12)))
    assert np.allclose(st.stats[:, om.TAU2_DT], k * dt * (tau ** 2).sum(1), rtol=1e-13)
    assert np.allclose(st.stats[:, om.WORK_ABS], k * dt * np.abs(tau[:, ai] * v[:, vi]).sum(1), rtol=1e-13)
    assert np.allclose(st.stats[:, om.DIST_XY], k * dt * np.hypot(v[:, 3], v[:, 4]), rtol=1e-13)
    assert np.array_equal(st.stats[:, om.SAT_MAX], (np.abs(tau[:, ai]) / eff).max(1))
    assert (st.steps == k).all() and (st.fail_step == 0).all() and (st.stats[:, [0, 1, 2, 3]] == 0).all()


def test_oracle_contact_counters():
    vi, ai, eff = model_maps()
    f = np.zeros((3, 4, 3))
    f[0, 0] = [0.0, 0.0, 50.0]; f[0, 1] = [1e-300, 0.0, 0.0]; f[0, 2] = [-0.0, 0.0, -0.0]; f[0, 3] = [3.0, 4.0, 12.0]
    f[1, :, 2] = 20.0
    contact = np.array([[1, 0, 1, 0], [0, 0, 0, 0], [1, 1, 1, 1]], np.uint8)
    st = om.State(3)
    for _ in range(2):
        om.step(st, 1e-3, 0.05, 0.3, vi, ai, eff, standing_q(3), np.zeros((3, 18)), standing_traj(3), contact, np.zeros((3, 12)),
                f.reshape(3, 12))
    assert list(st.stats[:, om.STANCE_UNLOADED]) == [2.0, 0.0, 8.0]     # robot 0: foot 2 (-0 counts as 0); robot 2: all four
    assert list(st.stats[:, om.SWING_LOADED]) == [4.0, 8.0, 0.0]        # robot 0: feet 1 (1e-300) and 3
    assert list(st.stats[:, om.F_MAX]) == [50.0, 20.0, 0.0]


def test_oracle_bookkeeping():
    """fail_step / fail_why are written once; why follows the latest step; a NaN state fails POS and ANG; +inf never fails."""
    vi, ai, eff = model_maps()
    n = 4
    st = om.State(n)
    z = np.zeros((n, 12))

    def step(q, status=None, pos_max=0.05, ang_max=0.3):
        om.step(st, 5e-3, pos_max, ang_max, vi, ai, eff, q, np.zeros((n, 18)), standing_traj(n), np.ones((n, 4)), z, z, status)

    step(standing_q(n))
    assert (st.why == 0).all() and (st.fail_step == 0).all()
    q = standing_q(n)
    q[0, 6] += 0.06                              # robot 0: POS
    q[1, :4] = axis_angle(np.array([1.0, 1.0, 0.0]), 0.31)     # robot 1: ANG
    q[3, :] = np.nan                             # robot 3: POS | ANG
    step(q, status=np.array([0, 0, 8, 0]))       # robot 2: STATUS
    assert list(st.fail_step) == [2, 2, 2, 2] and list(st.fail_why) == [1, 2, 4, 3] and list(st.why) == [1, 2, 4, 3]
    q2 = standing_q(n)
    q2[2, 6] += 1.0
    step(q2)
    assert list(st.fail_step) == [2, 2, 2, 2] and list(st.fail_why) == [1, 2, 4, 3] and list(st.why) == [0, 0, 1, 0]
    assert np.isnan(st.stats[3, om.SUM_POS2]) and st.stats[3, om.MAX_POS] == 0.0        # NaN is never a maximum
    fresh = om.State(n)
    om.step(fresh, 5e-3, np.inf, np.inf, vi, ai, eff, q, np.zeros((n, 18)), standing_traj(n), np.ones((n, 4)), z, z)
    assert list(fresh.why) == [0, 0, 0, 3] and list(fresh.fail_step) == [0, 0, 0, 1]   # inf bounds: only NaN still fails


@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_monitor.so"))
    lib.emu_monitor_step.argtypes = [C.c_longlong, C.c_double, C.c_double, C.c_double] + [C.c_void_p] * 15
    return lib


def emu_step(emu, st, dt, pos_max, ang_max, maps, q, v, traj, contact, tau, f, status=None):
    vi, ai, eff = maps
    args = [np.ascontiguousarray(x) for x in (q, v, traj, contact.astype(np.uint8), tau, f)]
    emu.emu_monitor_step(len(q), dt, pos_max, ang_max, P(vi), P(ai), P(eff), P(st.stats), P(st.steps), P(st.fail_step), P(st.fail_why),
                         P(st.why), *map(P, args), P(None if status is None else np.ascontiguousarray(status, np.int32)))


def random_records(rng, n, golden):
    g = np.load(GOLD / f"{golden}.npz")
    q, v, traj = (np.ascontiguousarray(np.resize(g[k], (n, g[k].shape[1]))) for k in ("q", "v", "traj"))
    q = q.copy()
    q[:, 4:7] = traj[:, 0:3] + rng.normal(0, 0.012, (n, 3))
    q[:, :4] *= rng.uniform(0.8, 1.2, (n, 1))
    contact = (rng.random((n, 4)) < 0.6).astype(np.uint8)
    f = rng.normal(0, 30, (n, 12)) * (rng.random((n, 4, 1)) < 0.5).repeat(3, 2).reshape(n, 12)
    tau = rng.normal(0, 15, (n, 12))
    status = np.where(rng.random(n) < 0.05, 1 << rng.integers(0, 12, n), 0).astype(np.int32)
    return q, v, traj, contact, tau, f, status


@pytest.mark.parametrize("robot,order,golden", [("mini_cheetah", "depth_first", "cfg4_mini_cheetah_walk"),
                                                ("mini_cheetah", "breadth_first", "cfg2_mini_cheetah_stand"),
                                                ("anymal_b", "depth_first", "cfg3_anymal_trot"),
                                                ("anymal_b", "breadth_first", "tl_anymal_trot")])
def test_emulated_monitor_matches_oracle(emu, robot, order, golden):
    """30 steps of 200 robots: counters, reasons, steps and fail_step exact; stats within 1e-13 relative."""
    maps = model_maps(robot, order)
    rng = np.random.default_rng(3)
    n = 200
    a, b = om.State(n), om.State(n)
    for k in range(30):
        q, v, traj, contact, tau, f, status = random_records(rng, n, golden)
        if k == 7:
            q[5] = np.nan
        om.step(a, 5e-3, 0.05, 0.3, *maps, q, v, traj, contact, tau, f, status)
        emu_step(emu, b, 5e-3, 0.05, 0.3, maps, q, v, traj, contact, tau, f, status)
        for key in ("steps", "fail_step", "fail_why", "why"):
            assert np.array_equal(getattr(a, key), getattr(b, key)), (k, key)
        for c in (om.STANCE_UNLOADED, om.SWING_LOADED):
            assert np.array_equal(a.stats[:, c], b.stats[:, c])
        ok = np.isfinite(a.stats)
        assert np.array_equal(ok, np.isfinite(b.stats))
        assert np.abs(a.stats[ok] - b.stats[ok]).max() <= 1e-13 * max(1.0, np.abs(a.stats[ok]).max())
        rel = np.abs(a.stats - b.stats) / np.maximum(np.abs(a.stats), 1e-300)
        assert (rel[ok] <= 1e-13).all()
    assert 0 < (a.fail_step > 0).sum() < n


# ------------------------------------------------------------------------------------------------------------------ GPU half
gpu = pytest.mark.gpu
Q0 = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4)
NOISE = np.array([0.01, 0.002, 0.01, 0.05, 0.02, 0.1])
MON_KEYS = ("stats", "steps", "fail_step", "fail_why")
ROLL_KEYS = ("q", "v", "t", "tau", "metrics", "status_or", "err_max", "f_contact")


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


def standing_sampler(ctl, bh=None):
    from quadruped_drake_b200 import planner as pl
    bh = float(grounded(ctl, 1, np.random.default_rng(0), 0.0)[0, 6]) if bh is None else bh
    return pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh))


@pytest.fixture(scope="module")
def world(ctl):
    """Variants, pushes, terrain and parameter sets of a 256-robot trotting robustness rollout, with a noisy delayed loop."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.capi import DEFAULT_PARAMS
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import PlantSet, Terrain, TerrainSet
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
    w = dict(q0=grounded(ctl, n, rng, 0.02), s=s, n=n,
             kw=dict(plant_set=ps, terrain_set=ts, param_set=pset, variant=(np.arange(n) % 2).astype(np.int32), push=push,
                     terrain=(np.arange(n) // 2 % 2).astype(np.int32), param_index=rng.integers(0, 4, n).astype(np.int32)))
    yield w
    pset.close(); ts.close(); ps.close(); s.close()


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
def test_null_monitor_is_rollout_loop(ctl, world):
    """wbc_rollout_monitor_host with mon == NULL: the bits and launch count of wbc_rollout_loop_host, all five kinds, with
    variants, pushes, terrain, parameter sets and a loop."""
    from quadruped_drake_b200.capi import WbcPlantOpts, WbcRolloutIO, WbcRolloutOpts
    n, steps = 64, 40
    rows = np.arange(n)
    q0, s, kw = world["q0"][:n], world["s"], world["kw"]
    pt, tr, cp, lp, keep = c_structs(kw, noisy_loop(world["n"], np.random.default_rng(5)), rows)
    for k, kind in enumerate(KIND_NAMES):
        outs, counts = [], []
        for fn, extra in (("wbc_rollout_loop_host", ()), ("wbc_rollout_monitor_host", (None,))):
            q, v, t = q0.copy(), np.zeros((n, 18)), np.zeros(n)
            r = [np.zeros((n, 12)), np.zeros((n, 4)), np.zeros(n, np.int32), np.zeros(n), np.zeros((steps, n, 4)), np.zeros((n, 12))]
            io = WbcRolloutIO(P(q), P(v), P(t), None, *map(P, r[:5]))
            o = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), P(r[5]))
            l0 = ctl.launches
            ctl._check(getattr(ctl.lib, fn)(ctl._h, k, s._p, n, steps, 5e-3, C.byref(io), C.byref(o), C.byref(pt), C.byref(tr),
                                            C.byref(cp), C.byref(lp), *extra), fn)
            counts.append(ctl.launches - l0)
            outs.append([q, v, t] + r)
        assert counts[0] == counts[1], kind
        for a, b in zip(*outs):
            assert np.array_equal(a, b), kind


@gpu
@pytest.mark.parametrize("kind", KIND_NAMES)
def test_monitor_leaves_every_output_alone(ctl, world, kind):
    """With a monitor every existing output has the bits of the run without one, with one more launch per step; graph replay,
    plain launches and the host entry give the same monitor state. Without f_contact and status_or (the library's scratch path)
    the monitor state is the same too."""
    import torch
    from quadruped_drake_b200.capi import WbcMonitor, WbcPlantOpts, WbcRolloutIO, WbcRolloutOpts
    from quadruped_drake_b200.rollout import Monitor, rollout
    n, steps, dt = world["n"], 150, 5e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    loop = noisy_loop(n, np.random.default_rng(6))
    l0 = ctl.launches
    ref = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, log_metrics=True, loop=loop, **kw)
    l1 = ctl.launches
    got = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, log_metrics=True, loop=loop, monitor=Monitor(), **kw)
    l2 = ctl.launches
    assert l2 - l1 == (l1 - l0) + steps
    for key in ROLL_KEYS + ("metrics_log",):
        assert np.array_equal(getattr(got, key), getattr(ref, key)), (kind, key)
    m = got.monitor
    assert (m.steps == steps).all() and np.isfinite(m.stats).all()
    assert np.array_equal(m.fail_why[m.fail_step == 0], np.zeros((m.fail_step == 0).sum(), np.int32))
    for graph in (True, False):
        q, v, t = (torch.from_numpy(x.copy()).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
        with torch.cuda.stream(torch.cuda.Stream()):
            r = rollout(ctl, s, kind, q, v, t, steps, dt, plant=True, use_graph=graph, loop=dev_loop(loop), monitor=Monitor(), **to_dev(kw))
        torch.cuda.synchronize()
        for key in ROLL_KEYS:
            assert np.array_equal(np_of(getattr(r, key)), getattr(ref, key)), (kind, graph, key)
        for key in MON_KEYS:
            assert np.array_equal(np_of(getattr(r.monitor, key)), getattr(m, key)), (kind, graph, key)
        assert np.array_equal(np_of(r.why), got.why)
    # the scratch path: no f_contact, no status_or, no why
    pt, tr, cp, lp, keep = c_structs(kw, loop, np.arange(n))
    q, v, t = q0.copy(), np.zeros((n, 18)), np.zeros(n)
    io = WbcRolloutIO(P(q), P(v), P(t), None, None, None, None, None, None)
    o = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    stats, st_, fs, fw = np.zeros((n, 11)), np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int32)
    mo = WbcMonitor(0.05, 0.3, P(stats), P(st_), P(fs), P(fw), None)
    ctl._check(ctl.lib.wbc_rollout_monitor_host(ctl._h, KIND_NAMES.index(kind), s._p, n, steps, dt, C.byref(io), C.byref(o), C.byref(pt),
                                                C.byref(tr), C.byref(cp), C.byref(lp), C.byref(mo)), "wbc_rollout_monitor_host")
    assert np.array_equal(q, ref.q)
    for key, x in zip(MON_KEYS, (stats, st_, fs, fw)):
        assert np.array_equal(x, getattr(m, key)), (kind, key)


@gpu
@pytest.mark.parametrize("kind", ["id", "pd"])
def test_fused_rollout_equals_a_manual_loop_and_the_oracle(ctl, world, kind):
    """The fused rollout has the bits of 1-step wbc_rollout_loop calls with a caller-owned LoopState, each followed by
    wbc_monitor_step on that step's records (plan sample, applied torque from the loop state, forces, status word); the oracle
    on the same records agrees within 1e-12."""
    import torch
    from quadruped_drake_b200.capi import WbcMonitor
    from quadruped_drake_b200.rollout import Loop, LoopState, Monitor, MonitorState, rollout
    n, steps, dt = 128, 120, 5e-3
    q0, s = world["q0"][:n], world["s"]
    kw = {k: (x[:n] if isinstance(x, np.ndarray) else x) for k, x in world["kw"].items()}
    loop = noisy_loop(n, np.random.default_rng(7))
    fused = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop, monitor=Monitor(), **kw)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    q, v, t = T(q0), T(np.zeros((n, 18))), T(np.zeros(n))
    dkw = to_dev(kw)
    dl = dev_loop(loop)
    dl.state = LoopState(n, like=q)
    ms = MonitorState(n, like=q)
    why = torch.zeros(n, dtype=torch.int32, device="cuda")
    mo = WbcMonitor(0.05, 0.3, p(ms.stats), p(ms.steps), p(ms.fail_step), p(ms.fail_why), p(why))
    traj = torch.empty((n, 54), dtype=torch.float64, device="cuda"); contact = torch.empty((n, 4), dtype=torch.uint8, device="cuda")
    rows = torch.arange(n, device="cuda")
    cs = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    recs = []
    for c in range(steps):
        ctl._check(ctl.lib.wbc_sample_trajectory(ctl._h, s._p, n, None, p(t), p(traj), p(contact), None, None, None, cs), "sample")
        r = rollout(ctl, s, kind, q, v, t, 1, dt, plant=True, loop=dl, **dkw)
        applied = dl.strength[:, None] * dl.state.hist[rows, (c - dl.delay.long()).clamp(min=0) % 16]
        applied = torch.where(((r.status_or & 4096) != 0)[:, None], torch.zeros_like(applied), applied).contiguous()
        f = r.f_contact.reshape(n, 12).contiguous()
        ctl._check(ctl.lib.wbc_monitor_step(ctl._h, n, dt, C.byref(mo), p(q), p(v), p(traj), p(contact), p(applied), p(f), p(r.status_or),
                                            cs), "wbc_monitor_step")
        recs.append([x.cpu().numpy().copy() for x in (q, v, traj, contact, applied, f, r.status_or)])
    torch.cuda.synchronize()
    assert np.array_equal(q.cpu().numpy(), fused.q)
    for key in MON_KEYS:
        assert np.array_equal(np_of(getattr(ms, key)), getattr(fused.monitor, key)), (kind, key)
    assert np.array_equal(why.cpu().numpy(), fused.why)
    ora = om.State(n)
    maps = model_maps()
    for rec in recs:
        om.step(ora, dt, 0.05, 0.3, *maps, *rec)
    for key in ("steps", "fail_step", "fail_why", "why"):
        assert np.array_equal(getattr(ora, key), getattr(fused.monitor, key) if key != "why" else fused.why), key
    got = fused.monitor.stats
    assert np.array_equal(ora.stats[:, [8, 9]], got[:, [8, 9]])
    assert (np.abs(ora.stats - got) <= 1e-12 * np.maximum(1.0, np.abs(ora.stats))).all()


@gpu
def test_continuation_and_permutation(ctl, world):
    """Four calls of 100 steps with a MonitorState (and a LoopState) equal one call of 400; permuting the robots with their loop
    streams permutes every monitor output."""
    from quadruped_drake_b200.rollout import Loop, LoopState, Monitor, MonitorState, rollout
    n, dt = world["n"], 5e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    loop = noisy_loop(n, np.random.default_rng(8))
    loop.state = LoopState(n)
    one = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 400, dt, plant=True, loop=loop, monitor=Monitor(), **kw)
    loop.state = LoopState(n)
    mon = Monitor(state=MonitorState(n))
    q, v, t = q0, np.zeros((n, 18)), np.zeros(n)
    for _ in range(4):
        r = rollout(ctl, s, "id", q, v, t, 100, dt, plant=True, loop=loop, monitor=mon, **kw)
        q, v, t = r.q, r.v, r.t
    assert r.monitor is mon.state
    for key in MON_KEYS:
        assert np.array_equal(getattr(mon.state, key), getattr(one.monitor, key)), key
    assert np.array_equal(r.why, one.why) and np.array_equal(r.q, one.q)
    perm = np.random.default_rng(9).permutation(n)
    pl = Loop(noise=loop.noise[perm], delay=loop.delay[perm], strength=loop.strength[perm], stream=loop.stream[perm], seed=loop.seed)
    loop.state = None
    a = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 200, dt, plant=True, loop=loop, monitor=Monitor(), **kw)
    pkw = {k: (x[perm] if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    b = rollout(ctl, s, "id", q0[perm], np.zeros((n, 18)), 0.0, 200, dt, plant=True, loop=pl, monitor=Monitor(), **pkw)
    for key in MON_KEYS:
        assert np.array_equal(getattr(a.monitor, key)[perm], getattr(b.monitor, key)), key
    assert np.array_equal(a.why[perm], b.why)


@gpu
def test_free_fall(ctl):
    """Robots released at rest 0.2 m above the ground under a zero-gain PD set: e_p follows the plant's discrete free fall
    g dt^2 k(k+1)/2, the first failure is POS at k = 20, every planned stance foot is unloaded and nothing is loaded or worked."""
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.rollout import Monitor, MonitorState, rollout
    n, dt, g = 4, 5e-3, 9.81
    s = standing_sampler(ctl, 0.5)
    zero = ParamSet(ctl, [{"pd_kp": 0.0, "pd_kd": 0.0}])
    q = np.tile(Q0, (n, 1))
    q[:, 6] = 0.5
    v, t = np.zeros((n, 18)), np.zeros(n)
    mon = Monitor(state=MonitorState(n))
    sum2 = 0.0
    for k in range(1, 31):
        r = rollout(ctl, s, "pd", q, v, t, 1, dt, plant=True, param_set=zero, monitor=mon)
        q, v, t = r.q, r.v, r.t
        drop = g * dt * dt * k * (k + 1) / 2
        sum2 += drop * drop
        assert np.abs(mon.state.max_pos - drop).max() < 1e-12, k
        assert np.abs(r.tau).max() == 0.0 and (r.status_or == 0).all()
        assert np.array_equal(r.why, np.full(n, 1 if drop > 0.05 else 0, np.int32)), k
    st = mon.state
    assert (st.fail_step == 20).all() and (st.fail_why == 1).all() and (st.steps == 30).all()
    assert np.abs(st.stats[:, 0] - sum2).max() < 1e-12
    assert (st.stance_unloaded == 120).all() and (st.f_max == 0).all() and (st.swing_loaded == 0).all() and (st.work_abs == 0).all()
    assert (st.max_ang < 1e-12).all()
    zero.close(); s.close()


@gpu
def test_pushes(ctl):
    """Jittered standing ID robots at dt = 5e-3, pushed over 0.1 s at t = 1 s: without a push none ever fails; at 5 N s every
    robot ends with why == 0; at 15 N s every robot has failed, none before t = 1 s."""
    from quadruped_drake_b200.rollout import Monitor, rollout
    per, dt, steps = 64, 5e-3, 1200
    rng = np.random.default_rng(10)
    q0 = grounded(ctl, 1, rng, 0.0)
    s = standing_sampler(ctl, float(q0[0, 6]))
    impulses = [0.0, 5.0, 15.0]
    n = per * len(impulses)
    q = np.tile(q0, (n, 1))
    q[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    push = np.array([[j / 0.1, 0, 0, 0, 0, 0.05, 1.0, 1.1] for j in impulses]).repeat(per, 0)
    r = rollout(ctl, s, "id", q, np.zeros((n, 18)), 0.0, steps, dt, plant=True, push=push, monitor=Monitor())
    m, cell = r.monitor, np.arange(n) // per
    assert (m.fail_step[cell == 0] == 0).all() and (r.why[cell == 0] == 0).all()
    assert (r.why[cell == 1] == 0).all()
    assert (m.fail_step[cell == 2] > 0).all() and (m.fail_time(0.0, dt)[cell == 2] >= 1.0 - 1e-9).all()
    s.close()


@gpu
def test_bad_parameter_index(ctl, world):
    """A robot with an out-of-range parameter index fails at step 1 with STATUS; its neighbours have the bits of the batch without
    it."""
    from quadruped_drake_b200.rollout import Monitor, rollout
    n, steps, dt = 64, 80, 5e-3
    q0, s = world["q0"][:n], world["s"]
    kw = {k: (x[:n].copy() if isinstance(x, np.ndarray) else x) for k, x in world["kw"].items()}
    kw["param_index"][[5, 40]] = [4, -1]
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, monitor=Monitor(), **kw)
    assert (r.monitor.fail_step[[5, 40]] == 1).all() and (r.monitor.fail_why[[5, 40]] & 4).all()
    rest = np.setdiff1d(np.arange(n), [5, 40])
    rkw = {k: (x[rest] if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    ref = rollout(ctl, s, "id", q0[rest], np.zeros((len(rest), 18)), 0.0, steps, dt, plant=True, monitor=Monitor(), **rkw)
    for key in MON_KEYS:
        assert np.array_equal(getattr(r.monitor, key)[rest], getattr(ref.monitor, key)), key
    assert np.array_equal(r.why[rest], ref.why)


@gpu
def test_end_state_verdict_matches_the_tools_rule(ctl):
    """A reduced study 3 of tools/bench_loop.py (ID, dt = 5e-3, noise scale x motor strength, 6 s): why == 0 is the tools'
    end-state rule on the final q and status_or, robot for robot (robots within 1e-9 of a bound skipped). The rule reads the OR of
    every step's status, the monitor the last step's: a robot whose status was set only before the last step is compared on its
    pose alone. Every robot failing at the end has fail_step > 0."""
    from quadruped_drake_b200.rollout import Loop, Monitor, rollout
    per, dt = 16, 5e-3
    rng = np.random.default_rng(11)
    q = grounded(ctl, 1, rng, 0.0)[0]
    s = standing_sampler(ctl, float(q[6]))
    cells = [(sc, st) for sc in (0.0, 4.0, 8.0) for st in (0.6, 1.0)]
    n = per * len(cells)
    q0 = np.tile(q, (n, 1))
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    noise = np.array([NOISE * sc for sc, _ in cells]).repeat(per, 0)
    strength = np.array([st for _, st in cells]).repeat(per)
    loop = Loop(noise=noise, delay=np.zeros(n, np.int32), strength=strength, seed=11)
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 1200, dt, plant=True, loop=loop, monitor=Monitor())
    qf = r.q
    dotq = np.abs((q0[:, 0:4] * qf[:, 0:4]).sum(axis=1)) / np.linalg.norm(qf[:, 0:4], axis=1)
    tilt = 2 * np.arccos(np.clip(dotq, -1, 1))
    pos = np.linalg.norm(qf[:, 4:7] - q0[:, 4:7], axis=1)
    up = (r.status_or == 0) & (pos < 0.05) & (tilt < 0.3)
    near = (np.abs(pos - 0.05) < 1e-9) | (np.abs(tilt - 0.3) < 1e-9)
    earlier = (r.status_or != 0) & ((r.why & 4) == 0)
    up[earlier] = (pos < 0.05)[earlier] & (tilt < 0.3)[earlier]
    assert np.array_equal((r.why == 0)[~near], up[~near])
    assert (r.monitor.fail_step[r.why != 0] > 0).all()
    assert up.any()
    s.close()


@gpu
def test_argument_errors(ctl, world):
    import torch
    from quadruped_drake_b200.capi import WbcMonitor, WbcPlantOpts, WbcRolloutIO, WbcRolloutOpts
    from quadruped_drake_b200.rollout import Monitor, MonitorState, rollout
    n = 4
    s = world["s"]
    q, v, t = world["q0"][:n].copy(), np.zeros((n, 18)), np.zeros(n)
    io = WbcRolloutIO(P(q), P(v), P(t), None, None, None, None, None, None)
    st = MonitorState(n)
    good = lambda **o: WbcMonitor(o.get("pos", 0.05), o.get("ang", 0.3), P(st.stats), o.get("steps", P(st.steps)), P(st.fail_step),  # noqa: E731
                                  P(st.fail_why), None)
    integ = WbcRolloutOpts(1, 0, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    ground = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    call = lambda o, m: ctl.lib.wbc_rollout_monitor_host(ctl._h, 0, s._p, n, 2, 5e-3, C.byref(io), C.byref(o), None, None, None, None,  # noqa: E731
                                                         C.byref(m))
    assert call(integ, good()) == 1 and b"ground plant" in ctl.lib.wbc_last_error(ctl._h)
    for m in (good(pos=np.nan), good(ang=-0.1), good(pos=-1e-300)):
        assert call(ground, m) == 1 and b"pos_max and ang_max" in ctl.lib.wbc_last_error(ctl._h)
    assert call(ground, good(steps=None)) == 1 and b"required" in ctl.lib.wbc_last_error(ctl._h)
    z = np.zeros((n, 12))
    assert ctl.lib.wbc_monitor_step_host(ctl._h, n, 5e-3, C.byref(good(ang=np.nan)), P(q), P(v), P(np.zeros((n, 54))),
                                         P(np.zeros((n, 4), np.uint8)), P(z), P(z), None) == 1
    assert np.array_equal(q, world["q0"][:n]) and (st.steps == 0).all()          # nothing ran
    tq, tv, tt = (torch.from_numpy(x.copy()).cuda() for x in (q, v, t))
    l0 = ctl.launches
    for field, bad in (("stats", lambda x: x.float()), ("stats", lambda x: x[:, :10].contiguous()), ("steps", lambda x: x.int()),
                       ("fail_step", lambda x: x.cpu()), ("fail_why", lambda x: x[: n - 1])):
        ms = MonitorState(n, like=tq)
        setattr(ms, field, bad(getattr(ms, field)))
        with pytest.raises(ValueError, match="monitor.state." + field):
            rollout(ctl, s, "id", tq, tv, tt, 2, 5e-3, plant=True, monitor=Monitor(state=ms))
    with pytest.raises(ValueError, match="monitor.state.stats"):
        rollout(ctl, s, "id", q, v, t, 2, 5e-3, plant=True, monitor=Monitor(state=MonitorState(n + 1)))
    assert ctl.launches == l0
