"""Uneven ground for the ground plant: per-robot planes and height fields (include/wbc.h, csrc/wbc_plant.cuh).

CPU half: the numpy terrain of oracle/terrain.py against its definition, the terrain plant step of the device code through the
host warp emulator (tests/emu/emu_plant_terrain.cpp) against the numpy plant step of the oracle on the same terrain
(oracle/terrain.py:plant_step, which runs the unchanged oracle/rollout.py:plant_step in the feet's terrain frames), the
flat terrain against the perturbed step's bits, and the freeze of a bad terrain index. GPU half: the same cases through the
C ABI, a flat terrain rollout against wbc_rollout_perturbed, and closed loops with known physical answers: standing on
inclines, sliding down a 20 degree incline, landing on an incline and standing on a step."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

Q0 = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4)      # simulate.py:171-176
DT = 5e-3
G = 9.81
PAYLOAD = dict(mass=1.2, com=(0.04, -0.02, 0.05), inertia=(2e-3, 3e-3, 4e-3, 1e-4, -2e-4, 3e-4))


def desc_of(robot):
    from quadruped_drake_b200.model import ROBOT_DIR
    from quadruped_drake_b200.urdf import load_description
    return load_description(ROBOT_DIR / f"{robot}.json")


def T(**kw):
    from quadruped_drake_b200.rollout import Terrain
    return Terrain(**kw)


def incline(deg, direction=(1.0, 0.0)):
    d = np.asarray(direction, float) / np.linalg.norm(direction)
    s = np.tan(np.radians(deg))
    return T(slope=(s * d[0], s * d[1]))


def step_terrain(height, robot="mini_cheetah"):
    """A step of `height` under the two left feet (y > 0): a grid along y with a 1 cm ramp between y = 0 and y = 0.01."""
    y = -0.3 + 0.01 * np.arange(61)
    row = np.where(y >= 0.01 - 1e-12, height, 0.0)
    return T(origin=(-1.0, -0.3), spacing=(2.0, 0.01), heights=np.tile(row[:, None], (1, 2)))


def bumpy():
    rng = np.random.default_rng(5)
    return T(z0=0.004, slope=(0.02, -0.03), origin=(-0.8, -0.8), spacing=(0.1, 0.1), heights=rng.uniform(-0.02, 0.02, (16, 16)))


def terrains():
    """(name, terrain) of the parity cases."""
    return [("flat", T()), ("x5", incline(5)), ("x20", incline(20)), ("diag5", incline(5, (1, 1))), ("diag20", incline(20, (1, -1))),
            ("bumpy", bumpy()), ("step3cm", step_terrain(0.03))]


def oracle_terrain(t):
    from oracle.terrain import Terrain
    return Terrain(z0=t.z0, slope=tuple(t.slope), origin=tuple(t.origin), spacing=tuple(t.spacing),
                   heights=None if t.heights is None else np.asarray(t.heights, float))


def terrain_descs(ts):
    """wbc_terrain_desc[] of the terrains (and the grids they point into, to keep alive)."""
    from quadruped_drake_b200.capi import WbcTerrainDesc
    grids = [None if t.heights is None else np.ascontiguousarray(t.heights, np.float64) for t in ts]
    arr = (WbcTerrainDesc * len(ts))(*[WbcTerrainDesc(t.z0, t.slope[0], t.slope[1], 0 if g is None else g.shape[1], 0 if g is None else g.shape[0],
                                                      t.origin[0], t.origin[1], t.spacing[0], t.spacing[1], None if g is None else g.ctypes.data)
                                       for t, g in zip(ts, grids)])
    return arr, grids


def ptr(a):
    from quadruped_drake_b200.capi import np_ptr
    return None if a is None else np_ptr(a)


def model_table(descs):
    from quadruped_drake_b200.model import WbcModelStruct, flatten
    return (WbcModelStruct * len(descs))(*[flatten(d).as_struct() for d in descs])


@pytest.fixture(scope="module")
def emu_tr(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_terrain.so"))
    lib.emu_plant_step_terrain.argtypes = ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_longlong, C.c_double, C.c_double, C.c_double, C.c_int] + [C.c_void_p] * 5)
    return lib


@pytest.fixture(scope="module")
def emu_pt(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_perturbed.so"))
    lib.emu_plant_step_perturbed.argtypes = ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_double,
                                              C.c_double, C.c_double, C.c_int] + [C.c_void_p] * 5)
    return lib


def emu_terrain(emu, descs, mu, variant, push, ts, index, t, q, v, tau):
    """One emulated terrain step; q, v, t updated in place -> f[N,4,3], status[N]. ts = None: flat ground (no set)."""
    n = len(q)
    f, st = np.zeros((n, 4, 3)), np.zeros(n, np.int32)
    mu_a = None if mu is None else np.ascontiguousarray(mu, np.float64)
    arr, keep = terrain_descs(ts) if ts is not None else (None, None)
    assert emu.emu_plant_step_terrain(model_table(descs), ptr(mu_a), len(descs), ptr(variant), ptr(push), arr, 0 if ts is None else len(ts),
                                      ptr(index), ptr(t), n, DT, 1.0, 0.2, 30, ptr(q), ptr(v), ptr(tau), ptr(f), ptr(st)) == 0
    return f, st


def foot_positions(P, q):
    return np.array([P.frame_position_quantities(q, np.zeros(18), fr)[0] for fr in P.foot_frames])


def place_feet(P, q, ot, lift=0.0):
    """Joint angles of q moved (Newton on the oracle's foot Jacobians, base fixed) so that every foot keeps its x, y and sits
    `lift` above the terrain ot."""
    from oracle import terrain as otr
    q = q.copy()
    for _ in range(8):
        quant = [P.frame_position_quantities(q, np.zeros(18), fr) for fr in P.foot_frames]
        p = np.array([x[0] for x in quant])
        target = p.copy()
        target[:, 2] = [otr.height(ot, x, y) + lift for x, y, _ in p]
        J = np.vstack([x[1][:, 6:] for x in quant])
        q[7:] += np.linalg.lstsq(J, (target - p).reshape(-1), rcond=None)[0]
    return q


def parity_cases(robot, tr):
    """Standing (feet on the terrain), airborne, sliding, penetrating and random states on terrain tr; a payload variant with
    mu 0.2, the nominal model with mu 1.0, active pushes."""
    from oracle.dynamics import Plant
    from quadruped_drake_b200 import load_robot
    P = Plant(desc_of(robot))
    ot = oracle_terrain(tr)
    rng = np.random.default_rng(23)
    n = 8
    q = np.tile(place_feet(P, load_robot(robot).nominal_q(), ot), (n, 1))
    v = np.zeros((n, 18))
    tau = rng.uniform(-3, 3, (n, 12))
    q[1, 6] += 0.1                                              # airborne
    v[2, 3:5] = [0.8, -0.4]                                     # sliding
    q[3, 6] -= 0.004                                            # penetrating
    q[4:, 7:] += rng.uniform(-0.2, 0.2, (n - 4, 12)); v[4:] = rng.uniform(-1, 1, (n - 4, 18))
    variant = np.array([1, 0, 1, 0, 1, 0, 1, 0], np.int32)
    t = np.full(n, 0.1)
    push = np.zeros((n, 8))
    push[:, 0:3] = rng.uniform(-40, 40, (n, 3))
    push[:, 3:6] = rng.uniform(-0.15, 0.15, (n, 3))
    push[:, 6], push[:, 7] = 0.0, 1.0
    return q, v, tau, variant, push, t


def variants(robot):
    from quadruped_drake_b200.model import with_payload
    d = desc_of(robot)
    return [("nominal", d, 1.0), ("payload", with_payload(d, **PAYLOAD), 0.2)]


class PushedPlant:
    """oracle.dynamics.Plant with a push (tau_g - J_p' F while the push window holds t), as in tests/test_plant_variants.py."""

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


def oracle_step(vs, variant, q, v, tau, push, t, ot):
    from oracle import terrain as otr
    from oracle.dynamics import Plant
    plants = [Plant(d) for _, d, _ in vs]
    return [otr.plant_step(PushedPlant(plants[variant[i]], push[i], t[i]), q[i], v[i], tau[i], DT, vs[variant[i]][2], 0.2, 30, terrain=ot)
            for i in range(len(q))]


def assert_matches_oracle(qn, vn, f, ref, what):
    for i, (qo, vo, fo) in enumerate(ref):
        assert np.abs(qn[i] - qo).max() < 1e-9 and np.abs(vn[i] - vo).max() < 1e-8, (what, i, np.abs(vn[i] - vo).max())
        assert np.abs(f[i] - fo).max() < 1e-6 * max(1.0, np.abs(fo).max()), (what, i)


# ------------------------------------------------------------------------------------------------------------------ CPU half
def test_grid_sampled_from_a_plane_reproduces_it_and_clamps_outside():
    from oracle import terrain as otr
    sx, sy, z0 = 0.21, -0.13, 0.05
    x0, y0, dx, dy, nx, ny = -0.7, -0.4, 0.11, 0.07, 13, 9
    xs, ys = x0 + dx * np.arange(nx), y0 + dy * np.arange(ny)
    grid = otr.Terrain(z0=z0, origin=(x0, y0), spacing=(dx, dy), heights=sx * xs[None, :] + sy * ys[:, None])
    plane = otr.Terrain(z0=z0, slope=(sx, sy))
    rng = np.random.default_rng(1)
    pts = np.c_[rng.uniform(xs[0], xs[-1], 200), rng.uniform(ys[0], ys[-1], 200)]
    pts = np.r_[pts, [[xs[-1], ys[-1]], [xs[0], ys[0]], [xs[-1], ys[3]]]]                 # far edges use the last cell
    for x, y in pts:
        assert abs(otr.height(grid, x, y) - otr.height(plane, x, y)) < 1e-12
        assert np.abs(otr.frame(grid, x, y) - otr.frame(plane, x, y)).max() < 1e-12
    for x, y, cx, cy in ((xs[-1] + 0.3, 0.0, xs[-1], 0.0), (xs[0] - 0.5, ys[0] - 1.0, xs[0], ys[0]), (0.1, ys[-1] + 2.0, 0.1, ys[-1])):
        h, g = otr.height_and_gradient(grid, x, y)
        assert abs(h - otr.height(plane, cx, cy)) < 1e-12
        assert (g[0] == 0.0) == (cx != x) and (g[1] == 0.0) == (cy != y)
        assert (cx != x or abs(g[0] - sx) < 1e-12) and (cy != y or abs(g[1] - sy) < 1e-12)


def test_frames_are_orthonormal_and_right_handed():
    from oracle import terrain as otr
    rng = np.random.default_rng(2)
    for _, t in terrains():
        ot = oracle_terrain(t)
        for x, y in rng.uniform(-1.2, 1.2, (50, 2)):
            R = otr.frame(ot, x, y)
            assert np.abs(R.T @ R - np.eye(3)).max() < 1e-14 and abs(np.linalg.det(R) - 1.0) < 1e-14 and R[2, 2] > 0
            assert abs(R[1, 0] + R[0, 2] * R[1, 2] / np.linalg.norm([1 - R[0, 2] ** 2, R[0, 2] * R[1, 2], R[0, 2] * R[2, 2]])) < 1e-15
    R = otr.frame(oracle_terrain(incline(20)), 0.3, 0.0)
    th = np.radians(20)
    assert np.abs(R[:, 2] - [-np.sin(th), 0, np.cos(th)]).max() < 1e-15 and np.abs(R[:, 0] - [np.cos(th), 0, np.sin(th)]).max() < 1e-15
    assert abs(otr.gap(oracle_terrain(incline(20)), np.array([0.3, 0.0, 1.0])) - (1.0 - 0.3 * np.tan(th)) * np.cos(th)) < 1e-15


def test_oracle_flat_terrain_keeps_the_bits():
    from oracle import rollout as ro
    from oracle.dynamics import Plant
    from oracle import terrain as otr
    P = Plant(desc_of("mini_cheetah"))
    q, v, tau, _, _, _ = parity_cases("mini_cheetah", T())
    for i in range(len(q)):
        a, b = ro.plant_step(P, q[i], v[i], tau[i], DT), otr.plant_step(P, q[i], v[i], tau[i], DT, terrain=otr.Terrain())
        assert all(np.array_equal(x, y) for x, y in zip(a, b)), i


@pytest.mark.parametrize("robot", ["mini_cheetah", "anymal_b"])
@pytest.mark.parametrize("tname", [n for n, _ in terrains()])
def test_emulated_terrain_step_matches_oracle(emu_tr, robot, tname):
    """Every terrain, payload variant at mu 0.2 and nominal at mu 1.0, active pushes; standing, airborne, sliding, penetrating
    and random states; two steps."""
    tr = dict(terrains())[tname]
    vs = variants(robot)
    q, v, tau, variant, push, t = parity_cases(robot, tr)
    ot = oracle_terrain(tr)
    index = np.ones(len(q), np.int32)                             # terrain 1 of a set [flat, tr]
    for step in range(2):
        ref = oracle_step(vs, variant, q, v, tau, push, t, ot)
        f, st = emu_terrain(emu_tr, [d for _, d, _ in vs], [m for _, _, m in vs], variant, push, [T(), tr], index, t, q, v, tau)
        assert (st == 0).all()
        assert_matches_oracle(q, v, f, ref, (robot, tname, step))


def test_emulated_flat_terrain_keeps_the_perturbed_bits(emu_tr, emu_pt):
    """No set, and a set of flat terrains: the bits of emu_plant_step_perturbed with the same variants and pushes."""
    vs = variants("mini_cheetah")
    descs, mus = [d for _, d, _ in vs], [m for _, _, m in vs]
    q, v, tau, variant, push, t = parity_cases("mini_cheetah", T())
    qa, va, ta = q.copy(), v.copy(), t.copy()
    fa, sa = np.zeros((len(q), 4, 3)), np.zeros(len(q), np.int32)
    assert emu_pt.emu_plant_step_perturbed(model_table(descs), ptr(np.array(mus)), 2, ptr(variant), ptr(push), ptr(ta), len(q), DT, 1.0, 0.2, 30,
                                           ptr(qa), ptr(va), ptr(tau), ptr(fa), ptr(sa)) == 0
    for ts, index in ((None, None), ([T(), T()], np.array([0, 1] * 4, np.int32))):
        qb, vb, tb = q.copy(), v.copy(), t.copy()
        fb, sb = emu_terrain(emu_tr, descs, mus, variant, push, ts, index, tb, qb, vb, tau)
        for a, b in ((qa, qb), (va, vb), (ta, tb), (fa, fb), (sa, sb)):
            assert np.array_equal(a, b)


def test_emulated_bad_terrain_index_freezes_only_that_robot(emu_tr):
    from quadruped_drake_b200.capi import ST_BADTERRAIN
    vs = variants("mini_cheetah")
    descs, mus = [d for _, d, _ in vs], [m for _, _, m in vs]
    ts = [incline(5), bumpy()]
    q, v, tau, variant, push, t = parity_cases("mini_cheetah", ts[0])
    index = np.array([0, 1, -1, 0, 2, 1, 0, 1 << 30], np.int32)
    bad = (index < 0) | (index >= 2)
    qa, va, ta = q.copy(), v.copy(), t.copy()
    fa, sa = emu_terrain(emu_tr, descs, mus, variant, push, ts, index, ta, qa, va, tau)
    qb, vb, tb = q[~bad].copy(), v[~bad].copy(), t[~bad].copy()
    fb, sb = emu_terrain(emu_tr, descs, mus, variant[~bad], push[~bad], ts, index[~bad], tb, qb, vb, tau[~bad])
    assert (sa[bad] & ST_BADTERRAIN).all() and (sa[~bad] == 0).all()
    assert np.array_equal(qa[bad], q[bad]) and np.array_equal(va[bad], v[bad]) and (fa[bad] == 0).all()
    for a, b in ((qa, qb), (va, vb), (ta, tb), (fa, fb), (sa, sb)):
        assert np.array_equal(a[~bad], b)


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
def test_terrain_plant_step_matches_oracle_on_gpu(ctl):
    """Every parity terrain through wbc_plant_step_terrain_host, and the device entry (torch tensors) gives the same bits."""
    import torch
    from quadruped_drake_b200.rollout import TerrainSet, plant_step
    vs = variants("mini_cheetah")
    ps = plant_set(ctl, [d for _, d, _ in vs], [m for _, _, m in vs])
    names, ts = zip(*terrains())
    tset = TerrainSet(ctl, list(ts))
    for k, (name, tr) in enumerate(terrains()):
        q, v, tau, variant, push, t = parity_cases("mini_cheetah", tr)
        index = np.full(len(q), k, np.int32)
        ref = oracle_step(vs, variant, q, v, tau, push, t, oracle_terrain(tr))
        qn, vn, f, st = plant_step(ctl, q, v, tau, DT, plant_set=ps, variant=variant, push=push, t=t, terrain_set=tset, terrain=index)
        assert (st == 0).all(), name
        assert_matches_oracle(qn, vn, f, ref, name)
        tq, tv, ttau, tt, tvar, tpush, tidx = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (q, v, tau, t, variant, push, index))
        _, _, tf, tst = plant_step(ctl, tq, tv, ttau, DT, plant_set=ps, variant=tvar, push=tpush, t=tt, terrain_set=tset, terrain=tidx)
        torch.cuda.synchronize()
        assert (tst.cpu().numpy() == 0).all()
        assert np.array_equal(tq.cpu().numpy(), qn) and np.array_equal(tv.cpu().numpy(), vn) and np.array_equal(tf.cpu().numpy(), f), name
    tset.close(); ps.close()


def grounded(ctl, n, rng=None, jitter=0.0):
    q0 = np.tile(Q0, (n, 1))
    if rng is not None and jitter > 0:
        q0[:, 7:] += rng.uniform(-jitter, jitter, (n, 12))
    pz = ctl.dynamics(q0, np.zeros((n, 18)))["p_feet"][:, :, 2]
    q0[:, 6] -= pz.min(axis=1)
    return q0


def run_torch(ctl, s, q0, steps, kind="id", dt=DT, **kw):
    import torch
    from quadruped_drake_b200.rollout import rollout
    n = len(q0)
    q, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    kw = {k: (torch.from_numpy(np.ascontiguousarray(x)).cuda() if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    with torch.cuda.stream(torch.cuda.Stream()):
        before = ctl.launches
        r = rollout(ctl, s, kind, q, v, t, steps, dt, plant=True, **kw)
    torch.cuda.synchronize()
    out = {k: x.cpu().numpy() for k, x in (("q", q), ("v", v), ("t", t), ("tau", r.tau), ("err_max", r.err_max), ("status", r.status_or),
                                             ("f", r.f_contact))}
    out["launches"] = ctl.launches - before
    return out


def standing_sampler(ctl, duration=6.0):
    from quadruped_drake_b200 import planner as pl
    bh = float(grounded(ctl, 1)[0, 6])
    return pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", duration, base_height=bh))


@gpu
def test_flat_terrain_rollout_keeps_the_perturbed_bits(ctl):
    """512 robots, 200 steps with variants and pushes: a set of flat terrains gives the bits of wbc_rollout_perturbed, with and
    without the graph, and the same launches per step."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.model import with_payload
    from quadruped_drake_b200.rollout import TerrainSet
    n, steps = 512, 200
    rng = np.random.default_rng(13)
    q0 = grounded(ctl, n, rng, 0.02)
    bh = float(grounded(ctl, 1)[0, 6])
    s = pl.TrajectorySampler(ctl, pl.make_gait_plan("mini_cheetah", "trot", goal=(1.5, 0.0), base_height=bh))
    d = desc_of("mini_cheetah")
    ps = plant_set(ctl, [d, with_payload(d, **PAYLOAD)], [1.0, 0.4])
    tset = TerrainSet(ctl, [T(), T()])
    variant = (np.arange(n) % 2).astype(np.int32)
    push = np.zeros((n, 8))
    push[:, 0:3] = rng.uniform(-30, 30, (n, 3)); push[:, 3:6] = rng.uniform(-0.1, 0.1, (n, 3))
    push[:, 6], push[:, 7] = 0.3, 0.8
    index = (np.arange(n) // 3 % 2).astype(np.int32)
    for graph in (False, True):
        a = run_torch(ctl, s, q0, steps, use_graph=graph, plant_set=ps, variant=variant, push=push)
        b = run_torch(ctl, s, q0, steps, use_graph=graph, plant_set=ps, variant=variant, push=push, terrain_set=tset, terrain=index)
        c = run_torch(ctl, s, q0, steps, use_graph=graph, plant_set=ps, variant=variant, push=push, terrain=np.zeros(n, np.int32))
        for k in ("q", "v", "t", "tau", "err_max", "status", "f"):
            assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], c[k]), (graph, k)
        assert a["launches"] == b["launches"] == c["launches"]
    tset.close(); ps.close(); s.close()


def placed_on(ctl, ot, n, lift=0.0, rng=None, jitter=0.0):
    """n robots with a level base at the plan's height over the terrain's origin and every foot placed on ot (+ lift)."""
    from oracle.dynamics import Plant
    from oracle import terrain as otr
    P = Plant(desc_of("mini_cheetah"))
    q = grounded(ctl, 1)[0]
    q[6] += otr.height(ot, 0.0, 0.0)
    q = place_feet(P, q, ot, lift)
    qs = np.tile(q, (n, 1))
    if rng is not None:
        qs[:, 7:] += rng.uniform(-jitter, jitter, (n, 12))
    return qs


def step_by_step(ctl, s, q0, steps, kind="id", dt=DT, **kw):
    """Rollouts of one step each (torch in place): yields (q before the step, q, f) per step."""
    import torch
    from quadruped_drake_b200.rollout import rollout
    n = len(q0)
    q, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    kw = {k: (torch.from_numpy(np.ascontiguousarray(x)).cuda() if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    status = np.zeros(n, np.int32)
    for _ in range(steps):
        qb = q.cpu().numpy()
        r = rollout(ctl, s, kind, q, v, t, 1, dt, plant=True, **kw)
        status |= r.status_or.cpu().numpy()
        yield qb, q.cpu().numpy(), v.cpu().numpy(), r.f_contact.cpu().numpy(), status


@gpu
@pytest.mark.parametrize("deg", [0.0, 5.0, 10.0])
def test_id_robots_stand_on_inclines(ctl, deg):
    """64 ID robots with jittered joints on an incline along x, mu = 1.0, 2 s: no status bit, the ground carries m g in world
    axes, and every foot force is in its tilted pyramid (R' f: normal >= 0, |t1|, |t2| <= mu n) in every step."""
    from quadruped_drake_b200.rollout import TerrainSet
    from oracle import terrain as otr
    n, m = 64, ctl.model.total_mass
    tr = incline(deg)
    ot = oracle_terrain(tr)
    R = otr.frame(ot, 0.0, 0.0)
    s = standing_sampler(ctl)
    tset = TerrainSet(ctl, [tr])
    q0 = placed_on(ctl, ot, n, rng=np.random.default_rng(7), jitter=0.02)
    for _, q, v, f, status in step_by_step(ctl, s, q0, 400, terrain_set=tset):
        loc = f @ R                                                # [n, 4, 3] in (t1, t2, n)
        scale = np.maximum(np.abs(loc).max(), 1.0)
        assert (loc[:, :, 2] >= -1e-9 * scale).all()
        assert (np.abs(loc[:, :, :2]) <= loc[:, :, 2:3] + 1e-9 * scale).all()
    assert (status == 0).all(), np.unique(status)
    total = f.sum(axis=1)
    assert (np.abs(total - [0.0, 0.0, m * G]) < 0.02 * m * G).all(), np.abs(total - [0, 0, m * G]).max() / (m * G)
    tset.close(); s.close()


def pd_on_incline(ctl, deg, n=16):
    """PD robots at the nominal joint angles with the base pitched to the incline and the feet on it."""
    from oracle.dynamics import Plant
    from oracle import terrain as otr
    P = Plant(desc_of("mini_cheetah"))
    ot = oracle_terrain(incline(deg))
    th = np.radians(deg)
    q = Q0.copy()
    q[0:4] = [np.cos(-th / 2), 0.0, np.sin(-th / 2), 0.0]
    gaps = [otr.gap(ot, p) for p in foot_positions(P, q)]
    q[6] -= np.mean(gaps) / np.cos(th)
    return np.tile(q, (n, 1)), ot


@gpu
def test_pd_robot_slides_down_a_20_degree_incline_at_the_coulomb_rate(ctl):
    """mu = 0.1 < tan 20: after 0.2 s the base accelerates down the slope at g (sin th - mu cos th) = 2.43 m/s^2 (3 %).
    mu = 0.5 > tan 20: the hind feet, which carry the robot, stick - they move less than 1 cm in 0.6 s. The base does not stay
    put: at the reference gains (Kp 30) the loaded hind knees give way, the front feet unload and slide off, and the robot tips
    over backwards within 1 s - friction-independent, it does the same at mu = 1.0 and stands on 10 degrees."""
    from quadruped_drake_b200.rollout import TerrainSet
    th = np.radians(20.0)
    q0, _ = pd_on_incline(ctl, 20.0)
    s = standing_sampler(ctl)
    tset = TerrainSet(ctl, [incline(20.0)])
    down = np.array([-np.cos(th), 0.0, -np.sin(th)])
    vel, status = {}, np.zeros(len(q0), np.int32)
    for k, (_, q, v, f, status) in enumerate(step_by_step(ctl, s, q0, 600, kind="pd", dt=1e-3, mu=0.1, terrain_set=tset)):
        if k + 1 in (200, 600):
            vel[k + 1] = v[:, 3:6] @ down
    assert (status == 0).all(), np.unique(status)
    acc = (vel[600] - vel[200]) / 0.4
    expect = G * (np.sin(th) - 0.1 * np.cos(th))
    assert (np.abs(acc - expect) < 0.03 * expect).all(), (acc, expect)
    c = run_torch(ctl, s, q0, 600, kind="pd", dt=1e-3, mu=0.5, terrain_set=tset)
    assert (c["status"] == 0).all()
    hind0, hind = (ctl.dynamics(x, np.zeros((len(x), 18)))["p_feet"][:, 2:4] for x in (q0, c["q"]))
    assert (np.linalg.norm(hind - hind0, axis=2) < 0.01).all(), np.linalg.norm(hind - hind0, axis=2).max()
    tset.close(); s.close()


def gaps_of(ctl, q, ot):
    from oracle import terrain as otr
    pf = ctl.dynamics(q, np.zeros((len(q), 18)))["p_feet"]
    return np.array([[otr.gap(ot, p) for p in row] for row in pf])


@gpu
@pytest.mark.parametrize("case", ["drop_on_10deg", "step_2cm"])
def test_no_foot_sinks_and_the_ground_carries_the_robot(ctl, case):
    """ID robots dropped from 3 cm onto a 10 degree incline, and standing with their two left feet on a 2 cm step: no foot more
    than 2 mm below its local terrain along the normal in any step, and after 2 s the ground carries m g (2 %)."""
    from quadruped_drake_b200.rollout import TerrainSet
    n, m = 16, ctl.model.total_mass
    tr = incline(10.0) if case == "drop_on_10deg" else step_terrain(0.02)
    ot = oracle_terrain(tr)
    q0 = placed_on(ctl, ot, n, lift=0.03 if case == "drop_on_10deg" else 0.0, rng=np.random.default_rng(9), jitter=0.01)
    s = standing_sampler(ctl)
    tset = TerrainSet(ctl, [tr])
    worst = 0.0
    for _, q, v, f, status in step_by_step(ctl, s, q0, 400, terrain_set=tset):
        worst = min(worst, gaps_of(ctl, q, ot).min())
    assert worst > -2e-3, worst
    assert (status == 0).all(), np.unique(status)
    total = f.sum(axis=1)
    assert (np.abs(total - [0.0, 0.0, m * G]) < 0.02 * m * G).all(), np.abs(total - [0, 0, m * G]).max() / (m * G)
    tset.close(); s.close()


@gpu
def test_bad_terrain_index_freezes_only_that_robot(ctl):
    from quadruped_drake_b200.capi import ST_BADTERRAIN
    from quadruped_drake_b200.rollout import TerrainSet
    n = 64
    s = standing_sampler(ctl)
    tset = TerrainSet(ctl, [incline(5.0), bumpy()])
    q0 = grounded(ctl, n, np.random.default_rng(4), 0.03)
    index = (np.arange(n) % 2).astype(np.int32)
    bad = np.zeros(n, bool); bad[[5, 30, 63]] = True
    index[5], index[30], index[63] = -1, 2, 1 << 30
    a = run_torch(ctl, s, q0, 60, terrain_set=tset, terrain=index)
    b = run_torch(ctl, s, q0[~bad], 60, terrain_set=tset, terrain=index[~bad])
    assert (a["status"][bad] & ST_BADTERRAIN).all() and not (a["status"][~bad] & ST_BADTERRAIN).any()
    assert np.array_equal(a["q"][bad], q0[bad]) and (a["v"][bad] == 0).all() and (a["f"][bad] == 0).all()
    for k in ("q", "v", "t", "tau", "err_max", "status", "f"):
        assert np.array_equal(a[k][~bad], b[k]), k
    tset.close(); s.close()


@gpu
def test_terrain_argument_errors_and_set_lifetime(built):
    """Each argument error returns WBC_ERR_ARG with a message; a set destroyed after its handle is safe."""
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.capi import WbcPlantOpts, WbcPlantTerrain, WbcRolloutIO, WbcRolloutOpts
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.rollout import TerrainSet, plant_step
    ctl = BatchedController("mini_cheetah", device=0)
    lib = ctl.lib
    g = np.zeros((4, 4))
    cases = [
        (T(origin=(0, 0), spacing=(0.1, 0.1), heights=np.zeros((4, 1))), "nx and ny"),
        (T(spacing=(0.0, 0.1), heights=g), "dx > 0"),
        (T(spacing=(0.1, -0.1), heights=g), "dx > 0"),
        (T(spacing=(0.1, 0.1), heights=np.where(np.eye(4) > 0, np.nan, 0.0)), "non-finite height"),
        (T(z0=float("inf")), "non-finite"),
    ]
    for tr, word in cases:
        arr, keep = terrain_descs([T(), tr])
        out = C.c_void_p()
        assert lib.wbc_terrain_set_create(ctl._h, 2, arr, C.byref(out)) == 1 and not out
        assert word in lib.wbc_last_error(ctl._h).decode(), (word, lib.wbc_last_error(ctl._h))
    arr, keep = terrain_descs([T(spacing=(0.1, 0.1), heights=g)])
    arr[0].heights = None                                                        # a grid without heights
    out = C.c_void_p()
    assert lib.wbc_terrain_set_create(ctl._h, 1, arr, C.byref(out)) == 1 and b"heights" in lib.wbc_last_error(ctl._h)
    assert lib.wbc_terrain_set_create(ctl._h, 0, arr, C.byref(out)) == 1
    tset = TerrainSet(ctl, [incline(5.0)])
    n = 4
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 1.0, base_height=0.3))
    tq, tv, tt = (torch.from_numpy(x).cuda() for x in (np.tile(Q0, (n, 1)), np.zeros((n, 18)), np.zeros(n)))
    io = WbcRolloutIO(tq.data_ptr(), tv.data_ptr(), tt.data_ptr(), None, None, None, None, None, None)
    tr = WbcPlantTerrain(tset._p, None)
    o = WbcRolloutOpts(1, 0, WbcPlantOpts(1.0, 0.2, 30, 0), None)                # plant = 0: no ground to shape
    assert lib.wbc_rollout_terrain(ctl._h, 0, s._p, n, 2, DT, C.byref(io), C.byref(o), None, C.byref(tr), None) == 1
    assert b"plant" in lib.wbc_last_error(ctl._h)
    if torch.cuda.device_count() > 1:                                            # a set from another device
        other = BatchedController("mini_cheetah", device=1)
        to = TerrainSet(other, [incline(5.0)])
        with pytest.raises(RuntimeError, match="another device"):
            plant_step(ctl, np.tile(Q0, (n, 1)), np.zeros((n, 18)), np.zeros((n, 12)), DT, terrain_set=to)
        to.close(); other.close()
    s.close()
    ctl.close()                                                                  # the set outlives its handle
    tset.close()
    c2 = BatchedController("mini_cheetah", device=0)
    t2 = TerrainSet(c2, [bumpy()])
    qn, vn, f, st = plant_step(c2, grounded(c2, 2), np.zeros((2, 18)), np.zeros((2, 12)), DT, terrain_set=t2, terrain=np.zeros(2, np.int32))
    assert (st == 0).all() and np.isfinite(qn).all()
    t2.close(); c2.close()
