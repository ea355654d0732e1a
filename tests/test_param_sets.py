"""Per-robot controller parameters (wbc_param_set_create, wbc_step_params[_host], wbc_rollout_params[_host]).

CPU half: the parameter-aware step of csrc/wbc_device.cuh (record selection, reduce, hand-over, solve, and the PD law) on the
host warp emulator (tests/emu/emu_step_params.cpp), each row against the oracle built with that row's parameters.
GPU half: a set whose records all equal the handle's params gives the bits of wbc_step on every path; rows assigned to K sets
give the bits of K handles created with those sets, for the step and for rollouts on both plants; optimality with per-row
parameters; bad indices and rejected descriptors."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from oracle import controllers as oc

GOLD = Path(__file__).parent / "golden"
KIND_NAMES = ["id", "clf", "pc", "mptc", "pd"]
ORACLES = {"id": oc.IDController, "clf": oc.CLFController, "pc": oc.PCController, "mptc": oc.MPTCController}
# the gains and weights a set varies (x 0.5 - 2)
SCALED = ["id_kp_body_p", "id_kd_body_p", "id_kp_body_rpy", "id_kd_body_rpy", "id_kp_foot", "id_kd_foot", "id_w_body", "id_w_foot",
          "clf_q_body_p", "clf_q_body_pd", "clf_q_body_rpy", "clf_q_body_rpyd", "clf_q_foot_p", "clf_q_foot_pd", "clf_w_delta",
          "pc_kp_body_p", "pc_kd_body_p", "pc_kp_body_rpy", "pc_kd_body_rpy", "pc_kp_foot", "pc_kd_foot", "pc_w_body", "pc_w_foot",
          "pd_kp", "pd_kd", "pd_clip"]


def param_sets(k, seed):
    """k override dicts for make_params: gains and weights x 0.5 - 2, mu 0.4 - 1.0, the CLF r, torque limits on for odd sets,
    and a shifted PD posture."""
    from quadruped_drake_b200.capi import DEFAULT_PARAMS
    rng = np.random.default_rng(seed)
    out = []
    for i in range(k):
        d = {n: DEFAULT_PARAMS[n] * float(rng.uniform(0.5, 2.0)) for n in SCALED}
        d.update(mu=float(rng.uniform(0.4, 1.0)), clf_r=float(rng.uniform(0.5, 2.0)), torque_limits=i % 2,
                 pd_q_nom=tuple(np.asarray(DEFAULT_PARAMS["pd_q_nom"]) + rng.uniform(-0.1, 0.1, 12)))
        out.append(d)
    return out


def oracle_kw(d):
    """The keys of a set the QP oracle takes (it has no iteration cap and no PD law)."""
    return {k: v for k, v in d.items() if k in oc.DEFAULTS}


def oracle_pd(robot, d, dof_order="depth_first"):
    q_nom = np.array([1.0, 0, 0, 0, 0, 0, 0.3] + list(d["pd_q_nom"]))
    return oc.BasicController(robot, dof_order, q_nom=q_nom, kp=d["pd_kp"], kd=d["pd_kd"], clip=d["pd_clip"])


def golden(case, n):
    g = np.load(GOLD / f"{case}.npz")
    return {k: np.ascontiguousarray(g[k][:n]) for k in ("q", "v", "traj", "contact")}


def robot_of(case):
    return "anymal_b" if "anymal" in case else "mini_cheetah"


def check_rows_against_oracle(robot, kind, g, sets, index, tau, vd, f, status):
    """Every row with status 0 within the golden bars of the oracle built with its set; at least 2/3 of the rows solve."""
    n = len(index)
    ok = 0
    for i in range(n):
        d = sets[index[i]]
        if kind == "pd":
            assert status[i] == 0
            ref = oracle_pd(robot, d).control_law(g["q"][i], g["v"][i])
            assert np.abs(tau[i] - ref).max() < 1e-12, i
            ok += 1
            continue
        if status[i] != 0:
            assert (tau[i] == 0).all() and (f[i] == 0).all() and (vd[i] == 0).all()
            continue
        o = ORACLES[kind](robot, **oracle_kw(d)).control_law(g["q"][i], g["v"][i], oc.traj_to_dict(g["traj"][i], g["contact"][i]))
        assert np.abs(tau[i] - o.tau).max() < 1e-5, (kind, i)
        assert np.abs(vd[i] - o.vd).max() < 1e-6, (kind, i)
        assert np.abs(f[i] - o.f).max() < 1e-5, (kind, i)
        ok += 1
    assert ok >= 2 * n // 3, (kind, ok, n)


# ------------------------------------------------------------------------------------------------------------------ CPU half
@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_params.so"))
    lib.emu_step_params.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
    return lib


def emu_step(emu, robot, kind, g, sets, index):
    from quadruped_drake_b200 import load_robot
    from quadruped_drake_b200.capi import KINDS, WbcIO, WbcParams, make_params, np_ptr
    ms = load_robot(robot).as_struct()
    arr = (WbcParams * len(sets))(*[make_params(**d) for d in sets])
    n = len(index)
    tau, met, st = np.zeros((n, 12)), np.zeros((n, 4)), np.full(n, -1, np.int32)
    vd, f, qi, lam = np.zeros((n, 18)), np.zeros((n, 4, 3)), np.zeros((n, 4)), np.zeros((n, 42))
    io = WbcIO(np_ptr(g["q"]), np_ptr(g["v"]), np_ptr(g["traj"]), np_ptr(g["contact"]), np_ptr(tau), np_ptr(met), np_ptr(st), np_ptr(vd),
               np_ptr(f), np_ptr(qi), np_ptr(lam))
    index = np.ascontiguousarray(index, np.int32)
    assert emu.emu_step_params(C.byref(ms), arr, len(sets), np_ptr(index), KINDS[kind], n, C.byref(io)) == 0
    return tau, vd, f.reshape(n, 4, 3), st, lam


@pytest.mark.parametrize("kind", KIND_NAMES)
@pytest.mark.parametrize("case", ["cfg3_anymal_trot", "cfg4_mini_cheetah_walk"])
def test_emulated_rows_match_oracle_with_their_params(emu, case, kind):
    """12 golden states, 6 sets: each row against the oracle built with its own set (bars of test_emulator.py; PD 1e-12)."""
    n, k = 12, 6
    g, sets = golden(case, n), param_sets(k, 11)
    index = np.random.default_rng(3).permutation(np.arange(n) % k).astype(np.int32)
    tau, vd, f, st, _ = emu_step(emu, robot_of(case), kind, g, sets, index)
    check_rows_against_oracle(robot_of(case), kind, g, sets, index, tau, vd, f, st)


@pytest.mark.parametrize("kind", ["id", "pc", "pd"])
def test_emulated_bad_index_gives_badparams_and_zero_outputs(emu, kind):
    from quadruped_drake_b200.capi import ST_BADPARAMS
    n, k = 6, 3
    g, sets = golden("cfg4_mini_cheetah_walk", n), param_sets(k, 5)
    good = np.array([0, 1, 2, 0, 1, 2], np.int32)
    bad = good.copy()
    bad[[1, 4]] = [-1, k]
    a = emu_step(emu, "mini_cheetah", kind, g, sets, good)
    b = emu_step(emu, "mini_cheetah", kind, g, sets, bad)
    assert (b[3][[1, 4]] == ST_BADPARAMS).all()
    for x in b[:3] + (b[4],):
        assert (x[[1, 4]] == 0).all()
    rest = [0, 2, 3, 5]
    for x, y in zip(a, b):
        assert np.array_equal(x[rest], y[rest])


# ------------------------------------------------------------------------------------------------------------------ GPU half
gpu = pytest.mark.gpu
K = 8


@pytest.fixture(scope="module")
def ctl(built):
    from quadruped_drake_b200.controller import BatchedController
    c = BatchedController("mini_cheetah", device=0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sets8():
    return param_sets(K, 2026)


@pytest.fixture(scope="module")
def handles(ctl, sets8):
    """One handle per set: the reference each row must reproduce bit for bit."""
    from quadruped_drake_b200.controller import BatchedController
    hs = [BatchedController("mini_cheetah", device=0, **d) for d in sets8]
    yield hs
    for h in hs:
        h.close()


@pytest.fixture(scope="module")
def states(ctl):
    from quadruped_drake_b200.synth import generate
    return generate(ctl.model, 65536 + 3, 77, "mixed", ctl.fk)


def outputs(o):
    return {k: (getattr(o, k).cpu().numpy() if hasattr(getattr(o, k), "cpu") else getattr(o, k))
            for k in ("tau", "metrics", "status", "vd", "f", "qp_info", "lam")}


def assert_same(a, b, what, keys=("tau", "metrics", "status", "vd", "f", "qp_info", "lam")):
    for k in keys:
        assert np.array_equal(a[k], b[k]), (what, k)


@gpu
@pytest.mark.parametrize("kind", KIND_NAMES)
def test_identity_set_gives_the_bits_of_wbc_step(ctl, states, kind):
    """Every record equal to the handle's params, robots spread over 3 such records: the bits of wbc_step on every output, at
    sizes across the chunk thresholds, with the same launch count."""
    import torch
    from quadruped_drake_b200.controller import ParamSet
    ps = ParamSet(ctl, [ctl.params] * 3)
    rng = np.random.default_rng(1)
    for n in (1000, 4096, 8192, 65536 + 3):
        q, v, traj, contact = (torch.from_numpy(np.ascontiguousarray(x[:n])).cuda() for x in states)
        idx = torch.from_numpy(rng.integers(0, 3, n).astype(np.int32)).cuda()
        l0 = ctl.launches
        a = outputs(ctl.step(kind, q, v, traj, contact, debug=True))
        l1 = ctl.launches
        b = outputs(ctl.step(kind, q, v, traj, contact, debug=True, param_set=ps, param_index=idx))
        torch.cuda.synchronize()
        assert ctl.launches - l1 == l1 - l0, (kind, n)
        if kind == "pd":
            assert np.array_equal(a["tau"], b["tau"]) and (b["status"] == 0).all()
        else:
            assert_same(a, b, (kind, n))
    ps.close()


def host_step(ctl, kind, q, v, traj, contact, pinned, param_set=None, index=None):
    """wbc_step_host / wbc_step_params_host with every buffer page-locked (pinned) or pageable."""
    from quadruped_drake_b200 import capi
    from quadruped_drake_b200.controller import _ctrl_params
    n = len(q)
    mk = (lambda s, dt=np.float64: capi.pinned_empty(s, dt)) if pinned else (lambda s, dt=np.float64: np.empty(s, dt))
    ins = []
    for x, dt in ((q, np.float64), (v, np.float64), (traj, np.float64), (contact, np.uint8)):
        a = mk(x.shape, dt)
        a[...] = x
        ins.append(a)
    out = {"tau": mk((n, 12)), "metrics": mk((n, 4)), "status": mk((n,), np.int32), "vd": mk((n, 18)), "f": mk((n, 4, 3)),
           "qp_info": mk((n, 4)), "lam": mk((n, 42))}
    out["status"][...] = -7
    p = capi.np_ptr
    io = capi.WbcIO(*(p(a) for a in ins), *(p(out[k]) for k in ("tau", "metrics", "status", "vd", "f", "qp_info", "lam")))
    k = capi.KINDS[kind]
    if index is None:
        ctl._check(ctl.lib.wbc_step_host(ctl._h, k, n, C.byref(io)), "wbc_step_host")
    else:
        idx = mk((n,), np.int32)
        idx[...] = index
        cp = _ctrl_params(param_set, p(idx))
        ctl._check(ctl.lib.wbc_step_params_host(ctl._h, k, n, C.byref(io), C.byref(cp)), "wbc_step_params_host")
    return {k: np.array(x) for k, x in out.items()}


@gpu
@pytest.mark.parametrize("kind", ["id", "pc", "pd"])
def test_identity_set_host_paths(ctl, states, kind):
    """wbc_step_params_host with page-locked buffers below and above the staging threshold and with pageable buffers: the
    bits of wbc_step_host."""
    from quadruped_drake_b200.controller import ParamSet
    ps = ParamSet(ctl, [ctl.params] * 2)
    rng = np.random.default_rng(2)
    for n, pinned in ((4096, True), (32768, True), (4096, False), (40000, False)):
        q, v, traj, contact = (x[:n] for x in states)
        idx = rng.integers(0, 2, n).astype(np.int32)
        a = host_step(ctl, kind, q, v, traj, contact, pinned)
        b = host_step(ctl, kind, q, v, traj, contact, pinned, ps, idx)
        if kind == "pd":
            assert np.array_equal(a["tau"], b["tau"]) and (b["status"] == 0).all(), (n, pinned)
        else:
            assert_same(a, b, (kind, n, pinned))
    ps.close()


@gpu
@pytest.mark.parametrize("kind", KIND_NAMES)
def test_rows_match_separate_handles(ctl, handles, sets8, states, kind):
    """4096 robots assigned at random to 8 sets: every row has the bits of the handle created with its set, stepped on its
    subset; the device entry gives the bits of the host entry."""
    import torch
    from quadruped_drake_b200.controller import ParamSet
    ps = ParamSet(ctl, sets8)
    n = 4096
    q, v, traj, contact = (x[:n] for x in states)
    idx = np.random.default_rng(9).integers(0, K, n).astype(np.int32)
    if kind == "pd":
        tau, st = ctl.step_pd(q, v, param_set=ps, param_index=idx)
        assert (st == 0).all()
        for k in range(K):
            sel = idx == k
            assert np.array_equal(tau[sel], handles[k].step_pd(q[sel], v[sel])), k
        tt, ts = ctl.step_pd(torch.from_numpy(q).cuda(), torch.from_numpy(v).cuda(), param_set=ps, param_index=torch.from_numpy(idx).cuda())
        assert np.array_equal(tt.cpu().numpy(), tau) and (ts.cpu().numpy() == 0).all()
        ps.close()
        return
    got = outputs(ctl.step(kind, q, v, traj, contact, debug=True, param_set=ps, param_index=idx))
    assert (got["status"] == 0).mean() > 0.9
    for k in range(K):
        sel = idx == k
        ref = outputs(handles[k].step(kind, q[sel], v[sel], traj[sel], contact[sel], debug=True))
        assert_same({key: x[sel] for key, x in got.items()}, ref, (kind, k))
    dev = outputs(ctl.step(kind, *(torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (q, v, traj, contact)), debug=True,
                           param_set=ps, param_index=torch.from_numpy(idx).cuda()))
    assert_same(dev, got, kind)
    ps.close()


def grounded(ctl, n, rng, jitter):
    q0 = np.tile(np.array([1.0, 0, 0, 0, 0, 0, 0.3] + [0.0, -0.8, 1.6] * 4), (n, 1))
    q0[:, 7:] += rng.uniform(-jitter, jitter, (n, 12))
    pz = ctl.dynamics(q0, np.zeros((n, 18)))["p_feet"][:, :, 2]
    q0[:, 6] -= pz.min(axis=1)
    return q0


def trot_sampler(ctl):
    from quadruped_drake_b200 import planner as pl
    bh = float(grounded(ctl, 1, np.random.default_rng(0), 0.0)[0, 6])
    return pl.TrajectorySampler(ctl, pl.make_gait_plan("mini_cheetah", "trot", goal=(1.5, 0.0), base_height=bh))


ROLL_KEYS = ("q", "v", "t", "tau", "metrics", "status_or", "err_max")


@gpu
@pytest.mark.parametrize("plant", ["plain", "variants", "terrain"])
def test_ground_plant_rollout_matches_separate_handles(ctl, handles, sets8, plant):
    """512 robots, 400 steps on the ground plant - nominal robots, payload variants with pushes, or variants with pushes on
    terrain: each robot has the bits of wbc_rollout_ex / wbc_rollout_perturbed / wbc_rollout_terrain on the handle of its set."""
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import PlantSet, Terrain, TerrainSet, rollout
    from quadruped_drake_b200.urdf import load_description
    n, steps, dt = 512, 400, 5e-3
    rng = np.random.default_rng(21)
    q0 = grounded(ctl, n, rng, 0.02)
    s = trot_sampler(ctl)
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    ps = PlantSet(ctl, [flatten(d), flatten(with_payload(d, 1.2, (0.04, -0.02, 0.05)))], [1.0, 0.6])
    ts = TerrainSet(ctl, [Terrain(), Terrain(slope=(np.tan(np.radians(5.0)), 0.0))])
    push = np.zeros((n, 8))
    push[:, 0:3] = rng.uniform(-40, 40, (n, 3)); push[:, 3:6] = rng.uniform(-0.1, 0.1, (n, 3))
    push[:, 6], push[:, 7] = 0.5, 0.7
    per_robot = {"variant": (np.arange(n) % 2).astype(np.int32), "push": push, "terrain": (np.arange(n) // 2 % 2).astype(np.int32)}
    kw = {"plain": {}, "variants": dict(plant_set=ps), "terrain": dict(plant_set=ps, terrain_set=ts)}[plant]
    rows = {"plain": [], "variants": ["variant", "push"], "terrain": ["variant", "push", "terrain"]}[plant]
    idx = rng.integers(0, K, n).astype(np.int32)
    pset = ParamSet(ctl, sets8)
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, param_set=pset, param_index=idx,
                **kw, **{k: per_robot[k] for k in rows})
    for k in range(K):
        sel = idx == k
        ref = rollout(handles[k], s, "id", q0[sel], np.zeros((sel.sum(), 18)), 0.0, steps, dt, plant=True, **kw,
                      **{key: per_robot[key][sel] for key in rows})
        for key in ROLL_KEYS + ("f_contact",):
            assert np.array_equal(getattr(r, key)[sel], getattr(ref, key)), (plant, k, key)
    pset.close(); ts.close(); ps.close(); s.close()


@gpu
def test_host_rollout_keeps_a_converted_plan_index(ctl, handles, sets8):
    """A host rollout with parameter sets and an int64 plan index (converted to int32 inside rollout) gives the bits of the
    per-set handles given the same plans."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.rollout import rollout
    n, steps, dt = 256, 200, 5e-3
    rng = np.random.default_rng(23)
    q0 = grounded(ctl, n, rng, 0.02)
    bh = float(grounded(ctl, 1, np.random.default_rng(0), 0.0)[0, 6])
    s = pl.TrajectorySampler(ctl, [pl.make_gait_plan("mini_cheetah", "trot", goal=(1.5, 0.0), base_height=bh),
                                   pl.make_motion_plan("mini_cheetah", "heave", 6.0, base_height=bh)])
    plan_index = np.arange(n) % 2                       # int64
    idx = rng.integers(0, K, n).astype(np.int32)
    pset = ParamSet(ctl, sets8)
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, dt, plan_index=plan_index, param_set=pset, param_index=idx.tolist())
    for k in range(K):
        sel = idx == k
        ref = rollout(handles[k], s, "id", q0[sel], np.zeros((sel.sum(), 18)), 0.0, steps, dt, plan_index=plan_index[sel].astype(np.int32))
        for key in ROLL_KEYS:
            assert np.array_equal(getattr(r, key)[sel], getattr(ref, key)), (k, key)
    pset.close(); s.close()


@gpu
def test_device_index_must_be_int32_cuda(ctl, sets8, states):
    """An index tensor of another dtype, device or shape is refused before anything is launched."""
    import torch
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.rollout import rollout
    ps = ParamSet(ctl, sets8)
    n = 64
    q, v, traj, contact = (torch.from_numpy(np.ascontiguousarray(x[:n])).cuda() for x in states)
    good = torch.zeros(n, dtype=torch.int32, device="cuda")
    for bad in (torch.zeros(n, dtype=torch.int64, device="cuda"), torch.zeros(n, dtype=torch.int32), good[: n - 1],
                torch.zeros(2 * n, dtype=torch.int32, device="cuda")[::2]):
        with pytest.raises(ValueError, match="int32"):
            ctl.step("id", q, v, traj, contact, param_set=ps, param_index=bad)
        with pytest.raises(ValueError, match="int32"):
            ctl.step_pd(q, v, param_set=ps, param_index=bad)
    s = trot_sampler(ctl)
    with pytest.raises(ValueError, match="int32"):
        rollout(ctl, s, "id", q.clone(), v.clone(), torch.zeros(n, dtype=torch.float64, device="cuda"), 2, 5e-3, param_set=ps,
                param_index=torch.arange(n, device="cuda"))
    ps.close(); s.close()


@gpu
def test_integrator_rollout_matches_separate_handles(ctl, handles, sets8):
    """The same with the integrator plant against wbc_rollout_ex; the device entry gives the host entry's bits."""
    import torch
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.rollout import rollout
    n, steps, dt = 512, 400, 5e-3
    rng = np.random.default_rng(22)
    q0 = grounded(ctl, n, rng, 0.02)
    s = trot_sampler(ctl)
    idx = rng.integers(0, K, n).astype(np.int32)
    pset = ParamSet(ctl, sets8)
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, dt, param_set=pset, param_index=idx)
    for k in range(K):
        sel = idx == k
        ref = rollout(handles[k], s, "id", q0[sel], np.zeros((sel.sum(), 18)), 0.0, steps, dt)
        for key in ROLL_KEYS:
            assert np.array_equal(getattr(r, key)[sel], getattr(ref, key)), (k, key)
    q, v, t = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
    with torch.cuda.stream(torch.cuda.Stream()):
        l0 = ctl.launches
        rollout(ctl, s, "id", q, v, t, steps, dt, param_set=pset, param_index=torch.from_numpy(idx).cuda())
        l1 = ctl.launches
        rollout(ctl, s, "id", q.clone().copy_(torch.from_numpy(q0)), v.clone().zero_(), t.clone().zero_(), steps, dt)
        l2 = ctl.launches
    torch.cuda.synchronize()
    assert np.array_equal(q.cpu().numpy(), r.q) and np.array_equal(v.cpu().numpy(), r.v)
    assert l1 - l0 == l2 - l1
    pset.close(); s.close()


@gpu
@pytest.mark.parametrize("kind", ["id", "clf", "pc", "mptc", "pd"])
def test_golden_parity_with_per_row_params(ctl, kind):
    """Golden states of mini_cheetah, 24 rows over 8 sets: each row within the parity bars of the oracle with its set."""
    from quadruped_drake_b200.controller import ParamSet
    sets = param_sets(K, 31)
    ps = ParamSet(ctl, sets)
    n = 24
    g = golden("cfg4_mini_cheetah_walk", n)
    idx = (np.arange(n) % K).astype(np.int32)
    if kind == "pd":
        tau, st = ctl.step_pd(g["q"], g["v"], param_set=ps, param_index=idx)
        check_rows_against_oracle("mini_cheetah", kind, g, sets, idx, tau, None, None, st)
    else:
        o = ctl.step(kind, g["q"], g["v"], g["traj"], g["contact"], debug=True, param_set=ps, param_index=idx)
        check_rows_against_oracle("mini_cheetah", kind, g, sets, idx, o.tau, o.vd, o.f, o.status)
    ps.close()


@gpu
@pytest.mark.parametrize("kind", ["id", "clf"])
def test_kkt_certificate_with_per_row_params(ctl, sets8, states, kind):
    """65536 + 3 instances over 8 sets: every solved row satisfies the KKT conditions of the reference QP with its own
    parameters, and rows with torque limits stay within the effort limits."""
    import kkt
    from types import SimpleNamespace
    from quadruped_drake_b200.controller import ParamSet
    ps = ParamSet(ctl, sets8)
    q, v, traj, contact = states
    n = len(q)
    idx = np.random.default_rng(4).integers(0, K, n).astype(np.int32)
    out = ctl.step(kind, q, v, traj, contact, debug=True, param_set=ps, param_index=idx)
    assert (out.status == 0).mean() > 0.9
    effort = np.asarray(ctl.model.as_struct().effort)
    act = np.asarray(ctl.model.as_struct().act_index)
    eff_act = np.empty(12)
    eff_act[act] = effort
    for k in range(K):
        sel = (idx == k) & (out.status == 0)
        if sets8[k]["torque_limits"]:
            assert (np.abs(out.tau[sel]) <= eff_act + 1e-9).all(), k
        for part in np.array_split(np.flatnonzero(sel), 4):
            o = SimpleNamespace(tau=out.tau[part], vd=out.vd[part], f=out.f[part], qp_info=out.qp_info[part], lam=out.lam[part])
            cert = kkt.certificate(kind, ctl.dynamics(q[part], v[part]), ctl.model, q[part], v[part], traj[part], contact[part], o,
                                   oracle_kw(sets8[k]))
            assert cert["stationarity"].max() < 1e-6 and cert["comp"].max() < 1e-6, (k, cert["stationarity"].max())
            assert cert["dual"].min() >= 0.0 and cert["eq"].max() < 1e-7 and cert["ineq"].max() < 1e-7
    ps.close()


@gpu
@pytest.mark.parametrize("kind", ["id", "pc", "pd"])
def test_bad_indices_are_flagged_and_neighbours_unaffected(ctl, sets8, states, kind):
    from quadruped_drake_b200.capi import ST_BADPARAMS
    from quadruped_drake_b200.controller import ParamSet
    ps = ParamSet(ctl, sets8)
    n = 5000
    q, v, traj, contact = (x[:n] for x in states)
    good = np.random.default_rng(6).integers(0, K, n).astype(np.int32)
    bad = good.copy()
    rows = [0, 17, 2048, 4999]
    bad[rows] = [-1, K, -5, K + 3]
    rest = np.setdiff1d(np.arange(n), rows)
    if kind == "pd":
        ta, sa = ctl.step_pd(q, v, param_set=ps, param_index=good)
        tb, sb = ctl.step_pd(q, v, param_set=ps, param_index=bad)
        assert (sb[rows] == ST_BADPARAMS).all() and (tb[rows] == 0).all() and (sb[rest] == 0).all()
        assert np.array_equal(ta[rest], tb[rest])
    else:
        a = outputs(ctl.step(kind, q, v, traj, contact, debug=True, param_set=ps, param_index=good))
        b = outputs(ctl.step(kind, q, v, traj, contact, debug=True, param_set=ps, param_index=bad))
        assert (b["status"][rows] & ST_BADPARAMS).all()
        for key in ("tau", "vd", "f", "lam"):
            assert (b[key][rows] == 0).all(), key
        assert_same({k: x[rest] for k, x in a.items()}, {k: x[rest] for k, x in b.items()}, kind)
    ps.close()


@gpu
def test_bad_index_robot_is_frozen_in_a_rollout(ctl, sets8):
    from quadruped_drake_b200.capi import ST_BADPARAMS
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.rollout import rollout
    n = 64
    q0 = grounded(ctl, n, np.random.default_rng(8), 0.02)
    s = trot_sampler(ctl)
    ps = ParamSet(ctl, sets8)
    idx = (np.arange(n) % K).astype(np.int32)
    idx[[5, 40]] = [-1, K]
    r = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 100, 5e-3, param_set=ps, param_index=idx)
    assert (r.status_or[[5, 40]] & ST_BADPARAMS).all()
    assert np.array_equal(r.q[[5, 40]], q0[[5, 40]]) and (r.v[[5, 40]] == 0).all()
    assert not (r.status_or[np.setdiff1d(np.arange(n), [5, 40])] & ST_BADPARAMS).any()
    ps.close(); s.close()


@gpu
def test_rejected_sets_and_arguments(ctl, built):
    import torch
    from quadruped_drake_b200.capi import WbcCtrlParams, WbcParams, WbcPlantPerturb, WbcRolloutIO, WbcRolloutOpts, make_params
    from quadruped_drake_b200.controller import ParamSet
    bad = [dict(reg_vd=1e-3), dict(reg_f=0.0), dict(id_kp_body_p=float("nan")), dict(pd_q_nom=(float("inf"),) + (0.0,) * 11),
           dict(max_iter=0), dict(torque_limits=2), dict(mu=-0.1), dict(clf_r=0.0), dict(clf_q_body_p=-1.0), dict(clf_w_delta=-1.0)]
    for d in bad:
        with pytest.raises(RuntimeError, match="wbc_param_set_create"):
            ParamSet(ctl, [{}, d])
    h = C.c_void_p()
    arr = (WbcParams * 1)(make_params())
    assert ctl.lib.wbc_param_set_create(ctl._h, 0, arr, C.byref(h)) == 1 and not h
    # perturbations on the integrator plant
    ps = ParamSet(ctl, [{}])
    s = trot_sampler(ctl)
    n = 4
    q, v, t = np.tile(grounded(ctl, 1, np.random.default_rng(0), 0.0), (n, 1)), np.zeros((n, 18)), np.zeros(n)
    io = WbcRolloutIO(q.ctypes.data, v.ctypes.data, t.ctypes.data, None, None, None, None, None, None)
    o = WbcRolloutOpts(1, 0)
    pt = WbcPlantPerturb(None, None, None)
    cp = WbcCtrlParams(ps._p, None)
    assert ctl.lib.wbc_rollout_params_host(ctl._h, 0, s._p, n, 2, 5e-3, C.byref(io), C.byref(o), C.byref(pt), None, C.byref(cp)) == 1
    assert b"ground plant" in ctl.lib.wbc_last_error(ctl._h)
    # a set from another device
    if torch.cuda.device_count() > 1:
        from quadruped_drake_b200.controller import BatchedController
        other = BatchedController("mini_cheetah", device=1)
        ps1 = ParamSet(other, [{}])
        with pytest.raises(RuntimeError, match="another device"):
            ctl.step("id", *(x[:n] for x in (q, v, np.zeros((n, 54)), np.ones((n, 4), np.uint8))), param_set=ps1)
        ps1.close(); other.close()
    ps.close(); s.close()
