"""Both variants of the solve kernel against the oracle: wbc_solve[_params]_kernel<KIND, VD>.

VD = true is launched when the caller asks for the accelerations (L stays in H, R^-1 in its own array); VD = false for every
other call (R^-1 overlaid on the dead factor, SolveSmem in csrc/wbc_device.cuh): the benchmark, wbc_step_host without vd, the
LeafSystem mirrors and every ground-plant rollout. Each check below runs in both variants, for every controller:

- golden vectors and the frozen deep-active-set instances of tests/golden/hard_tail.npz (tools/make_golden_hard.py: the 16
  status-0 instances with the most pivots of 13 seeded 65536-instance batches) at the golden bars, and bit for bit between the
  variants;
- the iteration cap: with max_iter = k (the pivots an instance takes) the bits of the default handle, with k - 1 exactly
  WBC_ST_MAXITER with zero outputs (include/wbc.h);
- every on/off subset of the optional outputs, ragged sizes, permutations, unaligned rows and host buffers (GPU).

CPU half on the host warp emulator (tests/emu), which picks the variant the way the library does; GPU half on the B200."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

GOLD = Path(__file__).parent / "golden"
OUTS = ("tau", "metrics", "status", "vd", "f", "qp_info", "lam")
OPTIONAL = ("vd", "f", "qp_info", "lam")
ST_MAXITER = 1
HARD = np.load(GOLD / "hard_tail.npz")
HARD_NAMES = [str(x) for x in HARD["names"]]


def robot_of(case):
    return "anymal_b" if "anymal" in case else "mini_cheetah"


def handle_kw(case):
    """dof order and torque box of a golden file (tools/make_golden.py)."""
    return dict(dof_order="breadth_first" if case.startswith("bf_") else "depth_first",
                **({"torque_limits": 1} if case.startswith("tl_") else {}))


def hard_combo(name, deepest=None):
    """Rows of one combination of hard_tail.npz (stored deepest first), its robot, kind and handle keywords."""
    c = HARD_NAMES.index(name)
    rows = np.flatnonzero(HARD["combo"] == c)
    rows = rows[np.argsort(-HARD["pivots"][rows], kind="stable")][:deepest]
    g = {k: np.ascontiguousarray(HARD[k][rows]) for k in ("q", "v", "traj", "contact", "tau", "vd", "f", "metrics", "objective", "ok")}
    kw = dict(dof_order=str(HARD["dof_orders"][c]), **({"torque_limits": 1} if HARD["torque_limits"][c] else {}))
    return g, str(HARD["robots"][c]), str(HARD["kinds"][c]), kw


def oracle_rows(g, kind, prefix=""):
    """Golden arrays of one kind under plain names (tau, vd, f, metrics, objective, ok)."""
    return {k: g[prefix + k] for k in ("tau", "vd", "f", "metrics", "objective", "ok")}


def assert_golden(kind, contact, ref, o):
    """The bars of test_emulator.py / test_gpu_parity.py on the rows the oracle certified: tau and f 1e-5, vd 1e-6 (where
    produced), objective 1e-6 relative (ID and CLF, as there), metrics 1e-12 (ID err) / 1e-8 relative (V, err, Vdot). Rows
    that fail carry zero torques; PC and MPTC in full flight are WBC_ST_UNSUPPORTED."""
    ok = ref["ok"]
    assert ok.mean() >= 0.75, ok.mean()
    assert (o["status"][ok] == 0).all(), np.unique(o["status"][ok], return_counts=True)
    if kind in ("pc", "mptc"):
        assert (o["status"][contact.sum(axis=1) == 0] == 64).all()
    assert np.abs(o["tau"] - ref["tau"])[ok].max() < 1e-5
    assert (o["tau"][o["status"] != 0] == 0).all()
    if o.get("f") is not None:
        assert np.abs(o["f"].reshape(-1, 4, 3) - ref["f"])[ok].max() < 1e-5
    if o.get("vd") is not None:
        assert np.abs(o["vd"] - ref["vd"])[ok].max() < 1e-6
    if o.get("qp_info") is not None and kind in ("id", "clf"):
        obj = ref["objective"][ok]
        assert np.abs(o["qp_info"][ok, 0] - obj).max() < 1e-6 * max(1.0, np.abs(obj).max())
    m, r = o["metrics"][ok], ref["metrics"][ok]
    if kind == "id":
        assert np.abs(m[:, 1] - r[:, 1]).max() < 1e-12
    else:
        assert (np.abs(m - r)[:, [0, 1, 3]] / np.maximum(1.0, np.abs(r[:, [0, 1, 3]]))).max() < 1e-8


def assert_same(a, b, what, keys=OUTS):
    for k in keys:
        if a.get(k) is not None and b.get(k) is not None:
            assert np.array_equal(a[k], b[k]), (what, k)


def assert_capped(o, rows, what):
    """WBC_ST_MAXITER exactly, and tau, f, vd (where requested) and lam zero (include/wbc.h)."""
    assert (o["status"][rows] == ST_MAXITER).all(), (what, o["status"][rows])
    for k in ("tau", "f", "vd", "lam"):
        if o.get(k) is not None:
            assert (o[k][rows] == 0).all(), (what, k)


def param_records(k, seed, torque_limits):
    """k parameter sets: task gains and weights x 0.5 - 2, mu 0.4 - 1.0, the combination's torque box."""
    from quadruped_drake_b200.capi import DEFAULT_PARAMS
    scaled = ["id_kp_body_p", "id_kd_body_p", "id_kp_body_rpy", "id_kd_body_rpy", "id_kp_foot", "id_kd_foot", "id_w_body", "id_w_foot",
              "clf_q_body_p", "clf_q_body_pd", "clf_q_body_rpy", "clf_q_body_rpyd", "clf_q_foot_p", "clf_q_foot_pd", "clf_w_delta",
              "pc_kp_body_p", "pc_kd_body_p", "pc_kp_body_rpy", "pc_kd_body_rpy", "pc_kp_foot", "pc_kd_foot", "pc_w_body", "pc_w_foot"]
    rng = np.random.default_rng(seed)
    return [dict({n: DEFAULT_PARAMS[n] * float(rng.uniform(0.5, 2.0)) for n in scaled}, mu=float(rng.uniform(0.4, 1.0)),
                 torque_limits=torque_limits) for _ in range(k)]


# ------------------------------------------------------------------------------------------------------------------ CPU half
# (case, kind) pairs of test_emulator.py
EMU_PAIRS = ([(c, "id") for c in ("cfg2_mini_cheetah_stand", "cfg3_anymal_trot", "cfg4_mini_cheetah_walk", "mixed_mini_cheetah")]
             + [(c, k) for c in ("cfg3_anymal_trot", "cfg4_mini_cheetah_walk") for k in ("clf", "pc", "mptc")]
             + [("bf_mini_cheetah_mixed", "id"), ("bf_anymal_trot", "clf"), ("bf_mini_cheetah_mixed", "pc"), ("tl_mini_cheetah_walk", "id"),
                ("tl_anymal_trot", "id"), ("fixtures_mini_cheetah", "id"), ("fixtures_mini_cheetah", "clf")])
EMU_ROWS = slice(24, 32)    # 8 instances per pair, past the ones test_emulator.py runs (~0.25 s per instance and variant)
EMU_DEEP = 4                # deepest instances per combination of hard_tail.npz


@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu.so"))
    lib.emu_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
    return lib


def emu_run(emu, robot, kind, g, with_vd, dof_order="depth_first", **params):
    """One emulated step with f, qp_info and lam on, vd on or off (which picks the solve variant). Outputs start as NaN / -7
    so that an output the step does not write cannot pass."""
    from quadruped_drake_b200 import load_robot
    from quadruped_drake_b200.capi import KINDS, NLAM, WbcIO, make_params, np_ptr
    ms, pr = load_robot(robot, dof_order=dof_order).as_struct(), make_params(**params)
    q, v, traj, contact = (np.ascontiguousarray(g[k]) for k in ("q", "v", "traj", "contact"))
    n = len(q)
    o = {"tau": np.full((n, 12), np.nan), "metrics": np.full((n, 4), np.nan), "status": np.full(n, -7, np.int32),
         "vd": np.full((n, 18), np.nan) if with_vd else None, "f": np.full((n, 4, 3), np.nan), "qp_info": np.full((n, 4), np.nan),
         "lam": np.full((n, NLAM), np.nan)}
    io = WbcIO(np_ptr(q), np_ptr(v), np_ptr(traj), np_ptr(contact), *(None if o[k] is None else np_ptr(o[k]) for k in OUTS[:3] + OPTIONAL))
    assert emu.emu_step(C.byref(ms), C.byref(pr), KINDS[kind], n, C.byref(io)) == 0
    return o


def golden_rows(case, rows=EMU_ROWS):
    g = np.load(GOLD / f"{case}.npz")
    return {k: (g[k][rows] if g[k].ndim and k not in ("dof_order", "params") else g[k]) for k in g.files}


@pytest.mark.parametrize("case,kind", EMU_PAIRS)
def test_emulated_golden_without_accelerations(emu, case, kind):
    """Goldens through the VD = false variant at the golden bars, and bit for bit the VD = true variant's outputs."""
    g = golden_rows(case)
    kw = handle_kw(case)
    a = emu_run(emu, robot_of(case), kind, g, False, **kw)
    b = emu_run(emu, robot_of(case), kind, g, True, **kw)
    ref = oracle_rows(g, kind, kind + "_")
    assert_golden(kind, g["contact"], ref, a)
    assert_golden(kind, g["contact"], ref, b)
    assert_same(a, b, (case, kind))


@pytest.mark.parametrize("name", HARD_NAMES)
def test_emulated_deep_instances_match_oracle(emu, name):
    """The deepest instances of hard_tail.npz (20+ pivots, drops and re-adds) in both variants against the oracle."""
    g, robot, kind, kw = hard_combo(name, EMU_DEEP)
    a = emu_run(emu, robot, kind, g, False, **kw)
    b = emu_run(emu, robot, kind, g, True, **kw)
    assert_golden(kind, g["contact"], oracle_rows(g, kind), a)
    assert_golden(kind, g["contact"], oracle_rows(g, kind), b)
    assert_same(a, b, name)


@pytest.mark.parametrize("kind", ["clf", "pc"])
def test_emulated_params_step_without_accelerations(built, kind):
    """The parameter-aware step (tests/emu/emu_step_params.cpp) in both variants: 12 golden states over 6 parameter records,
    bit for bit between the variants, and each row against the oracle built with its record."""
    from oracle import controllers as oc
    from quadruped_drake_b200 import load_robot
    from quadruped_drake_b200.capi import KINDS, NLAM, WbcIO, WbcParams, make_params, np_ptr
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_params.so"))
    lib.emu_step_params.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
    g = golden_rows("cfg4_mini_cheetah_walk", slice(0, 12))
    sets = param_records(6, 7, 0)
    index = np.ascontiguousarray(np.random.default_rng(4).permutation(np.arange(12) % 6), np.int32)
    ms, arr = load_robot("mini_cheetah").as_struct(), (WbcParams * 6)(*[make_params(**d) for d in sets])
    runs = []
    for with_vd in (False, True):
        o = {"tau": np.full((12, 12), np.nan), "metrics": np.full((12, 4), np.nan), "status": np.full(12, -7, np.int32),
             "vd": np.full((12, 18), np.nan) if with_vd else None, "f": np.full((12, 4, 3), np.nan), "qp_info": np.full((12, 4), np.nan),
             "lam": np.full((12, NLAM), np.nan)}
        io = WbcIO(*(np_ptr(np.ascontiguousarray(g[k])) for k in ("q", "v", "traj", "contact")),
                   *(None if o[k] is None else np_ptr(o[k]) for k in OUTS[:3] + OPTIONAL))
        assert lib.emu_step_params(C.byref(ms), arr, 6, np_ptr(index), KINDS[kind], 12, C.byref(io)) == 0
        runs.append(o)
    assert_same(runs[0], runs[1], kind)
    ctrl = {"clf": oc.CLFController, "pc": oc.PCController}[kind]
    solved = 0
    for i in range(12):
        if runs[0]["status"][i] != 0:
            continue
        d = {k: x for k, x in sets[index[i]].items() if k in oc.DEFAULTS}
        ref = ctrl("mini_cheetah", **d).control_law(g["q"][i], g["v"][i], oc.traj_to_dict(g["traj"][i], g["contact"][i]))
        assert np.abs(runs[0]["tau"][i] - ref.tau).max() < 1e-5 and np.abs(runs[1]["vd"][i] - ref.vd).max() < 1e-6, i
        assert np.abs(runs[0]["f"][i] - ref.f).max() < 1e-5, i
        solved += 1
    assert solved >= 8


CAP_GOLDEN = [("cfg4_mini_cheetah_walk", "clf"), ("cfg3_anymal_trot", "pc"), ("tl_anymal_trot", "id")]
CAP_DEEP = ["stand_mini_cheetah_clf_box", "stand_anymal_b_mptc", "stand_mini_cheetah_pc"]


@pytest.mark.parametrize("source", [f"{c}:{k}" for c, k in CAP_GOLDEN] + CAP_DEEP)
def test_emulated_iteration_cap(emu, source):
    """The instance with the most pivots k among the rows: max_iter = k gives the default bits, max_iter = k - 1 exactly
    WBC_ST_MAXITER with zero outputs, in both variants (qp_info is written whatever the status: not compared there)."""
    if ":" in source:
        case, kind = source.split(":")
        g, robot, kw = golden_rows(case), robot_of(case), handle_kw(case)
    else:
        g, robot, kind, kw = hard_combo(source, 1)
    base = emu_run(emu, robot, kind, g, True, **kw)
    piv = np.where(base["status"] == 0, base["qp_info"][:, 3], -1)
    i = int(np.argmax(piv))
    k = int(piv[i])
    assert k >= 2, (source, k)
    one = {key: g[key][i:i + 1] for key in ("q", "v", "traj", "contact")}
    for with_vd in (False, True):
        ref = emu_run(emu, robot, kind, one, with_vd, **kw)
        assert ref["status"][0] == 0 and ref["qp_info"][0, 3] == k
        assert_same(ref, emu_run(emu, robot, kind, one, with_vd, max_iter=k, **kw), (source, with_vd, k))
        assert_capped(emu_run(emu, robot, kind, one, with_vd, max_iter=k - 1, **kw), [0], (source, with_vd, k - 1))


# ------------------------------------------------------------------------------------------------------------------ GPU half
gpu = pytest.mark.gpu
GOLDEN_FILES = ["cfg2_mini_cheetah_stand", "cfg3_anymal_trot", "cfg4_mini_cheetah_walk", "mixed_mini_cheetah", "bf_mini_cheetah_mixed",
                "bf_anymal_trot", "tl_mini_cheetah_walk", "tl_anymal_trot", "fixtures_mini_cheetah"]
KINDS4 = ["id", "clf", "pc", "mptc"]


@pytest.fixture(scope="module")
def ctl_cache(built):
    from quadruped_drake_b200.controller import BatchedController
    cache = {}

    def get(robot, dof_order="depth_first", **params):
        key = (robot, dof_order, tuple(sorted(params.items())))
        if key not in cache:
            cache[key] = BatchedController(robot, device=0, dof_order=dof_order, **params)
        return cache[key]
    yield get
    for c in cache.values():
        c.close()


def np_outputs(o):
    return {k: (None if getattr(o, k) is None else np.asarray(getattr(o, k).cpu() if hasattr(getattr(o, k), "cpu") else getattr(o, k)))
            for k in OUTS}


def host_step(ctl, kind, ins, want=OPTIONAL, pinned=False, param_set=None, index=None, bufs=None):
    """wbc_step_host (wbc_step_params_host with a parameter set) with the optional outputs in `want`, every buffer pageable or
    page-locked. `bufs` (inputs and all outputs, reused across calls) avoids a page-locked allocation per call; outputs start as
    NaN / -7."""
    from quadruped_drake_b200 import capi
    from quadruped_drake_b200.controller import _ctrl_params
    n = len(ins[0])
    if bufs is None:
        bufs = host_buffers(ins, pinned)
    for k in OUTS:
        bufs[k][...] = -7 if k == "status" else np.nan
    p = capi.np_ptr
    io = capi.WbcIO(*(p(bufs[k]) for k in ("q", "v", "traj", "contact", "tau", "metrics", "status")),
                    *(p(bufs[k]) if k in want else None for k in OPTIONAL))
    kk = capi.KINDS[kind]
    if param_set is None:
        ctl._check(ctl.lib.wbc_step_host(ctl._h, kk, n, C.byref(io)), "wbc_step_host")
    else:
        idx = np.ascontiguousarray(index, np.int32)
        cp = _ctrl_params(param_set, p(idx))
        ctl._check(ctl.lib.wbc_step_params_host(ctl._h, kk, n, C.byref(io), C.byref(cp)), "wbc_step_params_host")
    return {k: (np.array(bufs[k]) if k in OUTS[:3] or k in want else None) for k in OUTS}


def host_buffers(ins, pinned):
    from quadruped_drake_b200 import capi
    n = len(ins[0])
    mk = (lambda s, dt=np.float64: capi.pinned_empty(s, dt)) if pinned else (lambda s, dt=np.float64: np.empty(s, dt))
    b = {}
    for k, x, dt in zip(("q", "v", "traj", "contact"), ins, (np.float64, np.float64, np.float64, np.uint8)):
        b[k] = mk(x.shape, dt)
        b[k][...] = x
    b.update(tau=mk((n, 12)), metrics=mk((n, 4)), status=mk((n,), np.int32), vd=mk((n, 18)), f=mk((n, 4, 3)), qp_info=mk((n, 4)),
             lam=mk((n, capi.NLAM)))
    return b


def dev_step(ctl, kind, tins, want):
    """wbc_step on device tensors through make_io with the optional outputs in `want` (torch's current stream)."""
    import torch
    from quadruped_drake_b200 import capi
    n, dev = tins[0].shape[0], tins[0].device
    shapes = {"tau": (n, 12), "metrics": (n, 4), "vd": (n, 18), "f": (n, 4, 3), "qp_info": (n, 4), "lam": (n, capi.NLAM)}
    o = {k: torch.full(shapes[k], float("nan"), dtype=torch.float64, device=dev) for k in ("tau", "metrics")}
    o["status"] = torch.full((n,), -7, dtype=torch.int32, device=dev)
    for k in OPTIONAL:
        o[k] = torch.full(shapes[k], float("nan"), dtype=torch.float64, device=dev) if k in want else None
    io = ctl.make_io(*tins, o["tau"], o["metrics"], o["status"], o["vd"], o["f"], o["qp_info"], o["lam"])
    stream = torch.cuda.current_stream(dev)
    assert ctl.lib.wbc_step(ctl._h, capi.KINDS[kind], n, C.byref(io), C.c_void_p(stream.cuda_stream)) == 0
    torch.cuda.synchronize()
    return {k: (None if x is None else x.cpu().numpy()) for k, x in o.items()}


@gpu
@pytest.mark.parametrize("kind", KINDS4)
@pytest.mark.parametrize("case", GOLDEN_FILES)
def test_benchmark_variant_matches_golden(ctl_cache, case, kind):
    """Every golden file stepped as the benchmark steps it (tau, metrics, status: the VD = false kernel) at the bars of
    test_gpu_parity.py, and bit for bit the debug=True step."""
    g = np.load(GOLD / f"{case}.npz")
    if f"{kind}_tau" not in g.files:
        pytest.skip("golden file holds no vectors of this controller")
    ctl = ctl_cache(robot_of(case), **handle_kw(case))
    a = np_outputs(ctl.step(kind, g["q"], g["v"], g["traj"], g["contact"]))
    b = np_outputs(ctl.step(kind, g["q"], g["v"], g["traj"], g["contact"], debug=True))
    assert a["vd"] is None and a["lam"] is None
    ref = oracle_rows(g, kind, kind + "_")
    assert ref["ok"].mean() > 0.95 or (kind in ("pc", "mptc") and (ref["ok"] | (g["contact"].sum(axis=1) == 0)).mean() > 0.95)
    assert_golden(kind, g["contact"], ref, a)
    assert_same(a, b, (case, kind), ("tau", "metrics", "status"))


SUBSET_CASE = {"id": "tl_anymal_trot", "clf": "cfg4_mini_cheetah_walk", "pc": "cfg3_anymal_trot", "mptc": "bf_mini_cheetah_mixed"}
SUBSETS = [tuple(k for j, k in enumerate(OPTIONAL) if (m >> j) & 1) for m in range(16)]
ZERO_COPY_LIMIT = {"id": 24576, "clf": 24576, "pc": 131072, "mptc": 131072}     # include/wbc.h


@gpu
@pytest.mark.parametrize("kind", KINDS4)
def test_optional_output_subsets(ctl_cache, kind):
    """All 16 on/off combinations of (vd, f, qp_info, lam): tau, metrics and status identical across them, and every requested
    output identical to the all-on call; on device tensors, and through wbc_step_host with pageable and page-locked buffers on
    each side of the zero-copy limit."""
    import torch
    case = SUBSET_CASE[kind]
    g = np.load(GOLD / f"{case}.npz")
    ctl = ctl_cache(robot_of(case), **handle_kw(case))
    tins = [torch.from_numpy(np.ascontiguousarray(g[k])).cuda() for k in ("q", "v", "traj", "contact")]
    full = dev_step(ctl, kind, tins, OPTIONAL)
    assert (full["status"] == 0).mean() > 0.5
    for want in SUBSETS:
        assert_same(dev_step(ctl, kind, tins, want), full, ("device", kind, want))
    from quadruped_drake_b200.synth import generate
    lim = ZERO_COPY_LIMIT[kind]
    for n in (lim - 1, lim + 5):
        ins = generate(ctl.model, n, 4000 + n, "walk", ctl.fk)
        ref = None
        for pinned in (False, True):
            bufs = host_buffers(ins, pinned)
            for want in SUBSETS[::-1]:                          # all-on first
                o = host_step(ctl, kind, ins, want, pinned, bufs=bufs)
                if ref is None:
                    ref = o
                    assert (ref["status"] == 0).mean() > 0.5
                assert_same(o, ref, ("host", kind, n, pinned, want))
            del bufs


@gpu
@pytest.mark.parametrize("name", HARD_NAMES)
def test_deep_instances_match_oracle(ctl_cache, name):
    """All 16 instances of a hard_tail.npz combination in both variants against the oracle (vd where it is produced), the
    variants bit for bit, and for ID and CLF the KKT certificate of the reference QP on the VD run."""
    import kkt
    from types import SimpleNamespace
    g, robot, kind, kw = hard_combo(name)
    ctl = ctl_cache(robot, **kw)
    ins = [g[k] for k in ("q", "v", "traj", "contact")]
    a = host_step(ctl, kind, ins, ("f", "qp_info", "lam"))
    b = np_outputs(ctl.step(kind, *ins, debug=True))
    assert_golden(kind, g["contact"], oracle_rows(g, kind), a)
    assert_golden(kind, g["contact"], oracle_rows(g, kind), b)
    assert_same(a, b, name)
    if kind in ("id", "clf"):
        ok = b["status"] == 0
        out = SimpleNamespace(**{k: b[k][ok] for k in ("tau", "vd", "f", "qp_info", "lam")})
        sel = [x[ok] for x in ins]
        params = {"torque_limits": 1} if kw.get("torque_limits") else None
        cert = kkt.certificate(kind, ctl.dynamics(sel[0], sel[1]), ctl.model, *sel, out, params)
        assert cert["stationarity"].max() < 1e-6 and cert["dual"].min() >= 0.0 and cert["comp"].max() < 1e-6
        assert cert["eq"].max() < 1e-7 and cert["ineq"].max() < 1e-7


@gpu
@pytest.mark.parametrize("name", HARD_NAMES)
def test_deep_batches_variants_agree(ctl_cache, name):
    """The whole 65536-instance batch a hard_tail.npz combination was chosen from (every pivot count up to the batch maximum):
    the VD = false step (f, qp_info, lam on) and the debug=True step agree bit for bit; and wbc_step_params with 8 parameter
    records in the VD = false variant gives, row by row, the bits of 8 handles created with those records."""
    from quadruped_drake_b200.controller import BatchedController, ParamSet
    from quadruped_drake_b200.synth import generate
    c = HARD_NAMES.index(name)
    robot, kind, dof_order = str(HARD["robots"][c]), str(HARD["kinds"][c]), str(HARD["dof_orders"][c])
    tl = int(HARD["torque_limits"][c])
    pattern = "mixed" if name.startswith("bf_") else "stand"
    ctl = ctl_cache(robot, dof_order, **({"torque_limits": 1} if tl else {}))
    ins = generate(ctl.model, int(HARD["n_batch"]), int(HARD["seeds"][c]), pattern, ctl.fk)
    want = ("f", "qp_info", "lam")
    a = host_step(ctl, kind, ins, want)
    b = np_outputs(ctl.step(kind, *ins, debug=True))
    assert (a["status"] == 0).mean() > 0.95
    assert_same(a, b, name)
    recs = param_records(8, 100 + c, tl)
    ps = ParamSet(ctl, recs)
    idx = np.random.default_rng(c).integers(0, 8, len(ins[0])).astype(np.int32)
    got = host_step(ctl, kind, ins, want, param_set=ps, index=idx)
    assert got["vd"] is None and (got["status"] == 0).mean() > 0.9
    for k, d in enumerate(recs):
        sel = idx == k
        h = BatchedController(robot, device=0, dof_order=dof_order, **d)
        try:
            ref = host_step(h, kind, [x[sel] for x in ins], want)
        finally:
            h.close()
        assert_same({key: (None if x is None else x[sel]) for key, x in got.items()}, ref, (name, k))
    ps.close()


@gpu
@pytest.mark.parametrize("name", ["stand_anymal_b_clf", "stand_mini_cheetah_pc"])
def test_iteration_cap_on_deep_instances(ctl_cache, name):
    """The 16 deepest instances of a combination, for every pivot count k among them: a handle with max_iter = k gives the
    default bits on the rows that take <= k pivots, a handle with max_iter = k - 1 gives exactly WBC_ST_MAXITER and zero
    outputs on the rows that take more; in both variants."""
    g, robot, kind, kw = hard_combo(name)
    ins = [g[k] for k in ("q", "v", "traj", "contact")]
    base = ctl_cache(robot, **kw)
    variants = {"vd_off": lambda c: host_step(c, kind, ins, ("f", "qp_info", "lam")),
                "vd_on": lambda c: np_outputs(c.step(kind, *ins, debug=True))}
    for vname, run in variants.items():
        ref = run(base)
        assert (ref["status"] == 0).all()
        piv = ref["qp_info"][:, 3].astype(int)
        assert piv.min() >= 2
        for k in np.unique(piv):
            at = run(ctl_cache(robot, max_iter=int(k), **kw))
            below = piv <= k
            assert_same({key: (None if x is None else x[below]) for key, x in at.items()},
                        {key: (None if x is None else x[below]) for key, x in ref.items()}, (name, vname, k))
            assert_capped(at, piv > k, (name, vname, k))
            capped = run(ctl_cache(robot, max_iter=int(k) - 1, **kw))
            assert_capped(capped, piv >= k, (name, vname, k - 1))
            less = piv < k
            assert_same({key: (None if x is None else x[less]) for key, x in capped.items()},
                        {key: (None if x is None else x[less]) for key, x in ref.items()}, (name, vname, k - 1))


@gpu
@pytest.mark.parametrize("kind", ["clf", "pc", "mptc"])
def test_shapes_for_every_kind(ctl_cache, kind):
    """Same bits as the same instances solved in another batch, in both variants: n = 1, 3, 5, 127 and 4099 (the chunked
    path, tail CTAs of the 4-warp reduce), a permutation, rows 8 bytes off the 16-byte boundary (per-lane input path) and
    page-locked host buffers (host-mapped reduce)."""
    import torch
    from quadruped_drake_b200.synth import generate
    ctl = ctl_cache("mini_cheetah")
    n = 4099
    q, v, traj, contact = ins = generate(ctl.model, n, 555, "mixed", ctl.fk)
    keys = {False: ("tau", "metrics", "status"), True: OUTS}
    for debug in (False, True):
        what = keys[debug]

        def step(*x):
            return np_outputs(ctl.step(kind, *x, debug=debug))
        full = step(*ins)
        assert ((full["status"] == 0) | (contact.sum(axis=1) == 0)).mean() > 0.95
        cut = lambda o, s: {k: (None if x is None else x[s]) for k, x in o.items()}  # noqa: E731
        pieces = [step(*(x[lo:hi] for x in ins)) for lo, hi in ((0, 127), (127, 2127), (2127, n))]
        for k in what:
            assert np.array_equal(np.concatenate([p[k] for p in pieces]), full[k]), (kind, debug, k)
        want = OPTIONAL if debug else ()
        assert_same(dev_step(ctl, kind, [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in ins], want), full,
                    (kind, debug, "device"), what)
        for m in (1, 3, 5):
            assert_same(step(*(x[:m] for x in ins)), cut(full, slice(0, m)), (kind, debug, m), what)
        perm = np.random.default_rng(1).permutation(127)
        assert_same(step(*(x[perm] for x in ins)), cut(full, perm), (kind, debug, "perm"), what)
        assert_same(host_step(ctl, kind, ins, want, pinned=True), full, (kind, debug, "pinned"), what)
        m = 1024

        def shifted(a, dtype):                   # device copy whose first element sits 8 bytes past a 16-byte boundary
            flat = torch.empty(a[:m].size + 16, dtype=dtype, device="cuda")
            off = 1 if dtype == torch.float64 else 8
            view = flat[off:off + a[:m].size]
            view.copy_(torch.from_numpy(np.ascontiguousarray(a[:m]).reshape(-1)))
            assert view.data_ptr() % 16 == 8
            return view.view(m, -1)
        tins = [shifted(q, torch.float64), shifted(v, torch.float64), shifted(traj, torch.float64), shifted(contact, torch.uint8)]
        assert_same(dev_step(ctl, kind, tins, want), cut(full, slice(0, m)), (kind, debug, "shifted"), what)
