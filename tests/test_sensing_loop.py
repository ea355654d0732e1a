"""Imperfect sensing and actuation in the ground-plant loop (wbc_rollout_loop[_host], wbc_loop_observe[_host]; include/wbc.h,
wbc_loop).

CPU half: Philox4x32-10, the normals, observe and actuate of csrc/wbc_loop.cuh on the host (tests/emu/emu_loop.cpp) against the
numpy restatement oracle/sensing.py, and the oracle's noise statistics.
GPU half: a zero profile gives the bits of wbc_rollout_params; the fused rollout equals a manual loop of existing entries; noise
depends on (seed, stream, tick) only; the observe entry against the oracle and its statistics; the closed loop against the
oracle controller and plant; bad profiles; argument errors."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from oracle import sensing as se

GOLD = Path(__file__).parent / "golden"
KIND_NAMES = ["id", "clf", "pc", "mptc", "pd"]
P = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731


# ------------------------------------------------------------------------------------------------------------------ CPU half
@pytest.fixture(scope="module")
def emu(built):
    lib = C.CDLL(str(Path(__file__).parent / "emu" / "libwbc_emu_loop.so"))
    vp = C.c_void_p
    lib.emu_philox.argtypes = [C.c_longlong, vp, vp, vp]
    lib.emu_normals.argtypes = [C.c_uint64, C.c_uint32, C.c_longlong, vp]
    lib.emu_observe.argtypes = [C.c_longlong, vp, vp, vp, vp, C.c_uint64, vp, vp, vp, vp, vp]
    lib.emu_actuate.argtypes = [C.c_longlong, vp, vp, vp, vp, vp, vp, vp, vp]
    return lib


def test_oracle_philox_known_answers():
    cases = [([0, 0, 0, 0], [0, 0], "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
             ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
             ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], "d16cfe09 94fdcceb 5001e420 24126ea1")]
    for ctr, key, want in cases:
        got = se.philox4x32_10(np.array(ctr, np.uint32), np.array(key, np.uint32))
        assert " ".join("%08x" % w for w in got) == want


def test_emulated_philox_matches_oracle_bit_for_bit(emu):
    rng = np.random.default_rng(0)
    n = 10_000
    ctr = rng.integers(0, 2**32, (n, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2**32, (n, 2), dtype=np.uint64).astype(np.uint32)
    out = np.zeros((n, 4), np.uint32)
    emu.emu_philox(n, P(ctr), P(key), P(out))
    assert np.array_equal(out, se.philox4x32_10(ctr, key))


def golden_states(case, n):
    g = np.load(GOLD / f"{case}.npz")
    return np.ascontiguousarray(g["q"][:n]), np.ascontiguousarray(g["v"][:n])


def emu_observe(emu, q, v, noise, seed, stream, tick, delay=None, strength=None):
    n = len(q)
    qo, vo = np.full_like(q, np.nan), np.full_like(v, np.nan)
    noise = np.ascontiguousarray(np.broadcast_to(noise, (n, 6)), np.float64)
    stream, tick = np.ascontiguousarray(stream, np.int32), np.ascontiguousarray(tick, np.int64)
    emu.emu_observe(n, P(noise), P(delay), P(strength), P(stream), seed, P(tick), P(q), P(v), P(qo), P(vo))
    return qo, vo


@pytest.mark.parametrize("case", ["cfg3_anymal_trot", "cfg4_mini_cheetah_walk"])
def test_emulated_observe_matches_oracle(emu, case):
    """Normals within 1e-14, q_obs / v_obs within 1e-13; blocks with sigma = 0 bit-exact; unit quaternions within 1e-15."""
    n = 48
    q, v = golden_states(case, n)
    rng = np.random.default_rng(1)
    noise = rng.uniform(0.0, 0.2, (n, 6)) * (rng.random((n, 6)) < 0.7)      # about a third of the blocks noise-free
    noise[:4] = 0.0
    stream = rng.integers(-2**31, 2**31, n).astype(np.int32)
    tick = rng.integers(0, 2**40, n)
    seed = 0x0123456789ABCDEF
    for i in range(0, n, 7):
        z = np.zeros(36)
        emu.emu_normals(seed, int(stream[i]) & 0xFFFFFFFF, int(tick[i]), P(z))
        assert np.abs(z - se.normals(seed, stream[i], tick[i])).max() < 1e-14
    qo, vo = emu_observe(emu, q, v, noise, seed, stream, tick)
    ro, rv = se.observe_batch(q, v, noise, seed, stream, tick)
    assert np.abs(qo - ro).max() < 1e-13 and np.abs(vo - rv).max() < 1e-13
    blocks = [(qo, q, slice(0, 4)), (qo, q, slice(4, 7)), (qo, q, slice(7, 19)), (vo, v, slice(0, 3)), (vo, v, slice(3, 6)),
              (vo, v, slice(6, 18))]
    for b, (got, true, sl) in enumerate(blocks):
        zero = noise[:, b] == 0.0
        assert np.array_equal(got[zero, sl], true[zero, sl]), b
        assert (got[~zero, sl] != true[~zero, sl]).any(axis=1).all(), b
    assert np.abs(np.linalg.norm(qo[noise[:, 0] > 0, :4], axis=1) - 1.0).max() < 1e-15


def test_oracle_noise_statistics():
    """10^5 normals of one stream over consecutive ticks: Kolmogorov-Smirnov against N(0, 1), mean and variance in 5 sigma."""
    from scipy import stats
    z = se.normals(2026, 7, np.arange(2778)).ravel()[:100_000]
    assert stats.kstest(z, "norm").pvalue > 1e-3
    n = len(z)
    assert abs(z.mean()) < 5 / np.sqrt(n)
    assert abs(z.var() - 1.0) < 5 * np.sqrt(2.0 / n)


def emu_actuate(emu, tau, delay, strength, noise, hist, tick):
    n = len(tau)
    applied, status = np.full((n, 12), np.nan), np.zeros(n, np.int32)
    emu.emu_actuate(n, P(delay), P(strength), P(noise), P(hist), P(tick), P(np.ascontiguousarray(tau)), P(applied), P(status))
    return applied, status


def test_emulated_actuate_matches_the_delay_rule(emu):
    """40 ticks, delays 0 / 1 / 7 / 15 x strengths 0 / 0.7 / 1.3: c < d, ring wrap-around; bit-exact against the oracle rule."""
    delays, strengths = [0, 1, 7, 15], [0.0, 0.7, 1.3]
    d = np.array([a for a in delays for _ in strengths], np.int32)
    s = np.array([b for _ in delays for b in strengths])
    n = len(d)
    hist, tick = np.zeros((n, 16, 12)), np.zeros(n, np.int64)
    acts = [se.Actuator(d[i], s[i]) for i in range(n)]
    rng = np.random.default_rng(2)
    for c in range(40):
        tau = rng.normal(0, 10, (n, 12))
        applied, status = emu_actuate(emu, tau, d, s, None, hist, tick)
        assert (status == 0).all() and (tick == c + 1).all()
        for i in range(n):
            assert np.array_equal(applied[i], acts[i].command(tau[i])), (c, i)
            assert np.array_equal(hist[i], acts[i].hist)


BAD_PROFILES = [("delay", -1), ("delay", 16), ("noise", np.nan), ("noise", -0.1), ("noise", np.inf), ("strength", np.inf),
                ("strength", -0.5), ("strength", np.nan), ("tick", -3)]


def test_emulated_bad_profiles_are_flagged(emu):
    """Each kind of bad profile: WBC_ST_BADLOOP, zero applied torque, hist and tick unchanged, observed without noise; the
    neighbours are unaffected."""
    n = len(BAD_PROFILES) + 2
    rng = np.random.default_rng(3)
    d, s = np.full(n, 2, np.int32), np.full(n, 0.9)
    noise = np.full((n, 6), 0.05)
    tick = np.full(n, 5, np.int64)
    for i, (what, val) in enumerate(BAD_PROFILES, start=1):
        {"delay": d, "strength": s, "tick": tick}.get(what, noise[:, 2])[i] = val
    hist = rng.normal(size=(n, 16, 12))
    h0, t0 = hist.copy(), tick.copy()
    tau = rng.normal(0, 10, (n, 12))
    applied, status = emu_actuate(emu, tau, d, s, noise, hist, tick)
    bad = np.arange(1, n - 1)
    assert (status[bad] == se.ST_BADLOOP).all() and (applied[bad] == 0).all()
    assert np.array_equal(hist[bad], h0[bad]) and np.array_equal(tick[bad], t0[bad])
    assert (status[[0, n - 1]] == 0).all() and (tick[[0, n - 1]] == 6).all()
    for i in (0, n - 1):
        assert np.array_equal(applied[i], 0.9 * h0[i, 3])
    q, v = golden_states("cfg4_mini_cheetah_walk", n)
    qo, vo = emu_observe(emu, q, v, noise, 1, np.arange(n), t0, d, s)
    assert np.array_equal(qo[bad], q[bad]) and np.array_equal(vo[bad], v[bad])
    ok = se.profile_ok(noise, d, s, t0)
    assert list(np.flatnonzero(ok)) == [0, n - 1]
    ro, rv = se.observe_batch(q, v, noise, 1, np.arange(n), t0, ok)
    assert np.abs(qo - ro).max() < 1e-13 and np.abs(vo - rv).max() < 1e-13 and not np.array_equal(qo[0], q[0])


# ------------------------------------------------------------------------------------------------------------------ GPU half
gpu = pytest.mark.gpu
Q0 = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4)
NOISE = np.array([0.01, 0.002, 0.01, 0.05, 0.02, 0.1])          # a moderate profile: 0.6 deg, 2 mm, 0.6 deg, ... per reading


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


def trot_sampler(ctl):
    from quadruped_drake_b200 import planner as pl
    bh = float(grounded(ctl, 1, np.random.default_rng(0), 0.0)[0, 6])
    return pl.TrajectorySampler(ctl, pl.make_gait_plan("mini_cheetah", "trot", goal=(1.5, 0.0), base_height=bh))


def param_sets(ctl, k, seed):
    from quadruped_drake_b200.capi import DEFAULT_PARAMS
    from quadruped_drake_b200.controller import ParamSet
    rng = np.random.default_rng(seed)
    names = ["id_kp_body_p", "id_kd_body_p", "id_kp_foot", "clf_q_body_p", "pc_kp_body_p", "pc_kd_foot", "pd_kp", "pd_kd"]
    return ParamSet(ctl, [{m: DEFAULT_PARAMS[m] * float(rng.uniform(0.7, 1.4)) for m in names} for _ in range(k)])


@pytest.fixture(scope="module")
def world(ctl):
    """The variants, pushes, terrain and parameter sets of a 512-robot robustness rollout."""
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import PlantSet, Terrain, TerrainSet
    from quadruped_drake_b200.urdf import load_description
    n = 512
    rng = np.random.default_rng(21)
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    ps = PlantSet(ctl, [flatten(d), flatten(with_payload(d, 1.2, (0.04, -0.02, 0.05)))], [1.0, 0.6])
    ts = TerrainSet(ctl, [Terrain(), Terrain(slope=(np.tan(np.radians(5.0)), 0.0))])
    pset = param_sets(ctl, 4, 5)
    push = np.zeros((n, 8))
    push[:, 0:3] = rng.uniform(-40, 40, (n, 3)); push[:, 3:6] = rng.uniform(-0.1, 0.1, (n, 3))
    push[:, 6], push[:, 7] = 0.5, 0.7
    w = dict(q0=grounded(ctl, n, rng, 0.02), s=trot_sampler(ctl),
             kw=dict(plant_set=ps, terrain_set=ts, param_set=pset, variant=(np.arange(n) % 2).astype(np.int32), push=push,
                     terrain=(np.arange(n) // 2 % 2).astype(np.int32), param_index=rng.integers(0, 4, n).astype(np.int32)))
    yield w
    pset.close(); ts.close(); ps.close(); w["s"].close()


ROLL_KEYS = ("q", "v", "t", "tau", "metrics", "status_or", "err_max", "f_contact")


def to_dev(kw):
    import torch
    return {k: (torch.from_numpy(np.ascontiguousarray(x)).cuda() if isinstance(x, np.ndarray) else x) for k, x in kw.items()}


def np_of(r, key):
    x = getattr(r, key)
    return x.cpu().numpy() if hasattr(x, "cpu") else x


@gpu
@pytest.mark.parametrize("kind", KIND_NAMES)
def test_zero_profile_gives_the_bits_of_rollout_params(ctl, world, kind):
    """sigma = 0, d = 0, strength 1 with variants, pushes, terrain and parameter sets: the bits of wbc_rollout_params on every
    output, host and device entries, graph and no graph; two more launches per step."""
    import torch
    from quadruped_drake_b200.rollout import Loop, rollout
    n, steps, dt = 512, 400, 5e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    zero = Loop(noise=np.zeros(6), delay=np.zeros(n, np.int32), strength=np.ones(n), seed=99)
    l0 = ctl.launches
    ref = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, log_metrics=True, **kw)
    l1 = ctl.launches
    got = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, log_metrics=True, loop=zero, **kw)
    l2 = ctl.launches
    assert l2 - l1 == (l1 - l0) + 2 * steps
    for key in ROLL_KEYS + ("metrics_log",):
        assert np.array_equal(np_of(got, key), np_of(ref, key)), (kind, key)
    for graph in (True, False):
        q, v, t = (torch.from_numpy(x.copy()).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
        dz = Loop(noise=torch.zeros((n, 6), dtype=torch.float64, device="cuda"), delay=torch.zeros(n, dtype=torch.int32, device="cuda"),
                  strength=torch.ones(n, dtype=torch.float64, device="cuda"), seed=99)
        with torch.cuda.stream(torch.cuda.Stream()):
            r = rollout(ctl, s, kind, q, v, t, steps, dt, plant=True, use_graph=graph, loop=dz, **to_dev(kw))
        torch.cuda.synchronize()
        for key in ROLL_KEYS:
            assert np.array_equal(np_of(r, key), np_of(ref, key)), (kind, graph, key)


def rollout_io(q, v, t, r=None):
    from quadruped_drake_b200.capi import WbcRolloutIO
    out = [None] * 5 if r is None else [P(r[k]) for k in ("tau", "metrics", "status_or", "err_max")] + [None]
    return WbcRolloutIO(P(q), P(v), P(t), None, *out)


@gpu
def test_null_loop_is_rollout_params(ctl, world):
    """wbc_rollout_loop_host with loop == NULL: the bits and the launch count of wbc_rollout_params_host."""
    from quadruped_drake_b200.capi import WbcCtrlParams, WbcPlantOpts, WbcRolloutOpts
    n, steps = 128, 50
    q0, s, kw = world["q0"][:n], world["s"], world["kw"]
    cp = WbcCtrlParams(kw["param_set"]._p, P(kw["param_index"][:n]))
    o = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    outs, counts = [], []
    for fn, extra in (("wbc_rollout_params_host", ()), ("wbc_rollout_loop_host", (None,))):
        q, v, t = q0.copy(), np.zeros((n, 18)), np.zeros(n)
        r = {"tau": np.zeros((n, 12)), "metrics": np.zeros((n, 4)), "status_or": np.zeros(n, np.int32), "err_max": np.zeros(n)}
        io = rollout_io(q, v, t, r)
        l0 = ctl.launches
        ctl._check(getattr(ctl.lib, fn)(ctl._h, 0, s._p, n, steps, 5e-3, C.byref(io), C.byref(o), None, None, C.byref(cp), *extra), fn)
        counts.append(ctl.launches - l0)
        outs.append([q, v, t] + list(r.values()))
    assert counts[0] == counts[1]
    for a, b in zip(*outs):
        assert np.array_equal(a, b)


def noisy_loop(n, rng, seed=7, dmax=15):
    from quadruped_drake_b200.rollout import Loop
    return Loop(noise=NOISE * rng.uniform(0.5, 2.0, (n, 1)), delay=rng.integers(0, dmax + 1, n).astype(np.int32),
                strength=rng.uniform(0.6, 1.4, n), stream=rng.integers(-2**31, 2**31, n).astype(np.int32), seed=seed)


@gpu
@pytest.mark.parametrize("kind", ["id", "pd"])
def test_fused_rollout_equals_a_manual_loop(ctl, world, kind):
    """256 robots x 200 steps with noise, delays 0-15 and strengths 0.6-1.4: the fused rollout has the bits of the loop
    sample -> wbc_loop_observe -> wbc_step_params -> a torch delay ring and scale -> wbc_plant_step_terrain. At dt = 1e-3, where
    most robots keep standing with a 15-step delay (DESIGN section 10), so the comparison covers live robots."""
    import torch
    from quadruped_drake_b200.capi import KINDS, WbcCtrlParams, WbcIO, WbcLoop, WbcPlantOpts, WbcPlantPerturb, WbcPlantTerrain
    from quadruped_drake_b200.rollout import rollout
    n, steps, dt = 256, 200, 1e-3
    rng = np.random.default_rng(31)
    q0, s = world["q0"][:n], world["s"]
    kw = {k: (x[:n] if isinstance(x, np.ndarray) else x) for k, x in world["kw"].items()}
    loop = noisy_loop(n, rng)
    r = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop, **kw)
    # the manual loop, on torch's current stream
    T = lambda x, dt_=None: torch.from_numpy(np.ascontiguousarray(x if dt_ is None else x.astype(dt_))).cuda()  # noqa: E731
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    q, v, t = T(q0), torch.zeros((n, 18), dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda")
    noise, delay, strength, stream = T(loop.noise), T(loop.delay), T(loop.strength), T(loop.stream)
    variant, push, terrain, pidx = T(kw["variant"]), T(kw["push"]), T(kw["terrain"]), T(kw["param_index"])
    traj = torch.empty((n, 54), dtype=torch.float64, device="cuda"); contact = torch.empty((n, 4), dtype=torch.uint8, device="cuda")
    qo, vo = torch.empty_like(q), torch.empty_like(v)
    tau, met = torch.zeros((n, 12), dtype=torch.float64, device="cuda"), torch.zeros((n, 4), dtype=torch.float64, device="cuda")
    st, st_or = torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")
    f = torch.zeros((n, 12), dtype=torch.float64, device="cuda")
    hist, tick = torch.zeros((n, 16, 12), dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.int64, device="cuda")
    scratch_hist = torch.zeros_like(hist)
    cs = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lp = WbcLoop(p(noise), p(delay), p(strength), p(stream), loop.seed, p(scratch_hist), p(tick))
    io = WbcIO(p(qo), p(vo), p(traj), p(contact), p(tau), p(met), p(st), None, None, None, None)
    cp = WbcCtrlParams(kw["param_set"]._p, p(pidx))
    po = WbcPlantOpts(1.0, 0.2, 30, 0)
    pt, tr = WbcPlantPerturb(kw["plant_set"]._p, p(variant), p(push)), WbcPlantTerrain(kw["terrain_set"]._p, p(terrain))
    rows = torch.arange(n, device="cuda")
    for c in range(steps):
        ctl._check(ctl.lib.wbc_sample_trajectory(ctl._h, s._p, n, None, p(t), p(traj), p(contact), None, None, None, cs), "sample")
        tick.fill_(c)
        ctl._check(ctl.lib.wbc_loop_observe(ctl._h, n, C.byref(lp), p(q), p(v), p(qo), p(vo), cs), "observe")
        ctl._check(ctl.lib.wbc_step_params(ctl._h, KINDS[kind], n, C.byref(io), C.byref(cp), cs), "step")
        hist[:, c % 16] = tau
        applied = (strength[:, None] * hist[rows, (c - delay.long()).clamp(min=0) % 16]).contiguous()
        ctl._check(ctl.lib.wbc_plant_step_terrain(ctl._h, n, dt, C.byref(po), C.byref(pt), C.byref(tr), p(q), p(v), p(applied), p(t),
                                                  p(st), p(st_or), p(f), cs), "plant")
    torch.cuda.synchronize()
    for key, x in (("q", q), ("v", v), ("t", t), ("tau", tau), ("status_or", st_or), ("f_contact", f.reshape(n, 4, 3))):
        assert np.array_equal(np_of(r, key), x.cpu().numpy()), (kind, key)
    assert (r.status_or == 0).mean() > 0.5


@gpu
def test_four_calls_with_a_state_equal_one_call(ctl, world):
    """A caller-owned LoopState continues the history: 4 x 100 steps give the bits of 1 x 400 steps (host and device)."""
    import torch
    from quadruped_drake_b200.rollout import LoopState, rollout
    n, dt = 256, 5e-3
    q0, s = world["q0"][:n], world["s"]
    kw = {k: (x[:n] if isinstance(x, np.ndarray) else x) for k, x in world["kw"].items()}
    loop = noisy_loop(n, np.random.default_rng(32))
    loop.state = LoopState(n)
    one = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, 400, dt, plant=True, loop=loop, **kw)
    assert (loop.state.tick == 400).all()
    loop.state = LoopState(n)
    q, v, t = q0, np.zeros((n, 18)), np.zeros(n)
    for _ in range(4):
        r = rollout(ctl, s, "id", q, v, t, 100, dt, plant=True, loop=loop, **kw)
        q, v, t = r.q, r.v, r.t
    for key in ("q", "v", "t", "tau", "f_contact"):
        assert np.array_equal(getattr(r, key), getattr(one, key)), key
    host_hist = loop.state.hist.copy()
    tq, tv, tt = (torch.from_numpy(x.copy()).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
    loop.state = LoopState(n, like=tq)
    dkw = to_dev(kw)
    for _ in range(4):
        rollout(ctl, s, "id", tq, tv, tt, 100, dt, plant=True, loop=loop, **dkw)
    torch.cuda.synchronize()
    assert np.array_equal(tq.cpu().numpy(), one.q) and np.array_equal(tv.cpu().numpy(), one.v)
    assert np.array_equal(loop.state.hist.cpu().numpy(), host_hist) and (loop.state.tick.cpu().numpy() == 400).all()


@gpu
def test_permuting_robots_with_their_streams_permutes_the_outputs(ctl, world):
    from quadruped_drake_b200.rollout import Loop, rollout
    n, steps, dt = 512, 200, 5e-3
    q0, s, kw = world["q0"], world["s"], world["kw"]
    loop = noisy_loop(n, np.random.default_rng(33))
    a = rollout(ctl, s, "id", q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop, **kw)
    perm = np.random.default_rng(34).permutation(n)
    pl = Loop(noise=loop.noise[perm], delay=loop.delay[perm], strength=loop.strength[perm], stream=loop.stream[perm], seed=loop.seed)
    pkw = {k: (x[perm] if isinstance(x, np.ndarray) else x) for k, x in kw.items()}
    b = rollout(ctl, s, "id", q0[perm], np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=pl, **pkw)
    for key in ROLL_KEYS:
        assert np.array_equal(getattr(a, key)[perm], getattr(b, key)), key


def rotvec(qo, q):
    """Rotation vector of q_obs (x) q^-1 (rows)."""
    inv = q[:, :4] * np.array([1.0, -1.0, -1.0, -1.0])
    d = np.stack([se.quat_mul(a, b) for a, b in zip(qo[:, :4], inv)])
    d *= np.sign(d[:, :1])
    s = np.linalg.norm(d[:, 1:], axis=1, keepdims=True)
    return 2.0 * np.arctan2(s, d[:, :1]) * d[:, 1:] / np.where(s > 0, s, 1.0)


@gpu
def test_observe_matches_oracle_and_its_statistics(ctl):
    """wbc_loop_observe against the oracle within 1e-13 (host and device entries); over 4096 robots x 64 ticks the per-block
    std is within 3 % of sigma and correlations across blocks, robots and ticks are below 0.02. Another seed or stream changes
    the noise."""
    import torch
    from quadruped_drake_b200.rollout import Loop, LoopState, observe
    n, ticks = 4096, 64
    q, v = golden_states("cfg4_mini_cheetah_walk", 64)
    q, v = np.ascontiguousarray(np.resize(q, (n, 19))), np.ascontiguousarray(np.resize(v, (n, 18)))
    sig = np.array([0.02, 0.01, 0.03, 0.2, 0.1, 0.5])
    loop = Loop(noise=sig, seed=0xDEADBEEF12345678, state=LoopState(n))
    loop.state.tick[:] = np.arange(n) * 1000
    qo, vo = observe(ctl, q, v, loop)
    ro, rv = se.observe_batch(q[:256], v[:256], sig, loop.seed, np.arange(256), loop.state.tick[:256])
    assert np.abs(qo[:256] - ro).max() < 1e-13 and np.abs(vo[:256] - rv).max() < 1e-13
    tq, tv = torch.from_numpy(q).cuda(), torch.from_numpy(v).cuda()
    dl = Loop(noise=sig, seed=loop.seed, state=LoopState(n, like=tq))
    E = np.empty((ticks, n, 36))
    for c in range(ticks):
        dl.state.tick.fill_(c)
        a, b = observe(ctl, tq, tv, dl)
        a, b = a.cpu().numpy(), b.cpu().numpy()
        E[c, :, 0:3] = rotvec(a, q) / sig[0]
        E[c, :, 3:6] = (a[:, 4:7] - q[:, 4:7]) / sig[1]
        E[c, :, 6:18] = (a[:, 7:] - q[:, 7:]) / sig[2]
        E[c, :, 18:21] = (b[:, 0:3] - v[:, 0:3]) / sig[3]
        E[c, :, 21:24] = (b[:, 3:6] - v[:, 3:6]) / sig[4]
        E[c, :, 24:36] = (b[:, 6:] - v[:, 6:]) / sig[5]
        if c == 0:
            z = se.normals(loop.seed, np.arange(8), 0)
            assert np.abs(E[0, :8, 3:] - z[:, 3:]).max() < 1e-6          # the normals themselves, in the documented order
    for blk in [slice(0, 3), slice(3, 6), slice(6, 18), slice(18, 21), slice(21, 24), slice(24, 36)]:
        assert abs(E[:, :, blk].std() - 1.0) < 0.03, blk
    flat = E.reshape(-1, 36)
    cb = np.corrcoef(flat.T)
    assert np.abs(cb - np.eye(36)).max() < 0.02
    cr = np.corrcoef(E[:, :-1].ravel(), E[:, 1:].ravel())[0, 1]
    ct = np.corrcoef(E[:-1].ravel(), E[1:].ravel())[0, 1]
    assert abs(cr) < 0.02 and abs(ct) < 0.02
    other_seed = Loop(noise=sig, seed=loop.seed + 1, state=LoopState(n, like=tq))
    other_stream = Loop(noise=sig, seed=loop.seed, stream=torch.arange(1, n + 1, dtype=torch.int32, device="cuda"), state=LoopState(n, like=tq))
    base = observe(ctl, tq, tv, Loop(noise=sig, seed=loop.seed, state=LoopState(n, like=tq)))[1].cpu().numpy()
    for lp in (other_seed, other_stream):
        x = observe(ctl, tq, tv, lp)[1].cpu().numpy()
        assert (x != base).any(axis=1).all()
    shifted = observe(ctl, tq[1:].contiguous(), tv[1:].contiguous(),
                      Loop(noise=sig, seed=loop.seed, stream=torch.arange(1, n, dtype=torch.int32, device="cuda"),
                           state=LoopState(n - 1, like=tq)))[1].cpu().numpy()
    assert np.array_equal(shifted, base[1:])                     # noise follows the stream, not the row


@gpu
@pytest.mark.parametrize("kind", ["id", "pd"])
def test_closed_loop_matches_oracle(ctl, kind):
    """Standing robots, 24 steps, noise, d = 3, strength 0.9: oracle noise + oracle controller + the delay rule +
    oracle/rollout.py:plant_step agree with the GPU rollout to q 1e-6, v and tau 1e-5. The PD law runs at dt = 1e-3: at 5e-3 its
    reference gains are unstable on the ground plant (DESIGN section 10)."""
    from oracle import controllers as oc, rollout as ro
    from oracle.dynamics import Plant
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.rollout import Loop, rollout
    n, steps, dt = 4, 24, (5e-3 if kind == "id" else 1e-3)
    rng = np.random.default_rng(41)
    q0 = grounded(ctl, n, rng, 0.01)
    bh = float(grounded(ctl, 1, rng, 0.0)[0, 6])
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh))
    loop = Loop(noise=NOISE, delay=np.full(n, 3, np.int32), strength=np.full(n, 0.9), stream=np.arange(10, 10 + n, dtype=np.int32),
                seed=5)
    r = rollout(ctl, s, kind, q0, np.zeros((n, 18)), 0.0, steps, dt, plant=True, loop=loop)
    assert (r.status_or == 0).all()
    plant = Plant("mini_cheetah")
    for i in range(n):
        ctrl = oc.IDController("mini_cheetah") if kind == "id" else oc.BasicController("mini_cheetah")
        act = se.Actuator(3, 0.9)
        q, v, t = q0[i].copy(), np.zeros(18), 0.0
        for c in range(steps):
            z = se.normals(loop.seed, loop.stream[i], c)
            qo, vo = se.observe(q, v, NOISE, z)
            if kind == "id":
                g = s.sample(np.array([t]))
                tau = ctrl.control_law(qo, vo, oc.traj_to_dict(g["traj"][0], g["contact"][0])).tau
            else:
                tau = ctrl.control_law(qo, vo)
            q, v, _ = ro.plant_step(plant, q, v, act.command(tau), dt)
            t += dt
        assert np.abs(r.q[i] - q).max() < 1e-6, (i, np.abs(r.q[i] - q).max())
        assert np.abs(r.v[i] - v).max() < 1e-5 and np.abs(r.tau[i] - tau).max() < 1e-5
    s.close()


@gpu
@pytest.mark.parametrize("what,val", BAD_PROFILES)
def test_bad_profile_in_a_rollout(ctl, world, what, val):
    """A bad profile: BADLOOP in status_or, zero applied torque (the robot moves as one with strength 0), hist and tick
    unchanged; the neighbours have the bits of the batch without the bad rows."""
    from quadruped_drake_b200.capi import ST_BADLOOP
    from quadruped_drake_b200.rollout import Loop, LoopState, rollout
    n, steps, dt = 64, 60, 5e-3
    q0, s = world["q0"][:n], world["s"]
    rng = np.random.default_rng(51)
    base = noisy_loop(n, rng, dmax=4)
    bad = [3, 40]
    rest = np.setdiff1d(np.arange(n), bad)

    def run(rows, edit=None):
        lp = Loop(noise=base.noise[rows].copy(), delay=base.delay[rows].copy(), strength=base.strength[rows].copy(),
                  stream=base.stream[rows].copy(), seed=base.seed, state=LoopState(len(rows)))
        lp.state.hist[:] = 0.25
        lp.state.tick[:] = 7
        if edit:
            edit(lp)
        return rollout(ctl, s, "id", q0[rows], np.zeros((len(rows), 18)), 0.0, steps, dt, plant=True, loop=lp), lp

    def make_bad(lp):
        k = {"delay": lp.delay, "strength": lp.strength, "tick": lp.state.tick}.get(what)
        if k is None:
            lp.noise[bad, 4] = val
        else:
            k[bad] = val

    r, lp = run(np.arange(n), make_bad)
    assert (r.status_or[bad] & ST_BADLOOP).all() and not (r.status_or[rest] & ST_BADLOOP).any()
    assert (lp.state.hist[bad] == 0.25).all() and np.array_equal(lp.state.tick[bad], np.full(2, val if what == "tick" else 7))
    ref, _ = run(rest)
    for key in ROLL_KEYS:
        assert np.array_equal(getattr(r, key)[rest], getattr(ref, key)), key

    def limp(lp2):
        lp2.noise[:] = 0.0
        lp2.strength[:] = 0.0
    zero, _ = run(np.array(bad), limp)
    assert np.array_equal(r.q[bad], zero.q) and np.array_equal(r.v[bad], zero.v)
    assert np.array_equal(r.status_or[bad], zero.status_or | ST_BADLOOP)


@gpu
def test_argument_errors(ctl, world):
    import torch
    from quadruped_drake_b200.capi import WbcLoop, WbcPlantOpts, WbcRolloutOpts
    from quadruped_drake_b200.rollout import Loop, LoopState, observe, rollout
    n = 4
    s = world["s"]
    q, v, t = world["q0"][:n].copy(), np.zeros((n, 18)), np.zeros(n)
    io = rollout_io(q, v, t)
    hist, tick = np.zeros((n, 16, 12)), np.zeros(n, np.int64)
    lp = WbcLoop(None, None, None, None, 0, None, None)
    integ = WbcRolloutOpts(1, 0, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    assert ctl.lib.wbc_rollout_loop_host(ctl._h, 0, s._p, n, 2, 5e-3, C.byref(io), C.byref(integ), None, None, None, C.byref(lp)) == 1
    assert b"ground plant" in ctl.lib.wbc_last_error(ctl._h)
    ground = WbcRolloutOpts(1, 1, WbcPlantOpts(1.0, 0.2, 30, 0), None)
    for one in (WbcLoop(None, None, None, None, 0, P(hist), None), WbcLoop(None, None, None, None, 0, None, P(tick))):
        assert ctl.lib.wbc_rollout_loop_host(ctl._h, 0, s._p, n, 2, 5e-3, C.byref(io), C.byref(ground), None, None, None, C.byref(one)) == 1
        assert b"hist and tick" in ctl.lib.wbc_last_error(ctl._h)
        assert ctl.lib.wbc_loop_observe_host(ctl._h, n, C.byref(one), P(q), P(v), P(q.copy()), P(v.copy())) == 1
    assert np.array_equal(q, world["q0"][:n])                    # nothing ran
    if torch.cuda.device_count() > 1:
        from quadruped_drake_b200.controller import BatchedController, ParamSet
        other = BatchedController("mini_cheetah", device=1)
        ps1 = ParamSet(other, [{}])
        with pytest.raises(RuntimeError, match="another device"):
            rollout(ctl, s, "id", q, v, t, 2, 5e-3, plant=True, param_set=ps1, loop=Loop(noise=NOISE))
        ps1.close(); other.close()
    tq, tv, tt = (torch.from_numpy(x.copy()).cuda() for x in (q, v, t))
    good = dict(noise=torch.zeros((n, 6), dtype=torch.float64, device="cuda"), delay=torch.zeros(n, dtype=torch.int32, device="cuda"),
                strength=torch.ones(n, dtype=torch.float64, device="cuda"), stream=torch.zeros(n, dtype=torch.int32, device="cuda"))
    bads = dict(noise=[good["noise"].float(), good["noise"][:, :5], good["noise"].t().contiguous().t(), good["noise"].cpu()],
                delay=[good["delay"].long(), good["delay"][: n - 1]], strength=[good["strength"].float(), good["strength"][None]],
                stream=[good["stream"].long()])
    l0 = ctl.launches
    for field, xs in bads.items():
        for x in xs:
            with pytest.raises(ValueError, match="loop." + field):
                rollout(ctl, s, "id", tq, tv, tt, 2, 5e-3, plant=True, loop=Loop(**{**good, field: x}))
            with pytest.raises(ValueError, match="loop." + field):
                observe(ctl, tq, tv, Loop(**{**good, field: x}))
    st = LoopState(n, like=tq)
    for h, tk in ((st.hist.float(), st.tick), (st.hist, st.tick.int()), (st.hist[:, :8].contiguous(), st.tick)):
        bad_state = LoopState(n, like=tq)
        bad_state.hist, bad_state.tick = h, tk
        with pytest.raises(ValueError, match="loop.state"):
            rollout(ctl, s, "id", tq, tv, tt, 2, 5e-3, plant=True, loop=Loop(state=bad_state))
    with pytest.raises(ValueError, match="loop.state"):
        rollout(ctl, s, "id", q, v, t, 2, 5e-3, plant=True, loop=Loop(state=LoopState(n + 1)))
    assert ctl.launches == l0
