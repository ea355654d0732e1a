"""Closed-loop batched rollout (SURVEY.md 8 f2): the caller of the control step, reference simulate.py:160-182.

    planner (device sampler) -> controller step -> semi-implicit Euler, n_steps times for N robots, no host round trips.

Two plants: `plant=False` advances the state with the QP's own contact-consistent accelerations ("planned contacts hold",
csrc/wbc_rollout.cuh); `plant=True` applies the controller's TORQUES to the simulated robot on flat ground (forward dynamics +
velocity-level contact with Coulomb friction, csrc/wbc_plant.cuh), so that a controller can fail physically. Everything runs
through `wbc_rollout_ex` in the C ABI. There is no CPU fallback.

Perturbed robots (`plant_set`, `variant`, `push`; ground plant only): the plant simulates a variant of the robot - a payload
(model.with_payload), other link masses or inertias - on the variant's own ground friction, and a push acts on the base during
a time window, while the controller keeps the handle's nominal model. They run through `wbc_rollout_perturbed` /
`wbc_plant_step_perturbed`.

Uneven ground (`terrain_set`, `terrain`; ground plant only): each robot stands on its own terrain - a plane plus an optional
height field (`Terrain`, defined in include/wbc.h) - while the controller keeps assuming flat ground. It runs through
`wbc_rollout_terrain` / `wbc_plant_step_terrain`, together with any variants and pushes.

Per-robot controller parameters (`param_set`, `param_index`; either plant): robot i is controlled with its own gains and weights
(controller.ParamSet). It runs through `wbc_rollout_params`, together with any variants, pushes and terrain.

Imperfect sensing and actuation (`loop`, a `Loop`; ground plant only): robot i's controller reads its state with Gaussian noise,
and its torque command reaches the plant `delay` control steps late, scaled by its motor strength (semantics in include/wbc.h,
wbc_loop). It runs through `wbc_rollout_loop`, together with any variants, pushes, terrain and parameter sets; `observe` runs the
sensing alone.

Rollout monitor (`monitor`, a `Monitor`; ground plant only): after every plant step each robot's true pose is compared with the
plan sample its controller tracked, the first failing step is kept, and tracking, effort and contact statistics accumulate in a
`MonitorState` on the device (semantics in include/wbc.h, wbc_monitor). It runs through `wbc_rollout_monitor`, together with
any loop, variants, pushes, terrain and parameter sets, and changes none of the other outputs.

Actuator model (`motor`, a `Motor`; ground plant only): between the actuated torque and the plant each joint's motor follows
its command through a first-order lag, saturates on a torque-speed envelope, and the joint adds viscous and Coulomb friction
(semantics in include/wbc.h, wbc_motor_desc). A `MotorSet` holds the records; without one every motor saturates at the URDF
effort. It runs through `wbc_rollout_motor`, together with any monitor, loop, variants, pushes, terrain and parameter sets;
`motor_apply` runs the motor alone.

State estimation (`estimator`, an `Estimator`; with a loop only): each robot's controller reads the base position and linear
velocity of a linear Kalman filter that fuses a synthesised accelerometer with leg kinematics, instead of observed ones
(semantics in include/wbc.h, wbc_estimator). An `EstimatorSet` holds the records (`estimator_desc`), an `EstimatorState` the
per-robot filter. It runs through `wbc_rollout_estimator`, together with any motor, monitor, variants, pushes, terrain and
parameter sets; `estimator_step` runs the filter alone.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi
from .capi import (KINDS, LOOP_HIST, MON_NSTAT, WbcCtrlParams, WbcEstimator, WbcEstimatorDesc, WbcLoop, WbcMonitor, WbcMotorDesc,
                   WbcPlantMotor, WbcPlantOpts, WbcPlantPerturb, WbcPlantTerrain, WbcRolloutIO, WbcRolloutOpts, WbcTerrainDesc, np_ptr)
from .controller import check_device_index
from .model import NQ, NU, NV, RobotModel, WbcModelStruct

Q0_MINI_CHEETAH = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4)     # simulate.py:171-176


def _is_torch(x):
    return type(x).__module__.startswith("torch")


class PlantSet:
    """Device-resident table of K robots for the ground plant (wbc_plant_set_create): models[k] (RobotModel or WbcModelStruct,
    with the controller's DOF and actuator order) is what the plant simulates for variant k, mu[k] its ground friction
    (None: the call's `mu` for every variant)."""

    def __init__(self, ctl, models, mu=None):
        self.ctl, self.lib = ctl, ctl.lib
        structs = [m.as_struct() if isinstance(m, RobotModel) else m for m in models]
        self.n_variants = len(structs)
        arr = (WbcModelStruct * self.n_variants)(*structs)
        self._mu = None if mu is None else np.ascontiguousarray(np.broadcast_to(np.asarray(mu, np.float64), (self.n_variants,)))
        self._p = C.c_void_p()
        self.ctl._check(self.lib.wbc_plant_set_create(ctl._h, self.n_variants, arr, None if self._mu is None else np_ptr(self._mu),
                                                      C.byref(self._p)), "wbc_plant_set_create")

    def close(self):
        if getattr(self, "_p", None):
            self.lib.wbc_plant_set_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class Terrain:
    """h(x, y) = z0 + slope[0] x + slope[1] y + H(x, y); H bilinear in heights[ny, nx] (None: no grid) with heights[0, 0] at
    `origin` and spacing (dx, dy). Outside the grid its edge values continue flat."""
    z0: float = 0.0
    slope: tuple = (0.0, 0.0)
    origin: tuple = (0.0, 0.0)
    spacing: tuple = (1.0, 1.0)
    heights: np.ndarray | None = None


class TerrainSet:
    """Device-resident table of T terrains for the ground plant (wbc_terrain_set_create); robot i stands on terrains[index[i]]."""

    def __init__(self, ctl, terrains):
        self.ctl, self.lib = ctl, ctl.lib
        self.n_terrains = len(terrains)
        grids = [None if t.heights is None else np.ascontiguousarray(t.heights, np.float64) for t in terrains]
        descs = []
        for t, g in zip(terrains, grids):
            ny, nx = (0, 0) if g is None else g.shape
            descs.append(WbcTerrainDesc(float(t.z0), float(t.slope[0]), float(t.slope[1]), nx, ny, float(t.origin[0]), float(t.origin[1]),
                                        float(t.spacing[0]), float(t.spacing[1]), None if g is None else g.ctypes.data))
        arr = (WbcTerrainDesc * self.n_terrains)(*descs)
        self._p = C.c_void_p()
        self.ctl._check(self.lib.wbc_terrain_set_create(ctl._h, self.n_terrains, arr, C.byref(self._p)), "wbc_terrain_set_create")

    def close(self):
        if getattr(self, "_p", None):
            self.lib.wbc_terrain_set_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _terrain(terrain_set, index, ptr):
    return WbcPlantTerrain(None if terrain_set is None else terrain_set._p, ptr(index))


def _terrain_index(n, index):
    return None if index is None else np.ascontiguousarray(np.broadcast_to(np.asarray(index, np.int32), (n,)))


def _perturb(plant_set, variant, push, ptr):
    return WbcPlantPerturb(None if plant_set is None else plant_set._p, ptr(variant), ptr(push))


def _perturb_arrays(n, variant, push):
    """Host copies in the layouts of the C ABI: variant [N] int32, push [N][8] float64 (None stays None)."""
    vi = None if variant is None else np.ascontiguousarray(np.broadcast_to(np.asarray(variant, np.int32), (n,)))
    pu = None if push is None else np.ascontiguousarray(np.broadcast_to(np.asarray(push, np.float64), (n, 8)))
    return vi, pu


class LoopState:
    """The persistent loop state of N robots: hist [N,16,12] float64, the ring of the last 16 commanded torques, and tick [N]
    int64, the number of commands issued so far; both zero. NumPy arrays, or torch tensors on the device of `like`. A rollout
    given a state continues it and leaves it advanced."""

    def __init__(self, n, like=None):
        if like is not None and _is_torch(like):
            import torch
            self.hist = torch.zeros((n, LOOP_HIST, 12), dtype=torch.float64, device=like.device)
            self.tick = torch.zeros(n, dtype=torch.int64, device=like.device)
        else:
            self.hist, self.tick = np.zeros((n, LOOP_HIST, 12)), np.zeros(n, np.int64)


@dataclass
class Loop:
    """Per-robot sensing and actuation of the ground-plant loop (include/wbc.h, wbc_loop). noise: standard deviations of base
    orientation (rad), base position (m), joint angles (rad), angular velocity (rad/s), linear velocity (m/s) and joint
    velocities (rad/s), shape (6,) for every robot or (N, 6); delay [N] int32 control steps in [0, 15]; strength [N] >= 0;
    stream [N] int32 noise stream ids (None: the row index); seed, 64 bits; state: a LoopState to continue (None: each call
    starts a fresh history). None for noise / delay / strength means no noise / no delay / strength 1. With torch inputs, torch
    values must be contiguous CUDA tensors of the ABI's dtype and shape; other values are broadcast and copied to the device."""
    noise: object = None
    delay: object = None
    strength: object = None
    stream: object = None
    seed: int = 0
    state: LoopState | None = None


_LOOP_FIELDS = (("noise", np.float64, 6), ("delay", np.int32, None), ("strength", np.float64, None), ("stream", np.int32, None))


def check_device_array(x, shape, dtype, what):
    """A per-robot array on the device must be a contiguous CUDA tensor of the ABI's dtype and shape: the kernels read it through
    its device pointer."""
    import torch
    dt = {np.float64: torch.float64, np.int32: torch.int32, np.int64: torch.int64}[dtype]
    if not (_is_torch(x) and x.is_cuda and x.is_contiguous() and x.dtype == dt and tuple(x.shape) == tuple(shape)):
        raise ValueError(f"{what} on the device must be a contiguous CUDA tensor {np.dtype(dtype).name}{list(shape)}")


def _loop_arrays(loop, n, dev=None):
    """The arrays of a Loop in the layouts of the C ABI (kept alive by the caller for the call): host arrays broadcast to N rows,
    or with dev != None torch tensors on that device (torch inputs checked, not converted)."""
    out = {}
    for name, dtype, width in _LOOP_FIELDS:
        x = getattr(loop, name)
        shape = (n,) if width is None else (n, width)
        if x is None:
            out[name] = None
        elif dev is not None and _is_torch(x):
            check_device_array(x, shape, dtype, f"loop.{name}")
            out[name] = x
        else:
            a = np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype), shape))
            if dev is not None:
                import torch
                a = torch.from_numpy(a.copy()).to(dev)
            out[name] = a
    st = loop.state
    if st is not None:
        if dev is not None:
            check_device_array(st.hist, (n, LOOP_HIST, 12), np.float64, "loop.state.hist")
            check_device_array(st.tick, (n,), np.int64, "loop.state.tick")
        elif not (isinstance(st.hist, np.ndarray) and st.hist.dtype == np.float64 and st.hist.shape == (n, LOOP_HIST, 12)
                  and st.hist.flags.c_contiguous and isinstance(st.tick, np.ndarray) and st.tick.dtype == np.int64
                  and st.tick.shape == (n,) and st.tick.flags.c_contiguous):
            raise ValueError(f"loop.state must hold contiguous host arrays hist float64[{n}, {LOOP_HIST}, 12] and tick int64[{n}]")
    return out


def _wbc_loop(loop, arrays, ptr):
    st = loop.state
    return WbcLoop(*(ptr(arrays[name]) for name, _, _ in _LOOP_FIELDS[:4]), int(loop.seed) & 0xFFFFFFFFFFFFFFFF,
                   None if st is None else ptr(st.hist), None if st is None else ptr(st.tick))


def observe(ctl, q, v, loop):
    """What the controllers of N robots read at their current ticks (wbc_loop_observe; the ticks are not advanced) -> q_obs [N,19],
    v_obs [N,18]. Host arrays go through the host entry; torch CUDA tensors stay on the device (torch's current stream)."""
    if _is_torch(q):
        import torch
        n, dev = q.shape[0], q.device
        check_device_array(q, (n, NQ), np.float64, "q")
        check_device_array(v, (n, NV), np.float64, "v")
        arrays = _loop_arrays(loop, n, dev)
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
        qo, vo = torch.empty_like(q), torch.empty_like(v)
        lp = _wbc_loop(loop, arrays, p)
        ctl._check(ctl.lib.wbc_loop_observe(ctl._h, n, C.byref(lp), p(q), p(v), p(qo), p(vo),
                                            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "wbc_loop_observe")
        return qo, vo
    q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, NQ)
    n = len(q)
    v = np.ascontiguousarray(v, dtype=np.float64).reshape(n, NV)
    arrays = _loop_arrays(loop, n)
    opt = lambda a: None if a is None else np_ptr(a)  # noqa: E731
    qo, vo = np.empty_like(q), np.empty_like(v)
    lp = _wbc_loop(loop, arrays, opt)
    ctl._check(ctl.lib.wbc_loop_observe_host(ctl._h, n, C.byref(lp), np_ptr(q), np_ptr(v), np_ptr(qo), np_ptr(vo)), "wbc_loop_observe_host")
    return qo, vo


class MonitorState:
    """The per-robot monitor state of N robots (include/wbc.h, wbc_monitor), zeroed, which is a fresh state: stats [N,11] float64
    (columns capi.MON_*), steps [N] int64, fail_step [N] int64 (0: not failed yet), fail_why [N] int32 (capi.MON_POS | MON_ANG |
    MON_STATUS). NumPy arrays, or torch tensors on the device of `like`. A rollout given a state continues it."""

    def __init__(self, n, like=None):
        if like is not None and _is_torch(like):
            import torch
            z = lambda shape, dt_: torch.zeros(shape, dtype=dt_, device=like.device)  # noqa: E731
            self.stats, self.steps = z((n, MON_NSTAT), torch.float64), z(n, torch.int64)
            self.fail_step, self.fail_why = z(n, torch.int64), z(n, torch.int32)
        else:
            self.stats, self.steps = np.zeros((n, MON_NSTAT)), np.zeros(n, np.int64)
            self.fail_step, self.fail_why = np.zeros(n, np.int64), np.zeros(n, np.int32)

    @property
    def failed(self):
        return self.fail_step > 0

    def fail_time(self, t0=0.0, dt=5e-3):
        """Time at which each robot was first found failed, t0 + fail_step dt (the end of that step); +inf if it never failed."""
        if _is_torch(self.fail_step):
            import torch
            t = t0 + self.fail_step.to(torch.float64) * dt
            return torch.where(self.fail_step > 0, t, torch.full_like(t, float("inf")))
        return np.where(self.fail_step > 0, t0 + self.fail_step * dt, np.inf)

    rms_pos = property(lambda s: (s.stats[:, capi.MON_SUM_POS2] / s.steps) ** 0.5)
    rms_ang = property(lambda s: (s.stats[:, capi.MON_SUM_ANG2] / s.steps) ** 0.5)
    max_pos = property(lambda s: s.stats[:, capi.MON_MAX_POS])
    max_ang = property(lambda s: s.stats[:, capi.MON_MAX_ANG])
    tau2_dt = property(lambda s: s.stats[:, capi.MON_TAU2_DT])
    work_abs = property(lambda s: s.stats[:, capi.MON_WORK_ABS])
    sat_max = property(lambda s: s.stats[:, capi.MON_SAT_MAX])
    f_max = property(lambda s: s.stats[:, capi.MON_F_MAX])
    stance_unloaded = property(lambda s: s.stats[:, capi.MON_STANCE_UNLOADED])
    swing_loaded = property(lambda s: s.stats[:, capi.MON_SWING_LOADED])
    dist_xy = property(lambda s: s.stats[:, capi.MON_DIST_XY])


@dataclass
class Monitor:
    """Failure bounds of the rollout monitor: base position error (m) and orientation error (rad) against the plan sample; +inf
    turns a bound off. state: a MonitorState to continue (None: each call starts a fresh one)."""
    pos_max: float = 0.05
    ang_max: float = 0.3
    state: MonitorState | None = None


_MON_FIELDS = (("stats", np.float64, (MON_NSTAT,)), ("steps", np.int64, ()), ("fail_step", np.int64, ()), ("fail_why", np.int32, ()))


def _monitor_state(monitor, n, like=None):
    """The monitor's state, checked (or a fresh one): torch CUDA tensors when `like` is a torch tensor, host arrays otherwise."""
    st = monitor.state if monitor.state is not None else MonitorState(n, like)
    for name, dtype, width in _MON_FIELDS:
        x, shape = getattr(st, name), (n, *width)
        if like is not None and _is_torch(like):
            check_device_array(x, shape, dtype, f"monitor.state.{name}")
        elif not (isinstance(x, np.ndarray) and x.dtype == dtype and x.shape == shape and x.flags.c_contiguous):
            raise ValueError(f"monitor.state.{name} must be a contiguous host array {np.dtype(dtype).name}{list(shape)}")
    return st


def _wbc_monitor(monitor, st, why, ptr):
    return WbcMonitor(float(monitor.pos_max), float(monitor.ang_max), ptr(st.stats), ptr(st.steps), ptr(st.fail_step), ptr(st.fail_why),
                      ptr(why))


def motor_desc(model, peak_scale=1.0, speed_knee=np.inf, speed_free=np.inf, lag=0.0, damping=0.0, coulomb=0.0, coulomb_speed=0.0):
    """One motor record (WbcMotorDesc) for the joints of `model` (a RobotModel, or a BatchedController's): peak torque
    peak_scale x the URDF effort; every other field a scalar for all 12 joints or an array in the model's joint order. The
    defaults are the motor of a NULL set: saturation at the effort and nothing else; peak_scale = inf is the ideal motor."""
    d = WbcMotorDesc()
    vals = dict(peak=peak_scale * np.asarray(model.effort, np.float64), speed_knee=speed_knee, speed_free=speed_free, lag=lag,
                damping=damping, coulomb=coulomb, coulomb_speed=coulomb_speed)
    for name, x in vals.items():
        getattr(d, name)[:] = [float(y) for y in np.broadcast_to(np.asarray(x, np.float64), (NU,))]
    return d


class MotorSet:
    """Device-resident table of K motor records (wbc_motor_set_create); robot i's motors are descs[index[i]]."""

    def __init__(self, ctl, descs):
        self.ctl, self.lib = ctl, ctl.lib
        self.n_sets = len(descs)
        arr = (WbcMotorDesc * self.n_sets)(*descs)
        self._p = C.c_void_p()
        self.ctl._check(self.lib.wbc_motor_set_create(ctl._h, self.n_sets, arr, C.byref(self._p)), "wbc_motor_set_create")

    def close(self):
        if getattr(self, "_p", None):
            self.lib.wbc_motor_set_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MotorState:
    """The motor state of N robots: tau_m [N,12] float64, each actuator's last motor torque (actuator order), and count [N] int64,
    the number of motor steps so far; both zero (a fresh state). NumPy arrays, or torch tensors on the device of `like`. A rollout
    given a state continues it and leaves it advanced."""

    def __init__(self, n, like=None):
        if like is not None and _is_torch(like):
            import torch
            self.tau_m = torch.zeros((n, NU), dtype=torch.float64, device=like.device)
            self.count = torch.zeros(n, dtype=torch.int64, device=like.device)
        else:
            self.tau_m, self.count = np.zeros((n, NU)), np.zeros(n, np.int64)


@dataclass
class Motor:
    """Per-robot actuator model of the ground-plant loop. set: a MotorSet (None: saturation at the URDF effort); index [N] int32
    record of each robot (None: record 0); state: a MotorState to continue (None: each call starts a fresh one)."""
    set: MotorSet | None = None
    index: object = None
    state: MotorState | None = None


def _motor_arrays(motor, n, dev=None):
    """(index, state) of a Motor in the layouts of the C ABI, checked: the index broadcast to N rows (a host copy, or on `dev`
    torch tensors are checked, not converted), the state as given."""
    idx, st = motor.index, motor.state
    if dev is not None:
        check_device_index(idx, n, "motor.index")
        if st is not None:
            check_device_array(st.tau_m, (n, NU), np.float64, "motor.state.tau_m")
            check_device_array(st.count, (n,), np.int64, "motor.state.count")
        return idx, st
    if st is not None and not (isinstance(st.tau_m, np.ndarray) and st.tau_m.dtype == np.float64 and st.tau_m.shape == (n, NU)
                               and st.tau_m.flags.c_contiguous and isinstance(st.count, np.ndarray) and st.count.dtype == np.int64
                               and st.count.shape == (n,) and st.count.flags.c_contiguous):
        raise ValueError(f"motor.state must hold contiguous host arrays tau_m float64[{n}, {NU}] and count int64[{n}]")
    return _terrain_index(n, idx), st


def _wbc_motor(motor, idx, st, ptr):
    return WbcPlantMotor(None if motor.set is None else motor.set._p, ptr(idx), None if st is None else ptr(st.tau_m),
                         None if st is None else ptr(st.count))


def motor_apply(ctl, v, tau, motor, dt=5e-3):
    """The motor alone on one step (wbc_motor_apply) -> (tau_plant [N,12], status [N] int32: ST_BADMOTOR for a bad index). v [N,18]
    the true joint velocities, tau [N,12] the torque reaching the motors (actuator order); motor.state is required and advanced
    (its tau_m is the motor torque). Host arrays go through the host entry; torch CUDA tensors stay on the device (torch's
    current stream)."""
    if motor.state is None:
        raise ValueError("motor_apply: motor.state is required (a MotorState)")
    if _is_torch(v):
        import torch
        n, dev = v.shape[0], v.device
        check_device_array(v, (n, NV), np.float64, "v")
        check_device_array(tau, (n, NU), np.float64, "tau")
        idx, st = _motor_arrays(motor, n, dev)
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
        out, status = torch.empty_like(tau), torch.zeros(n, dtype=torch.int32, device=dev)
        mt = _wbc_motor(motor, idx, st, p)
        ctl._check(ctl.lib.wbc_motor_apply(ctl._h, n, float(dt), C.byref(mt), p(v), p(tau), p(out), p(status),
                                           C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "wbc_motor_apply")
        return out, status
    v = np.ascontiguousarray(v, dtype=np.float64).reshape(-1, NV)
    n = len(v)
    tau = np.ascontiguousarray(tau, dtype=np.float64).reshape(n, NU)
    idx, st = _motor_arrays(motor, n)
    opt = lambda a: None if a is None else np_ptr(a)  # noqa: E731
    out, status = np.empty_like(tau), np.zeros(n, np.int32)
    mt = _wbc_motor(motor, idx, st, opt)
    ctl._check(ctl.lib.wbc_motor_apply_host(ctl._h, n, float(dt), C.byref(mt), np_ptr(v), np_ptr(tau), np_ptr(out), np_ptr(status)),
               "wbc_motor_apply_host")
    return out, status


# Defaults in the spirit of the linear Kalman filter of the open-source MIT Cheetah software (oracle/estimator.py); not measured.
ESTIMATOR_DEFAULTS = dict(q_pos=0.02, q_vel=0.1, q_foot=0.02, r_pos=0.002, r_vel=0.05, r_height=0.005, swing_scale=100.0, p0_pos=0.01,
                          p0_vel=0.1, p0_foot=0.01)


def estimator_desc(**kw):
    """One estimator record (WbcEstimatorDesc): ESTIMATOR_DEFAULTS with the given fields replaced. Process stds q_pos (m/sqrt(s)),
    q_vel (m/s/sqrt(s)), q_foot (m/sqrt(s)); measurement stds r_pos (m), r_vel (m/s), r_height (m), +inf drops those rows;
    swing_scale >= 1 multiplies the stds of a foot planned in swing; p0_pos, p0_vel, p0_foot the stds of the prime."""
    vals = dict(ESTIMATOR_DEFAULTS)
    for k, x in kw.items():
        if k not in vals:
            raise TypeError(f"estimator_desc: unknown field {k!r}")
        vals[k] = float(x)
    return WbcEstimatorDesc(**vals)


class EstimatorSet:
    """Device-resident table of K estimator records (wbc_estimator_set_create); robot i's filter uses descs[index[i]]."""

    def __init__(self, ctl, descs):
        self.ctl, self.lib = ctl, ctl.lib
        self.n_sets = len(descs)
        arr = (WbcEstimatorDesc * self.n_sets)(*descs)
        self._p = C.c_void_p()
        self.ctl._check(self.lib.wbc_estimator_set_create(ctl._h, self.n_sets, arr, C.byref(self._p)), "wbc_estimator_set_create")

    def close(self):
        if getattr(self, "_p", None):
            self.lib.wbc_estimator_set_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_EST_FIELDS = (("x", np.float64, (18,)), ("P", np.float64, (18, 18)), ("v_prev", np.float64, (3,)), ("count", np.int64, ()),
               ("stats", np.float64, (4,)))


class EstimatorState:
    """The filter state of N robots: x [N,18] (base position, base velocity, feet LF RF LH RH; world), P [N,18,18], v_prev [N,3],
    count [N] int64 (0: the next step primes the filter) and stats [N,4] (sum |p err|^2, max |p err|, sum |v err|^2, max |v err|);
    all zero. NumPy arrays, or torch tensors on the device of `like`. A rollout given a state continues it and leaves it advanced."""

    def __init__(self, n, like=None):
        for name, dtype, width in _EST_FIELDS:
            if like is not None and _is_torch(like):
                import torch
                x = torch.zeros((n, *width), dtype={np.float64: torch.float64, np.int64: torch.int64}[dtype], device=like.device)
            else:
                x = np.zeros((n, *width), dtype)
            setattr(self, name, x)

    rms_pos = property(lambda s: (s.stats[:, 0] / s.count) ** 0.5)
    max_pos = property(lambda s: s.stats[:, 1])
    rms_vel = property(lambda s: (s.stats[:, 2] / s.count) ** 0.5)
    max_vel = property(lambda s: s.stats[:, 3])


@dataclass
class Estimator:
    """Per-robot state estimation of the ground-plant loop. set: an EstimatorSet (required); index [N] int32 record of each robot
    (None: record 0); accel_noise [N] accelerometer noise std in m/s^2 (None: none); state: an EstimatorState to continue (None:
    each call primes a fresh filter in library scratch, and keeps no statistics)."""
    set: EstimatorSet
    index: object = None
    accel_noise: object = None
    state: EstimatorState | None = None


def _estimator_arrays(est, n, dev=None):
    """(index, accel_noise, state) of an Estimator in the layouts of the C ABI, checked: index and accel_noise broadcast to N rows
    (host copies, or on `dev` torch tensors checked, not converted), the state as given."""
    if not isinstance(est.set, EstimatorSet):
        raise ValueError("estimator.set must be an EstimatorSet")
    st = est.state
    if dev is not None:
        check_device_index(est.index, n, "estimator.index")
        if est.accel_noise is not None:
            check_device_array(est.accel_noise, (n,), np.float64, "estimator.accel_noise")
        if st is not None:
            for name, dtype, width in _EST_FIELDS:
                check_device_array(getattr(st, name), (n, *width), dtype, f"estimator.state.{name}")
        return est.index, est.accel_noise, st
    if st is not None:
        for name, dtype, width in _EST_FIELDS:
            x = getattr(st, name)
            if not (isinstance(x, np.ndarray) and x.dtype == dtype and x.shape == (n, *width) and x.flags.c_contiguous):
                raise ValueError(f"estimator.state.{name} must be a contiguous host array {np.dtype(dtype).name}{[n, *width]}")
    an = None if est.accel_noise is None else np.ascontiguousarray(np.broadcast_to(np.asarray(est.accel_noise, np.float64), (n,)))
    return _terrain_index(n, est.index), an, st


def _wbc_estimator(est, idx, an, st, ptr):
    s = (None,) * 5 if st is None else tuple(ptr(getattr(st, name)) for name, _, _ in _EST_FIELDS)
    return WbcEstimator(est.set._p, ptr(idx), ptr(an), *s)


def estimator_step(ctl, q, v, q_obs, v_obs, contact, estimator, loop=None, dt=5e-3):
    """The estimator alone on one step (wbc_estimator_step) -> (q_obs, v_obs, status_or [N] int32: ST_BADESTIM for a bad index or
    a failed step). q [N,19], v [N,18] the true state at the start of the step; q_obs, v_obs what the loop observed (the returned
    arrays carry the estimate in [4:7] and [3:6]); contact [N,4] uint8 the planned stance flags; loop gives the seed, streams and
    ticks (read, not advanced; None: seed 0, row streams, tick 0). estimator.state is required and advanced. Host arrays go
    through the host entry (q_obs, v_obs copied); torch CUDA tensors stay on the device and q_obs, v_obs are updated in place."""
    if estimator.state is None:
        raise ValueError("estimator_step: estimator.state is required (an EstimatorState)")
    if _is_torch(q):
        import torch
        n, dev = q.shape[0], q.device
        check_device_array(q, (n, NQ), np.float64, "q")
        check_device_array(v, (n, NV), np.float64, "v")
        check_device_array(q_obs, (n, NQ), np.float64, "q_obs")
        check_device_array(v_obs, (n, NV), np.float64, "v_obs")
        if not (_is_torch(contact) and contact.is_cuda and contact.is_contiguous() and contact.dtype == torch.uint8
                and tuple(contact.shape) == (n, 4)):
            raise ValueError("contact on the device must be a contiguous CUDA tensor uint8[N, 4]")
        idx, an, st = _estimator_arrays(estimator, n, dev)
        arrays = None if loop is None else _loop_arrays(loop, n, dev)      # (kept alive for the call)
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
        status = torch.zeros(n, dtype=torch.int32, device=dev)
        es = _wbc_estimator(estimator, idx, an, st, p)
        lp = None if loop is None else C.byref(_wbc_loop(loop, arrays, p))
        ctl._check(ctl.lib.wbc_estimator_step(ctl._h, n, float(dt), C.byref(es), lp, p(q), p(v), p(q_obs), p(v_obs), p(contact), p(status),
                                              C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "wbc_estimator_step")
        return q_obs, v_obs, status
    q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, NQ)
    n = len(q)
    v = np.ascontiguousarray(v, dtype=np.float64).reshape(n, NV)
    qo, vo = np.array(q_obs, dtype=np.float64).reshape(n, NQ), np.array(v_obs, dtype=np.float64).reshape(n, NV)
    ct = np.ascontiguousarray(contact, dtype=np.uint8).reshape(n, 4)
    idx, an, st = _estimator_arrays(estimator, n)
    arrays = None if loop is None else _loop_arrays(loop, n)
    opt = lambda a: None if a is None else np_ptr(a)  # noqa: E731
    status = np.zeros(n, np.int32)
    es = _wbc_estimator(estimator, idx, an, st, opt)
    lp = None if loop is None else C.byref(_wbc_loop(loop, arrays, opt))
    ctl._check(ctl.lib.wbc_estimator_step_host(ctl._h, n, float(dt), C.byref(es), lp, np_ptr(q), np_ptr(v), np_ptr(qo), np_ptr(vo),
                                               np_ptr(ct), np_ptr(status)), "wbc_estimator_step_host")
    return qo, vo, status


class RolloutResult:
    __slots__ = ("q", "v", "t", "tau", "metrics", "status_or", "err_max", "metrics_log", "f_contact", "monitor", "why", "estimator")

    def __init__(self, **kw):
        for k in self.__slots__:
            setattr(self, k, kw.get(k))


def _opts(use_graph, plant, mu, erp, iters, f_ptr=None):
    return WbcRolloutOpts(1 if use_graph else 0, 1 if plant else 0, WbcPlantOpts(float(mu), float(erp), int(iters), 0), f_ptr)


def rollout(ctl, sampler, kind, q, v, t, n_steps, dt=5e-3, plan_index=None, log_metrics=False, use_graph=True, plant=False,
            mu=1.0, erp=0.2, iters=30, plant_set=None, variant=None, push=None, terrain_set=None, terrain=None, param_set=None,
            param_index=None, loop=None, monitor=None, motor=None, estimator=None) -> RolloutResult:
    """Advance N robots by n_steps control periods of length dt (simulate.py:20-21: dt = 5e-3, 6 s = 1200 steps).
    NumPy inputs are copied (host entry); torch CUDA tensors are updated IN PLACE on torch's current stream.
    plant=True: ground-contact simulation driven by the torques (mu: ground friction, simulate.py:44-46); the result then
    carries the last step's ground forces `f_contact[N,4,3]`.
    Perturbed robots (plant=True only): plant_set (PlantSet or None: the nominal model), variant [N] int32 (None: variant 0),
    push [N,8] = force (world) | point (base frame) | t_on | t_off (None: no pushes); torch tensors on the device with torch
    inputs, arrays otherwise. A robot with an out-of-range variant index is frozen and flagged ST_BADVARIANT.
    Uneven ground (plant=True only): terrain_set (TerrainSet or None: flat ground), terrain [N] int32 (None: terrain 0); an
    out-of-range terrain index freezes that robot, flagged ST_BADTERRAIN.
    Per-robot controller parameters (either plant): param_set (controller.ParamSet or None: the handle's params), param_index
    [N] int32 (None: set 0); a robot with an out-of-range index gets zero torques, flagged ST_BADPARAMS.
    Imperfect sensing and actuation (plant=True only): loop (a Loop) gives each robot's state noise, command delay and motor
    strength; `tau` is then the last COMMANDED torque. A robot with a bad profile is flagged ST_BADLOOP and gets zero torque.
    Rollout monitor (plant=True only): monitor (a Monitor) accumulates per-robot failure and effort statistics; the result then
    carries `monitor` (its MonitorState, advanced) and `why` [N] int32, the failure reasons at the last step.
    Actuator model (plant=True only): motor (a Motor) puts each robot's motors between the actuated torque and the plant; `tau`
    stays the last COMMANDED torque, and a monitor sees the motor torque. A robot with a bad record index is flagged ST_BADMOTOR
    and gets zero torque.
    State estimation (plant=True and a loop only): estimator (an Estimator) gives each robot's controller the filter's base
    position and linear velocity; the result then carries `estimator` (its EstimatorState, advanced, or None). A robot with a bad
    record index or a failed filter step is controlled from the observed state and flagged ST_BADESTIM."""
    if estimator is not None and (loop is None or not plant):
        raise ValueError("rollout: an estimator needs loop= (its observed state, seed, streams and ticks) and plant=True")
    on_terrain = terrain_set is not None or terrain is not None
    perturbed = plant_set is not None or variant is not None or push is not None
    per_robot = param_set is not None or param_index is not None
    k = KINDS[kind] if isinstance(kind, str) else int(kind)
    if _is_torch(q):
        import torch
        n, dev = q.shape[0], q.device
        mk = lambda shape, dt_=torch.float64: torch.empty(shape, dtype=dt_, device=dev)  # noqa: E731
        r = RolloutResult(q=q, v=v, t=t, tau=mk((n, NU)), metrics=mk((n, 4)), status_or=mk((n,), torch.int32), err_max=mk((n,)),
                          metrics_log=mk((n_steps, n, 4)) if log_metrics else None, f_contact=mk((n, 4, 3)) if plant else None)
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
        io = WbcRolloutIO(p(q), p(v), p(t), p(plan_index), p(r.tau), p(r.metrics), p(r.status_or), p(r.err_max), p(r.metrics_log))
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        o = _opts(use_graph, plant, mu, erp, iters, p(r.f_contact))
        if monitor is not None or motor is not None or estimator is not None:
            ea = None if estimator is None else _estimator_arrays(estimator, n, dev)
            if monitor is not None:
                r.monitor, r.why = _monitor_state(monitor, n, q), mk((n,), torch.int32)
            arrays = None if loop is None else _loop_arrays(loop, n, dev)      # (kept alive for the call)
            pt = C.byref(_perturb(plant_set, variant, push, p)) if perturbed else None
            tr = C.byref(_terrain(terrain_set, terrain, p)) if on_terrain else None
            check_device_index(param_index, n)
            cp = C.byref(WbcCtrlParams(None if param_set is None else param_set._p, p(param_index))) if per_robot else None
            lp = None if loop is None else C.byref(_wbc_loop(loop, arrays, p))
            mo = None if monitor is None else C.byref(_wbc_monitor(monitor, r.monitor, r.why, p))
            if estimator is not None:
                mt = None if motor is None else C.byref(_wbc_motor(motor, *_motor_arrays(motor, n, dev), p))
                es = C.byref(_wbc_estimator(estimator, *ea, p))
                r.estimator = estimator.state
                ctl._check(ctl.lib.wbc_rollout_estimator(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt,
                                                         tr, cp, lp, mo, mt, es, stream), "wbc_rollout_estimator")
            elif motor is None:
                ctl._check(ctl.lib.wbc_rollout_monitor(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt, tr,
                                                       cp, lp, mo, stream), "wbc_rollout_monitor")
            else:
                mt = C.byref(_wbc_motor(motor, *_motor_arrays(motor, n, dev), p))
                ctl._check(ctl.lib.wbc_rollout_motor(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt, tr,
                                                     cp, lp, mo, mt, stream), "wbc_rollout_motor")
        elif loop is not None:
            arrays = _loop_arrays(loop, n, dev)            # (kept alive for the call)
            pt = C.byref(_perturb(plant_set, variant, push, p)) if perturbed else None
            tr = C.byref(_terrain(terrain_set, terrain, p)) if on_terrain else None
            check_device_index(param_index, n)
            cp = C.byref(WbcCtrlParams(None if param_set is None else param_set._p, p(param_index))) if per_robot else None
            lp = _wbc_loop(loop, arrays, p)
            ctl._check(ctl.lib.wbc_rollout_loop(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt, tr, cp,
                                                C.byref(lp), stream), "wbc_rollout_loop")
        elif per_robot:
            pt = C.byref(_perturb(plant_set, variant, push, p)) if perturbed else None
            tr = C.byref(_terrain(terrain_set, terrain, p)) if on_terrain else None
            check_device_index(param_index, n)
            cp = WbcCtrlParams(None if param_set is None else param_set._p, p(param_index))
            ctl._check(ctl.lib.wbc_rollout_params(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt, tr,
                                                  C.byref(cp), stream), "wbc_rollout_params")
        elif on_terrain:
            pt, tr = _perturb(plant_set, variant, push, p), _terrain(terrain_set, terrain, p)
            ctl._check(ctl.lib.wbc_rollout_terrain(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), C.byref(pt),
                                                   C.byref(tr), stream), "wbc_rollout_terrain")
        elif perturbed:
            pt = _perturb(plant_set, variant, push, p)
            ctl._check(ctl.lib.wbc_rollout_perturbed(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), C.byref(pt),
                                                     stream), "wbc_rollout_perturbed")
        else:
            ctl._check(ctl.lib.wbc_rollout_ex(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), stream), "wbc_rollout_ex")
        return r
    q = np.array(q, dtype=np.float64).reshape(-1, NQ)
    n = len(q)
    v = np.array(v, dtype=np.float64).reshape(n, NV)
    t = np.array(np.broadcast_to(np.asarray(t, dtype=np.float64), (n,)))
    pi = None if plan_index is None else np.ascontiguousarray(plan_index, dtype=np.int32).reshape(n)
    r = RolloutResult(q=q, v=v, t=t, tau=np.empty((n, NU)), metrics=np.empty((n, 4)), status_or=np.empty(n, np.int32), err_max=np.empty(n),
                      metrics_log=np.empty((n_steps, n, 4)) if log_metrics else None, f_contact=np.zeros((n, 4, 3)) if plant else None)
    opt = lambda a: None if a is None else np_ptr(a)  # noqa: E731
    io = WbcRolloutIO(np_ptr(q), np_ptr(v), np_ptr(t), opt(pi), np_ptr(r.tau), np_ptr(r.metrics), np_ptr(r.status_or), np_ptr(r.err_max),
                      opt(r.metrics_log))
    o = _opts(use_graph, plant, mu, erp, iters, opt(r.f_contact))
    if monitor is not None or motor is not None or estimator is not None:
        ea = None if estimator is None else _estimator_arrays(estimator, n)      # (kept alive for the call)
        if monitor is not None:
            r.monitor, r.why = _monitor_state(monitor, n), np.zeros(n, np.int32)
        vi, pu = _perturb_arrays(n, variant, push)      # (kept alive for the call)
        ti, ci = _terrain_index(n, terrain), _terrain_index(n, param_index)
        arrays = None if loop is None else _loop_arrays(loop, n)
        pt = C.byref(_perturb(plant_set, vi, pu, opt)) if perturbed else None
        tr = C.byref(_terrain(terrain_set, ti, opt)) if on_terrain else None
        cp = C.byref(WbcCtrlParams(None if param_set is None else param_set._p, opt(ci))) if per_robot else None
        lp = None if loop is None else C.byref(_wbc_loop(loop, arrays, opt))
        mo = None if monitor is None else C.byref(_wbc_monitor(monitor, r.monitor, r.why, opt))
        if estimator is not None:
            mi, ms = (None, None) if motor is None else _motor_arrays(motor, n)      # (kept alive for the call)
            mt = None if motor is None else C.byref(_wbc_motor(motor, mi, ms, opt))
            es = C.byref(_wbc_estimator(estimator, *ea, opt))
            r.estimator = estimator.state
            ctl._check(ctl.lib.wbc_rollout_estimator_host(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt,
                                                          tr, cp, lp, mo, mt, es), "wbc_rollout_estimator_host")
        elif motor is None:
            ctl._check(ctl.lib.wbc_rollout_monitor_host(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt, tr,
                                                        cp, lp, mo), "wbc_rollout_monitor_host")
        else:
            mi, ms = _motor_arrays(motor, n)             # (kept alive for the call)
            mt = C.byref(_wbc_motor(motor, mi, ms, opt))
            ctl._check(ctl.lib.wbc_rollout_motor_host(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt, tr,
                                                      cp, lp, mo, mt), "wbc_rollout_motor_host")
    elif loop is not None:
        vi, pu = _perturb_arrays(n, variant, push)      # (kept alive for the call)
        ti, ci = _terrain_index(n, terrain), _terrain_index(n, param_index)
        arrays = _loop_arrays(loop, n)
        pt = C.byref(_perturb(plant_set, vi, pu, opt)) if perturbed else None
        tr = C.byref(_terrain(terrain_set, ti, opt)) if on_terrain else None
        cp = C.byref(WbcCtrlParams(None if param_set is None else param_set._p, opt(ci))) if per_robot else None
        lp = _wbc_loop(loop, arrays, opt)
        ctl._check(ctl.lib.wbc_rollout_loop_host(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt, tr, cp,
                                                 C.byref(lp)), "wbc_rollout_loop_host")
    elif per_robot:
        vi, pu = _perturb_arrays(n, variant, push)      # (kept alive for the call)
        ti, ci = _terrain_index(n, terrain), _terrain_index(n, param_index)
        pt = C.byref(_perturb(plant_set, vi, pu, opt)) if perturbed else None
        tr = C.byref(_terrain(terrain_set, ti, opt)) if on_terrain else None
        cp = WbcCtrlParams(None if param_set is None else param_set._p, opt(ci))
        ctl._check(ctl.lib.wbc_rollout_params_host(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), pt, tr,
                                                   C.byref(cp)), "wbc_rollout_params_host")
    elif on_terrain:
        pt, tr = _perturb(plant_set, *_perturb_arrays(n, variant, push), opt), _terrain(terrain_set, _terrain_index(n, terrain), opt)
        ctl._check(ctl.lib.wbc_rollout_terrain_host(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), C.byref(pt),
                                                    C.byref(tr)), "wbc_rollout_terrain_host")
    elif perturbed:
        pt = _perturb(plant_set, *_perturb_arrays(n, variant, push), opt)
        ctl._check(ctl.lib.wbc_rollout_perturbed_host(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o), C.byref(pt)),
                   "wbc_rollout_perturbed_host")
    else:
        ctl._check(ctl.lib.wbc_rollout_ex_host(ctl._h, k, sampler._p, n, int(n_steps), float(dt), C.byref(io), C.byref(o)), "wbc_rollout_ex_host")
    return r


def plant_step(ctl, q, v, tau, dt=5e-3, mu=1.0, erp=0.2, iters=30, ctrl_status=None, plant_set=None, variant=None, push=None, t=None,
               terrain_set=None, terrain=None):
    """One time step of N simulated robots on flat ground -> q+[N,19], v+[N,18], f_contact[N,4,3] (ground forces LF RF LH RH,
    world axes), status[N]. Host arrays go through wbc_plant_step_host (q, v copied); torch CUDA tensors are updated IN PLACE
    on torch's current stream (wbc_plant_step). plant_set / variant / push as in `rollout` (wbc_plant_step_perturbed); t [N] is
    each robot's time at the start of the step, required with pushes (a torch tensor is advanced by dt in place). terrain_set /
    terrain as in `rollout` (wbc_plant_step_terrain)."""
    on_terrain = terrain_set is not None or terrain is not None
    perturbed = plant_set is not None or variant is not None or push is not None
    o = WbcPlantOpts(float(mu), float(erp), int(iters), 0)
    if _is_torch(q):
        import torch
        n, dev = q.shape[0], q.device
        f, st = torch.zeros((n, 4, 3), dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.int32, device=dev)
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        args = (p(q), p(v), p(tau), p(t), p(ctrl_status), p(st), p(f), stream)
        if on_terrain:
            pt, tr = _perturb(plant_set, variant, push, p), _terrain(terrain_set, terrain, p)
            ctl._check(ctl.lib.wbc_plant_step_terrain(ctl._h, n, float(dt), C.byref(o), C.byref(pt), C.byref(tr), *args), "wbc_plant_step_terrain")
        elif perturbed:
            pt = _perturb(plant_set, variant, push, p)
            ctl._check(ctl.lib.wbc_plant_step_perturbed(ctl._h, n, float(dt), C.byref(o), C.byref(pt), *args), "wbc_plant_step_perturbed")
        else:
            ctl._check(ctl.lib.wbc_plant_step(ctl._h, n, float(dt), C.byref(o), *args), "wbc_plant_step")
        return q, v, f, st
    q = np.array(q, dtype=np.float64).reshape(-1, NQ)
    n = len(q)
    v = np.array(v, dtype=np.float64).reshape(n, NV)
    tau = np.ascontiguousarray(tau, dtype=np.float64).reshape(n, NU)
    f, st = np.zeros((n, 4, 3)), np.zeros(n, np.int32)
    cs = None if ctrl_status is None else np.ascontiguousarray(ctrl_status, dtype=np.int32).reshape(n)
    opt = lambda a: None if a is None else np_ptr(a)  # noqa: E731
    ta = None if t is None else np.array(np.broadcast_to(np.asarray(t, dtype=np.float64), (n,)))
    args = (np_ptr(q), np_ptr(v), np_ptr(tau), opt(ta), opt(cs), np_ptr(st), np_ptr(f))
    if on_terrain:
        pt, tr = _perturb(plant_set, *_perturb_arrays(n, variant, push), opt), _terrain(terrain_set, _terrain_index(n, terrain), opt)
        ctl._check(ctl.lib.wbc_plant_step_terrain_host(ctl._h, n, float(dt), C.byref(o), C.byref(pt), C.byref(tr), *args),
                   "wbc_plant_step_terrain_host")
    elif perturbed:
        pt = _perturb(plant_set, *_perturb_arrays(n, variant, push), opt)
        ctl._check(ctl.lib.wbc_plant_step_perturbed_host(ctl._h, n, float(dt), C.byref(o), C.byref(pt), *args), "wbc_plant_step_perturbed_host")
    else:
        ctl._check(ctl.lib.wbc_plant_step_host(ctl._h, n, float(dt), C.byref(o), *args), "wbc_plant_step_host")
    return q, v, f, st


def integrate(ctl, q, v, vd, dt, t=None):
    """One semi-implicit Euler step on torch CUDA tensors, in place (wbc_integrate)."""
    import torch
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream(q.device).cuda_stream)
    ctl._check(ctl.lib.wbc_integrate(ctl._h, q.shape[0], float(dt), p(q), p(v), p(vd), p(t), stream), "wbc_integrate")
