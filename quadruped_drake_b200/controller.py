"""Host-side mirror of the reference controller interface, on top of the C ABI.

`BatchedController` is the pydrake-free batch entry (SURVEY.md 8b):

    step(kind, q[N,19], v[N,18], traj[N,54], contact[N,4]) -> tau[N,12], metrics[N,4], status[N]

on NumPy arrays (host buffers; copies happen inside `wbc_step_host`) or torch CUDA tensors
(device pointers, launched on torch's current stream). `ParamSet` holds K gain / weight sets on the device; with
`param_set=` / `param_index=` each robot of one step runs with its own set (`wbc_step_params[_host]`).

`IDController`, `CLFController`, `PCController` keep the reference constructor
`(plant, dt, use_lcm=False)` and port layout (reference controllers/basic_controller.py:21-77,
inverse_dynamics_controller.py:10-23): in0 "quad_state" (37), in1 "trunk_input" (abstract dict,
reference planners/simple.py:45-85), out0 "quad_torques" (12), out1 "output_metrics" (4). With
pydrake importable they are real LeafSystems; without it they expose the same callbacks
(`DoSetControlTorques`, `SetLoggingOutputs`, `ControlLaw`) over minimal port stand-ins.
Solver failure raises AssertionError exactly where the reference asserts
(inverse_dynamics_controller.py:224); the batch entry reports it in `status` instead.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .capi import KINDS, WbcCtrlParams, WbcIO, WbcParams, make_params, np_ptr
from .model import NQ, NTRAJ, NU, NV, RobotModel, load_robot

FEET = ["lf", "rf", "lh", "rh"]


def dict_to_traj(d):
    """Reference trunk dict (planners/simple.py:45-85) -> (traj[54], contact[4]) in the wbc.h layout."""
    t = np.zeros(NTRAJ)
    for k, key in enumerate(["p_body", "pd_body", "pdd_body", "rpy_body", "rpyd_body", "rpydd_body"]):
        t[3 * k:3 * k + 3] = np.asarray(d[key], float).ravel()
    for i, f in enumerate(FEET):
        t[18 + 3 * i:21 + 3 * i] = np.asarray(d["p_" + f], float).ravel()
        t[30 + 3 * i:33 + 3 * i] = np.asarray(d["pd_" + f], float).ravel()
        t[42 + 3 * i:45 + 3 * i] = np.asarray(d["pdd_" + f], float).ravel()
    return t, np.array([1 if c else 0 for c in d["contact_states"]], dtype=np.uint8)


def traj_to_dict(traj, contact, f_plan=None, u2_max=0.0):
    """(traj[54], contact[4]) -> the reference trunk dict (planners/simple.py:45-85, planners/towr.py:112-148)."""
    t = np.asarray(traj, float).ravel()
    d = {"p_body": t[0:3].copy(), "pd_body": t[3:6].copy(), "pdd_body": t[6:9].copy(),
         "rpy_body": t[9:12].copy(), "rpyd_body": t[12:15].copy(), "rpydd_body": t[15:18].copy()}
    for i, f in enumerate(FEET):
        d["p_" + f] = t[18 + 3 * i:21 + 3 * i].copy()
        d["pd_" + f] = t[30 + 3 * i:33 + 3 * i].copy()
        d["pdd_" + f] = t[42 + 3 * i:45 + 3 * i].copy()
    d["contact_states"] = [bool(c) for c in np.asarray(contact).ravel()]
    d["f_cj"] = np.zeros((3, 4)) if f_plan is None else np.asarray(f_plan, float).reshape(4, 3).T.copy()
    d["u2_max"] = u2_max
    return d


def _is_torch(x):
    return type(x).__module__.startswith("torch")


class StepOutput:
    __slots__ = ("tau", "metrics", "status", "vd", "f", "qp_info", "lam")

    def __init__(self, tau, metrics, status, vd=None, f=None, qp_info=None, lam=None):
        self.tau, self.metrics, self.status, self.vd, self.f, self.qp_info, self.lam = tau, metrics, status, vd, f, qp_info, lam

    def __iter__(self):
        return iter((self.tau, self.metrics, self.status))


class ParamSet:
    """Device-resident table of K controller parameter sets (wbc_param_set_create) on the device of `ctl`: params[k] is a
    dict of overrides for `make_params` or a `WbcParams` struct. Robot i of a step or rollout given `param_set=` runs with
    params[param_index[i]]; an index outside [0, K) is flagged ST_BADPARAMS with zero outputs."""

    def __init__(self, ctl, params):
        self.ctl, self.lib = ctl, ctl.lib
        structs = [p if isinstance(p, WbcParams) else make_params(**p) for p in params]
        self.n_sets = len(structs)
        arr = (WbcParams * self.n_sets)(*structs)
        self._p = C.c_void_p()
        self.ctl._check(self.lib.wbc_param_set_create(ctl._h, self.n_sets, arr, C.byref(self._p)), "wbc_param_set_create")

    def close(self):
        if getattr(self, "_p", None):
            self.lib.wbc_param_set_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _ctrl_params(param_set, index_ptr):
    return WbcCtrlParams(None if param_set is None else param_set._p, index_ptr)


def check_device_index(index, n, what="param_index"):
    """A per-robot index on the device must be a contiguous int32 CUDA tensor of shape (N,): the kernels read it as int32
    through its device pointer."""
    import torch
    if index is not None and not (_is_torch(index) and index.is_cuda and index.is_contiguous() and index.dtype == torch.int32
                                  and tuple(index.shape) == (n,)):
        raise ValueError(f"{what} on the device must be a contiguous CUDA tensor int32[{n}]")


def _param_index(n, index):
    """Host copy of a per-robot set index in the layout of the C ABI (int32 [N]); None stays None."""
    return None if index is None else np.ascontiguousarray(np.broadcast_to(np.asarray(index, np.int32), (n,)))


class BatchedController:
    """One handle of libwbc_b200.so on one device."""

    def __init__(self, robot="mini_cheetah", device=0, dof_order="depth_first", **params):
        self.lib = capi.load_library()
        self.model = robot if isinstance(robot, RobotModel) else load_robot(robot, dof_order=dof_order)
        self.params = make_params(**params)
        self.device = int(device)
        self._h = C.c_void_p()
        ms = self.model.as_struct()
        rc = self.lib.wbc_create(C.byref(ms), C.byref(self.params), self.device, C.byref(self._h))
        if rc != 0:
            msg = self.lib.wbc_last_error(self._h).decode() if self._h else "allocation failed"
            if self._h:
                self.lib.wbc_destroy(self._h)
                self._h = C.c_void_p()
            raise RuntimeError(f"wbc_create failed ({rc}): {msg}")

    def close(self):
        if getattr(self, "_h", None):
            self.lib.wbc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {self.lib.wbc_last_error(self._h).decode()}")

    @property
    def launches(self) -> int:
        return int(self.lib.wbc_launch_count(self._h))

    # ------------------------------------------------------------------ batch step
    def step(self, kind, q, v, traj, contact, debug=False, param_set=None, param_index=None) -> StepOutput:
        """param_set (ParamSet or None: the handle's params) / param_index [N] (None: set 0): per-robot controller parameters
        through wbc_step_params[_host]; a torch index is an int32 CUDA tensor. Left at None, wbc_step[_host] runs."""
        k = KINDS[kind] if isinstance(kind, str) else int(kind)
        per_robot = param_set is not None or param_index is not None
        if _is_torch(q):
            return self._step_torch(k, q, v, traj, contact, debug, param_set, param_index, per_robot)
        q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, NQ)
        n = q.shape[0]
        v = np.ascontiguousarray(v, dtype=np.float64).reshape(n, NV)
        traj = np.ascontiguousarray(traj, dtype=np.float64).reshape(n, NTRAJ)
        contact = np.ascontiguousarray(np.asarray(contact) != 0, dtype=np.uint8).reshape(n, 4)
        tau, met, st = np.empty((n, NU)), np.empty((n, 4)), np.empty(n, dtype=np.int32)
        vd = np.empty((n, NV)) if debug else None
        f = np.empty((n, 4, 3)) if debug else None
        qi = np.empty((n, 4)) if debug else None
        lam = np.empty((n, capi.NLAM)) if debug else None
        io = WbcIO(np_ptr(q), np_ptr(v), np_ptr(traj), np_ptr(contact), np_ptr(tau), np_ptr(met), np_ptr(st),
                   np_ptr(vd) if debug else None, np_ptr(f) if debug else None, np_ptr(qi) if debug else None,
                   np_ptr(lam) if debug else None)
        if per_robot:
            pi = _param_index(n, param_index)
            cp = _ctrl_params(param_set, None if pi is None else np_ptr(pi))
            self._check(self.lib.wbc_step_params_host(self._h, k, n, C.byref(io), C.byref(cp)), "wbc_step_params_host")
        else:
            self._check(self.lib.wbc_step_host(self._h, k, n, C.byref(io)), "wbc_step_host")
        return StepOutput(tau, met, st, vd, f, qi, lam)

    def step_plan(self, kind, sampler, q, v, t, plan_index=None, tau=None, metrics=None, status=None) -> StepOutput:
        """Control step with the trunk targets sampled from a device-resident plan (`planner.TrajectorySampler`) at the
        per-instance times t[N]: the host sends q, v, t only (wbc_step_plan_host). Host arrays; outputs may be passed in."""
        k = KINDS[kind] if isinstance(kind, str) else int(kind)
        q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, NQ)
        n = q.shape[0]
        v = np.ascontiguousarray(v, dtype=np.float64).reshape(n, NV)
        t = np.ascontiguousarray(t, dtype=np.float64).reshape(n)
        pi = None if plan_index is None else np.ascontiguousarray(plan_index, dtype=np.int32).reshape(n)
        tau = np.empty((n, NU)) if tau is None else tau
        metrics = np.empty((n, 4)) if metrics is None else metrics
        status = np.empty(n, dtype=np.int32) if status is None else status
        self._check(self.lib.wbc_step_plan_host(self._h, k, sampler._p, n, np_ptr(q), np_ptr(v), np_ptr(t), None if pi is None else np_ptr(pi),
                                                np_ptr(tau), np_ptr(metrics), np_ptr(status)), "wbc_step_plan_host")
        return StepOutput(tau, metrics, status)

    def step_pd(self, q, v, param_set=None, param_index=None):
        """BasicController.ControlLaw (basic_controller.py:322-352) for a batch of host states -> tau[N,12]. With param_set /
        param_index (as in `step`) each robot uses its set's pd_kp, pd_kd, pd_clip and pd_q_nom, and the call returns
        (tau, status[N]) with ST_BADPARAMS for an index out of range. Torch CUDA tensors (in place of the arrays, param_index
        int32) always go through wbc_step_params on torch's current stream and return (tau, status)."""
        if _is_torch(q):
            import torch
            n = q.shape[0]
            for t, w in ((q, NQ), (v, NV)):
                if not (_is_torch(t) and t.is_cuda and t.is_contiguous() and t.dtype == torch.float64 and tuple(t.shape) == (n, w)):
                    raise ValueError("device inputs must be contiguous CUDA tensors: q f64[N,19], v f64[N,18]")
            check_device_index(param_index, n)
            tau = torch.empty((n, NU), dtype=torch.float64, device=q.device)
            st = torch.empty((n,), dtype=torch.int32, device=q.device)
            p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
            io = WbcIO(p(q), p(v), None, None, p(tau), None, p(st), None, None, None)
            cp = _ctrl_params(param_set, p(param_index))
            stream = torch.cuda.current_stream(q.device).cuda_stream
            self._check(self.lib.wbc_step_params(self._h, capi.WBC_CTRL_PD, n, C.byref(io), C.byref(cp), C.c_void_p(stream)), "wbc_step_params")
            return tau, st
        q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, NQ)
        n = q.shape[0]
        v = np.ascontiguousarray(v, dtype=np.float64).reshape(n, NV)
        tau = np.empty((n, NU))
        if param_set is not None or param_index is not None:
            st = np.empty(n, dtype=np.int32)
            pi = _param_index(n, param_index)
            io = WbcIO(np_ptr(q), np_ptr(v), None, None, np_ptr(tau), None, np_ptr(st), None, None, None)
            cp = _ctrl_params(param_set, None if pi is None else np_ptr(pi))
            self._check(self.lib.wbc_step_params_host(self._h, capi.WBC_CTRL_PD, n, C.byref(io), C.byref(cp)), "wbc_step_params_host")
            return tau, st
        io = WbcIO(np_ptr(q), np_ptr(v), None, None, np_ptr(tau), None, None, None, None, None)
        self._check(self.lib.wbc_step_host(self._h, capi.WBC_CTRL_PD, n, C.byref(io)), "wbc_step_host")
        return tau

    def _step_torch(self, k, q, v, traj, contact, debug, param_set=None, param_index=None, per_robot=False):
        import torch
        n = q.shape[0]
        for t, w, dt in ((q, NQ, torch.float64), (v, NV, torch.float64), (traj, NTRAJ, torch.float64), (contact, 4, torch.uint8)):
            if not (t.is_cuda and t.is_contiguous() and t.dtype == dt and t.shape == (n, w)):
                raise ValueError("device inputs must be contiguous CUDA tensors: q f64[N,19], v f64[N,18], traj f64[N,54], contact u8[N,4]")
        check_device_index(param_index, n)
        dev = q.device
        tau = torch.empty((n, NU), dtype=torch.float64, device=dev)
        met = torch.empty((n, 4), dtype=torch.float64, device=dev)
        st = torch.empty((n,), dtype=torch.int32, device=dev)
        vd = torch.empty((n, NV), dtype=torch.float64, device=dev) if debug else None
        f = torch.empty((n, 4, 3), dtype=torch.float64, device=dev) if debug else None
        qi = torch.empty((n, 4), dtype=torch.float64, device=dev) if debug else None
        lam = torch.empty((n, capi.NLAM), dtype=torch.float64, device=dev) if debug else None
        io = self.make_io(q, v, traj, contact, tau, met, st, vd, f, qi, lam)
        stream = torch.cuda.current_stream(dev).cuda_stream
        if per_robot:
            cp = _ctrl_params(param_set, None if param_index is None else C.c_void_p(param_index.data_ptr()))
            self._check(self.lib.wbc_step_params(self._h, k, n, C.byref(io), C.byref(cp), C.c_void_p(stream)), "wbc_step_params")
        else:
            self._check(self.lib.wbc_step(self._h, k, n, C.byref(io), C.c_void_p(stream)), "wbc_step")
        return StepOutput(tau, met, st, vd, f, qi, lam)

    @staticmethod
    def make_io(q, v, traj, contact, tau, met, st, vd=None, f=None, qi=None, lam=None) -> WbcIO:
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        return WbcIO(p(q), p(v), p(traj), p(contact), p(tau), p(met), p(st), p(vd), p(f), p(qi), p(lam))

    def time_step(self, kind, io: WbcIO, n: int, reps: int, stream=0) -> float:
        """Mean device milliseconds per launch over `reps` back-to-back launches (CUDA events on `stream`)."""
        k = KINDS[kind] if isinstance(kind, str) else int(kind)
        ms = C.c_double()
        self._check(self.lib.wbc_time_step(self._h, k, n, C.byref(io), reps, C.c_void_p(stream), C.byref(ms)), "wbc_time_step")
        return ms.value

    # ------------------------------------------------------------------ dynamics parity entry
    def dynamics(self, q, v):
        """CalcDynamics + CalcFramePositionQuantities x4 (basic_controller.py:101-115,173-196) for a batch
        of host states -> dict(M, Cv, tau_g, J_feet, Jdv_feet, p_feet) in Drake velocity order."""
        q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, NQ)
        n = q.shape[0]
        v = np.ascontiguousarray(v, dtype=np.float64).reshape(n, NV)
        out = dict(M=np.empty((n, NV, NV)), Cv=np.empty((n, NV)), tau_g=np.empty((n, NV)),
                   J_feet=np.empty((n, 4, 3, NV)), Jdv_feet=np.empty((n, 4, 3)), p_feet=np.empty((n, 4, 3)))
        fn = self.lib.wbc_dynamics_host
        fn.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 8
        fn.restype = C.c_int
        self._check(fn(self._h, n, np_ptr(q), np_ptr(v), np_ptr(out["M"]), np_ptr(out["Cv"]), np_ptr(out["tau_g"]),
                       np_ptr(out["J_feet"]), np_ptr(out["Jdv_feet"]), np_ptr(out["p_feet"])), "wbc_dynamics_host")
        return out

    def coriolis(self, q, v):
        """CalcCoriolisMatrix + CalcFrameJacobianDot x4 (basic_controller.py:117-132,198-220) -> C[n,18,18], Jd[n,4,3,18]."""
        q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, NQ)
        n = q.shape[0]
        v = np.ascontiguousarray(v, dtype=np.float64).reshape(n, NV)
        Cm, Jd = np.empty((n, NV, NV)), np.empty((n, 4, 3, NV))
        self._check(self.lib.wbc_coriolis_host(self._h, n, np_ptr(q), np_ptr(v), np_ptr(Cm), np_ptr(Jd)), "wbc_coriolis_host")
        return Cm, Jd

    def fk(self, q, v):
        """Foot positions and velocities (for synth.generate)."""
        d = self.dynamics(q, v)
        return d["p_feet"], np.einsum("nkij,nj->nki", d["J_feet"], np.asarray(v, float).reshape(len(d["M"]), NV))


def measure_fp64_peak(device=0) -> float:
    lib = capi.load_library()
    t = C.c_double()
    rc = lib.wbc_measure_fp64_peak(int(device), C.byref(t))
    if rc != 0:
        raise RuntimeError(f"wbc_measure_fp64_peak failed ({rc})")
    return t.value


# ----------------------------------------------------------------------- LeafSystem mirror
try:  # pragma: no cover - pydrake is not in the build image
    from pydrake.all import AbstractValue, BasicVector, LeafSystem
    _HAVE_DRAKE = True
except Exception:  # noqa: BLE001
    _HAVE_DRAKE = False

    class BasicVector:
        def __init__(self, n):
            self._v = np.zeros(int(n))

        def SetFromVector(self, v):
            self._v[:] = np.asarray(v, float).ravel()

        def get_value(self):
            return self._v

        def size(self):
            return self._v.size

    class AbstractValue:
        def __init__(self, v):
            self._v = v

        @staticmethod
        def Make(v):
            return AbstractValue(v)

        def get_value(self):
            return self._v

    class _Port:
        def __init__(self, name, index, model_value, calc=None):
            self.name, self.index, self.model_value, self.calc = name, index, model_value, calc

        def get_name(self):
            return self.name

        def get_index(self):
            return self.index

    class Context:
        """Stand-in for a Drake context: holds the fixed input-port values."""
        def __init__(self):
            self.inputs = {}

        def FixValue(self, index, value):
            self.inputs[index] = value

    class LeafSystem:
        def __init__(self):
            self._in, self._out = [], []

        def DeclareVectorInputPort(self, name, model):
            self._in.append(_Port(name, len(self._in), model))
            return self._in[-1]

        def DeclareAbstractInputPort(self, name, model):
            self._in.append(_Port(name, len(self._in), model))
            return self._in[-1]

        def DeclareVectorOutputPort(self, name, model, calc):
            self._out.append(_Port(name, len(self._out), model, calc))
            return self._out[-1]

        def get_input_port(self, i):
            return self._in[i]

        def get_output_port(self, i):
            return self._out[i]

        def GetInputPort(self, name):
            return next(p for p in self._in if p.name == name)

        def GetOutputPort(self, name):
            return next(p for p in self._out if p.name == name)

        def CreateDefaultContext(self):
            return Context()

        def EvalVectorInput(self, context, i):
            b = BasicVector(len(context.inputs[i]))
            b.SetFromVector(context.inputs[i])
            return b

        def EvalAbstractInput(self, context, i):
            return AbstractValue(context.inputs[i])

        def EvalOutput(self, context, i):
            port = self._out[i]
            out = BasicVector(port.model_value.size())
            port.calc(context, out)
            return out.get_value().copy()


def dict_to_traj_batch(d, n):
    """Trunk dict of arrays with a leading instance axis (SURVEY 8b: N > 1 under Drake) -> traj[N,54], contact[N,4].
    A dict without the leading axis (the reference's single-robot dict) is broadcast to all N instances."""
    traj, contact = np.zeros((n, NTRAJ)), np.zeros((n, 4), np.uint8)
    for k, key in enumerate(["p_body", "pd_body", "pdd_body", "rpy_body", "rpyd_body", "rpydd_body"]):
        traj[:, 3 * k:3 * k + 3] = np.asarray(d[key], float).reshape(-1, 3)
    for i, f in enumerate(FEET):
        traj[:, 18 + 3 * i:21 + 3 * i] = np.asarray(d["p_" + f], float).reshape(-1, 3)
        traj[:, 30 + 3 * i:33 + 3 * i] = np.asarray(d["pd_" + f], float).reshape(-1, 3)
        traj[:, 42 + 3 * i:45 + 3 * i] = np.asarray(d["pdd_" + f], float).reshape(-1, 3)
    contact[:] = np.asarray(d["contact_states"]).reshape(-1, 4) != 0
    return traj, contact


class _QPController(LeafSystem):
    KIND = "id"
    HAS_TRUNK_PORT = True

    def __init__(self, plant, dt, use_lcm=False, device=0, dof_order="depth_first", n_instances=1, **params):
        """`(plant, dt, use_lcm)` as in the reference (basic_controller.py:21). `plant`: a pydrake MultibodyPlant (its DOF
        order is read from the plant itself, SURVEY E.1), a robot name, or a RobotModel. `n_instances` > 1 widens the ports
        to 37N / 12N / 4N instance-major vectors and the trunk dict to arrays with a leading N axis (SURVEY 8b)."""
        LeafSystem.__init__(self)
        self.dt = dt
        self.plant = plant
        self.n = int(n_instances)
        if self.n < 1:
            raise ValueError("n_instances must be >= 1")
        from . import drake_bridge
        if drake_bridge.is_drake_plant(plant):
            # live plant: velocity / actuator numbering from GetJointByName(j).velocity_start() and MakeActuationMatrix()
            name = drake_bridge.robot_of_plant(plant)
            robot = load_robot(name)
            robot.v_index, robot.act_index = drake_bridge.derive_v_index(plant, name)
        else:
            robot = plant if isinstance(plant, (str, RobotModel)) else getattr(plant, "wbc_robot", "mini_cheetah")
        self.batched = BatchedController(robot, device=device, dof_order=dof_order, **params)
        self.DeclareVectorInputPort("quad_state", BasicVector((NQ + NV) * self.n))
        self.DeclareVectorOutputPort("quad_torques", BasicVector(NU * self.n), self.DoSetControlTorques)
        self.V = self.err = self.res = self.Vdot = 0.0 if self.n == 1 else np.zeros(self.n)
        self.DeclareVectorOutputPort("output_metrics", BasicVector(4 * self.n), self.SetLoggingOutputs)
        if self.HAS_TRUNK_PORT:
            self.DeclareAbstractInputPort("trunk_input", AbstractValue.Make({}))
        self.last_status = 0
        # page-locked step buffers and the wbc_io over them, made once: a control step writes the state and the trunk targets
        # into them and calls wbc_step_host, whose kernels read / write them directly (no per-step allocation or staging copy)
        n = self.n
        widths = (NQ, NV, NTRAJ, NU, 4)                                # q, v, traj, tau, metrics: doubles; then status, contact
        slab = capi.pinned_empty((n * (sum(widths) + 1),))             # ONE page-locked allocation (each costs milliseconds)
        slab[:] = 0.0
        views, o = [], 0
        for w in widths:
            views.append(slab[o:o + n * w].reshape(n, w))
            o += n * w
        self._hq, self._hv, self._ht, self._htau, self._hmet = views
        tail = slab[o:o + n].view(np.uint8)                            # 8 n bytes: n int32 status words, then 4 n contact flags
        self._hst, self._hc = tail[:4 * n].view(np.int32), tail[4 * n:8 * n].reshape(n, 4)
        self._slab = slab
        self._hio = WbcIO(np_ptr(self._hq), np_ptr(self._hv), np_ptr(self._ht), np_ptr(self._hc), np_ptr(self._htau), np_ptr(self._hmet),
                          np_ptr(self._hst), None, None, None)
        self._kind = KINDS[self.KIND]
        # LCM bridge (basic_controller.py:54-61): messages are decoded / encoded by the device codecs of wire.py. The
        # LCM runtime itself is optional: without it, feed `lcm_callback` yourself and read `published`.
        self.use_lcm = use_lcm
        if use_lcm and self.n != 1:
            raise ValueError("the LCM bridge carries one robot (basic_controller.py:79-87)")
        self.q, self.v = np.zeros(NQ), np.zeros(NV)
        self.published = []
        self.lc = None
        if use_lcm:
            from .wire import WireCodec
            self.wire = WireCodec(self.batched)
            try:  # pragma: no cover - no LCM runtime in the build image
                import lcm
                self.lc = lcm.LCM()
                self.lc.subscribe("robot_current_state", self.lcm_callback)
            except ImportError:
                self.lc = None

    def lcm_callback(self, channel, data):
        """basic_controller.py:79-87: latest robot state from a `robot_state_control_lcmt` message."""
        msg = np.frombuffer(bytes(data), np.uint8)
        if msg.size != 204:
            raise ValueError("Decode error")
        d = self.wire.decode_robot_state(msg[None])
        if d["status"][0] != 0:
            raise ValueError("Decode error")          # robot_state_control_lcmt.py:40
        self.q, self.v = d["q"][0].copy(), d["v"][0].copy()

    def SetLoggingOutputs(self, context, output):
        if self.n == 1:
            output.SetFromVector(np.asarray([self.V, self.err, self.res, self.Vdot], float))
        else:   # instance-major [V, err, res, Vdot] per robot
            output.SetFromVector(np.stack([np.broadcast_to(x, (self.n,)) for x in (self.V, self.err, self.res, self.Vdot)], axis=1).ravel())

    def DoSetControlTorques(self, context, output):
        if self.use_lcm:
            # basic_controller.py:291-297,307-317: state from LCM, torques out over LCM (velocity order), zeros to Drake
            if self.lc is not None:  # pragma: no cover
                self.lc.handle()
            u = self.ControlLaw(context, self.q, self.v)
            msgs, st = self.wire.encode_robot_state(None, None, np.asarray(u, float)[None], tau_in_actuator_order=True)
            if st[0] != 0:
                raise OverflowError("float too large to pack with f format")
            data = msgs[0].tobytes()
            self.published.append(("robot_control_input", data))
            del self.published[:-16]
            if self.lc is not None:  # pragma: no cover
                self.lc.publish("robot_control_input", data)
            output.SetFromVector(np.zeros(NU))
            return
        state = np.asarray(self.EvalVectorInput(context, 0).get_value(), float)
        if self.n == 1:
            q, v = state[:NQ], state[-NV:]               # basic_controller.py:299-302
        else:
            x = state.reshape(self.n, NQ + NV)
            q, v = x[:, :NQ], x[:, NQ:]
        output.SetFromVector(np.asarray(self.ControlLaw(context, q, v)).ravel())

    _TRUNK_KEYS = (["p_body", "pd_body", "pdd_body", "rpy_body", "rpyd_body", "rpydd_body"] + ["p_" + f for f in FEET]
                   + ["pd_" + f for f in FEET] + ["pdd_" + f for f in FEET])      # row order of traj[54] viewed as [18, 3]

    def ControlLaw(self, context, q, v):
        trunk = self.EvalAbstractInput(context, 1).get_value()
        if self.n == 1:
            try:        # one conversion for the 18 three-vectors of the dict (lists, (3,) or (3,1) arrays alike)
                self._ht[0] = np.array([trunk[k] for k in self._TRUNK_KEYS], dtype=np.float64).reshape(NTRAJ)
                self._hc[0] = trunk["contact_states"]
            except ValueError:
                self._ht[0], self._hc[0] = dict_to_traj(trunk)
            self._hq[0], self._hv[0] = q, v
        else:
            self._ht[:], self._hc[:] = dict_to_traj_batch(trunk, self.n)
            self._hq[:], self._hv[:] = q, v
        b = self.batched
        b._check(b.lib.wbc_step_host(b._h, self._kind, self.n, C.byref(self._hio)), "wbc_step_host")
        st = self._hst
        self.last_status = int(st[0]) if self.n == 1 else st.copy()
        # reference: `assert result.is_success()` (inverse_dynamics_controller.py:224); a zero / non-finite quaternion, gimbal
        # lock (CalcRpyDtFromAngularVelocityInParent) and PC in full flight (pc_controller.py:248-249) raise inside Drake /
        # NumPy there, so every status bit raises here
        if st.any():
            bad = np.nonzero(st)[0]
            raise AssertionError(f"QP solve failed for instance(s) {bad[:8].tolist()} (status "
                                 f"{int(st[bad[0]])}: {capi.status_names(int(st[bad[0]]))})")
        self._log(self._hmet[0] if self.n == 1 else self._hmet.T)
        return self._htau[0].copy() if self.n == 1 else self._htau.copy()

    def _log(self, m):
        self.err, self.res = self._f(m[1]), self._f(m[2])

    @staticmethod
    def _f(x):
        return float(x) if np.ndim(x) == 0 else np.array(x, float)


class IDController(_QPController):
    """Drop-in for reference controllers/inverse_dynamics_controller.py:IDController."""
    KIND = "id"


class CLFController(_QPController):
    """Drop-in for reference controllers/clf_controller.py:CLFController."""
    KIND = "clf"

    def _log(self, m):
        self.V, self.err, self.Vdot = self._f(m[0]), self._f(m[1]), self._f(m[3])


class PCController(_QPController):
    """Drop-in for reference controllers/pc_controller.py:PCController."""
    KIND = "pc"

    def _log(self, m):
        self.V, self.err, self.Vdot = self._f(m[0]), self._f(m[1]), self._f(m[3])


class MPTCController(PCController):
    """Drop-in for reference controllers/mptc_controller.py:MPTCController."""
    KIND = "mptc"


class BasicController(_QPController):
    """Drop-in for reference controllers/basic_controller.py:BasicController (joint-space PD, :322-352)."""
    KIND = "pd"
    HAS_TRUNK_PORT = False            # the reference BasicController declares no trunk input (basic_controller.py:33-50)

    def ControlLaw(self, context, q, v):
        if self.n == 1:
            return self.batched.step_pd(np.asarray(q)[None], np.asarray(v)[None])[0].copy()
        return self.batched.step_pd(q, v)
