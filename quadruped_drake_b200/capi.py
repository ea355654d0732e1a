"""ctypes binding of include/wbc.h (libwbc_b200.so). No torch types cross this boundary.

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a). There is no CPU
fallback: if the shared library is missing or no CUDA device is usable, loading raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from .model import WbcModelStruct

import os

# WBC_LIB lets experiments point at an alternative build of the same library (e.g. different launch bounds)
LIB_PATH = Path(os.environ.get("WBC_LIB") or (Path(__file__).resolve().parent / "csrc" / "libwbc_b200.so"))

WBC_CTRL_ID, WBC_CTRL_CLF, WBC_CTRL_PC, WBC_CTRL_MPTC, WBC_CTRL_PD = 0, 1, 2, 3, 4
KINDS = {"id": WBC_CTRL_ID, "clf": WBC_CTRL_CLF, "pc": WBC_CTRL_PC, "mptc": WBC_CTRL_MPTC, "pd": WBC_CTRL_PD}
ST_MAXITER, ST_INFEASIBLE, ST_RANKDEF, ST_GIMBAL, ST_NOTPD, ST_BADQUAT, ST_UNSUPPORTED, ST_DIVERGED = 1, 2, 4, 8, 16, 32, 64, 128
ST_NONFINITE = 256
ST_BADVARIANT = 512
ST_BADTERRAIN = 1024
ST_BADPARAMS = 2048
ST_BADLOOP = 4096
ST_BADMOTOR = 8192
ST_BADESTIM = 16384
ST_BADCONTACT = 32768
LOOP_HIST = 16
# contact detector (include/wbc.h, wbc_contact): consumers of the detected flags, and the columns of its per-robot stats
CONTACT_FEED_ESTIMATOR, CONTACT_FEED_CONTROLLER = 1, 2
CONTACT_NSTAT = 6
# rollout monitor (include/wbc.h, wbc_monitor): failure reasons and the columns of its per-robot stats
MON_POS, MON_ANG, MON_STATUS = 1, 2, 4
MON_NSTAT = 11
(MON_SUM_POS2, MON_MAX_POS, MON_SUM_ANG2, MON_MAX_ANG, MON_TAU2_DT, MON_WORK_ABS, MON_SAT_MAX, MON_F_MAX, MON_STANCE_UNLOADED,
 MON_SWING_LOADED, MON_DIST_XY) = range(MON_NSTAT)
NLAM = 42
_ST_NAMES = {ST_MAXITER: "MAXITER", ST_INFEASIBLE: "INFEASIBLE", ST_RANKDEF: "RANKDEF", ST_GIMBAL: "GIMBAL", ST_NOTPD: "NOTPD",
             ST_BADQUAT: "BADQUAT", ST_UNSUPPORTED: "UNSUPPORTED", ST_DIVERGED: "DIVERGED",
             ST_NONFINITE: "NONFINITE", ST_BADVARIANT: "BADVARIANT", ST_BADTERRAIN: "BADTERRAIN",
             ST_BADPARAMS: "BADPARAMS", ST_BADLOOP: "BADLOOP", ST_BADMOTOR: "BADMOTOR",
             ST_BADESTIM: "BADESTIM", ST_BADCONTACT: "BADCONTACT"}


def status_names(status: int) -> str:
    return "|".join(n for b, n in _ST_NAMES.items() if status & b) or "OK"

_PARAM_DOUBLES = [
    "id_kp_body_p", "id_kd_body_p", "id_kp_body_rpy", "id_kd_body_rpy", "id_kp_foot", "id_kd_foot", "id_w_body", "id_w_foot",
    "clf_q_body_p", "clf_q_body_pd", "clf_q_body_rpy", "clf_q_body_rpyd", "clf_q_foot_p", "clf_q_foot_pd", "clf_r", "clf_w_delta",
    "pc_kp_body_p", "pc_kd_body_p", "pc_kp_body_rpy", "pc_kd_body_rpy", "pc_kp_foot", "pc_kd_foot", "pc_w_body", "pc_w_foot",
    "mu", "contact_damping", "reg_f", "reg_tau", "reg_vd",
]


class WbcParams(C.Structure):
    """ctypes mirror of `wbc_params`."""
    _fields_ = [(n, C.c_double) for n in _PARAM_DOUBLES] + [("torque_limits", C.c_int32), ("max_iter", C.c_int32),
                                                              ("pd_kp", C.c_double), ("pd_kd", C.c_double), ("pd_clip", C.c_double),
                                                              ("pd_q_nom", C.c_double * 12)]


# Reference constants (SURVEY.md Appendix G); kept here so the struct can be filled without the library.
DEFAULT_PARAMS = dict(
    id_kp_body_p=500.0, id_kd_body_p=50.0, id_kp_body_rpy=500.0, id_kd_body_rpy=50.0,
    id_kp_foot=100.0, id_kd_foot=20.0, id_w_body=10.0, id_w_foot=1.0,
    clf_q_body_p=5000.0, clf_q_body_pd=200.0, clf_q_body_rpy=5000.0, clf_q_body_rpyd=200.0,
    clf_q_foot_p=200.0, clf_q_foot_pd=20.0, clf_r=1.0, clf_w_delta=1000.0,
    pc_kp_body_p=100.0, pc_kd_body_p=10.0, pc_kp_body_rpy=100.0, pc_kd_body_rpy=10.0,
    pc_kp_foot=200.0, pc_kd_foot=20.0, pc_w_body=10.0, pc_w_foot=1.0,
    mu=0.7, contact_damping=100.0, reg_f=1e-6, reg_tau=0.0, reg_vd=0.0, torque_limits=0, max_iter=200,
    pd_kp=30.0, pd_kd=1.5, pd_clip=150.0, pd_q_nom=(0.0, -0.8, 1.6) * 4,
)


def make_params(**overrides) -> WbcParams:
    vals = dict(DEFAULT_PARAMS)
    unknown = set(overrides) - set(vals)
    if unknown:
        raise KeyError(f"unknown controller parameters: {sorted(unknown)}")
    vals.update(overrides)
    p = WbcParams()
    for k, v in vals.items():
        if k == "pd_q_nom":
            for i, x in enumerate(v):
                p.pd_q_nom[i] = float(x)
        else:
            setattr(p, k, int(v) if k in ("torque_limits", "max_iter") else float(v))
    return p


class WbcIO(C.Structure):
    """ctypes mirror of `wbc_io`; pointers are raw addresses (host or device)."""
    _fields_ = [("q", C.c_void_p), ("v", C.c_void_p), ("traj", C.c_void_p), ("contact", C.c_void_p),
                ("tau", C.c_void_p), ("metrics", C.c_void_p), ("status", C.c_void_p),
                ("vd", C.c_void_p), ("f", C.c_void_p), ("qp_info", C.c_void_p), ("lam", C.c_void_p)]


class WbcRolloutIO(C.Structure):
    """ctypes mirror of `wbc_rollout_io`."""
    _fields_ = [(n, C.c_void_p) for n in ("q", "v", "t", "plan_index", "tau", "metrics", "status_or", "err_max", "metrics_log")]


class WbcPlantOpts(C.Structure):
    """ctypes mirror of `wbc_plant_opts` (ground friction, penetration correction, Gauss-Seidel sweeps)."""
    _fields_ = [("mu", C.c_double), ("erp", C.c_double), ("iters", C.c_int32), ("reserved", C.c_int32)]


class WbcRolloutOpts(C.Structure):
    """ctypes mirror of `wbc_rollout_opts`."""
    _fields_ = [("use_graph", C.c_int32), ("plant", C.c_int32), ("plant_opts", WbcPlantOpts), ("f_contact", C.c_void_p)]


class WbcPlantPerturb(C.Structure):
    """ctypes mirror of `wbc_plant_perturb` (variant set, per-robot variant index, per-robot push rows)."""
    _fields_ = [("set", C.c_void_p), ("variant", C.c_void_p), ("push", C.c_void_p)]


class WbcTerrainDesc(C.Structure):
    """ctypes mirror of `wbc_terrain_desc` (plane z0 + sx x + sy y, optional height grid [ny][nx] at (x0, y0), spacing dx, dy)."""
    _fields_ = [("z0", C.c_double), ("sx", C.c_double), ("sy", C.c_double), ("nx", C.c_int32), ("ny", C.c_int32),
                ("x0", C.c_double), ("y0", C.c_double), ("dx", C.c_double), ("dy", C.c_double), ("heights", C.c_void_p)]


class WbcPlantTerrain(C.Structure):
    """ctypes mirror of `wbc_plant_terrain` (terrain set, per-robot terrain index)."""
    _fields_ = [("set", C.c_void_p), ("index", C.c_void_p)]


class WbcCtrlParams(C.Structure):
    """ctypes mirror of `wbc_ctrl_params` (parameter set, per-robot set index)."""
    _fields_ = [("set", C.c_void_p), ("index", C.c_void_p)]


class WbcLoop(C.Structure):
    """ctypes mirror of `wbc_loop` (per-robot noise, delay, strength and stream; the seed; the loop state hist / tick)."""
    _fields_ = [("noise", C.c_void_p), ("delay", C.c_void_p), ("strength", C.c_void_p), ("stream", C.c_void_p), ("seed", C.c_uint64),
                ("hist", C.c_void_p), ("tick", C.c_void_p)]


class WbcMotorDesc(C.Structure):
    """ctypes mirror of `wbc_motor_desc`: seven per-joint arrays [12] in the model's joint order."""
    _fields_ = [(name, C.c_double * 12) for name in ("peak", "speed_knee", "speed_free", "lag", "damping", "coulomb", "coulomb_speed")]


class WbcPlantMotor(C.Structure):
    """ctypes mirror of `wbc_plant_motor` (set, index [N]; the state tau_m [N][12] and count [N], both or neither)."""
    _fields_ = [("set", C.c_void_p), ("index", C.c_void_p), ("tau_m", C.c_void_p), ("count", C.c_void_p)]


class WbcEstimatorDesc(C.Structure):
    """ctypes mirror of `wbc_estimator_desc`: process, measurement and initial standard deviations, and the swing scale."""
    _fields_ = [(name, C.c_double) for name in ("q_pos", "q_vel", "q_foot", "r_pos", "r_vel", "r_height", "swing_scale", "p0_pos",
                                                "p0_vel", "p0_foot")]


class WbcContactDesc(C.Structure):
    """ctypes mirror of `wbc_contact_desc`: force filter time constant (s) and the stance thresholds f_on >= f_off (N)."""
    _fields_ = [(name, C.c_double) for name in ("tau_f", "f_on", "f_off")]


class WbcContact(C.Structure):
    """ctypes mirror of `wbc_contact` (set, index [N], feed; the state q_prev [N][19], v_prev [N][18], tau_prev [N][12],
    f_true [N][12], f_hat [N][12], flag [N][4] and count [N], all or none; stats [N][6] or NULL)."""
    _fields_ = [("set", C.c_void_p), ("index", C.c_void_p), ("feed", C.c_int32)] + \
        [(name, C.c_void_p) for name in ("q_prev", "v_prev", "tau_prev", "f_true", "f_hat", "flag", "count", "stats")]


class WbcEstimator(C.Structure):
    """ctypes mirror of `wbc_estimator` (set, index [N], accel_noise [N]; the state x [N][18], P [N][18][18], v_prev [N][3] and
    count [N], all or none; stats [N][4] or NULL)."""
    _fields_ = [(name, C.c_void_p) for name in ("set", "index", "accel_noise", "x", "P", "v_prev", "count", "stats")]


class WbcMonitor(C.Structure):
    """ctypes mirror of `wbc_monitor` (failure bounds; the per-robot state stats / steps / fail_step / fail_why; optional why)."""
    _fields_ = [("pos_max", C.c_double), ("ang_max", C.c_double), ("stats", C.c_void_p), ("steps", C.c_void_p),
                ("fail_step", C.c_void_p), ("fail_why", C.c_void_p), ("why", C.c_void_p)]


def np_ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


_lib = None


def load_library() -> C.CDLL:
    """Load libwbc_b200.so and declare every symbol of include/wbc.h. Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(f"{LIB_PATH} is not built - run `python -c 'import __graft_entry__ as g; g.build()'`. "
                           "There is no CPU fallback for the controller path.")
    lib = C.CDLL(str(LIB_PATH))
    H = C.c_void_p
    i64, i32, dp = C.c_int64, C.c_int, C.c_void_p
    lib.wbc_default_params.argtypes = [C.POINTER(WbcParams)]
    lib.wbc_create.argtypes = [C.POINTER(WbcModelStruct), C.POINTER(WbcParams), i32, C.POINTER(H)]
    lib.wbc_destroy.argtypes = [H]
    lib.wbc_last_error.argtypes = [H]
    lib.wbc_last_error.restype = C.c_char_p
    lib.wbc_dynamics.argtypes = [H, i64, dp, dp, dp, dp, dp, dp, dp, dp, dp]
    lib.wbc_coriolis.argtypes = [H, i64, dp, dp, dp, dp, dp]
    lib.wbc_coriolis_host.argtypes = [H, i64, dp, dp, dp, dp]
    lib.wbc_coriolis_host.restype = C.c_int
    lib.wbc_step.argtypes = [H, i32, i64, C.POINTER(WbcIO), dp]
    for name in ("wbc_step_id", "wbc_step_clf", "wbc_step_pc", "wbc_step_mptc"):
        getattr(lib, name).argtypes = [H, i64, dp, dp, dp, dp, dp, dp, dp, dp]
        getattr(lib, name).restype = C.c_int
    lib.wbc_step_pd.argtypes = [H, i64, dp, dp, dp, dp]
    lib.wbc_step_pd.restype = C.c_int
    lib.wbc_step_host.argtypes = [H, i32, i64, C.POINTER(WbcIO)]
    lib.wbc_time_step.argtypes = [H, i32, i64, C.POINTER(WbcIO), i32, dp, C.POINTER(C.c_double)]
    lib.wbc_profile_step.argtypes = [H, i32, i64, C.POINTER(WbcIO), i32, dp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.wbc_profile_step.restype = C.c_int
    lib.wbc_measure_fp64_peak.argtypes = [i32, C.POINTER(C.c_double)]
    lib.wbc_dynamics_host.argtypes = [H, i64] + [dp] * 8
    lib.wbc_dynamics_host.restype = C.c_int
    lib.wbc_host_alloc.argtypes = [C.c_size_t]
    lib.wbc_host_alloc.restype = C.c_void_p
    lib.wbc_host_free.argtypes = [C.c_void_p]
    lib.wbc_host_free.restype = None
    u8 = dp
    lib.wbc_lcm_decode_trunk_state.argtypes = [H, i64, u8, dp, dp, dp, dp, dp, dp, dp]
    lib.wbc_lcm_encode_trunk_state.argtypes = [H, i64, dp, dp, dp, dp, dp, u8, dp]
    lib.wbc_lcm_decode_robot_state.argtypes = [H, i64, u8, dp, dp, dp, dp, dp]
    lib.wbc_lcm_encode_robot_state.argtypes = [H, i64, dp, dp, dp, i32, u8, dp, dp]
    lib.wbc_lcm_decode_trunk_state_host.argtypes = [H, i64, u8, dp, dp, dp, dp, dp, dp]
    lib.wbc_lcm_encode_trunk_state_host.argtypes = [H, i64, dp, dp, dp, dp, dp, u8]
    lib.wbc_lcm_decode_robot_state_host.argtypes = [H, i64, u8, dp, dp, dp, dp]
    lib.wbc_lcm_encode_robot_state_host.argtypes = [H, i64, dp, dp, dp, i32, u8, dp]
    lib.wbc_plan_destroy.argtypes = [dp]
    lib.wbc_plan_destroy.restype = C.c_int
    lib.wbc_sample_trajectory.argtypes = [H, dp, i64, dp, dp, dp, dp, dp, dp, dp, dp]
    lib.wbc_sample_trajectory_host.argtypes = [H, dp, i64, dp, dp, dp, dp, dp, dp, dp]
    lib.wbc_sample_trajectory.restype = lib.wbc_sample_trajectory_host.restype = lib.wbc_plan_create.restype = C.c_int
    lib.wbc_step_plan_host.argtypes = [H, i32, dp, i64, dp, dp, dp, dp, dp, dp, dp]
    lib.wbc_step_plan_host.restype = C.c_int
    lib.wbc_integrate.argtypes = [H, i64, C.c_double, dp, dp, dp, dp, dp]
    lib.wbc_rollout.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), i32, dp]
    lib.wbc_rollout_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), i32]
    lib.wbc_integrate.restype = lib.wbc_rollout.restype = lib.wbc_rollout_host.restype = C.c_int
    lib.wbc_default_plant_opts.argtypes = [C.POINTER(WbcPlantOpts)]
    lib.wbc_plant_step.argtypes = [H, i64, C.c_double, C.POINTER(WbcPlantOpts), dp, dp, dp, dp, dp, dp, dp, dp]
    lib.wbc_plant_step_host.argtypes = [H, i64, C.c_double, C.POINTER(WbcPlantOpts), dp, dp, dp, dp, dp, dp, dp]
    lib.wbc_rollout_ex.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts), dp]
    lib.wbc_rollout_ex_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts)]
    lib.wbc_default_plant_opts.restype = lib.wbc_plant_step.restype = lib.wbc_plant_step_host.restype = C.c_int
    lib.wbc_rollout_ex.restype = lib.wbc_rollout_ex_host.restype = C.c_int
    lib.wbc_plant_set_create.argtypes = [H, C.c_int32, C.POINTER(WbcModelStruct), dp, C.POINTER(H)]
    lib.wbc_plant_set_destroy.argtypes = [dp]
    lib.wbc_plant_step_perturbed.argtypes = [H, i64, C.c_double, C.POINTER(WbcPlantOpts), C.POINTER(WbcPlantPerturb)] + [dp] * 8
    lib.wbc_plant_step_perturbed_host.argtypes = [H, i64, C.c_double, C.POINTER(WbcPlantOpts), C.POINTER(WbcPlantPerturb)] + [dp] * 7
    lib.wbc_rollout_perturbed.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                          C.POINTER(WbcPlantPerturb), dp]
    lib.wbc_rollout_perturbed_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                               C.POINTER(WbcPlantPerturb)]
    lib.wbc_terrain_set_create.argtypes = [H, C.c_int32, C.POINTER(WbcTerrainDesc), C.POINTER(H)]
    lib.wbc_terrain_set_destroy.argtypes = [dp]
    lib.wbc_plant_step_terrain.argtypes = [H, i64, C.c_double, C.POINTER(WbcPlantOpts), C.POINTER(WbcPlantPerturb),
                                           C.POINTER(WbcPlantTerrain)] + [dp] * 8
    lib.wbc_plant_step_terrain_host.argtypes = [H, i64, C.c_double, C.POINTER(WbcPlantOpts), C.POINTER(WbcPlantPerturb),
                                                C.POINTER(WbcPlantTerrain)] + [dp] * 7
    lib.wbc_rollout_terrain.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                        C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), dp]
    lib.wbc_rollout_terrain_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                             C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain)]
    lib.wbc_param_set_create.argtypes = [H, C.c_int32, C.POINTER(WbcParams), C.POINTER(H)]
    lib.wbc_param_set_destroy.argtypes = [dp]
    lib.wbc_step_params.argtypes = [H, i32, i64, C.POINTER(WbcIO), C.POINTER(WbcCtrlParams), dp]
    lib.wbc_step_params_host.argtypes = [H, i32, i64, C.POINTER(WbcIO), C.POINTER(WbcCtrlParams)]
    lib.wbc_rollout_params.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                       C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams), dp]
    lib.wbc_rollout_params_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                            C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams)]
    lib.wbc_rollout_loop.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                     C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams), C.POINTER(WbcLoop), dp]
    lib.wbc_rollout_loop_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                          C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams), C.POINTER(WbcLoop)]
    lib.wbc_loop_observe.argtypes = [H, i64, C.POINTER(WbcLoop), dp, dp, dp, dp, dp]
    lib.wbc_loop_observe_host.argtypes = [H, i64, C.POINTER(WbcLoop), dp, dp, dp, dp]
    lib.wbc_rollout_monitor.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                        C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams), C.POINTER(WbcLoop),
                                        C.POINTER(WbcMonitor), dp]
    lib.wbc_rollout_monitor_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                             C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams),
                                             C.POINTER(WbcLoop), C.POINTER(WbcMonitor)]
    lib.wbc_monitor_step.argtypes = [H, i64, C.c_double, C.POINTER(WbcMonitor)] + [dp] * 8
    lib.wbc_monitor_step_host.argtypes = [H, i64, C.c_double, C.POINTER(WbcMonitor)] + [dp] * 7
    lib.wbc_motor_set_create.argtypes = [H, C.c_int32, C.POINTER(WbcMotorDesc), C.POINTER(H)]
    lib.wbc_motor_set_destroy.argtypes = [dp]
    lib.wbc_rollout_motor.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                      C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams), C.POINTER(WbcLoop),
                                      C.POINTER(WbcMonitor), C.POINTER(WbcPlantMotor), dp]
    lib.wbc_rollout_motor_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                           C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams),
                                           C.POINTER(WbcLoop), C.POINTER(WbcMonitor), C.POINTER(WbcPlantMotor)]
    lib.wbc_motor_apply.argtypes = [H, i64, C.c_double, C.POINTER(WbcPlantMotor)] + [dp] * 5
    lib.wbc_motor_apply_host.argtypes = [H, i64, C.c_double, C.POINTER(WbcPlantMotor)] + [dp] * 4
    lib.wbc_estimator_set_create.argtypes = [H, C.c_int32, C.POINTER(WbcEstimatorDesc), C.POINTER(H)]
    lib.wbc_estimator_set_destroy.argtypes = [dp]
    lib.wbc_rollout_estimator.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                          C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams),
                                          C.POINTER(WbcLoop), C.POINTER(WbcMonitor), C.POINTER(WbcPlantMotor), C.POINTER(WbcEstimator), dp]
    lib.wbc_rollout_estimator_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                               C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams),
                                               C.POINTER(WbcLoop), C.POINTER(WbcMonitor), C.POINTER(WbcPlantMotor), C.POINTER(WbcEstimator)]
    lib.wbc_estimator_step.argtypes = [H, i64, C.c_double, C.POINTER(WbcEstimator), C.POINTER(WbcLoop)] + [dp] * 7
    lib.wbc_estimator_step_host.argtypes = [H, i64, C.c_double, C.POINTER(WbcEstimator), C.POINTER(WbcLoop)] + [dp] * 6
    lib.wbc_contact_set_create.argtypes = [H, C.c_int32, C.POINTER(WbcContactDesc), C.POINTER(H)]
    lib.wbc_contact_set_destroy.argtypes = [dp]
    lib.wbc_rollout_contact.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                        C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams),
                                        C.POINTER(WbcLoop), C.POINTER(WbcMonitor), C.POINTER(WbcPlantMotor), C.POINTER(WbcEstimator),
                                        C.POINTER(WbcContact), dp]
    lib.wbc_rollout_contact_host.argtypes = [H, i32, dp, i64, C.c_int32, C.c_double, C.POINTER(WbcRolloutIO), C.POINTER(WbcRolloutOpts),
                                             C.POINTER(WbcPlantPerturb), C.POINTER(WbcPlantTerrain), C.POINTER(WbcCtrlParams),
                                             C.POINTER(WbcLoop), C.POINTER(WbcMonitor), C.POINTER(WbcPlantMotor), C.POINTER(WbcEstimator),
                                             C.POINTER(WbcContact)]
    lib.wbc_contact_step.argtypes = [H, i64, C.c_double, C.POINTER(WbcContact)] + [dp] * 6
    lib.wbc_contact_step_host.argtypes = [H, i64, C.c_double, C.POINTER(WbcContact)] + [dp] * 5
    for name in PERTURB_SYMBOLS + TERRAIN_SYMBOLS + PARAM_SYMBOLS + LOOP_SYMBOLS + MONITOR_SYMBOLS + MOTOR_SYMBOLS + ESTIMATOR_SYMBOLS + \
            CONTACT_SYMBOLS:
        getattr(lib, name).restype = C.c_int
    for name in WIRE_SYMBOLS:
        getattr(lib, name).restype = C.c_int
    lib.wbc_multi_create.argtypes = [C.POINTER(WbcModelStruct), C.POINTER(WbcParams), i32, C.POINTER(C.c_int), C.POINTER(H)]
    lib.wbc_multi_destroy.argtypes = [H]
    lib.wbc_multi_last_error.argtypes = [H]
    lib.wbc_multi_last_error.restype = C.c_char_p
    lib.wbc_multi_device_count.argtypes = [H]
    lib.wbc_multi_launch_count.argtypes = [H]
    lib.wbc_multi_launch_count.restype = C.c_int64
    lib.wbc_multi_step_host.argtypes = [H, i32, i64, C.POINTER(WbcIO)]
    lib.wbc_multi_create.restype = lib.wbc_multi_destroy.restype = lib.wbc_multi_device_count.restype = lib.wbc_multi_step_host.restype = C.c_int
    lib.wbc_launch_count.argtypes = [H]
    lib.wbc_launch_count.restype = C.c_int64
    for name in ("wbc_default_params", "wbc_create", "wbc_destroy", "wbc_dynamics", "wbc_coriolis", "wbc_step",
                 "wbc_step_id", "wbc_step_clf", "wbc_step_pc", "wbc_step_host", "wbc_time_step", "wbc_measure_fp64_peak"):
        getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


WIRE_SYMBOLS = ["wbc_lcm_decode_trunk_state", "wbc_lcm_encode_trunk_state", "wbc_lcm_decode_robot_state", "wbc_lcm_encode_robot_state",
                "wbc_lcm_decode_trunk_state_host", "wbc_lcm_encode_trunk_state_host", "wbc_lcm_decode_robot_state_host",
                "wbc_lcm_encode_robot_state_host"]
ROLLOUT_SYMBOLS = ["wbc_integrate", "wbc_rollout", "wbc_rollout_host", "wbc_rollout_ex", "wbc_rollout_ex_host", "wbc_plant_step",
                   "wbc_plant_step_host", "wbc_default_plant_opts"]
PERTURB_SYMBOLS = ["wbc_plant_set_create", "wbc_plant_set_destroy", "wbc_plant_step_perturbed", "wbc_plant_step_perturbed_host",
                   "wbc_rollout_perturbed", "wbc_rollout_perturbed_host"]
TERRAIN_SYMBOLS = ["wbc_terrain_set_create", "wbc_terrain_set_destroy", "wbc_plant_step_terrain", "wbc_plant_step_terrain_host",
                   "wbc_rollout_terrain", "wbc_rollout_terrain_host"]
PARAM_SYMBOLS = ["wbc_param_set_create", "wbc_param_set_destroy", "wbc_step_params", "wbc_step_params_host", "wbc_rollout_params",
                 "wbc_rollout_params_host"]
LOOP_SYMBOLS = ["wbc_rollout_loop", "wbc_rollout_loop_host", "wbc_loop_observe", "wbc_loop_observe_host"]
MONITOR_SYMBOLS = ["wbc_rollout_monitor", "wbc_rollout_monitor_host", "wbc_monitor_step", "wbc_monitor_step_host"]
MOTOR_SYMBOLS = ["wbc_motor_set_create", "wbc_motor_set_destroy", "wbc_rollout_motor", "wbc_rollout_motor_host", "wbc_motor_apply",
                 "wbc_motor_apply_host"]
ESTIMATOR_SYMBOLS = ["wbc_estimator_set_create", "wbc_estimator_set_destroy", "wbc_rollout_estimator", "wbc_rollout_estimator_host",
                     "wbc_estimator_step", "wbc_estimator_step_host"]
CONTACT_SYMBOLS = ["wbc_contact_set_create", "wbc_contact_set_destroy", "wbc_rollout_contact", "wbc_rollout_contact_host",
                   "wbc_contact_step", "wbc_contact_step_host"]
TRAJ_SYMBOLS = ROLLOUT_SYMBOLS + PERTURB_SYMBOLS + TERRAIN_SYMBOLS + PARAM_SYMBOLS + LOOP_SYMBOLS + MONITOR_SYMBOLS + MOTOR_SYMBOLS + ESTIMATOR_SYMBOLS + CONTACT_SYMBOLS + ["wbc_step_plan_host", "wbc_plan_create", "wbc_plan_destroy", "wbc_sample_trajectory", "wbc_sample_trajectory_host"]
MULTI_SYMBOLS = ["wbc_multi_create", "wbc_multi_destroy", "wbc_multi_last_error", "wbc_multi_device_count", "wbc_multi_launch_count",
                 "wbc_multi_step_host"]
EXPORTED_SYMBOLS = WIRE_SYMBOLS + TRAJ_SYMBOLS + MULTI_SYMBOLS + ["wbc_default_params", "wbc_create", "wbc_destroy", "wbc_last_error", "wbc_dynamics", "wbc_coriolis",
                    "wbc_step", "wbc_step_id", "wbc_step_clf", "wbc_step_pc", "wbc_step_mptc", "wbc_step_pd", "wbc_step_host", "wbc_time_step", "wbc_profile_step",
                    "wbc_measure_fp64_peak", "wbc_launch_count", "wbc_dynamics_host", "wbc_coriolis_host", "wbc_host_alloc", "wbc_host_free"]


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """NumPy array over page-locked host memory (wbc_host_alloc); freed when the array is collected."""
    lib = load_library()
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    ptr = lib.wbc_host_alloc(max(nbytes, 1))
    if not ptr:
        raise MemoryError("wbc_host_alloc failed")
    buf = (C.c_char * max(nbytes, 1)).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    import weakref
    weakref.finalize(buf, lib.wbc_host_free, ptr)
    return arr
