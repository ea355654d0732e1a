"""ORACLE (test infrastructure only): numpy restatement of the rollout monitor of the ground-plant loop (include/wbc.h,
wbc_monitor; csrc/wbc_monitor.cuh), written from its definition. Per control step, after the plant step:

    e_p     = |q[4:7] - traj[0:3]|
    e_theta = 2 atan2(|u|, |w|),  (w, u) = conj(q_ref) (x) q / |q|,  q_ref = qz(yaw) (x) qy(pitch) (x) qx(roll) of traj[9:12]
    reasons = POS if !(e_p <= pos_max) | ANG if !(e_theta <= ang_max) | STATUS if the step's status word != 0
    steps += 1; the first step with a reason sets fail_step = steps and fail_why = reasons, once; why = reasons
    stats: sums and maxima (m = e > m ? e : m) of e_p^2, e_p, e_theta^2, e_theta, dt sum tau^2, dt sum_j |tau_act[j] v_vidx[j]|,
           max_j |tau_act[j]| / effort_j, max_foot |f|, stance feet with f == 0, swing feet with f != 0, dt |v[3:5]|
"""
from __future__ import annotations

import numpy as np

POS, ANG, STATUS = 1, 2, 4
NSTAT = 11
(SUM_POS2, MAX_POS, SUM_ANG2, MAX_ANG, TAU2_DT, WORK_ABS, SAT_MAX, F_MAX, STANCE_UNLOADED, SWING_LOADED, DIST_XY) = range(NSTAT)


def quat_mul(a, b):
    """Hamilton product of [..., 4] quaternions [w x y z]."""
    aw, ax, ay, az = np.moveaxis(np.asarray(a, np.float64), -1, 0)
    bw, bx, by, bz = np.moveaxis(np.asarray(b, np.float64), -1, 0)
    return np.stack([aw * bw - ax * bx - ay * by - az * bz, aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx, aw * bz + ax * by - ay * bx + az * bw], axis=-1)


def rpy_quat(rpy):
    """Quaternion of Drake's RollPitchYaw [..., 3]: qz(yaw) (x) qy(pitch) (x) qx(roll)."""
    rpy = np.asarray(rpy, np.float64)
    h = 0.5 * rpy
    z = np.zeros(rpy.shape[:-1])
    qx = np.stack([np.cos(h[..., 0]), np.sin(h[..., 0]), z, z], axis=-1)
    qy = np.stack([np.cos(h[..., 1]), z, np.sin(h[..., 1]), z], axis=-1)
    qz = np.stack([np.cos(h[..., 2]), z, z, np.sin(h[..., 2])], axis=-1)
    return quat_mul(quat_mul(qz, qy), qx)


def quat_matrix(q):
    """Rotation matrix of a unit quaternion [w x y z]."""
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def errors(q, traj):
    """e_p, e_theta of rows q [N,19] against traj [N,54]."""
    q, traj = np.atleast_2d(q), np.atleast_2d(traj)
    ep = np.linalg.norm(q[:, 4:7] - traj[:, 0:3], axis=1)
    qh = q[:, 0:4] / np.linalg.norm(q[:, 0:4], axis=1, keepdims=True)
    ref = rpy_quat(traj[:, 9:12]) * np.array([1.0, -1.0, -1.0, -1.0])
    d = quat_mul(ref, qh)
    eth = 2.0 * np.arctan2(np.linalg.norm(d[:, 1:], axis=1), np.abs(d[:, 0]))
    return ep, eth


class State:
    """The per-robot monitor state of N robots; zeroed is fresh."""

    def __init__(self, n):
        self.stats, self.steps = np.zeros((n, NSTAT)), np.zeros(n, np.int64)
        self.fail_step, self.fail_why, self.why = np.zeros(n, np.int64), np.zeros(n, np.int32), np.zeros(n, np.int32)


def _max(e, m):
    return np.where(e > m, e, m)


def step(st, dt, pos_max, ang_max, v_index, act_index, effort, q, v, traj, contact, tau, f, status=None):
    """One monitored step of N robots (rows): q [N,19], v [N,18] post-step, traj [N,54], contact [N,4], tau [N,12] applied
    (actuator order), f [N,12] world ground forces, status [N] (None: 0). Updates st in place."""
    q, v, traj, tau, f = (np.atleast_2d(np.asarray(x, np.float64)) for x in (q, v, traj, tau, f))
    contact = np.atleast_2d(contact) != 0
    n = len(q)
    status = np.zeros(n, np.int64) if status is None else np.asarray(status)
    ep, eth = errors(q, traj)
    with np.errstate(invalid="ignore"):
        why = (np.where(~(ep <= pos_max), POS, 0) | np.where(~(eth <= ang_max), ANG, 0) | np.where(status != 0, STATUS, 0)).astype(np.int32)
    st.steps += 1
    first = (why != 0) & (st.fail_step == 0)
    st.fail_step[first] = st.steps[first]
    st.fail_why[first] = why[first]
    st.why[:] = why
    tj = tau[:, np.asarray(act_index)]                      # torque of joint j
    vj = v[:, np.asarray(v_index)]
    ff = f.reshape(n, 4, 3)
    zero = (ff == 0.0).all(axis=2)
    s = st.stats
    with np.errstate(invalid="ignore", divide="ignore"):
        s[:, SUM_POS2] += ep * ep
        s[:, MAX_POS] = _max(ep, s[:, MAX_POS])
        s[:, SUM_ANG2] += eth * eth
        s[:, MAX_ANG] = _max(eth, s[:, MAX_ANG])
        s[:, TAU2_DT] += dt * (tau * tau).sum(axis=1)
        s[:, WORK_ABS] += dt * np.abs(tj * vj).sum(axis=1)
        sat = np.zeros(n)
        for j in range(12):
            sat = _max(np.abs(tj[:, j]) / effort[j], sat)
        s[:, SAT_MAX] = _max(sat, s[:, SAT_MAX])
        fm = np.zeros(n)
        for k in range(4):
            fm = _max(np.linalg.norm(ff[:, k], axis=1), fm)
        s[:, F_MAX] = _max(fm, s[:, F_MAX])
        s[:, STANCE_UNLOADED] += (contact & zero).sum(axis=1)
        s[:, SWING_LOADED] += (~contact & ~zero).sum(axis=1)
        s[:, DIST_XY] += dt * np.sqrt(v[:, 3] ** 2 + v[:, 4] ** 2)
    return st
