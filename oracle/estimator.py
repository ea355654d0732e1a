"""ORACLE (test infrastructure only): numpy restatement of the state estimator of the ground-plant loop (include/wbc.h,
wbc_estimator_desc / wbc_estimator; csrc/wbc_estimator.cuh), written from its definition. Robot i with record r, at loop tick c:

    state     x = [p (3), v (3), foot LF, RF, LH, RH (4 x 3)] (world), P [18][18], v_prev [3], count
    legs      r_k(q), J_k(q) thetadot: foot k relative to the base origin, base axes, from joint_xyz / joint_axis / foot_xyz
    accel     a_w = (v[3:6] - v_prev) / dt;  f_b = R_true' (a_w - g) + sigma_acc z,  z = normals of Philox draws 18 and 19 of the
              loop counter (j, stream, c_lo, c_hi); the filter input a = R_obs f_b + g
    prime     (count <= 0) p = q_obs[4:7], v = v_obs[3:6], foot_k = p + R_obs r_k(q_obs), P = diag(p0_pos^2, p0_vel^2, p0_foot^2);
              output unchanged, v_prev = v[3:6], count = 1
    predict   v += dt a; p += dt v (the plant's semi-implicit Euler); P = A P A' + Q, Q = dt diag(q_pos^2, q_vel^2, (q_foot s_k)^2)
    update    28 rows, leg by leg: y_p = R_obs r_k (pred. foot_k - p), y_v = -(w_obs x R_obs r_k + R_obs J_k thetadot_obs)
              (pred. v), y_z = 0 (pred. foot_k,z); std r_pos s_k, r_vel s_k, r_height s_k; +inf drops the row
              S = H P H' + R, K = P H' S^-1, x += K (y - H x), P = (I - K H) P, then P = (P + P') / 2
    s_k       1 for a foot planned in stance, swing_scale for one planned in swing
    output    q_obs[4:7] = p, v_obs[3:6] = v; v_prev = v[3:6]; count += 1; stats += |p - p_true|^2, max, |v - v_true|^2, max
    failure   a pivot of S (the innovation variance of a scalar update) not > 0, or x / P not finite: output unchanged,
              WBC_ST_BADESTIM, count = 0, x / P / v_prev / stats unchanged
    bad index WBC_ST_BADESTIM, nothing changes

The pivots of the LDL' factorisation of S in row order are the innovation variances of the sequential scalar updates the kernel
makes, so both fail on the same steps in exact arithmetic.

DEFAULTS are in the spirit of the linear Kalman filter of the open-source MIT Cheetah software (a small process noise on the base,
a trusted leg-kinematics position, a loose leg velocity, a tight flat-ground height, swing feet scaled far out); they are not
measured on any robot."""
from __future__ import annotations

import numpy as np

from . import sensing

ST_BADESTIM = 16384
FIELDS = ("q_pos", "q_vel", "q_foot", "r_pos", "r_vel", "r_height", "swing_scale", "p0_pos", "p0_vel", "p0_foot")
DEFAULTS = dict(q_pos=0.02, q_vel=0.1, q_foot=0.02, r_pos=0.002, r_vel=0.05, r_height=0.005, swing_scale=100.0, p0_pos=0.01,
                p0_vel=0.1, p0_foot=0.01)
ACCEL_DRAWS = (18, 19)


def desc(**kw):
    """A record {field: value}: DEFAULTS with the given fields replaced."""
    d = dict(DEFAULTS)
    for k, x in kw.items():
        if k not in d:
            raise KeyError(k)
        d[k] = float(x)
    return d


def desc_problem(d):
    """Why a record cannot be used, or None (the checks of wbc_estimator_set_create)."""
    vals = [float(d[k]) for k in FIELDS]
    if any(np.isnan(x) or x < 0 for x in vals):
        return "NaN or negative"
    if not all(np.isfinite(d[k]) for k in ("q_pos", "q_vel", "q_foot", "p0_pos", "p0_vel", "p0_foot")):
        return "non-finite process or initial std"
    if not (np.isfinite(d["swing_scale"]) and d["swing_scale"] >= 1.0):
        return "swing_scale"
    return None


def quat_matrix(q4):
    """R of a [w x y z] quaternion, normalised first."""
    n = np.sqrt(q4 @ q4)
    w, x, y, z = q4 / n
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _rot(axis, th):
    a = np.asarray(axis, float)
    K = np.array([[0.0, -a[2], a[1]], [a[2], 0.0, -a[0]], [-a[1], a[0], 0.0]])
    return np.cos(th) * np.eye(3) + np.sin(th) * K + (1.0 - np.cos(th)) * np.outer(a, a)


def leg_kinematics(model, q, v, leg):
    """Foot `leg` relative to the base origin in base axes, r_k, and its velocity from the joint rates, J_k thetadot (base axes):
    the chain of joint_xyz / joint_axis / foot_xyz with joint k's angle q[v_index[k] + 1] and rate v[v_index[k]]."""
    R, rho = np.eye(3), np.zeros(3)
    axes, origins, rates = [], [], []
    for j in range(3):
        k = 3 * leg + j
        rho = rho + R @ np.asarray(model.joint_xyz[k], float)
        axes.append(R @ np.asarray(model.joint_axis[k], float))
        origins.append(rho.copy())
        rates.append(v[model.v_index[k]])
        R = R @ _rot(model.joint_axis[k], q[model.v_index[k] + 1])
    r = rho + R @ np.asarray(model.foot_xyz[leg], float)
    jv = sum(np.cross(a, r - o) * w for a, o, w in zip(axes, origins, rates))
    return r, jv


def draws(seed, stream, c, js):
    """The normal pairs of Philox draws js of the loop counter (j, stream, c_lo, c_hi) under the loop key -> [len(js), 2]."""
    s = int(seed) & 0xFFFFFFFFFFFFFFFF
    cu = int(c) & 0xFFFFFFFFFFFFFFFF
    ctr = np.array([[j, int(stream) & 0xFFFFFFFF, cu & 0xFFFFFFFF, cu >> 32] for j in js], np.uint64)
    key = np.broadcast_to(np.array([s & 0xFFFFFFFF, s >> 32], np.uint64), (len(js), 2))
    ua, ub = sensing.uniforms(sensing.philox4x32_10(ctr, key))
    r = np.sqrt(-2.0 * np.log(ua))
    return np.stack([r * np.cos(np.pi * (2.0 * ub)), r * np.sin(np.pi * (2.0 * ub))], axis=-1)


def accel_normals(seed, stream, c):
    """The three normals of the accelerometer noise at step c: draw 18 (z0, z1) and the first of draw 19."""
    return draws(seed, stream, c, ACCEL_DRAWS).reshape(-1)[:3]


class State:
    """The filter state of one robot: x [18], P [18, 18], v_prev [3], count, stats [4]."""

    def __init__(self, x=None, P=None, v_prev=None, count=0, stats=None):
        self.x = np.zeros(18) if x is None else np.array(x, float)
        self.P = np.zeros((18, 18)) if P is None else np.array(P, float)
        self.v_prev = np.zeros(3) if v_prev is None else np.array(v_prev, float)
        self.count = int(count)
        self.stats = np.zeros(4) if stats is None else np.array(stats, float)

    def copy(self):
        return State(self.x, self.P, self.v_prev, self.count, self.stats)


def measurements(d, model, q_obs, v_obs, contact):
    """(H [28, 18], y [28], std [28]) of the update, leg by leg: 3 position rows, 3 velocity rows, 1 height row."""
    R = quat_matrix(np.asarray(q_obs[0:4], float))
    w = np.asarray(v_obs[0:3], float)
    H, y, sd = np.zeros((28, 18)), np.zeros(28), np.zeros(28)
    for k in range(4):
        s = 1.0 if contact[k] else d["swing_scale"]
        r, jv = leg_kinematics(model, q_obs, v_obs, k)
        rw = R @ r
        yv = -(np.cross(w, rw) + R @ jv)
        m = 7 * k
        for a in range(3):
            H[m + a, 6 + 3 * k + a], H[m + a, a] = 1.0, -1.0
            y[m + a], sd[m + a] = rw[a], d["r_pos"] * s
            H[m + 3 + a, 3 + a] = 1.0
            y[m + 3 + a], sd[m + 3 + a] = yv[a], d["r_vel"] * s
        H[m + 6, 6 + 3 * k + 2] = 1.0
        y[m + 6], sd[m + 6] = 0.0, d["r_height"] * s
    return H, y, sd


def _pivots(S):
    """The pivots of the LDL' factorisation of S in row order (no pivoting)."""
    S = np.array(S, float)
    out = []
    for m in range(len(S)):
        p = S[m, m]
        out.append(p)
        if not p > 0.0:
            break
        S[m + 1:, m + 1:] -= np.outer(S[m + 1:, m], S[m, m + 1:]) / p
    return np.array(out)


def step(d, model, dt, q, v, q_obs, v_obs, contact, st, seed=0, stream=0, c=0, sigma_acc=0.0):
    """One estimator step of one robot with record d (None: bad index). Returns (q_obs', v_obs', state', status); `st` is not
    modified."""
    q, v = np.asarray(q, float), np.asarray(v, float)
    qo, vo = np.array(q_obs, float), np.array(v_obs, float)
    st = st.copy()
    if d is None:
        return qo, vo, st, ST_BADESTIM
    g = np.asarray(model.gravity, float)
    Ro = quat_matrix(qo[0:4])
    if st.count <= 0:
        x = np.zeros(18)
        x[0:3], x[3:6] = qo[4:7], vo[3:6]
        for k in range(4):
            x[6 + 3 * k:9 + 3 * k] = x[0:3] + Ro @ leg_kinematics(model, qo, vo, k)[0]
        st.x = x
        st.P = np.diag([d["p0_pos"] ** 2] * 3 + [d["p0_vel"] ** 2] * 3 + [d["p0_foot"] ** 2] * 12)
        st.v_prev, st.count = v[3:6].copy(), 1
        _stats(st, q, v)
        return qo, vo, st, 0
    a_w = (v[3:6] - st.v_prev) / dt
    f_b = quat_matrix(q[0:4]).T @ (a_w - g)
    if sigma_acc != 0.0:
        f_b = f_b + sigma_acc * accel_normals(seed, stream, c)
    acc = Ro @ f_b + g
    x = st.x.copy()
    x[3:6] = x[3:6] + dt * acc
    x[0:3] = x[0:3] + dt * x[3:6]
    A = np.eye(18)
    A[0:3, 3:6] = dt * np.eye(3)
    sk = [1.0 if contact[k] else d["swing_scale"] for k in range(4)]
    Q = dt * np.diag([d["q_pos"] ** 2] * 3 + [d["q_vel"] ** 2] * 3 + sum(([(d["q_foot"] * s) ** 2] * 3 for s in sk), []))
    P = A @ st.P @ A.T + Q
    H, y, sd = measurements(d, model, qo, vo, contact)
    keep = np.isfinite(sd)
    H, y, Rm = H[keep], y[keep], np.diag(sd[keep] ** 2)
    ok = True
    if len(y):
        S = H @ P @ H.T + Rm
        ok = bool((_pivots(S) > 0.0).all())
        if ok:
            K = np.linalg.solve(S, H @ P).T
            x = x + K @ (y - H @ x)
            P = (np.eye(18) - K @ H) @ P
    if ok:
        P = 0.5 * (P + P.T)
        ok = bool(np.isfinite(x).all() and np.isfinite(P).all())
    if not ok:
        st.count = 0
        return qo, vo, st, ST_BADESTIM
    st.x, st.P, st.v_prev, st.count = x, P, v[3:6].copy(), st.count + 1
    qo[4:7], vo[3:6] = x[0:3], x[3:6]
    _stats(st, q, v)
    return qo, vo, st, 0


def _stats(st, q, v):
    ep, ev = np.linalg.norm(st.x[0:3] - q[4:7]), np.linalg.norm(st.x[3:6] - v[3:6])
    st.stats[0] += ep * ep
    st.stats[1] = max(st.stats[1], ep)
    st.stats[2] += ev * ev
    st.stats[3] = max(st.stats[3], ev)
