"""ORACLE (test infrastructure only): numpy restatement of the actuator model of the ground-plant loop (include/wbc.h,
wbc_motor_desc / wbc_plant_motor; csrc/wbc_motor.cuh), written from its definition. Per robot i with record r = set[index[i]],
joint k (the model's joint order), actuator a = act_index[k]:

    w = v[i][v_index[k]] (the true velocity at the start of the step), u = the torque reaching actuator a
    lag:      s = u if count[i] == 0 or lag_k == 0, else m + alpha (u - m), m = tau_m[i][a], alpha = -expm1(-dt / lag_k)
    envelope: L = peak_k, except where s and w are non-zero and of one sign and |w| > speed_knee_k: there L = 0 if
              |w| >= speed_free_k, else peak_k (speed_free_k - |w|) / (speed_free_k - speed_knee_k) (peak_k if speed_free_k = inf)
    out = s if |s| <= L else copysign(L, s) (NaN stays NaN); tau_m[i][a] = out
    friction: f = -damping_k w - coulomb_k clamp(w / coulomb_speed_k, -1, 1), a zero coefficient left out; plant = out + f
              (out itself with both coefficients zero); count[i] += 1
    bad index (outside [0, K)): plant torque 0, status WBC_ST_BADMOTOR, tau_m and count unchanged
    NULL set: one record, peak = the model's effort, speed_knee = speed_free = inf, lag = damping = coulomb = 0

The products and sums are evaluated in the order written, one rounding each, as the kernel does."""
from __future__ import annotations

import numpy as np

ST_BADMOTOR = 8192
FIELDS = ("peak", "speed_knee", "speed_free", "lag", "damping", "coulomb", "coulomb_speed")


def record(effort, peak_scale=1.0, speed_knee=np.inf, speed_free=np.inf, lag=0.0, damping=0.0, coulomb=0.0, coulomb_speed=0.0):
    """A record {field: [12]}: peak = peak_scale x effort, the other fields broadcast to the 12 joints."""
    vals = dict(peak=peak_scale * np.asarray(effort, float), speed_knee=speed_knee, speed_free=speed_free, lag=lag, damping=damping,
                coulomb=coulomb, coulomb_speed=coulomb_speed)
    return {k: np.array(np.broadcast_to(np.asarray(x, float), (12,))) for k, x in vals.items()}


def lag(u, m, first, lag_k, dt):
    """The filtered command s: u where `first` (count == 0) or lag_k == 0, else m + alpha (u - m)."""
    on = ~first & (lag_k != 0.0)
    with np.errstate(all="ignore"):
        alpha = -np.expm1(-dt / np.where(on, lag_k, 1.0))
        return np.where(on, m + alpha * (u - m), u)


def envelope(s, w, peak, knee, free):
    """The torque limit L of the torque-speed envelope."""
    aw = np.abs(w)
    motoring = ((s > 0.0) & (w > 0.0)) | ((s < 0.0) & (w < 0.0))
    with np.errstate(all="ignore"):
        fall = np.where(free == np.inf, peak, peak * (free - aw) / (free - knee))
    return np.where(motoring & (aw > knee), np.where(aw >= free, 0.0, fall), peak)


def clamp(s, lim):
    """s clamped to [-L, L]; a NaN s stays NaN."""
    return np.where(np.abs(s) > lim, np.copysign(lim, s), s)


def plant_input(out, w, damping, coulomb, cspeed):
    """out + friction; a zero coefficient adds nothing."""
    with np.errstate(all="ignore"):
        x = w / np.where(coulomb != 0.0, cspeed, 1.0)
        x = np.where(x > 1.0, 1.0, np.where(x < -1.0, -1.0, x))
        fd = -(damping * w)
        fc = coulomb * x
        f = np.where(damping != 0.0, np.where(coulomb != 0.0, fd - fc, fd), -fc)
        return np.where((damping != 0.0) | (coulomb != 0.0), out + f, out)


def apply(records, index, tau_m, count, dt, v_index, act_index, v, u):
    """One motor step of N robots. records: list of K records (the NULL set is [record(effort)]); index [N] or None; tau_m [N,12]
    (actuator order) and count [N] are advanced in place; v [N,18]; u [N,12] (actuator order) -> (tau_plant [N,12] actuator
    order, status [N] int32)."""
    n = len(v)
    K = len(records)
    idx = np.zeros(n, np.int64) if index is None else np.asarray(index, np.int64)
    ok = (idx >= 0) & (idx < K)
    r = np.where(ok, idx, 0)
    rec = {f: np.stack([records[j][f] for j in range(K)])[r] for f in FIELDS}      # [N, 12], joint order
    ai, vi = np.asarray(act_index), np.asarray(v_index)
    w = v[:, vi]
    uk, mk = u[:, ai], tau_m[:, ai]
    s = lag(uk, mk, (count == 0)[:, None], rec["lag"], dt)
    out = clamp(s, envelope(s, w, rec["peak"], rec["speed_knee"], rec["speed_free"]))
    tp = plant_input(out, w, rec["damping"], rec["coulomb"], rec["coulomb_speed"])
    plant = np.zeros_like(u)
    plant[:, ai] = np.where(ok[:, None], tp, 0.0)
    new_m = tau_m.copy()
    new_m[:, ai] = out
    tau_m[ok] = new_m[ok]
    count[ok] += 1
    return plant, np.where(ok, 0, ST_BADMOTOR).astype(np.int32)
