"""ORACLE (test infrastructure only): numpy restatement of the contact detector of the ground-plant loop (include/wbc.h,
wbc_contact_desc / wbc_contact; csrc/wbc_contact.cuh), written from its definition on oracle.dynamics.Plant. Robot i with record r:

    state     q_prev [19], v_prev [18] (what it read at its previous step), tau_prev [12] (measured torque, actuator order),
              f_true [4, 3] (the plant's forces of its latest step), f_hat [4, 3], flag [4], count, stats [6]
    prime     (count <= 0) flag = plan, f_hat = 0, q_prev = q, v_prev = v, count = 1
    residual  M, Cv, tau_g, S = calc_dynamics(q_prev, v_prev);  r = M (v - v_prev) - dt (S' tau_prev - Cv - tau_g)
    per leg   J_leg = foot k's translational Jacobian (frame_position_quantities at q_prev) over leg k's joint columns;
              singular when |det J_leg| <= 1e-9 |a0| |a1| |a2| (a_j its columns): f_hat, flag held, no statistics;
              else J_leg' p = r[leg columns], f_raw = p / dt (world axes)
    filter    f_hat = f_raw on the first estimate after a prime or with tau_f = 0, else f_hat += alpha (f_raw - f_hat),
              alpha = -expm1(-dt / tau_f)
    flags     0 -> 1 when f_hat_z >= f_on, 1 -> 0 when f_hat_z <= f_off
    stats     += sum_k |f_raw - f_true|^2, max= |f_raw - f_true|, += true stance, true swing, false stance, false swing (a foot is
              loaded when any component of f_true is non-zero)
    then      q_prev = q, v_prev = v, count += 1
    failure   a non-finite f_raw of a non-singular leg: count = 0, everything else unchanged, ST_BADCONTACT, output = plan
    bad index ST_BADCONTACT, nothing changes, output = plan

The plant's step (oracle/rollout.py:plant_step) is v+ = v + dt M^-1 (S' tau - Cv - tau_g) + M^-1 J_c' p, so with the true state and
the torque the plant received the joint rows of leg k read r_k = J_leg' p_k: f_raw is the plant's f_contact up to rounding.

DEFAULTS are untuned: a 10 ms force filter, and thresholds of about a quarter and a tenth of a mini_cheetah foot's standing load
(about 22 N)."""
from __future__ import annotations

import numpy as np

ST_BADCONTACT = 32768
FEED_ESTIMATOR, FEED_CONTROLLER = 1, 2
FIELDS = ("tau_f", "f_on", "f_off")
DEFAULTS = dict(tau_f=0.01, f_on=6.0, f_off=2.0)
SINGULAR_SINVOL = 1e-9


def desc(**kw):
    """A record {field: value}: DEFAULTS with the given fields replaced."""
    d = dict(DEFAULTS)
    for k, x in kw.items():
        if k not in d:
            raise KeyError(k)
        d[k] = float(x)
    return d


def desc_problem(d):
    """Why a record cannot be used, or None (the checks of wbc_contact_set_create)."""
    if not (np.isfinite(d["tau_f"]) and d["tau_f"] >= 0.0):
        return "tau_f"
    if np.isnan(d["f_on"]) or np.isnan(d["f_off"]):
        return "NaN threshold"
    if not d["f_off"] <= d["f_on"]:
        return "f_off > f_on"
    return None


def leg_columns(plant, k):
    """The v indices of the joints that move foot k, from the hip down."""
    i = plant.index[plant.foot_frames[k]]
    cols = []
    while i > 0:
        if plant.vidx[i] is not None:
            cols.append(plant.vidx[i])
        i = plant.parent[i]
    return cols[::-1]


def raw_forces(plant, q_prev, v_prev, v, tau_prev, dt):
    """(f_raw [4, 3], singular [4]) of the momentum residual between (q_prev, v_prev) and v under the torque tau_prev."""
    q_prev, v_prev, v = (np.asarray(x, float) for x in (q_prev, v_prev, v))
    M, Cv, tau_g, S = plant.calc_dynamics(q_prev, v_prev)
    r = M @ (v - v_prev) - dt * (S.T @ np.asarray(tau_prev, float) - Cv - tau_g)
    f, singular = np.zeros((4, 3)), np.zeros(4, bool)
    for k, frame in enumerate(plant.foot_frames):
        cols = leg_columns(plant, k)
        Jl = plant.frame_position_quantities(q_prev, v_prev, frame)[1][:, cols]
        singular[k] = abs(np.linalg.det(Jl)) <= SINGULAR_SINVOL * np.prod(np.linalg.norm(Jl, axis=0))
        if not singular[k]:
            f[k] = np.linalg.solve(Jl.T, r[cols]) / dt
    return f, singular


class State:
    """The detector state of one robot."""

    def __init__(self, q_prev=None, v_prev=None, tau_prev=None, f_true=None, f_hat=None, flag=None, count=0, stats=None):
        self.q_prev = np.zeros(19) if q_prev is None else np.array(q_prev, float)
        self.v_prev = np.zeros(18) if v_prev is None else np.array(v_prev, float)
        self.tau_prev = np.zeros(12) if tau_prev is None else np.array(tau_prev, float)
        self.f_true = np.zeros((4, 3)) if f_true is None else np.array(f_true, float).reshape(4, 3)
        self.f_hat = np.zeros((4, 3)) if f_hat is None else np.array(f_hat, float).reshape(4, 3)
        self.flag = np.zeros(4, np.uint8) if flag is None else np.array(flag, np.uint8)
        self.count = int(count)
        self.stats = np.zeros(6) if stats is None else np.array(stats, float)

    def copy(self):
        return State(self.q_prev, self.v_prev, self.tau_prev, self.f_true, self.f_hat, self.flag, self.count, self.stats)


def step(d, plant, dt, q, v, plan, st):
    """One detector step of one robot with record d (None: bad index). Returns (detected [4] uint8, state', status); `st` is not
    modified."""
    plan = (np.asarray(plan) != 0).astype(np.uint8)
    st = st.copy()
    if d is None:
        return plan, st, ST_BADCONTACT
    if st.count <= 0:
        st.flag, st.f_hat, st.q_prev, st.v_prev, st.count = plan.copy(), np.zeros((4, 3)), np.array(q, float), np.array(v, float), 1
        return plan, st, 0
    f_raw, singular = raw_forces(plant, st.q_prev, st.v_prev, v, st.tau_prev, dt)
    if (~singular & ~np.isfinite(f_raw).all(axis=1)).any():
        st.count = 0
        return plan, st, ST_BADCONTACT
    raw = st.count == 1 or d["tau_f"] == 0.0
    alpha = 1.0 if raw else -np.expm1(-dt / d["tau_f"])
    for k in range(4):
        if singular[k]:
            continue
        st.f_hat[k] = f_raw[k] if raw else st.f_hat[k] + alpha * (f_raw[k] - st.f_hat[k])
        if st.flag[k]:
            st.flag[k] = 0 if st.f_hat[k, 2] <= d["f_off"] else 1
        else:
            st.flag[k] = 1 if st.f_hat[k, 2] >= d["f_on"] else 0
        e = f_raw[k] - st.f_true[k]
        st.stats[0] += e @ e
        st.stats[1] = max(st.stats[1], np.sqrt(e @ e))
        loaded, f = bool((st.f_true[k] != 0.0).any()), bool(st.flag[k])
        st.stats[2 + (0 if f and loaded else 1 if not f and not loaded else 2 if f else 3)] += 1
    st.q_prev, st.v_prev, st.count = np.array(q, float), np.array(v, float), st.count + 1
    return st.flag.copy(), st, 0


def record(st, tau_meas, f_contact):
    """The record step after the plant: the measured torque and the plant's forces into the state (a copy is returned)."""
    st = st.copy()
    st.tau_prev, st.f_true = np.array(tau_meas, float), np.array(f_contact, float).reshape(4, 3)
    return st
