// wbc_monitor.cuh — the rollout monitor of the ground-plant loop (include/wbc.h, wbc_monitor): after each plant step it
// compares robot i's true state with the plan sample its controller tracked, decides whether the robot has failed, and folds
// tracking, effort and contact statistics into caller-owned per-robot accumulators. The semantics are stated once in
// include/wbc.h and restated in numpy by oracle/monitor.py.
//
// One kernel, one thread per robot, in the style of wbcloop::observe_kernel. The device functions also compile on the host
// (tests/emu/emu_monitor.cpp), which defines WBC_DEV.
#pragma once
#include <stdint.h>
#include <math.h>
#include "wbc.h"

#ifndef WBC_DEV
#define WBC_DEV __device__ __forceinline__
#endif

namespace wbcmon {

// Device view of a wbc_monitor, with the step length and the handle's joint maps and effort limits (by value).
struct MonArgs {
  double pos_max, ang_max, dt;
  double* stats; long long* steps; long long* fail_step; int32_t* fail_why; int32_t* why;
  int v_index[WBC_NU], act_index[WBC_NU];
  double effort[WBC_NU];
};

WBC_DEV double max_rule(double e, double m) { return e > m ? e : m; }

// Rotation angle in [0, pi] between the unit quaternion of q[0:4] and the quaternion of RollPitchYaw rpy (Drake:
// qz(yaw) (x) qy(pitch) (x) qx(roll)): 2 atan2(|u|, |w|) of (w, u) = conj(q_ref) (x) q_hat.
WBC_DEV double orientation_error(const double* q, const double* rpy) {
  double sr, cr, sp, cp, sy, cy;
  sincos(0.5 * rpy[0], &sr, &cr);
  sincos(0.5 * rpy[1], &sp, &cp);
  sincos(0.5 * rpy[2], &sy, &cy);
  const double rw = cy * cp * cr + sy * sp * sr, rx = cy * cp * sr - sy * sp * cr;
  const double ry = cy * sp * cr + sy * cp * sr, rz = sy * cp * cr - cy * sp * sr;
  const double inv = 1.0 / sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  const double bw = q[0] * inv, bx = q[1] * inv, by = q[2] * inv, bz = q[3] * inv;
  // conj(r) (x) b = (rw bw + r.b, rw b - bw r - r x b)
  const double w = rw * bw + rx * bx + ry * by + rz * bz;
  const double ux = rw * bx - bw * rx - (ry * bz - rz * by);
  const double uy = rw * by - bw * ry - (rz * bx - rx * bz);
  const double uz = rw * bz - bw * rz - (rx * by - ry * bx);
  return 2.0 * atan2(sqrt(ux * ux + uy * uy + uz * uz), fabs(w));
}

// One monitored step of robot i: q [19], v [18] after the plant step; traj [54], contact [4] the plan sample its controller
// tracked; tau [12] the applied torque (actuator order); f [12] the plant's ground forces (world axes); s the step's status word.
WBC_DEV void monitor_instance(const MonArgs& a, long long i, const double* __restrict__ q, const double* __restrict__ v,
                              const double* __restrict__ traj, const uint8_t* __restrict__ contact, const double* __restrict__ tau,
                              const double* __restrict__ f, int s) {
  const double* qi = q + i * WBC_NQ;
  const double* vi = v + i * WBC_NV;
  const double* tr = traj + i * WBC_NTRAJ;
  const double* ti = tau + i * WBC_NU;
  const double* fi = f + i * 12;
  const double dx = qi[4] - tr[0], dy = qi[5] - tr[1], dz = qi[6] - tr[2];
  const double ep = sqrt(dx * dx + dy * dy + dz * dz);
  const double eth = orientation_error(qi, tr + 9);
  int why = 0;
  if (!(ep <= a.pos_max)) why |= WBC_MON_POS;
  if (!(eth <= a.ang_max)) why |= WBC_MON_ANG;
  if (s != 0) why |= WBC_MON_STATUS;
  const long long k = a.steps[i] + 1;
  a.steps[i] = k;
  if (why != 0 && a.fail_step[i] == 0) { a.fail_step[i] = k; a.fail_why[i] = why; }
  if (a.why) a.why[i] = why;
  double tau2 = 0.0, work = 0.0, sat = 0.0;
#pragma unroll
  for (int c = 0; c < WBC_NU; ++c) tau2 += ti[c] * ti[c];
#pragma unroll
  for (int j = 0; j < WBC_NU; ++j) {              // joint j: its actuator's torque, its velocity, its effort limit
    const double t = ti[a.act_index[j]];
    work += fabs(t * vi[a.v_index[j]]);
    sat = max_rule(fabs(t) / a.effort[j], sat);
  }
  double fmax = 0.0, unloaded = 0.0, loaded = 0.0;
#pragma unroll
  for (int ft = 0; ft < 4; ++ft) {
    const double fx = fi[3 * ft], fy = fi[3 * ft + 1], fz = fi[3 * ft + 2];
    fmax = max_rule(sqrt(fx * fx + fy * fy + fz * fz), fmax);
    const bool zero = fx == 0.0 && fy == 0.0 && fz == 0.0;
    if (contact[i * 4 + ft] != 0 && zero) unloaded += 1.0;
    if (contact[i * 4 + ft] == 0 && !zero) loaded += 1.0;
  }
  double* st = a.stats + i * WBC_MON_NSTAT;
  st[WBC_MON_SUM_POS2] += ep * ep;
  st[WBC_MON_MAX_POS] = max_rule(ep, st[WBC_MON_MAX_POS]);
  st[WBC_MON_SUM_ANG2] += eth * eth;
  st[WBC_MON_MAX_ANG] = max_rule(eth, st[WBC_MON_MAX_ANG]);
  st[WBC_MON_TAU2_DT] += a.dt * tau2;
  st[WBC_MON_WORK_ABS] += a.dt * work;
  st[WBC_MON_SAT_MAX] = max_rule(sat, st[WBC_MON_SAT_MAX]);
  st[WBC_MON_F_MAX] = max_rule(fmax, st[WBC_MON_F_MAX]);
  st[WBC_MON_STANCE_UNLOADED] += unloaded;
  st[WBC_MON_SWING_LOADED] += loaded;
  st[WBC_MON_DIST_XY] += a.dt * sqrt(vi[3] * vi[3] + vi[4] * vi[4]);
}

#ifdef __CUDACC__
// status: the step's status words (NULL: 0). word (the rollout's per-step word; status is then unused): read, ORed into
// status_or when given, and zeroed for the next step.
__global__ void __launch_bounds__(256) monitor_kernel(const MonArgs a, long long n, const double* __restrict__ q,
                                                      const double* __restrict__ v, const double* __restrict__ traj,
                                                      const uint8_t* __restrict__ contact, const double* __restrict__ tau,
                                                      const double* __restrict__ f, const int32_t* __restrict__ status,
                                                      int32_t* __restrict__ word, int32_t* __restrict__ status_or) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int s = word ? word[i] : status ? status[i] : 0;
  monitor_instance(a, i, q, v, traj, contact, tau, f, s);
  if (word) {
    if (status_or) status_or[i] |= s;
    word[i] = 0;
  }
}
#endif

}  // namespace wbcmon
