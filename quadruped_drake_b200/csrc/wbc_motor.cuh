// wbc_motor.cuh — the actuator model of the ground-plant loop (include/wbc.h, wbc_motor_desc / wbc_plant_motor): between the
// actuated torque and the plant, each joint's motor follows its command through a first-order lag, saturates on a
// torque-speed envelope, and the joint adds viscous and Coulomb friction. The semantics are stated once in include/wbc.h and
// restated in numpy by oracle/motor.py.
//
// One kernel. Joints are independent, so each robot gets a 16-lane group of one warp: lanes 0-11 each do one joint, and two
// robots share a warp. The per-robot words (count, the status word) are read and written by the group's lane 0 only. The device
// functions also compile on the host (tests/emu/emu_motor.cpp), which defines WBC_DEV.
#pragma once
#include <stdint.h>
#include <math.h>
#include "wbc.h"

#ifndef WBC_DEV
#define WBC_DEV __device__ __forceinline__
#endif

namespace wbcmotor {

// Device view of a wbc_plant_motor: the record table (NULL: one record of the handle's effort limits, every other field off),
// the per-robot state, the step length, and the handle's joint maps and effort limits (by value).
struct MotorArgs {
  const wbc_motor_desc* set; const int32_t* index; int n_sets;
  double* tau_m; long long* count;
  double dt;
  int v_index[WBC_NU], act_index[WBC_NU];
  double effort[WBC_NU];
};

// Products and sums written as separate roundings: the kernel must not contract them into FMAs, so that it rounds as the host
// restatement does.
#ifdef __CUDACC__
WBC_DEV double mul_rn(double a, double b) { return __dmul_rn(a, b); }
WBC_DEV double add_rn(double a, double b) { return __dadd_rn(a, b); }
#else
WBC_DEV double mul_rn(double a, double b) { return a * b; }
WBC_DEV double add_rn(double a, double b) { return a + b; }
#endif

// Why a record cannot be used, or nullptr (host code: wbc_motor_set_create checks every record with it).
inline const char* desc_problem(const wbc_motor_desc& d) {
  const auto nonneg_finite = [](double x) { return x >= 0.0 && x <= 1.7976931348623157e308; };
  for (int k = 0; k < WBC_NU; ++k) {
    if (!(d.peak[k] >= 0.0)) return "wbc_motor_set_create: peak must be >= 0 (+inf: no limit)";
    if (!(d.speed_knee[k] >= 0.0) || !(d.speed_free[k] >= 0.0))
      return "wbc_motor_set_create: speed_knee and speed_free must be >= 0 (+inf: off)";
    if (!(d.speed_knee[k] <= d.speed_free[k])) return "wbc_motor_set_create: speed_knee must be <= speed_free";
    if (!nonneg_finite(d.lag[k]) || !nonneg_finite(d.damping[k]) || !nonneg_finite(d.coulomb[k]) || !nonneg_finite(d.coulomb_speed[k]))
      return "wbc_motor_set_create: lag, damping, coulomb and coulomb_speed must be finite and >= 0";
    if (d.coulomb[k] > 0.0 && !(d.coulomb_speed[k] > 0.0)) return "wbc_motor_set_create: coulomb > 0 needs coulomb_speed > 0";
  }
  return nullptr;
}

// Robot i's record, or -1 for an index outside [0, n_sets).
WBC_DEV int motor_record(const MotorArgs& a, long long i) {
  const int r = a.index ? a.index[i] : 0;
  return r >= 0 && r < a.n_sets ? r : -1;
}

// Joint k of robot i with record r (-1: bad index) at filter count c: reads u = tau_in[i][a] and w, writes tau_m[i][a] and the
// plant input tau_plant[i][a] (a = act_index[k]).
WBC_DEV void motor_joint(const MotorArgs& a, long long i, int k, int r, long long c, const double* __restrict__ v,
                         const double* __restrict__ tau_in, double* __restrict__ tau_plant) {
  const int ai = a.act_index[k];
  const long long o = i * WBC_NU + ai;
  if (r < 0) {
    tau_plant[o] = 0.0;
    return;
  }
  const double inf = INFINITY;
  const wbc_motor_desc* d = a.set ? a.set + r : nullptr;
  const double peak = d ? d->peak[k] : a.effort[k];
  const double knee = d ? d->speed_knee[k] : inf, sfree = d ? d->speed_free[k] : inf;
  const double lag = d ? d->lag[k] : 0.0, damping = d ? d->damping[k] : 0.0;
  const double coulomb = d ? d->coulomb[k] : 0.0, cspeed = d ? d->coulomb_speed[k] : 0.0;
  const double w = v[i * WBC_NV + a.v_index[k]];
  const double u = tau_in[o];
  double s = u;
  if (c != 0 && lag != 0.0) {
    const double m = a.tau_m[o];
    const double alpha = -expm1(-a.dt / lag);
    s = add_rn(m, mul_rn(alpha, u - m));
  }
  double lim = peak;
  const double aw = fabs(w);
  if (((s > 0.0 && w > 0.0) || (s < 0.0 && w < 0.0)) && aw > knee)
    lim = aw >= sfree ? 0.0 : sfree == inf ? peak : mul_rn(peak, sfree - aw) / (sfree - knee);
  const double out = fabs(s) > lim ? copysign(lim, s) : s;     // a NaN s fails the test and stays
  a.tau_m[o] = out;
  double tp = out;
  if (damping != 0.0 || coulomb != 0.0) {
    double f = damping != 0.0 ? -mul_rn(damping, w) : 0.0;
    if (coulomb != 0.0) {
      double x = w / cspeed;
      x = x > 1.0 ? 1.0 : x < -1.0 ? -1.0 : x;
      f = damping != 0.0 ? add_rn(f, -mul_rn(coulomb, x)) : -mul_rn(coulomb, x);
    }
    tp = add_rn(out, f);
  }
  tau_plant[o] = tp;
}

// Robot i's per-robot words after its joints: count advances, or a bad index sets WBC_ST_BADMOTOR in status (when given).
WBC_DEV void motor_finish(const MotorArgs& a, long long i, int r, long long c, int32_t* __restrict__ status) {
  if (r < 0) {
    if (status) status[i] |= WBC_ST_BADMOTOR;
  } else {
    a.count[i] = c + 1;
  }
}

#ifdef __CUDACC__
constexpr int MOTOR_BLOCK = 256;        // 16 robots per CTA

__global__ void __launch_bounds__(MOTOR_BLOCK) motor_kernel(const MotorArgs a, long long n, const double* __restrict__ v,
                                                            const double* __restrict__ tau_in, double* __restrict__ tau_plant,
                                                            int32_t* __restrict__ status) {
  const long long i = ((long long)blockIdx.x * MOTOR_BLOCK + threadIdx.x) >> 4;
  const int k = threadIdx.x & 15;
  int r = -1;
  long long c = 0;
  if (k == 0 && i < n) {
    r = motor_record(a, i);
    if (r >= 0) c = a.count[i];
  }
  r = __shfl_sync(0xffffffffu, r, 0, 16);        // every grid warp is whole: all 32 lanes take part
  c = __shfl_sync(0xffffffffu, c, 0, 16);
  if (i >= n) return;
  if (k < WBC_NU) motor_joint(a, i, k, r, c, v, tau_in, tau_plant);
  if (k == 0) motor_finish(a, i, r, c, status);
}
#endif

}  // namespace wbcmotor
