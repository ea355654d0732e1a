// wbc_estimator.cuh — state estimation in the ground-plant loop (include/wbc.h, wbc_estimator_desc / wbc_estimator): a per-robot
// linear Kalman filter over base position, base velocity and the four foot positions fuses a synthesised accelerometer with leg
// kinematics, and the controller reads its estimate of the base position and linear velocity. The semantics are stated once in
// include/wbc.h and restated in numpy by oracle/estimator.py.
//
// One kernel, one warp per robot. Lanes 0-3 each evaluate one leg's kinematics and its seven measurement rows; lane 0 the
// accelerometer and the state prediction. Lane r < 18 holds row r of the covariance in registers: the prediction is a row pass
// (a shuffle) and a column pass, and each of the 28 rows is a scalar update (P h from the lane's own row, published through
// shared memory, the gain, a rank-one downdate of the row), so that no 28 x 28 system is factored. Rows stay out of shared
// memory because the downdates would otherwise make the kernel bound by shared-memory bandwidth; the symmetrisation at the end
// goes through it once. The device functions also compile on the host
// (tests/emu/emu_estimator.cpp), which defines WBC_DEV, the warp collectives and sincospi.
#pragma once
#include <stdint.h>
#include <math.h>
#include "wbc.h"
#include "wbc_loop.cuh"

#ifndef WBC_DEV
#define WBC_DEV __device__ __forceinline__
#endif

namespace wbcest {

constexpr int NX = 18;             // p (3), v (3), feet (4 x 3)
constexpr int NY = 28;             // 7 rows per leg: foot position (3), foot velocity (3), foot height (1)
constexpr int ACCEL_DRAW = 18;     // Philox draws 18 and 19 of the loop counter: after the loop's 18

// Device view of a wbc_estimator with its loop and the handle's kinematic model (by value).
struct EstArgs {
  const wbc_estimator_desc* set; const int32_t* index; int n_sets;
  const double* accel_noise;
  double* x; double* P; double* v_prev; long long* count; double* stats;
  double dt;
  unsigned long long seed; const int32_t* stream; const long long* tick;
  double gravity[3];
  double joint_xyz[WBC_NU][3], joint_axis[WBC_NU][3], foot_xyz[WBC_NLEG][3];
  int v_index[WBC_NU];
};

// Per-warp shared memory: the covariance (padded rows), the state, P h of the current row, and the measurement table.
struct EstSmem {
  double P[NX][NX + 1];
  double x[NX];
  double ph[NX];
  double y[NY], sd[NY];
  double sk[WBC_NLEG];
};

// Why a record cannot be used, or nullptr (host code: wbc_estimator_set_create checks every record with it).
inline const char* desc_problem(const wbc_estimator_desc& d) {
  const double v[10] = {d.q_pos, d.q_vel, d.q_foot, d.r_pos, d.r_vel, d.r_height, d.swing_scale, d.p0_pos, d.p0_vel, d.p0_foot};
  for (double x : v)
    if (!(x >= 0.0)) return "wbc_estimator_set_create: a field is NaN or negative";
  const double fin[6] = {d.q_pos, d.q_vel, d.q_foot, d.p0_pos, d.p0_vel, d.p0_foot};
  for (double x : fin)
    if (!(x <= 1.7976931348623157e308)) return "wbc_estimator_set_create: process and initial stds must be finite";
  if (!(d.swing_scale >= 1.0 && d.swing_scale <= 1.7976931348623157e308))
    return "wbc_estimator_set_create: swing_scale must be finite and >= 1";
  return nullptr;
}

// Robot i's record, or -1 for an index outside [0, n_sets).
WBC_DEV int est_record(const EstArgs& a, long long i) {
  const int r = a.index ? a.index[i] : 0;
  return r >= 0 && r < a.n_sets ? r : -1;
}

// Rotation matrix (row-major) of a quaternion, normalised first.
WBC_DEV void quat_rot(const double* q, double R[9]) {
  const double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  const double w = q[0] / n, x = q[1] / n, y = q[2] / n, z = q[3] / n;
  R[0] = 1 - 2 * (y * y + z * z); R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
  R[3] = 2 * (x * y + w * z); R[4] = 1 - 2 * (x * x + z * z); R[5] = 2 * (y * z - w * x);
  R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = 1 - 2 * (x * x + y * y);
}

WBC_DEV void mat_vec(const double R[9], const double a[3], double o[3]) {
  for (int r = 0; r < 3; ++r) o[r] = R[3 * r] * a[0] + R[3 * r + 1] * a[1] + R[3 * r + 2] * a[2];
}

WBC_DEV void cross3(const double a[3], const double b[3], double o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}

// Foot `leg` relative to the base origin in base axes (r) and its velocity from the joint rates (jv, base axes), from the joint
// angles of q [19] and rates of v [18]: the leg chain of joint_xyz / joint_axis / foot_xyz, written standalone.
WBC_DEV void leg_kinematics(const EstArgs& a, const double* q, const double* v, int leg, double r[3], double jv[3]) {
  double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, rho[3] = {0, 0, 0};
  double ax[3][3], org[3][3], rate[3];
  for (int j = 0; j < 3; ++j) {
    const int k = 3 * leg + j;
    double t[3];
    mat_vec(R, a.joint_xyz[k], t);
    for (int c = 0; c < 3; ++c) rho[c] += t[c];
    const double* la = a.joint_axis[k];
    mat_vec(R, la, ax[j]);
    for (int c = 0; c < 3; ++c) org[j][c] = rho[c];
    rate[j] = v[a.v_index[k]];
    double sn, cs;
    sincos(q[a.v_index[k] + 1], &sn, &cs);
    const double oc = 1.0 - cs;
    // Rot(la, th) = cs I + sn [la]x + (1 - cs) la la'
    const double G[9] = {cs + oc * la[0] * la[0], -sn * la[2] + oc * la[0] * la[1], sn * la[1] + oc * la[0] * la[2],
                         sn * la[2] + oc * la[1] * la[0], cs + oc * la[1] * la[1], -sn * la[0] + oc * la[1] * la[2],
                         -sn * la[1] + oc * la[2] * la[0], sn * la[0] + oc * la[2] * la[1], cs + oc * la[2] * la[2]};
    double Rn[9];
    for (int rr = 0; rr < 3; ++rr)
      for (int cc = 0; cc < 3; ++cc) Rn[3 * rr + cc] = R[3 * rr] * G[cc] + R[3 * rr + 1] * G[3 + cc] + R[3 * rr + 2] * G[6 + cc];
    for (int e = 0; e < 9; ++e) R[e] = Rn[e];
  }
  double t[3];
  mat_vec(R, a.foot_xyz[leg], t);
  for (int c = 0; c < 3; ++c) { r[c] = rho[c] + t[c]; jv[c] = 0.0; }
  for (int j = 0; j < 3; ++j) {
    const double d[3] = {r[0] - org[j][0], r[1] - org[j][1], r[2] - org[j][2]};
    double cr[3];
    cross3(ax[j], d, cr);
    for (int c = 0; c < 3; ++c) jv[c] += cr[c] * rate[j];
  }
}

// The three accelerometer normals of robot `stream` at step c: draw 18 (two) and the first of draw 19.
WBC_DEV void accel_normals(unsigned long long seed, uint32_t stream, long long c, double z[3]) {
  double z3;
  for (int j = 0; j < 2; ++j) {
    uint32_t w[4] = {(uint32_t)(ACCEL_DRAW + j), stream, (uint32_t)(unsigned long long)c, (uint32_t)((unsigned long long)c >> 32)};
    wbcloop::philox4x32_10(w, (uint32_t)seed, (uint32_t)(seed >> 32));
    if (j == 0) wbcloop::normal_pair(w, z[0], z[1]);
    else wbcloop::normal_pair(w, z[2], z3);
  }
}

// One estimator step of robot i on warp lane `lane` (every lane of the warp calls it; sm is the warp's shared memory).
WBC_DEV void estimate_robot(const EstArgs& a, long long i, int lane, EstSmem& sm, const double* __restrict__ q,
                            const double* __restrict__ v, double* __restrict__ q_obs, double* __restrict__ v_obs,
                            const uint8_t* __restrict__ contact, int32_t* __restrict__ status_or) {
  const int r = est_record(a, i);
  if (r < 0) {
    if (lane == 0 && status_or) status_or[i] |= WBC_ST_BADESTIM;
    return;
  }
  const wbc_estimator_desc& d = a.set[r];
  const double* qi = q + i * WBC_NQ;
  const double* vi = v + i * WBC_NV;
  double* qo = q_obs + i * WBC_NQ;
  double* vo = v_obs + i * WBC_NV;
  double* xg = a.x + i * NX;
  double* Pg = a.P + i * NX * NX;
  double* vp = a.v_prev + i * 3;
  const long long count = a.count[i];
  const bool prime = count <= 0;
  double Ro[9];
  quat_rot(qo, Ro);
  // ---- legs: lane k < 4 gives foot k's world offset R_obs r_k and its measurement rows
  if (lane < WBC_NLEG) {
    const int k = lane;
    double rk[3], jv[3], rw[3], t[3], u[3];
    leg_kinematics(a, qo, vo, k, rk, jv);
    mat_vec(Ro, rk, rw);
    const double s = contact[i * WBC_NLEG + k] ? 1.0 : d.swing_scale;
    sm.sk[k] = s;
    cross3(vo, rw, t);                       // w_obs x R_obs r_k
    mat_vec(Ro, jv, u);
    for (int c = 0; c < 3; ++c) {
      sm.y[7 * k + c] = rw[c];
      sm.sd[7 * k + c] = d.r_pos * s;
      sm.y[7 * k + 3 + c] = -(t[c] + u[c]);
      sm.sd[7 * k + 3 + c] = d.r_vel * s;
    }
    sm.y[7 * k + 6] = 0.0;
    sm.sd[7 * k + 6] = d.r_height * s;
    // the prime's feet: p + R_obs r_k
    if (prime)
      for (int c = 0; c < 3; ++c) sm.x[6 + 3 * k + c] = qo[4 + c] + rw[c];
  }
  // ---- lane 0: the base state (prime, or the prediction with the synthesised accelerometer)
  if (lane == 0) {
    if (prime) {
      for (int c = 0; c < 3; ++c) { sm.x[c] = qo[4 + c]; sm.x[3 + c] = vo[3 + c]; }
    } else {
      double Rt[9], aw[3], fb[3], acc[3];
      quat_rot(qi, Rt);
      for (int c = 0; c < 3; ++c) aw[c] = (vi[3 + c] - vp[c]) / a.dt - a.gravity[c];
      for (int c = 0; c < 3; ++c) fb[c] = Rt[c] * aw[0] + Rt[3 + c] * aw[1] + Rt[6 + c] * aw[2];     // R_true' (a_w - g)
      const double sa = a.accel_noise ? a.accel_noise[i] : 0.0;
      if (sa != 0.0) {
        double z[3];
        const long long c = a.tick ? a.tick[i] : 0;
        accel_normals(a.seed, a.stream ? (uint32_t)a.stream[i] : (uint32_t)i, c, z);
        for (int e = 0; e < 3; ++e) fb[e] = fb[e] + sa * z[e];
      }
      mat_vec(Ro, fb, acc);
      for (int c = 0; c < 3; ++c) {
        const double vn = xg[3 + c] + a.dt * (acc[c] + a.gravity[c]);
        sm.x[3 + c] = vn;
        sm.x[c] = xg[c] + a.dt * vn;
      }
    }
  }
  if (!prime && lane >= 6 && lane < NX) sm.x[lane] = xg[lane];
  // ---- covariance: lane r < 18 holds row r in registers (Pr); the prime's diagonal, or A P A' + Q (row pass p += dt v, then
  //      column pass)
  double Pr[NX];
#pragma unroll
  for (int c = 0; c < NX; ++c) {
    if (prime) {
      const double s0 = c < 3 ? d.p0_pos : c < 6 ? d.p0_vel : d.p0_foot;
      Pr[c] = c == lane ? s0 * s0 : 0.0;
    } else {
      Pr[c] = lane < NX ? Pg[lane * NX + c] : 0.0;
    }
  }
  __syncwarp();
  bool ok = true;
  if (!prime) {
#pragma unroll
    for (int c = 0; c < NX; ++c) {
      const double below = __shfl_sync(0xffffffffu, Pr[c], lane + 3 < 32 ? lane + 3 : lane);   // row lane + 3
      if (lane < 3) Pr[c] += a.dt * below;
    }
    const double qs = lane < 3 ? d.q_pos : lane < 6 ? d.q_vel : lane < NX ? d.q_foot * sm.sk[(lane - 6) / 3] : 0.0;
#pragma unroll
    for (int c = 0; c < NX; ++c) {
      if (c < 3) Pr[c] += a.dt * Pr[c + 3];
      if (c == lane) Pr[c] += a.dt * (qs * qs);
    }
    // ---- the 28 rows as scalar updates: h = e_plus - e_minus (minus < 0: none)
    for (int m = 0; m < NY && ok; ++m) {
      const double sd = sm.sd[m];
      if (!(sd <= 1.7976931348623157e308)) continue;               // +inf drops the row
      const int k = m / 7, e = m % 7;
      const int plus = e < 3 ? 6 + 3 * k + e : e < 6 ? e : 6 + 3 * k + 2;
      const int minus = e < 3 ? e : -1;
      double pp = 0.0, pm = 0.0;
#pragma unroll
      for (int c = 0; c < NX; ++c) {
        if (c == plus) pp = Pr[c];
        if (c == minus) pm = Pr[c];
      }
      const double phr = minus >= 0 ? pp - pm : pp;
      if (lane < NX) sm.ph[lane] = phr;
      __syncwarp();
      const double S = (minus >= 0 ? sm.ph[plus] - sm.ph[minus] : sm.ph[plus]) + sd * sd;
      const double innov = sm.y[m] - (minus >= 0 ? sm.x[plus] - sm.x[minus] : sm.x[plus]);
      ok = S > 0.0;                                                 // the same value in every lane
      __syncwarp();
      if (ok && lane < NX) {
        const double K = phr / S;
        sm.x[lane] += K * innov;
#pragma unroll
        for (int c = 0; c < NX; ++c) Pr[c] -= K * sm.ph[c];
      }
      __syncwarp();
    }
    // symmetrise through shared memory: lane r owns the pairs (r, c > r)
    if (lane < NX)
      for (int c = 0; c < NX; ++c) sm.P[lane][c] = Pr[c];
    __syncwarp();
    if (ok && lane < NX)
      for (int c = lane + 1; c < NX; ++c) {
        const double s = 0.5 * (sm.P[lane][c] + sm.P[c][lane]);
        sm.P[lane][c] = s;
        sm.P[c][lane] = s;
      }
    __syncwarp();
    bool fin = true;
    if (lane < NX) {
      fin = fabs(sm.x[lane]) <= 1.7976931348623157e308;
      for (int c = 0; c < NX; ++c) fin = fin && fabs(sm.P[lane][c]) <= 1.7976931348623157e308;
    }
    ok = ok && __all_sync(0xffffffffu, fin);
  } else {
    if (lane < NX)
      for (int c = 0; c < NX; ++c) sm.P[lane][c] = Pr[c];
    __syncwarp();
  }
  if (!ok) {
    if (lane == 0) {
      a.count[i] = 0;
      if (status_or) status_or[i] |= WBC_ST_BADESTIM;
    }
    return;
  }
  if (lane < NX) {
    xg[lane] = sm.x[lane];
    for (int c = 0; c < NX; ++c) Pg[lane * NX + c] = sm.P[lane][c];
  }
  if (lane == 0) {
    for (int c = 0; c < 3; ++c) vp[c] = vi[3 + c];
    a.count[i] = prime ? 1 : count + 1;
    if (!prime)
      for (int c = 0; c < 3; ++c) { qo[4 + c] = sm.x[c]; vo[3 + c] = sm.x[3 + c]; }
    if (a.stats) {
      double ep = 0.0, ev = 0.0;
      for (int c = 0; c < 3; ++c) {
        const double dp = sm.x[c] - qi[4 + c], dv = sm.x[3 + c] - vi[3 + c];
        ep += dp * dp;
        ev += dv * dv;
      }
      double* s = a.stats + i * 4;
      s[0] += ep;
      s[1] = fmax(s[1], sqrt(ep));
      s[2] += ev;
      s[3] = fmax(s[3], sqrt(ev));
    }
  }
}

#ifdef __CUDACC__
constexpr int EST_BLOCK = 128;        // 4 robots per CTA

__global__ void __launch_bounds__(EST_BLOCK) estimate_kernel(const EstArgs a, long long n, const double* __restrict__ q,
                                                             const double* __restrict__ v, double* __restrict__ q_obs,
                                                             double* __restrict__ v_obs, const uint8_t* __restrict__ contact,
                                                             int32_t* __restrict__ status_or) {
  __shared__ EstSmem sm[EST_BLOCK / 32];
  const long long i = ((long long)blockIdx.x * EST_BLOCK + threadIdx.x) >> 5;
  if (i >= n) return;                     // whole warps leave together
  estimate_robot(a, i, threadIdx.x & 31, sm[threadIdx.x >> 5], q, v, q_obs, v_obs, contact, status_or);
}
#endif

}  // namespace wbcest
