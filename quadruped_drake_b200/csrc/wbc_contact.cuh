// wbc_contact.cuh — contact detection in the ground-plant loop (include/wbc.h, wbc_contact_desc / wbc_contact): per robot, each
// foot's ground force is estimated from the joint torques and the motion they produced, and a hysteresis on its world-z component
// gives the foot's stance flag. The semantics are stated once in include/wbc.h and restated in numpy by oracle/contact.py.
//
// Two kernels. contact_detect_kernel is one warp per robot: it stages q_prev, v_prev into a WarpSmem and runs the controllers'
// dynamics_phase<DYN_STEP> (M's block-arrow parts Mb / Mleg, hb / hj = Cv + tau_g with the controller sign, the foot Jacobian leg
// blocks L), the same block the plant steps with; lanes 0-3 then form the joint rows of the momentum residual of one leg each and
// solve its 3 x 3 system by cofactors, all in FP64. contact_record_kernel is elementwise and runs after the plant: it copies the
// measured torque and the plant's forces into the state. The device functions also compile on the host
// (tests/emu/emu_contact.cpp, with the warp collectives of cuda_emu.h).
#pragma once
#include "wbc_device.cuh"

namespace wbccontact {
using namespace wbc;

constexpr int NSTAT = 6;                 // sum |err|^2, max |err|, true stance, true swing, false stance, false swing
constexpr double SINGULAR_SINVOL = 1e-9; // a leg is singular when |det J_leg| <= 1e-9 |a0| |a1| |a2|

// Device view of a wbc_contact (the state arrays are always given here: the library substitutes its scratch).
struct ContactArgs {
  const wbc_contact_desc* set; const int32_t* index; int n_sets;
  double* q_prev; double* v_prev; double* tau_prev; double* f_true; double* f_hat; uint8_t* flag; long long* count; double* stats;
  double dt;
};

// Why a record cannot be used, or nullptr (host code: wbc_contact_set_create checks every record with it).
inline const char* desc_problem(const wbc_contact_desc& d) {
  if (!(d.tau_f >= 0.0 && d.tau_f <= 1.7976931348623157e308)) return "wbc_contact_set_create: tau_f must be finite and >= 0";
  if (d.f_on != d.f_on || d.f_off != d.f_off) return "wbc_contact_set_create: f_on and f_off must not be NaN";
  if (!(d.f_off <= d.f_on)) return "wbc_contact_set_create: f_off <= f_on is required";
  return nullptr;
}

// Robot i's record, or -1 for an index outside [0, n_sets).
WBC_DEV int contact_record(const ContactArgs& a, long long i) {
  const int r = a.index ? a.index[i] : 0;
  return r >= 0 && r < a.n_sets ? r : -1;
}

// One detector step of robot i on warp lane `lane` (every lane of the warp calls it; s is the warp's shared memory). q, v: what
// the detector reads; plan: the plan's flags; detected [N][4] gets the step's flags, ctrl [N][4] (or null) plan AND detected.
WBC_DEV void detect_robot(const ContactArgs& a, const wbc_model& md, long long i, int lane, WarpSmem& s, const double* __restrict__ q,
                          const double* __restrict__ v, const uint8_t* __restrict__ plan, uint8_t* __restrict__ detected,
                          uint8_t* __restrict__ ctrl, int32_t* __restrict__ status_or) {
  const int r = contact_record(a, i);
  const uint8_t planned = lane < WBC_NLEG ? (plan[i * WBC_NLEG + lane] != 0) : 0;
  if (r < 0) {
    if (lane < WBC_NLEG) {
      detected[i * WBC_NLEG + lane] = planned;
      if (ctrl) ctrl[i * WBC_NLEG + lane] = planned;
    }
    if (lane == 0 && status_or) status_or[i] |= WBC_ST_BADCONTACT;
    return;
  }
  const double* qi = q + i * WBC_NQ;
  const double* vi = v + i * WBC_NV;
  double* qp = a.q_prev + i * WBC_NQ;
  double* vp = a.v_prev + i * WBC_NV;
  const long long count = a.count[i];
  __syncwarp();                                      // every lane has read count before lane 0 rewrites it
  if (count <= 0) {                                  // prime: the plan's flags, no force, the state read now
    if (lane < WBC_NLEG) {
      a.flag[i * WBC_NLEG + lane] = planned;
      detected[i * WBC_NLEG + lane] = planned;
      if (ctrl) ctrl[i * WBC_NLEG + lane] = planned;
    }
    if (lane < 12) a.f_hat[i * 12 + lane] = 0.0;
    if (lane < WBC_NQ) qp[lane] = qi[lane];
    if (lane < WBC_NV) vp[lane] = vi[lane];
    if (lane == 0) a.count[i] = 1;
    return;
  }
  if (lane < WBC_NQ) s.q[lane] = qp[lane];
  if (lane < WBC_NV) s.v[lane] = vp[lane];
  __syncwarp();
  int dyn_status = 0;                                // (a bad quaternion shows as a non-finite or wrong force, not as a bit)
  dynamics_phase<DYN_STEP>(s, md, lane, dyn_status, nullptr);
  // ---- lane k < 4: leg k's joint rows r_k of M (v - v_prev) - dt (B tau_prev - h), then J_leg' p = r_k by cofactors
  double f_raw[3] = {0.0, 0.0, 0.0};
  bool singular = true, bad = false;
  if (lane < WBC_NLEG) {
    const int k = lane;
    double dvb[6], dvj[3], rk[3];
#pragma unroll
    for (int c = 0; c < 6; ++c) dvb[c] = vi[c] - s.v[c];
#pragma unroll
    for (int y = 0; y < 3; ++y) { const int e = md.v_index[3 * k + y]; dvj[y] = vi[e] - s.v[e]; }
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      const int j = 3 * k + x;
      double acc = -a.dt * (a.tau_prev[i * WBC_NU + md.act_index[j]] - s.hj[j]);
#pragma unroll
      for (int c = 0; c < 6; ++c) acc = fma(s.Mb[6 + j][c], dvb[c], acc);
#pragma unroll
      for (int y = 0; y < 3; ++y) acc = fma(s.Mleg[k][x <= y ? sym3(x, y) : sym3(y, x)], dvj[y], acc);
      rk[x] = acc;
    }
    const double(&L)[3][3] = s.L[k];                 // rows: world axes, columns: the leg's joints
    const double C[3][3] = {{L[1][1] * L[2][2] - L[1][2] * L[2][1], L[1][2] * L[2][0] - L[1][0] * L[2][2], L[1][0] * L[2][1] - L[1][1] * L[2][0]},
                            {L[0][2] * L[2][1] - L[0][1] * L[2][2], L[0][0] * L[2][2] - L[0][2] * L[2][0], L[0][1] * L[2][0] - L[0][0] * L[2][1]},
                            {L[0][1] * L[1][2] - L[0][2] * L[1][1], L[0][2] * L[1][0] - L[0][0] * L[1][2], L[0][0] * L[1][1] - L[0][1] * L[1][0]}};
    const double det = L[0][0] * C[0][0] + L[0][1] * C[0][1] + L[0][2] * C[0][2];
    double vol = 1.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) vol *= sqrt(L[0][c] * L[0][c] + L[1][c] * L[1][c] + L[2][c] * L[2][c]);
    singular = fabs(det) <= SINGULAR_SINVOL * vol;
    // (L')^-1 = C / det: p = C r / det, f = p / dt
    const double scale = 1.0 / (det * a.dt);
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      f_raw[x] = (C[x][0] * rk[0] + C[x][1] * rk[1] + C[x][2] * rk[2]) * scale;
      if (!singular && !(fabs(f_raw[x]) <= 1.7976931348623157e308)) bad = true;
    }
  }
  const bool fail = __any_sync(WBC_FULL, bad);
  __syncwarp();                                      // every lane has read v_prev before it is overwritten below
  if (fail) {
    if (lane < WBC_NLEG) {
      detected[i * WBC_NLEG + lane] = planned;
      if (ctrl) ctrl[i * WBC_NLEG + lane] = planned;
    }
    if (lane == 0) {
      a.count[i] = 0;
      if (status_or) status_or[i] |= WBC_ST_BADCONTACT;
    }
    return;
  }
  // ---- filter, hysteresis and statistics of foot k = lane
  double e2 = 0.0, ts = 0.0, tw = 0.0, fs = 0.0, fw = 0.0;
  if (lane < WBC_NLEG) {
    const int k = lane;
    const wbc_contact_desc d = a.set[r];
    uint8_t f = a.flag[i * WBC_NLEG + k];
    if (!singular) {
      double* fh = a.f_hat + i * 12 + 3 * k;
      const bool raw = count == 1 || d.tau_f == 0.0;
      const double alpha = raw ? 1.0 : -expm1(-a.dt / d.tau_f);
#pragma unroll
      for (int x = 0; x < 3; ++x) fh[x] = raw ? f_raw[x] : fh[x] + alpha * (f_raw[x] - fh[x]);
      f = f ? (fh[2] <= d.f_off ? 0 : 1) : (fh[2] >= d.f_on ? 1 : 0);
      a.flag[i * WBC_NLEG + k] = f;
      if (a.stats) {
        const double* ft = a.f_true + i * 12 + 3 * k;
#pragma unroll
        for (int x = 0; x < 3; ++x) e2 += (f_raw[x] - ft[x]) * (f_raw[x] - ft[x]);
        const bool loaded = ft[0] != 0.0 || ft[1] != 0.0 || ft[2] != 0.0;
        ts = f && loaded; tw = !f && !loaded; fs = f && !loaded; fw = !f && loaded;
      }
    }
    detected[i * WBC_NLEG + k] = f;
    if (ctrl) ctrl[i * WBC_NLEG + k] = planned & f;
  }
  if (a.stats) {                                     // lanes 0-3 into lane 0 (lanes >= 4 hold zeros)
    double m2 = e2;
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
      e2 += __shfl_xor_sync(WBC_FULL, e2, o);
      m2 = fmax(m2, __shfl_xor_sync(WBC_FULL, m2, o));
      ts += __shfl_xor_sync(WBC_FULL, ts, o); tw += __shfl_xor_sync(WBC_FULL, tw, o);
      fs += __shfl_xor_sync(WBC_FULL, fs, o); fw += __shfl_xor_sync(WBC_FULL, fw, o);
    }
    if (lane == 0) {
      double* st = a.stats + i * NSTAT;
      st[0] += e2; st[1] = fmax(st[1], sqrt(m2));
      st[2] += ts; st[3] += tw; st[4] += fs; st[5] += fw;
    }
  }
  if (lane < WBC_NQ) qp[lane] = qi[lane];
  if (lane < WBC_NV) vp[lane] = vi[lane];
  if (lane == 0) a.count[i] = count + 1;
}

// The record step of element t = 12 i + j: robot i's measured torque and the plant's force component j (a bad index: untouched).
WBC_DEV void record_element(const ContactArgs& a, long long t, const double* __restrict__ tau_meas, const double* __restrict__ f_contact) {
  if (contact_record(a, t / 12) < 0) return;
  a.tau_prev[t] = tau_meas[t];
  a.f_true[t] = f_contact[t];
}

#ifdef __CUDACC__
constexpr int CONTACT_BLOCK = 128;       // 4 robots per CTA: the model (1928 B) is staged once for four warps
static_assert(sizeof(wbc_model) % 8 == 0, "the model is staged as doubles");

__global__ void __launch_bounds__(CONTACT_BLOCK) contact_detect_kernel(const ContactArgs a, const wbc_model* __restrict__ gmd, long long n,
                                                                       const double* __restrict__ q, const double* __restrict__ v,
                                                                       const uint8_t* __restrict__ plan, uint8_t* __restrict__ detected,
                                                                       uint8_t* __restrict__ ctrl, int32_t* __restrict__ status_or) {
  __shared__ __align__(16) wbc_model md;
  __shared__ WarpSmem sm[CONTACT_BLOCK / 32];
  for (int e = threadIdx.x; e < (int)(sizeof(wbc_model) / 8); e += CONTACT_BLOCK)
    reinterpret_cast<double*>(&md)[e] = reinterpret_cast<const double*>(gmd)[e];
  __syncthreads();
  const long long i = ((long long)blockIdx.x * CONTACT_BLOCK + threadIdx.x) >> 5;
  if (i >= n) return;                     // whole warps leave together
  detect_robot(a, md, i, threadIdx.x & 31, sm[threadIdx.x >> 5], q, v, plan, detected, ctrl, status_or);
}

__global__ void contact_record_kernel(const ContactArgs a, long long n, const double* __restrict__ tau_meas,
                                      const double* __restrict__ f_contact) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n * WBC_NU) record_element(a, t, tau_meas, f_contact);
}
#endif

}  // namespace wbccontact
