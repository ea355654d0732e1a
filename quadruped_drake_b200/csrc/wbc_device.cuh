// wbc_device.cuh — per-warp whole-body controller step (sm_100a, FP64 on the CUDA cores).
//
// One warp owns one robot instance from load to store; nothing but the 860 B/step of
// algorithmic I/O touches HBM. Phases (see DESIGN.md):
//   1. dynamics   composite spatial inertias about the base origin, world axes
//                 (replaces basic_controller.py:101-115 CalcDynamics and :173-196 foot queries)
//   2. equalities [A|b] of the tau-eliminated QP, one column per lane, in shared memory
//   3. Gauss-Jordan with column pivoting -> z = z0 + Z w  (12 or 13 free variables)
//   4. reduced rows Y = [a_b; f / swing-task; tau; extra] as affine maps of w
//   5. reduced Hessian / gradient, Cholesky, J = L^-T
//   6. Goldfarb-Idnani dual active set on w (exact optimum; replaces OsqpSolver().Solve,
//      inverse_dynamics_controller.py:223)
//   7. tau / metrics / status
//
// The file is plain CUDA C++ restricted to warp-synchronous primitives so that
// tests/emu/ can compile it for the host with a lock-step warp emulator.
#pragma once
#include <stdint.h>
#include <math.h>
#include <stddef.h>
#include <type_traits>
#include "wbc.h"

#ifndef WBC_DEV
#define WBC_DEV __device__ __forceinline__
#endif
#ifndef WBC_FULL
#define WBC_FULL 0xffffffffu
#endif

namespace wbc {

constexpr int NF = 13;      // reduced dimension (12 free variables for ID/PC, 13 for CLF; padded to 13)
constexpr int YS = 15;      // row stride of Y: 13 coefficients + constant + 1 pad (odd stride: row-per-lane access is bank-conflict free)
constexpr int YROWS = 32;   // 0-5 a_b | 6-17 leg rows (f of a stance leg / task accel of a swing leg) | 18-29 tau | 30,31 extra
constexpr int AR = 6;       // rows of the reduced base system (the stance-leg rows are eliminated analytically)
constexpr int AC = 32;      // columns of [A|b]: lane c owns column c, lane 31 the right-hand side
// A stance leg is RANKDEF when |det L_k| <= RANKDEF_SINVOL * |c0| |c1| |c2| (c_j the columns of its 3x3 foot Jacobian block).
// The contact rows are solved through L_k^-1, so the error of the leg's joint accelerations grows like 1 / det. Against the
// oracle (stretched-knee sweep of tests/test_edge_states.py) the vd error of PC reaches 1.6e-7 at a sine-volume of 1.5e-3 on
// mini_cheetah; from 2e-3 up every unflagged instance of both robots is 10x inside the 1e-5 (tau) / 1e-6 (vd) parity bars.
// That flags knees within about 4e-3 rad (mini_cheetah) / 5e-3 rad (anymal_b) of the stretched pose.
constexpr double RANKDEF_SINVOL = 2e-3;

// Host-precomputed constants (wbc_create): per-channel CARE solution of the double integrator and the
// decay rate gamma of clf_controller.py:170-188 (closed form, SURVEY Appendix C.2).
struct Derived {
  double clf_p[3][3];     // channel type (0 rpy, 1 base position, 2 swing foot) x (p11, p12, p22)
  double clf_gamma[2];    // [no swing foot, at least one swing foot]
};

// Host side (wbc_create and the test emulator).
// Scalar double-integrator CARE (clf_controller.py:170-187 with block-diagonal Q, R = r I, SURVEY C.2):
// p12 = sqrt(qp r), p22 = sqrt(r (qd + 2 p12)), p11 = p12 p22 / r; gamma = lambda_min(Q) / lambda_max(P) (:188).
inline void derive_constants(const wbc_params& p, wbc::Derived& d) {
  const double qp[3] = {p.clf_q_body_rpy, p.clf_q_body_p, p.clf_q_foot_p};
  const double qd[3] = {p.clf_q_body_rpyd, p.clf_q_body_pd, p.clf_q_foot_pd};
  double lmax[3];
  for (int t = 0; t < 3; ++t) {
    const double r = p.clf_r;
    const double p12 = sqrt(qp[t] * r), p22 = sqrt(r * (qd[t] + 2.0 * p12)), p11 = p12 * p22 / r;
    d.clf_p[t][0] = p11; d.clf_p[t][1] = p12; d.clf_p[t][2] = p22;
    lmax[t] = 0.5 * (p11 + p22) + sqrt(0.25 * (p11 - p22) * (p11 - p22) + p12 * p12);
  }
  auto mn = [](double a, double b) { return a < b ? a : b; };
  auto mx = [](double a, double b) { return a > b ? a : b; };
  const double qmin_body = mn(mn(qp[0], qd[0]), mn(qp[1], qd[1]));
  const double qmin_all = mn(qmin_body, mn(qp[2], qd[2]));
  d.clf_gamma[0] = qmin_body / mx(lmax[0], lmax[1]);
  d.clf_gamma[1] = qmin_all / mx(mx(lmax[0], lmax[1]), lmax[2]);
}


struct StepArgs {
  const double* q; const double* v; const double* traj; const uint8_t* contact;
  double* tau; double* metrics; int32_t* status; double* vd; double* f; double* qp_info; double* lam;
  long long n; int kind;
};

// Per-warp shared memory of the reduce half (phases 0-4): inputs, dynamics block, the reduced base system and the reduced
// problem it leaves behind (9.9 KB).
struct alignas(16) WarpSmem {
  // ---- inputs
  double q[WBC_NQ], v[WBC_NV], traj[WBC_NTRAJ];
  // ---- dynamics block (internal joint order k = 3*leg + j)
  double Mb[18][6];      // Mb[c][r] = M[r][c] for r < 6 (base rows of the mass matrix, column major)
  double Mleg[4][6];     // per-leg 3x3 block, upper triangle (0,0)(0,1)(0,2)(1,1)(1,2)(2,2)
  double hb[6], hj[12];  // bias: C v + tau_g (controller sign)
  double rho[4][3];      // foot position relative to the base origin, world axes
  double L[4][3][3];     // leg block of the foot Jacobian: L[leg][row][joint]
  double Jdv[4][3], vf[4][3];
  double Ld[4][3][3];    // time derivative of L (PC only): Ld[leg][row][joint]
  double task[16];       // 7-15: base rotation matrix (column major)
  double y[YROWS];       // scratch (CLF: kappa per task row)
  // ---- reduced base system [B | c0] over u = [a_b(6); per leg f_k (stance) or a_k (swing)] and its reduction
  double A[AR][AC];
  double AK[4][3][7];    // stance leg k: a_k = AK[k][:, 6] - AK[k][:, 0:6] a_b   (= L_k^-1 (r_k - Jb_k a_b))
  // ---- reduced problem ([Y | cw | ct] contiguous and 16-byte aligned: one bulk copy in the split path)
  alignas(16) double Y[YROWS][YS];
  double cw[YROWS], ct[YROWS];   // cost weight / target of each Y row: 1/2 cw (y - ct)^2
};

// Per-warp shared memory of the solve kernel of the split path (phases 5-7 only): the reduced problem (Y, cw, ct - one
// contiguous 4 KB block, filled by a single bulk copy of the record the reduce kernel wrote) and the Goldfarb-Idnani state.
template <bool VD>
struct alignas(16) SolveSmemT {
  alignas(16) double Y[YROWS][YS];
  double cw[YROWS], ct[YROWS];
  double H[NF][NF];                       // reduced Hessian -> its Cholesky factor L (lower triangle, in place); once W is
                                          // built L is dead unless the accelerations are requested (x recovery), so without
                                          // VD the rows of R^-1 (below) live here
  double Rp[NF * (NF + 3) / 2];           // R of the active set, transposed and packed: column c keeps rows 0..c+1 (the
                                          // sub-diagonal entry exists only while a dropped column is rotated away)
  double d[NF];                           // 1 / L[k][k]
  union { double g[NF]; double dm[NF]; }; // start-up: b = W'e / then the current d = J'n
  union { double npv[NF]; double x[NF]; };// recovered w (exit only)
  double u[NF], y[YROWS];
  int act[NF];
  alignas(8) unsigned long long mbar;     // completion barrier of the bulk copy
  double Ris[VD ? NF * NF : 1];           // R^-1 of the active set, row k in lane k's row (stride NF: conflict free)
  static constexpr bool kVd = VD;
};
template <class SM> WBC_DEV double* ri_rows(SM& s) { return SM::kVd ? &s.Ris[0] : &s.H[0][0]; }
using SolveSmem = SolveSmemT<false>;      // step without accelerations (the benchmark path): 28 warps / SM
using SolveSmemVd = SolveSmemT<true>;     // vd requested (rollout, debug outputs): L is kept for the x recovery, 24 warps / SM
static_assert(sizeof(SolveSmem) <= 7312, "28 single-warp CTAs of the solve kernel must fit one SM (228 KB, 1 KB reserved per CTA)");
// entry (row, col) of R, row <= col + 1
template <class SM> WBC_DEV double& Rent(SM& s, int col, int row) { return s.Rp[col * (col + 3) / 2 + row]; }
constexpr int REC_Y = YROWS * YS + 2 * YROWS;   // doubles of [Y | cw | ct]
constexpr int REC_MISC = 16;                    // status, cmask, nf, nextra, ok, extra_bound, err, Vl, PFl, csum, Vpc
constexpr int REC_DOUBLES = REC_Y + REC_MISC;   // one record of the reduce -> solve hand-over (4224 B)
constexpr int VDMAP_DOUBLES = 18 * YS;          // accelerations [a_b; joints] as affine maps of w (only when vd is requested)

// ------------------------------------------------------------------ small vector helpers
struct V3 { double x, y, z; };
WBC_DEV V3 mk(double x, double y, double z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
WBC_DEV V3 operator+(V3 a, V3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
WBC_DEV V3 operator-(V3 a, V3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
WBC_DEV V3 operator*(double s, V3 a) { return mk(s * a.x, s * a.y, s * a.z); }
WBC_DEV V3 cross(V3 a, V3 b) { return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
WBC_DEV double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
WBC_DEV double comp(V3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
struct M3 { V3 c0, c1, c2; };  // columns
WBC_DEV V3 mul(const M3& R, V3 a) { return a.x * R.c0 + a.y * R.c1 + a.z * R.c2; }
struct S6 { double xx, yy, zz, xy, xz, yz; };  // symmetric 3x3
WBC_DEV V3 mul(const S6& I, V3 a) {
  return mk(I.xx * a.x + I.xy * a.y + I.xz * a.z, I.xy * a.x + I.yy * a.y + I.yz * a.z, I.xz * a.x + I.yz * a.y + I.zz * a.z);
}
WBC_DEV V3 ld3(const double* p) { return mk(p[0], p[1], p[2]); }

// Fast reciprocal / reciprocal square root: hardware approximation + two Newton steps (full double precision for the
// normal-range operands that occur here; an IEEE division expands to ~25 instructions, this to ~7).
#ifdef __CUDA_ARCH__
WBC_DEV double frcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
}
WBC_DEV double frsqrt(double x) {
  double r;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  // Newton for 1/sqrt: r <- r (1.5 - 0.5 x r^2), written as r + r * (0.5 - 0.5 x r^2)
  double h = 0.5 * x;
  double e = fma(-h * r, r, 0.5);
  r = fma(r, e, r);
  e = fma(-h * r, r, 0.5);
  return fma(r, e, r);
}
#else
WBC_DEV double frcp(double x) { return 1.0 / x; }
WBC_DEV double frsqrt(double x) { return 1.0 / sqrt(x); }
#endif

// Asynchronous 8-byte global -> shared copy (LDGSTS): the trajectory row is requested at the start of a step and only
// waited for after the dynamics phase, so its latency (microseconds when the buffers live in page-locked host memory)
// hides behind the arithmetic that does not need it.
#ifdef __CUDA_ARCH__
WBC_DEV void async_copy8(double* smem_dst, const double* gsrc) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gsrc) : "memory");
}
WBC_DEV void async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
#else
WBC_DEV void async_copy8(double* smem_dst, const double* gsrc) { *smem_dst = *gsrc; }
WBC_DEV void async_wait_all() {}
#endif

template <typename T> WBC_DEV T shfl(T v, int src) { return __shfl_sync(WBC_FULL, v, src); }
WBC_DEV double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(WBC_FULL, v, o);
  return v;
}
// Arg-max / arg-min of a NON-NEGATIVE double over the warp with two 32-bit redux.sync reductions (IEEE order of
// non-negative doubles = unsigned order of their bit patterns): high words first, then the low words of the lanes that
// tie on the high word; the winner is the lowest such lane. Returns the extreme value (exact) and its lane.
WBC_DEV double warp_max_lane(double v, int& lane_out) {
  const unsigned hi = (unsigned)__double2hiint(v), lo = (unsigned)__double2loint(v);
  const unsigned mhi = __reduce_max_sync(WBC_FULL, hi);
  const unsigned mlo = __reduce_max_sync(WBC_FULL, hi == mhi ? lo : 0u);
  lane_out = __ffs((int)__ballot_sync(WBC_FULL, hi == mhi && lo == mlo)) - 1;
  return __hiloint2double((int)mhi, (int)mlo);
}
// Arg-max of a NON-NEGATIVE double on its high word only (one redux instead of two): the winner is within 2^-20 relative of
// the maximum, which is all a pivot rule needs. Returns the winning lane, `any` = some lane holds a value >= 2^-1022 * 2^32.
WBC_DEV int warp_argmax_hi(double v, bool& any) {
  const unsigned hi = (unsigned)__double2hiint(v);
  const unsigned mhi = __reduce_max_sync(WBC_FULL, hi);
  any = mhi != 0u;
  return __ffs((int)__ballot_sync(WBC_FULL, hi == mhi)) - 1;
}
WBC_DEV double warp_min_lane(double v, int& lane_out) {
  const unsigned hi = (unsigned)__double2hiint(v), lo = (unsigned)__double2loint(v);
  const unsigned mhi = __reduce_min_sync(WBC_FULL, hi);
  const unsigned mlo = __reduce_min_sync(WBC_FULL, hi == mhi ? lo : 0xffffffffu);
  lane_out = __ffs((int)__ballot_sync(WBC_FULL, hi == mhi && lo == mlo)) - 1;
  return __hiloint2double((int)mhi, (int)mlo);
}

// Spatial inertia about the base origin P, world axes: mass, first moment h = m c, rotational part.
struct SpI { double m; V3 h; S6 I; };
// World-frame spatial inertia of a link with body-frame CoM `com`, inertia about CoM `Ic`,
// pose (R, rho) relative to P.
WBC_DEV SpI link_inertia(double m, V3 com, const double* ic, const M3& R, V3 rho) {
  SpI s; s.m = m;
  V3 c = rho + mul(R, com);
  s.h = m * c;
  // R Ic R^T
  S6 Ic; Ic.xx = ic[0]; Ic.yy = ic[1]; Ic.zz = ic[2]; Ic.xy = ic[3]; Ic.xz = ic[4]; Ic.yz = ic[5];
  // T = R * Ic (columns of T = R * columns of Ic)
  V3 t0 = mul(R, mk(Ic.xx, Ic.xy, Ic.xz)), t1 = mul(R, mk(Ic.xy, Ic.yy, Ic.yz)), t2 = mul(R, mk(Ic.xz, Ic.yz, Ic.zz));
  // (T R^T)_{ab} = sum_k T_{ak} R_{bk};  R_{bk} = component b of column k
  auto e = [&](int a, int b) {
    return comp(t0, a) * comp(R.c0, b) + comp(t1, a) * comp(R.c1, b) + comp(t2, a) * comp(R.c2, b);
  };
  double cc = dot(c, c);
  s.I.xx = e(0, 0) + m * (cc - c.x * c.x); s.I.yy = e(1, 1) + m * (cc - c.y * c.y); s.I.zz = e(2, 2) + m * (cc - c.z * c.z);
  s.I.xy = e(0, 1) - m * c.x * c.y; s.I.xz = e(0, 2) - m * c.x * c.z; s.I.yz = e(1, 2) - m * c.y * c.z;
  return s;
}
// momentum-like product I * [w; u] -> (n, f)
WBC_DEV void spi_mul(const SpI& s, V3 w, V3 u, V3& n, V3& f) {
  n = mul(s.I, w) + cross(s.h, u);
  f = s.m * u - cross(s.h, w);
}
WBC_DEV SpI spi_add(const SpI& a, const SpI& b) {
  SpI s; s.m = a.m + b.m; s.h = a.h + b.h;
  s.I.xx = a.I.xx + b.I.xx; s.I.yy = a.I.yy + b.I.yy; s.I.zz = a.I.zz + b.I.zz;
  s.I.xy = a.I.xy + b.I.xy; s.I.xz = a.I.xz + b.I.xz; s.I.yz = a.I.yz + b.I.yz;
  return s;
}
#define WBC_SPI_SHFL(OP, s, arg, W)                                                                          \
  {                                                                                                          \
    SpI t_;                                                                                                  \
    t_.m = OP(WBC_FULL, s.m, arg, W); t_.h.x = OP(WBC_FULL, s.h.x, arg, W); t_.h.y = OP(WBC_FULL, s.h.y, arg, W); \
    t_.h.z = OP(WBC_FULL, s.h.z, arg, W); t_.I.xx = OP(WBC_FULL, s.I.xx, arg, W); t_.I.yy = OP(WBC_FULL, s.I.yy, arg, W); \
    t_.I.zz = OP(WBC_FULL, s.I.zz, arg, W); t_.I.xy = OP(WBC_FULL, s.I.xy, arg, W); t_.I.xz = OP(WBC_FULL, s.I.xz, arg, W); \
    t_.I.yz = OP(WBC_FULL, s.I.yz, arg, W); tmp_spi = t_;                                                    \
  }
#define WBC_V3_SHFL(OP, a, arg, W) mk(OP(WBC_FULL, (a).x, arg, W), OP(WBC_FULL, (a).y, arg, W), OP(WBC_FULL, (a).z, arg, W))

WBC_DEV int sym3(int i, int j) {  // upper-triangle index of a 3x3 symmetric block, i <= j
  return i == 0 ? j : (i == 1 ? 2 + j : 5);
}

// Output selector for the dynamics parity entry.
struct DynOut { double* M; double* Cv; double* taug; double* Jfeet; double* Jdv; double* pfeet; };

// ------------------------------------------------------------------------------ phase 1
// Modes of dynamics_phase
constexpr int DYN_STEP = 0;    // step kernels: gravity folded into the bias (hb/hj = Cv + tau_g)
constexpr int DYN_PARITY = 1;  // wbc_dynamics: hb/hj = Cv only, tau_g (controller sign) to taug_sm[18] (internal order)
constexpr int DYN_BIAS = 2;    // bias only: b = C(q, vel) vel for the velocity `vel_int` (internal order) -> bias_out[18]
constexpr int DYN_STEP_JD = 3; // DYN_STEP plus the Jdot leg blocks Ld (PC controller)
constexpr int DYN_PC = 4;      // DYN_STEP_JD or DYN_BIAS chosen at RUN time (`bias_rt`): one copy of the code for all four
                               // passes of the PC reduce kernel, which is bound by instruction fetch

// Fills the dynamics block of `s` for the state in s.q / s.v (see the modes above).
template <int MODE>
WBC_DEV void dynamics_phase(WarpSmem& s, const wbc_model& md, int lane, int& status, double* taug_sm,
                            const double* vel_int = nullptr, double* bias_out = nullptr, bool bias_rt = false) {
  // compile-time constants for the templated modes; DYN_PC decides at run time
  const bool GRAV = (MODE == DYN_STEP || MODE == DYN_STEP_JD) || (MODE == DYN_PC && !bias_rt);
  const bool BIAS_ONLY = (MODE == DYN_BIAS) || (MODE == DYN_PC && bias_rt);
  const bool WITH_JD = (MODE == DYN_STEP_JD) || (MODE == DYN_PC && !bias_rt);
  const int leg = lane >> 3, j = lane & 7;
  const bool link = j < 3;
  const int jl = link ? j : 2;
  // base rotation from the (normalised) quaternion
  double qw = s.q[0], qx = s.q[1], qy = s.q[2], qz = s.q[3];
  double nn = qw * qw + qx * qx + qy * qy + qz * qz;
  if (!(nn > 1e-300) || !(nn < 1e300)) { status |= WBC_ST_BADQUAT; nn = 1.0; qw = 1.0; qx = qy = qz = 0.0; }
  double inv = frsqrt(nn);
  qw *= inv; qx *= inv; qy *= inv; qz *= inv;
  M3 R0;
  R0.c0 = mk(1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy + qw * qz), 2 * (qx * qz - qw * qy));
  R0.c1 = mk(2 * (qx * qy - qw * qz), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz + qw * qx));
  R0.c2 = mk(2 * (qx * qz + qw * qy), 2 * (qy * qz - qw * qx), 1 - 2 * (qx * qx + qy * qy));
  const V3 wb = BIAS_ONLY ? ld3(&vel_int[0]) : ld3(&s.v[0]), vb = BIAS_ONLY ? ld3(&vel_int[3]) : ld3(&s.v[3]);
  const V3 grav = ld3(md.gravity);
  V3 aw0 = mk(0, 0, 0);
  V3 av0 = mk(0, 0, 0) - cross(wb, vb);
  if (GRAV) av0 = av0 - grav;

  // ---- leg chain: lane j advances through joints 0..j of its leg and stops at its own link, so only one frame /
  //      twist / acceleration is live per lane (lanes 3..7 shadow the shank lane and contribute zeros)
  M3 R = R0; V3 rho = mk(0, 0, 0);
  V3 vw = wb, vv = vb, aw = aw0, av = av0;
  V3 a = mk(0, 0, 0), b = mk(0, 0, 0), org = mk(0, 0, 0);
  V3 wpar = wb, vorg = vb;      // (WITH_JD) angular velocity of the own joint's parent and velocity of its origin
  // each link lane evaluates sin / cos of its OWN joint once; the chain below fetches joint jj's pair from lane (leg, jj)
  double sn_own, cs_own;
  sincos(s.q[md.v_index[3 * leg + jl] + 1], &sn_own, &cs_own);
#pragma unroll
  for (int jj = 0; jj < 3; ++jj) {
    const double sn = __shfl_sync(WBC_FULL, sn_own, jj, 8), cs = __shfl_sync(WBC_FULL, cs_own, jj, 8);
    if (jj <= jl) {
      const int k = 3 * leg + jj;
      rho = rho + mul(R, ld3(md.joint_xyz[k]));
      const V3 la = ld3(md.joint_axis[k]);
      a = mul(R, la);
      const int vi = md.v_index[k];
      const double thd = BIAS_ONLY ? vel_int[6 + k] : s.v[vi];
      // R <- R * Rot(la, th):  Rot e_m = cs e_m + sn (la x e_m) + (1-cs) la (la . e_m)
      const double oc = 1.0 - cs;
      V3 r0 = mk(cs + oc * la.x * la.x, sn * la.z + oc * la.y * la.x, -sn * la.y + oc * la.z * la.x);
      V3 r1 = mk(-sn * la.z + oc * la.x * la.y, cs + oc * la.y * la.y, sn * la.x + oc * la.z * la.y);
      V3 r2 = mk(sn * la.y + oc * la.x * la.z, -sn * la.x + oc * la.y * la.z, cs + oc * la.z * la.z);
      M3 Rn; Rn.c0 = mul(R, r0); Rn.c1 = mul(R, r1); Rn.c2 = mul(R, r2);
      R = Rn;
      b = cross(rho, a);                     // S = [a; rho x a]
      org = rho;
      if (WITH_JD) { wpar = vw; vorg = vv + cross(vw, rho); }
      // acc += (vel x S) thd ; vel += S thd
      aw = aw + thd * cross(vw, a);
      av = av + thd * (cross(vw, b) + cross(vv, a));
      vw = vw + thd * a; vv = vv + thd * b;
    }
  }
  // ---- own link: spatial inertia about P and inertial force
  const int bi = 1 + 3 * leg + jl;
  SpI Il = link_inertia(md.mass[bi], ld3(md.com[bi]), md.inertia_com[bi], R, rho);
  V3 pn, pf, fn, ff;
  spi_mul(Il, vw, vv, pn, pf);
  spi_mul(Il, aw, av, fn, ff);
  fn = fn + cross(vw, pn) + cross(vv, pf);
  ff = ff + cross(vw, pf);
  if (!link) {
    Il.m = 0; Il.h = mk(0, 0, 0); Il.I.xx = Il.I.yy = Il.I.zz = Il.I.xy = Il.I.xz = Il.I.yz = 0;
    fn = mk(0, 0, 0); ff = mk(0, 0, 0);
  }
  // composite over the sub-chain: lane j gets links j..2 (lanes 3..7 hold zeros)
  SpI Ic = Il, tmp_spi;
  V3 fcn = fn, fcf = ff;
  WBC_SPI_SHFL(__shfl_down_sync, Il, 1, 8); Ic = spi_add(Ic, tmp_spi);
  WBC_SPI_SHFL(__shfl_down_sync, Il, 2, 8); Ic = spi_add(Ic, tmp_spi);
  fcn = fcn + WBC_V3_SHFL(__shfl_down_sync, fn, 1, 8) + WBC_V3_SHFL(__shfl_down_sync, fn, 2, 8);
  fcf = fcf + WBC_V3_SHFL(__shfl_down_sync, ff, 1, 8) + WBC_V3_SHFL(__shfl_down_sync, ff, 2, 8);
  // ---- mass-matrix columns of joint (leg, j): F_j = I^c_j S_j; leg block entries S_i . F_j with the ancestors' screw
  //      axes S_i = [a_i; b_i] fetched from lanes j-1, j-2 of the leg group
  V3 Fn, Ff;
  spi_mul(Ic, a, b, Fn, Ff);
  const V3 a1 = WBC_V3_SHFL(__shfl_up_sync, a, 1, 8), b1 = WBC_V3_SHFL(__shfl_up_sync, b, 1, 8);
  const V3 a2 = WBC_V3_SHFL(__shfl_up_sync, a, 2, 8), b2 = WBC_V3_SHFL(__shfl_up_sync, b, 2, 8);
  if (link && BIAS_ONLY) bias_out[6 + 3 * leg + j] = dot(a, fcn) + dot(b, fcf);
  if (link && !BIAS_ONLY) {
    const int c = 6 + 3 * leg + j;
    s.Mb[c][0] = Fn.x; s.Mb[c][1] = Fn.y; s.Mb[c][2] = Fn.z; s.Mb[c][3] = Ff.x; s.Mb[c][4] = Ff.y; s.Mb[c][5] = Ff.z;
    s.Mleg[leg][sym3(j, j)] = dot(a, Fn) + dot(b, Ff);
    if (j >= 1) s.Mleg[leg][sym3(j - 1, j)] = dot(a1, Fn) + dot(b1, Ff);
    if (j >= 2) s.Mleg[leg][sym3(j - 2, j)] = dot(a2, Fn) + dot(b2, Ff);
    s.hj[3 * leg + j] = dot(a, fcn) + dot(b, fcf);
    if (taug_sm && !BIAS_ONLY) {
      // controller-sign gravity term: -S . [h x g ; m g]
      taug_sm[6 + 3 * leg + j] = -(dot(a, cross(Ic.h, grav)) + Ic.m * dot(b, grav));
    }
  }
  // ---- totals: leg composites sit in lanes j == 0; butterfly over the four legs, then add the base body
  SpI It = Ic; V3 ftn = fcn, ftf = fcf;
  if (j != 0) { It.m = 0; It.h = mk(0, 0, 0); It.I.xx = It.I.yy = It.I.zz = It.I.xy = It.I.xz = It.I.yz = 0; ftn = mk(0, 0, 0); ftf = mk(0, 0, 0); }
#pragma unroll
  for (int o = 8; o <= 16; o <<= 1) {
    SpI cur = It;
    WBC_SPI_SHFL(__shfl_xor_sync, cur, o, 32); It = spi_add(It, tmp_spi);
    V3 tn = WBC_V3_SHFL(__shfl_xor_sync, ftn, o, 32), tf = WBC_V3_SHFL(__shfl_xor_sync, ftf, o, 32);
    ftn = ftn + tn; ftf = ftf + tf;
  }
  // broadcast from lane 0 (lanes with j != 0 hold partial garbage-free zeros + others)
  {
    SpI cur = It;
    WBC_SPI_SHFL(__shfl_sync, cur, 0, 32); It = tmp_spi;
    ftn = WBC_V3_SHFL(__shfl_sync, ftn, 0, 32); ftf = WBC_V3_SHFL(__shfl_sync, ftf, 0, 32);
  }
  {
    SpI Ib = link_inertia(md.mass[0], ld3(md.com[0]), md.inertia_com[0], R0, mk(0, 0, 0));
    V3 bn, bf, gn, gf;
    spi_mul(Ib, wb, vb, bn, bf);
    spi_mul(Ib, aw0, av0, gn, gf);
    gn = gn + cross(wb, bn) + cross(vb, bf);
    gf = gf + cross(wb, bf);
    It = spi_add(It, Ib); ftn = ftn + gn; ftf = ftf + gf;
  }
  if (lane < 6 && BIAS_ONLY) bias_out[lane] = lane < 3 ? comp(ftn, lane) : comp(ftf, lane - 3);
  if (lane < 6 && !BIAS_ONLY) {
    // column c of [[I, skew(h)], [-skew(h), m 1]]
    const int c = lane;
    double col[6];
    if (c < 3) {
      V3 e = mk(c == 0, c == 1, c == 2);
      V3 top = mul(It.I, e), bot = mk(0, 0, 0) - cross(It.h, e);
      col[0] = top.x; col[1] = top.y; col[2] = top.z; col[3] = bot.x; col[4] = bot.y; col[5] = bot.z;
    } else {
      V3 e = mk(c == 3, c == 4, c == 5);
      V3 top = cross(It.h, e), bot = It.m * e;
      col[0] = top.x; col[1] = top.y; col[2] = top.z; col[3] = bot.x; col[4] = bot.y; col[5] = bot.z;
    }
#pragma unroll
    for (int r = 0; r < 6; ++r) s.Mb[c][r] = col[r];
    s.hb[c] = c < 3 ? comp(ftn, c) : comp(ftf, c - 3);
    if (taug_sm && !BIAS_ONLY) {
      V3 tg = cross(It.h, grav);
      taug_sm[c] = c < 3 ? -comp(tg, c) : -It.m * comp(grav, c - 3);
    }
  }
  // ---- foot point: computed on the shank lane (j == 2 holds the full chain), broadcast inside the leg group
  V3 rf = rho + mul(R, ld3(md.foot_xyz[leg]));
  V3 vfoot = vv + cross(vw, rf);
  V3 jdv = av + cross(aw, rf) + cross(vw, vfoot);
  if (GRAV) jdv = jdv + grav;
  rf = WBC_V3_SHFL(__shfl_sync, rf, 2, 8);
  vfoot = WBC_V3_SHFL(__shfl_sync, vfoot, 2, 8);
  jdv = WBC_V3_SHFL(__shfl_sync, jdv, 2, 8);
  if (link && WITH_JD) {
    // d/dt of column j of L: (omega_parent x a_j) x (p_f - o_j) + a_j x (pdot_f - odot_j)   (SURVEY Appendix F)
    const V3 Ldc = cross(cross(wpar, a), rf - org) + cross(a, vfoot - vorg);
    s.Ld[leg][0][j] = Ldc.x; s.Ld[leg][1][j] = Ldc.y; s.Ld[leg][2][j] = Ldc.z;
  }
  if (link && !BIAS_ONLY) {
    const V3 Lc = cross(a, rf - org);
    s.L[leg][0][j] = Lc.x; s.L[leg][1][j] = Lc.y; s.L[leg][2][j] = Lc.z;
    s.rho[leg][j] = comp(rf, j);
    s.Jdv[leg][j] = comp(jdv, j);
    s.vf[leg][j] = comp(vfoot, j);
  }
  // base rotation for the task-space block: stash R0 in task[7..15]
  if (lane == 0 && !BIAS_ONLY) {
    s.task[7] = R0.c0.x; s.task[8] = R0.c0.y; s.task[9] = R0.c0.z;
    s.task[10] = R0.c1.x; s.task[11] = R0.c1.y; s.task[12] = R0.c1.z;
    s.task[13] = R0.c2.x; s.task[14] = R0.c2.y; s.task[15] = R0.c2.z;
  }
  __syncwarp();
}

// The PC / MPTC reduce kernel runs the dynamics four times per instance (state pass + three bias passes of the
// polarisation); they all go through this one out-of-line copy.
#ifdef __CUDACC__
__device__ __noinline__
#else
static
#endif
void dynamics_pc_pass(WarpSmem& s, const wbc_model& md, int lane, int& status, const double* vel_int, double* bias_out, bool bias,
                      double* taug_out = nullptr) {
  dynamics_phase<DYN_PC>(s, md, lane, status, taug_out, vel_int, bias_out, bias);
}

// --------------------------------------------------------------------------- task space
// RollPitchYaw(R) and the rate map N (inverse_dynamics_controller.py:163-166, SURVEY A.7).
struct BodyTask { double rpy[3], rpyd[3]; double N[3][3]; };
WBC_DEV void body_task(const WarpSmem& s, int lane, int& status, BodyTask& t) {
  const double r00 = s.task[7], r10 = s.task[8], r20 = s.task[9], r21 = s.task[12], r22 = s.task[15];
  const double cp = sqrt(r00 * r00 + r10 * r10);
  // spread the three atan2 over three lanes
  const int m = lane % 3;
  double num = m == 0 ? r21 : (m == 1 ? -r20 : r10);
  double den = m == 0 ? r22 : (m == 1 ? cp : r00);
  double ang = atan2(num, den);
  t.rpy[0] = shfl(ang, 0); t.rpy[1] = shfl(ang, 1); t.rpy[2] = shfl(ang, 2);
  double cy, sy;
  const double icp = cp < 1e-6 ? 0.0 : frcp(cp);       // one reciprocal serves cos / sin of the yaw and the rate map below
  if (cp < 1e-6) { status |= WBC_ST_GIMBAL; cy = 1.0; sy = 0.0; }
  else { cy = r00 * icp; sy = r10 * icp; }
  const double sp = -r20;
  t.N[0][0] = cy * cp; t.N[0][1] = -sy; t.N[0][2] = 0.0;
  t.N[1][0] = sy * cp; t.N[1][1] = cy;  t.N[1][2] = 0.0;
  t.N[2][0] = -sp;     t.N[2][1] = 0.0; t.N[2][2] = 1.0;
  // rpyd = N^-1 omega
  const double wx = s.v[0], wy = s.v[1], wz = s.v[2];
  t.rpyd[0] = (cy * wx + sy * wy) * icp;
  t.rpyd[1] = -sy * wx + cy * wy;
  t.rpyd[2] = wz + sp * t.rpyd[0];
}

// ------------------------------------------------------------------------------ phase 2+3
// skew(r)[i][c] with skew(r) = [[0,-rz,ry],[rz,0,-rx],[-ry,rx,0]]
WBC_DEV double skew_ent(V3 r, int i, int c) {
  if (i == c) return 0.0;
  const double m = comp(r, 3 - i - c);
  return ((i + 1) % 3 == c) ? -m : m;
}
WBC_DEV int stance_slot(unsigned cmask, int k) {  // index of foot k among the stance feet, -1 if swing
  return ((cmask >> k) & 1) ? __popc(cmask & ((1u << k) - 1)) : -1;
}
WBC_DEV int stance_foot(unsigned cmask, int slot) {  // foot index of the slot-th stance foot
  int k = 0, cnt = 0;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) { if ((cmask >> kk) & 1) { if (cnt == slot) k = kk; ++cnt; } }
  return k;
}

// Equality constraints of the tau-eliminated QP (SURVEY Appendix C.1 with tau = M_j vd + h_j - L' f substituted):
//   contact rows  Jb_k a_b + L_k a_k = r_k := -Jdv_k - Kd J_k v     (AddContactConstraint, stance feet)
//   base rows     M_bb a_b + sum_k M_bk a_k - sum_stance Jb_k' f_k = -h_b   (base rows of AddDynamicsConstraint)
// The contact rows are solved analytically for the stance-leg joint accelerations through the leg's own 3x3 Jacobian
// block, a_k = L_k^-1 (r_k - Jb_k a_b) (stored as AK), which leaves 6 base rows over the 18 variables
// u = [a_b; per leg: f_k if stance, a_k if swing] (+ delta for CLF). Column `lane` of that 6 x 18 system [B | c0]
// (c0 in lane 31) goes to shared memory for the pivoted Gauss-Jordan below.
WBC_DEV void build_base_system(WarpSmem& s, int lane, unsigned cmask, double kd, int& status) {
  // ---- AK rows: lane 3k+i computes row i of L_k^-1 = (c_{i+1} x c_{i+2}) / det, c_j the columns of L_k
  bool bad = false;
  if (lane < 12) {
    const int k = lane / 3, i = lane % 3;
    if ((cmask >> k) & 1) {
      const int i1 = (i + 1) % 3, i2 = (i + 2) % 3;
      const V3 ci = mk(s.L[k][0][i], s.L[k][1][i], s.L[k][2][i]);
      const V3 c1 = mk(s.L[k][0][i1], s.L[k][1][i1], s.L[k][2][i1]);
      const V3 c2 = mk(s.L[k][0][i2], s.L[k][1][i2], s.L[k][2][i2]);
      const V3 cx = cross(c1, c2);
      const double det = dot(ci, cx);
      // singular stance leg (stretched knee): |det| against the product of the column norms, i.e. the sine-volume of the
      // leg's columns, so that the test does not depend on the leg's size; compared squared (no square root)
      const double vol2 = dot(ci, ci) * dot(c1, c1) * dot(c2, c2);
      bad = !(det * det > RANKDEF_SINVOL * RANKDEF_SINVOL * vol2);
      const V3 li = frcp(bad ? 1.0 : det) * cx;                // row i of L_k^-1
      const V3 rh = ld3(s.rho[k]);
      // Li Jb = [-Li skew(rho) | Li];  li' skew(rho) = (li x rho)'  ->  row of -Li skew(rho) = rho x li
      const V3 lxr = cross(rh, li);
      s.AK[k][i][0] = lxr.x; s.AK[k][i][1] = lxr.y; s.AK[k][i][2] = lxr.z;
      s.AK[k][i][3] = li.x; s.AK[k][i][4] = li.y; s.AK[k][i][5] = li.z;
      const V3 r = mk(-s.Jdv[k][0] - kd * s.vf[k][0], -s.Jdv[k][1] - kd * s.vf[k][1], -s.Jdv[k][2] - kd * s.vf[k][2]);
      s.AK[k][i][6] = dot(li, r);
    }
  }
  if (__any_sync(WBC_FULL, bad)) status |= WBC_ST_RANKDEF;
  __syncwarp();
  const int c = lane;
  double col[AR];
#pragma unroll
  for (int r = 0; r < AR; ++r) col[r] = 0.0;
  if (c < 6 || c == 31) {
    const int cc = c < 6 ? c : 6;                              // AK column: 0-5 -> S_b, 6 -> right-hand side
#pragma unroll
    for (int r = 0; r < 6; ++r) col[r] = c < 6 ? s.Mb[c][r] : -s.hb[r];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (!((cmask >> k) & 1)) continue;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const double ak = s.AK[k][a][cc];
#pragma unroll
        for (int r = 0; r < 6; ++r) col[r] = fma(-s.Mb[6 + 3 * k + a][r], ak, col[r]);
      }
    }
  } else if (c < 18) {
    const int k = (c - 6) / 3, i = (c - 6) % 3;
    if ((cmask >> k) & 1) {
      const V3 rh = ld3(s.rho[k]);                             // -Jb_k' e_i = [skew(rho)[i][0:3] ; -e_i]
#pragma unroll
      for (int r = 0; r < 3; ++r) { col[r] = skew_ent(rh, i, r); col[3 + r] = (r == i) ? -1.0 : 0.0; }
    } else {
#pragma unroll
      for (int r = 0; r < 6; ++r) col[r] = s.Mb[c][r];
    }
  }
#pragma unroll
  for (int r = 0; r < AR; ++r) s.A[r][c] = col[r];
  __syncwarp();
}

// Gauss-Jordan, one pivot per row, pivot column = largest remaining entry of that row.
// Finished pivot columns are left stale (never read again). Returns the bit mask of pivot columns.
// `rowmap` packs, 3 bits per variable, 1 + the pivot row of the variable (0 = free): warp uniform, so the null-space entries
// below index it with shifts instead of a shared-memory table.
WBC_DEV unsigned gauss_jordan(WarpSmem& s, int lane, int m, int n, int& status, unsigned long long& rowmap) {
  unsigned used = 0;
  rowmap = 0ull;
  for (int r = 0; r < m; ++r) {
    const double arc0 = s.A[r][lane];
    const bool eligible = lane < n && !((used >> lane) & 1);
    int pcol;
    const double best = warp_max_lane(eligible ? fabs(arc0) : 0.0, pcol);
    if (!(best > 1e-9)) {            // rows are O(0.01..10) (kg, kg m, lever arms): anything below is round-off
      status |= WBC_ST_RANKDEF;
      continue;
    }
    const double piv = shfl(arc0, pcol);
    const double arc = arc0 * frcp(piv);
    if (lane != pcol) {
      // row r itself is updated with factor A[r][pcol] = piv: arc0 - piv*arc = 0, so overwrite it afterwards
#pragma unroll
      for (int i = 0; i < AR; ++i) {
        if (i < m) {
          const double f = s.A[i][pcol];
          s.A[i][lane] = fma(-f, arc, s.A[i][lane]);
        }
      }
      s.A[r][lane] = arc;
    }
    rowmap |= (unsigned long long)(r + 1) << (3 * pcol);
    used |= 1u << pcol;
    __syncwarp();
  }
  return used;
}

// Entry (var, column `lane`) of Z (free lanes) or of z0 (lane 31).
// Lane 31 holds the right-hand side in the same column index, with the opposite sign convention.
WBC_DEV double zent(const WarpSmem& s, int lane, int var, unsigned long long rowmap) {
  const int r = (int)((rowmap >> (3 * var)) & 7ull) - 1;
  const double a = s.A[r >= 0 ? r : 0][lane];
  return r >= 0 ? (lane == 31 ? a : -a) : (var == lane ? 1.0 : 0.0);
}

// ------------------------------------------------------------------------------ phase 5
// Lower-triangle pairs (i >= k) of an N x N matrix owned by a lane: entries e = lane, lane+32, lane+64 of the N (N + 1) / 2
// (N = active reduced dimension: 12 for ID / PC / MPTC, 13 for CLF; the storage stride stays NF).
struct TriPairs { int i[3], k[3]; };
template <int N> WBC_DEV TriPairs tri_pairs(int lane) {
  TriPairs t;
#pragma unroll
  for (int h = 0; h < 3; ++h) {
    const int e = lane + 32 * h;
    int ii = 0;
#pragma unroll
    for (int c = 1; c < N; ++c) ii += (c * (c + 1) / 2 <= e) ? 1 : 0;
    t.i[h] = e < N * (N + 1) / 2 ? ii : -1;
    t.k[h] = e - ii * (ii + 1) / 2;
  }
  return t;
}

// H = sum_r cw_r Y_r' Y_r (+ identity on padded dims) and e_r = cw_r (y0_r - ct_r) (left in s.y for the solver start-up, which
// needs b = L^-1 Y'e = W'e). The weight is constant inside a row class - body rows 0-5, the three rows of a leg, the torque
// rows - so each class is summed unweighted and scaled once.
template <int N, class SM> WBC_DEV void reduced_hessian(SM& s, int lane, int nf, bool tau_rows, bool extra, const TriPairs& tp) {
  s.y[lane] = s.cw[lane] * (s.Y[lane][NF] - s.ct[lane]);
  const double wb = s.cw[0], wl0 = s.cw[6], wl1 = s.cw[9], wl2 = s.cw[12], wl3 = s.cw[15];
#pragma unroll
  for (int h = 0; h < 3; ++h) {
    const int i = tp.i[h], k = tp.k[h];
    if (i < 0) continue;
    const double* yi = &s.Y[0][i];
    const double* yk = &s.Y[0][k];
    auto term = [&](int r) { return yi[r * YS] * yk[r * YS]; };
    auto leg = [&](int r) { return fma(yi[(r + 2) * YS], yk[(r + 2) * YS], fma(yi[(r + 1) * YS], yk[(r + 1) * YS], term(r))); };
    const double b0 = fma(yi[2 * YS], yk[2 * YS], fma(yi[1 * YS], yk[1 * YS], term(0)));
    const double b1 = fma(yi[5 * YS], yk[5 * YS], fma(yi[4 * YS], yk[4 * YS], term(3)));
    double acc = wb * (b0 + b1);
    acc = fma(wl0, leg(6), acc); acc = fma(wl1, leg(9), acc); acc = fma(wl2, leg(12), acc); acc = fma(wl3, leg(15), acc);
    if (tau_rows) {
      double t0 = 0.0, t1 = 0.0;
#pragma unroll
      for (int r = 18; r < 30; r += 2) { t0 = fma(yi[r * YS], yk[r * YS], t0); t1 = fma(yi[(r + 1) * YS], yk[(r + 1) * YS], t1); }
      acc = fma(s.cw[18], t0 + t1, acc);
    }
    if (extra) acc = fma(s.cw[30] * yi[30 * YS], yk[30 * YS], fma(s.cw[31] * yi[31 * YS], yk[31 * YS], acc));
    if (i >= nf) acc = (i == k) ? 1.0 : 0.0;
    s.H[i][k] = acc;
  }
  __syncwarp();
}

// In-place Cholesky (lower) of s.H, then J = L^-T (J J' = H^-1) and the unconstrained minimiser x.
template <int N, class SM> WBC_DEV void cholesky_factor(SM& s, int lane, int& status, const TriPairs& tp) {
  // Right-looking elimination on the UNSCALED columns, H[i][k] -= H[i][j] H[k][j] / d_j: one shared-memory round trip per
  // step (the pivot reciprocal is the only dependent special-function chain); the columns are scaled by 1 / sqrt(d_j)
  // afterwards, all at once.
  for (int j = 0; j < N; ++j) {
    const double dj = s.H[j][j];
    if (!(dj > 1e-300)) { status |= WBC_ST_NOTPD; }
    const double rd = frcp(dj > 1e-300 ? dj : 1.0);
#pragma unroll
    for (int h = 0; h < 3; ++h) {
      const int i = tp.i[h], k = tp.k[h];
      if (i >= 0 && k > j) s.H[i][k] = fma(-s.H[i][j] * rd, s.H[k][j], s.H[i][k]);
    }
    __syncwarp();
  }
  if (lane < N) { const double dk = s.H[lane][lane]; s.d[lane] = frsqrt(dk > 1e-300 ? dk : 1.0); }   // 1 / L[k][k]
  __syncwarp();
#pragma unroll
  for (int h = 0; h < 3; ++h) {
    const int i = tp.i[h], k = tp.k[h];
    if (i >= 0) s.H[i][k] *= s.d[k];
  }
  __syncwarp();
}
// ------------------------------------------------------------------------------ phase 6
// Inequality i is  ca*y[ra] + cb*y[rb] <= bound  with y = Y w + y0.
struct Ineq { int ra, rb; double ca, cb, bound; };
struct IneqSet {
  unsigned cmask; double mu; int nfric; int nextra; int ntl; const double* effort;
  double extra_bound[2];
};
WBC_DEV Ineq get_ineq(const IneqSet& S, int i) {
  Ineq q; q.ra = q.rb = 0; q.ca = q.cb = 0.0; q.bound = 0.0;
  if (i < S.nfric) {
    // friction pyramid of the (i/4)-th stance foot (inverse_dynamics_controller.py:66-86)
    int sl = i >> 2, t = i & 3, k = 0, cnt = 0;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) { if ((S.cmask >> kk) & 1) { if (cnt == sl) k = kk; ++cnt; } }
    q.ra = 6 + 3 * k + (t >> 1); q.ca = (t & 1) ? -1.0 : 1.0;
    q.rb = 6 + 3 * k + 2; q.cb = -S.mu; q.bound = 0.0;
  } else if (i < S.nfric + S.nextra) {
    const int e = i - S.nfric;
    q.ra = 30 + e; q.ca = 1.0; q.bound = S.extra_bound[e];
  } else {
    const int e = i - S.nfric - S.nextra;   // torque limits: +-tau_k <= effort_k
    const int k = e % 12;
    q.ra = 18 + k; q.ca = e < 12 ? 1.0 : -1.0; q.bound = S.effort[k];
  }
  return q;
}

// Triangular solves with the Cholesky factor L (s.H lower triangle in place, s.d its inverse diagonal): lane k owns
// component k, the finished component is broadcast by shuffle.
template <int N, class SM> WBC_DEV double tri_fwd_lane(const SM& s, int lane, double rhs) {
  // solves L b = rhs (rhs_k in lane k < N); returns b_lane
  const bool row = lane < N;
  const int li = row ? lane : N - 1;
  const double dinv = s.d[li];
  double acc = row ? rhs : 0.0, bl = 0.0;
#pragma unroll
  for (int j = 0; j < N; ++j) {
    const double bj = shfl(acc * dinv, j);
    if (lane == j) bl = bj;
    else if (lane > j) acc = fma(-s.H[li][j], bj, acc);
  }
  return bl;
}
template <int N, class SM> WBC_DEV double tri_bwd_lane(const SM& s, int lane, double rhs) {
  // solves L' x = rhs; returns x_lane
  const bool row = lane < N;
  const int li = row ? lane : N - 1;
  const double dinv = s.d[li];
  double acc = row ? rhs : 0.0, xl = 0.0;
#pragma unroll
  for (int j = N - 1; j >= 0; --j) {
    const double xj = shfl(acc * dinv, j);
    if (lane == j) xl = xj;
    else if (lane < j) acc = fma(-s.H[j][li], xj, acc);
  }
  return xl;
}

// ------------------------------------------------------------------------------ phase 6: Goldfarb-Idnani on W = Y J
// Dual active-set method on  min 1/2 w'Hw + g'w  s.t. the IneqSet (exact optimum; replaces OsqpSolver().Solve,
// inverse_dynamics_controller.py:223), written on W = Y J (32 x N, J J' = H^-1) instead of on J itself. Every quantity an
// iteration needs is a function of W:
//   d = J'n_p = -(ca W[ra] + cb W[rb])             two rows of W (the constraint combines two rows of Y)
//   Y z = W[:, q:] d[q:]                           -> y += t Y z is one FMA per lane; w itself is never formed
//   J <- J Q (Householder on add, Givens on drop)  -> W <- W Q, a row update that keeps all 32 lanes busy
// so the N x N matrix-vector products, the J update and the y = Y w + y0 product of the textbook form (about 265
// shared-memory wavefronts per iteration, the limiter measured on that form) reduce to ~85 wavefronts and half the
// instructions. W is built IN PLACE over Y (W = Y L^-T, forward substitution along each row); the free-part chains enter an
// unrolled sequence at column q (q is warp uniform) with static shared-memory offsets - no masks, no selects.
// On entry s.H holds the Cholesky factor L (lower, in place), s.d its inverse diagonal, s.y the weighted residuals e.
// On exit s.y = Y w + y0 and the multipliers are in s.u / s.act; w is recovered (x = H^-1 Y' C (y - y0), Y read back from
// the hand-over record `Yg`) only when the caller asks for the accelerations.
template <int N, class SM> WBC_DEV int gi_solve_ws(SM& s, int lane, const IneqSet& S, int max_iter, int& status, int& q_out,
                                                  double& minslack, const double* Yg) {
  const int mi = S.nfric + S.nextra + S.ntl;
  const bool row = lane < N;
  const int li = row ? lane : N - 1;
  const Ineq c0 = get_ineq(S, lane < mi ? lane : 0);
  const bool have0 = lane < mi;
  double* Wl = &s.Y[lane][0];                    // row `lane` of W (after the substitution below)
  // ---- W = Y L^-T in place (forward substitution along the row, L broadcast from shared memory). The unconstrained minimiser
  //      needs b = L^-1 g with g = Y'e, i.e. b = W'e: lane k < N sums column k of W against e (left in s.y by
  //      reduced_hessian) - no triangular solve - and then y = y0 - W b with the row still in registers.
  double yl;
  {
    double w[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
      double acc = Wl[k];
#pragma unroll
      for (int j = 0; j < k; ++j) acc = fma(-w[j], s.H[k][j], acc);
      w[k] = acc * s.d[k];
    }
#pragma unroll
    for (int k = 0; k < N; ++k) Wl[k] = w[k];
    __syncwarp();
    {
      const double* wc = &s.Y[0][li];
      double b0 = 0.0, b1 = 0.0;
#pragma unroll
      for (int r = 0; r < 18; r += 2) { b0 = fma(wc[r * YS], s.y[r], b0); b1 = fma(wc[(r + 1) * YS], s.y[r + 1], b1); }
      if (s.cw[18] != 0.0) {
#pragma unroll
        for (int r = 18; r < 30; r += 2) { b0 = fma(wc[r * YS], s.y[r], b0); b1 = fma(wc[(r + 1) * YS], s.y[r + 1], b1); }
      }
      b0 = fma(wc[30 * YS], s.y[30], b0); b1 = fma(wc[31 * YS], s.y[31], b1);
      if (row) s.dm[lane] = b0 + b1;
    }
    __syncwarp();
    double ya = Wl[NF], ya1 = 0.0;
#pragma unroll
    for (int k = 0; k < N; ++k) { if (k & 1) ya1 = fma(-w[k], s.dm[k], ya1); else ya = fma(-w[k], s.dm[k], ya); }
    yl = ya + ya1;
    __syncwarp();                                  // every lane has consumed e (s.y) and b (s.dm)
    s.y[lane] = yl;
  }
  __syncwarp();
  // |J'n_i|^2 = n_i' H^-1 n_i of the constraint(s) this lane watches: invariant under the orthogonal updates of J, so it is
  // formed once from the initial W (no warp reduction per pivot); scale of the "no free direction left" test below
  double ddl0 = 0.0, ddl1 = 0.0;
  {
    const double* wa = &s.Y[c0.ra][0];
    const double* wb = &s.Y[c0.rb][0];
#pragma unroll
    for (int k = 0; k < N; ++k) { const double t = fma(c0.ca, wa[k], c0.cb * wb[k]); ddl0 = fma(t, t, ddl0); }
    if (mi > 32) {
      const Ineq c1 = get_ineq(S, lane + 32 < mi ? lane + 32 : 0);
      const double* va = &s.Y[c1.ra][0];
      const double* vb = &s.Y[c1.rb][0];
#pragma unroll
      for (int k = 0; k < N; ++k) { const double t = fma(c1.ca, va[k], c1.cb * vb[k]); ddl1 = fma(t, t, ddl1); }
    }
  }
  // ---- R^-1 rows start at zero (without VD they overlay L, which is dead from here on: W, b and y are formed)
  double* const Ril = ri_rows(s) + li * NF;      // row `lane` of R^-1 (entries j < lane stay exactly zero)
  {
    double* r0 = ri_rows(s);
    for (int e = lane; e < NF * NF; e += 32) r0[e] = 0.0;
  }
  __syncwarp();
  int q = 0, iters = 0;
  unsigned long long activemask = 0ull;
  double ul = 0.0;                  // lane k < q: multiplier of active slot k
  int actl = 0;                     // constraint id in slot `lane`
  minslack = 0.0;
  // most violated inequality (y lives in shared memory: every lane reads the two rows its constraint combines); the winner
  // is chosen on the high word of the violation (one redux)
  double violl = 0.0;
  auto select = [&](bool& any, int& p_out, int& wl) {
    double viol = 0.0; int who = lane;
    if (have0 && !((activemask >> lane) & 1ull)) {
      const double ta = c0.ca * s.y[c0.ra], tb = c0.cb * s.y[c0.rb];
      const double sl = c0.bound - ta - tb;
      if (sl < -1e-10 * (1.0 + fabs(c0.bound) + fabs(ta) + fabs(tb))) viol = -sl;
    }
    if (mi > 32) {
      const Ineq c1 = get_ineq(S, lane + 32 < mi ? lane + 32 : 0);
      if (lane + 32 < mi && !((activemask >> (lane + 32)) & 1ull)) {
        const double ta = c1.ca * s.y[c1.ra], tb = c1.cb * s.y[c1.rb];
        const double sl = c1.bound - ta - tb;
        if (sl < -1e-10 * (1.0 + fabs(c1.bound) + fabs(ta) + fabs(tb)) && -sl > viol) { viol = -sl; who = lane + 32; }
      }
    }
    violl = viol;
    wl = warp_argmax_hi(viol, any);
    p_out = (mi > 32) ? shfl(who, wl) : wl;
  };
  bool any; int p, wlane;
  select(any, p, wlane);
  for (;;) {
    if (!any) break;
    // descriptor of the pivot: the lane that watches constraint p (< 32) already holds it
    Ineq cp;
    if (p < 32) {
      const int rr = shfl(c0.ra | (c0.rb << 8), p);
      cp.ra = rr & 0xff; cp.rb = rr >> 8;
      cp.ca = shfl(c0.ca, p); cp.cb = shfl(c0.cb, p); cp.bound = shfl(c0.bound, p);
    } else {
      cp = get_ineq(S, p);
    }
    const double nca = -cp.ca, ncb = -cp.cb;
    double up = 0.0;
    bool fail = false;
    const double dd = (p < 32) ? shfl(ddl0, p & 31) : shfl(ddl1, p & 31);   // |J'n_p|^2
    for (;;) {
      if (++iters > max_iter) { status |= WBC_ST_MAXITER; fail = true; break; }
      // ---- d = J'n = -(ca W[ra] + cb W[rb]); lane k owns d_k and publishes it
      const double dself = fma(nca, s.Y[cp.ra][li], ncb * s.Y[cp.rb][li]);
      if (row) s.dm[lane] = dself;
      __syncwarp();
      // free part k >= q: the unrolled chain is entered at k = q
      double zn = 0.0, zn1 = 0.0, wd = 0.0, wd1 = 0.0;    // |d[q:]|^2 and (Y z)_lane = W[lane][q:] . d[q:]
      switch (q) {
#define WBC_ACC(K)                                                                                   \
        case K:                                                                                      \
          if (K < N) {                                                                               \
            const double dk_ = s.dm[K < N ? K : 0];                                                  \
            if (K & 1) { zn1 = fma(dk_, dk_, zn1); wd1 = fma(Wl[K < N ? K : 0], dk_, wd1); }         \
            else { zn = fma(dk_, dk_, zn); wd = fma(Wl[K < N ? K : 0], dk_, wd); }                   \
          }
        WBC_ACC(0) WBC_ACC(1) WBC_ACC(2) WBC_ACC(3) WBC_ACC(4) WBC_ACC(5) WBC_ACC(6) WBC_ACC(7) WBC_ACC(8) WBC_ACC(9) WBC_ACC(10)
        WBC_ACC(11) WBC_ACC(12)
#undef WBC_ACC
        default: break;
      }
      // ---- r = R^-1 d[:q]: lane k owns r_k = R^-1[k][:q] . d[:q] - an FMA chain per lane on its own row of R^-1 (no
      //      shuffle-serialised back substitution); entered at j = q - 1, entries left of the diagonal are zero
      double rk = 0.0, rk1 = 0.0;
      switch (q) {
#define WBC_RI(K)                                                                                    \
        case K + 1:                                                                                  \
          if (K < N) {                                                                               \
            if (K & 1) rk1 = fma(Ril[K < N ? K : 0], s.dm[K < N ? K : 0], rk1);                      \
            else rk = fma(Ril[K < N ? K : 0], s.dm[K < N ? K : 0], rk);                              \
          }
        WBC_RI(12) WBC_RI(11) WBC_RI(10) WBC_RI(9) WBC_RI(8) WBC_RI(7) WBC_RI(6) WBC_RI(5) WBC_RI(4) WBC_RI(3) WBC_RI(2) WBC_RI(1)
        WBC_RI(0)
#undef WBC_RI
        default: break;
      }
      zn += zn1; wd += wd1; rk += rk1;
      const int qc = q < N ? q : N - 1;
      const double dq = s.dm[qc], wq = Wl[qc];
      const double sp = cp.bound - cp.ca * s.y[cp.ra] - cp.cb * s.y[cp.rb];
      // special-function chains of this pivot, issued together so that they overlap the ratio-test reduction:
      // 1 / |d2|^2 (step length), 1 / |d2| (Householder scale and the new diagonal of R^-1), 1 / (v'v / 2)
      const bool zok = zn > 1e-14 * fmax(dd, 1e-300);
      const double zs = zok ? zn : 1.0;
      const double izn = frcp(zs);
      const double rs = frsqrt(zs);                        // 1 / |d2|
      const double nrm = zs * rs;                          // |d2|
      const double alpha = dq > 0.0 ? -nrm : nrm;
      const double hv = fma(-dq, alpha, zs);               // |v|^2 / 2 = zn - dq alpha  (> 0: no cancellation by the sign choice)
      const double ihv = frcp(hv);
      int l;
      const double t1 = warp_min_lane((lane < q && rk > 0.0) ? fmax(ul * frcp(rk), 0.0) + 0.0 : INFINITY, l);
      const double t2 = zok ? -sp * izn : INFINITY;
      const double t = fmin(t1, t2);
      if (!(t < INFINITY)) { status |= WBC_ST_INFEASIBLE; fail = true; break; }
      const bool dual_only = !(t2 < INFINITY);
      if (lane < q) ul -= t * rk;
      up += t;
      __syncwarp();                                        // every lane has read y[ra], y[rb] of this pivot
      if (!dual_only) { yl = fma(t, wd, yl); s.y[lane] = yl; }
      if (!dual_only && t2 <= t1) {
        // ---- full step: add p. The next pivot is selected here, from the y just published: its reductions are independent
        //      of the Householder update below and overlap it.
        activemask |= 1ull << p;
        if (lane == 0 && q < N - 1) s.dm[qc] = dq - alpha;     // the published d becomes the Householder vector v = d[q:] - alpha e_q
        __syncwarp();
        bool nany; int np, nwl;
        select(nany, np, nwl);
        // Householder on d[q:] -> (alpha, 0, ..), W[:, q:] <- W[:, q:] (I - 2 v v'/v'v), v = d[q:] - alpha e_q
        double rqq = dq, irq = dq > 0.0 ? rs : -rs;        // one free column left: R[q][q] = d_q = +-|d2|
        if (q < N - 1) {
          const double sc = (wd - alpha * wq) * ihv;       // 2 (W[lane] . v) / v'v,  W[lane] . v = wd - alpha W[lane][q]
          switch (q) {                                     // W[k] -= sc v_k, k >= q
#define WBC_UPD(K) case K: if (K < N) Wl[K < N ? K : 0] = fma(-sc, s.dm[K < N ? K : 0], Wl[K < N ? K : 0]);
            WBC_UPD(0) WBC_UPD(1) WBC_UPD(2) WBC_UPD(3) WBC_UPD(4) WBC_UPD(5) WBC_UPD(6) WBC_UPD(7) WBC_UPD(8) WBC_UPD(9) WBC_UPD(10)
            WBC_UPD(11) WBC_UPD(12)
#undef WBC_UPD
            default: break;
          }
          rqq = alpha; irq = dq > 0.0 ? -rs : rs;          // 1 / alpha
        }
        // R gains the column (d[:q]; rqq); R^-1 gains the column (-r / rqq; 1 / rqq)
        if (lane < q) { Rent(s, q, lane) = dself; Ril[qc] = -rk * irq; }
        if (lane == q) { Rent(s, q, q) = rqq; Ril[qc] = irq; ul = up; actl = p; }
        ++q;
        any = nany; p = np; wlane = nwl;
        __syncwarp();
        break;
      }
      // ---- drop the blocking constraint l (position in the active list)
      {
        __syncwarp();                                      // every lane is done reading R^-1 and d
        const int dropped = shfl(actl, l);
        activemask &= ~(1ull << dropped);
        // shift the columns right of l one place left: the triangle becomes upper Hessenberg from column l on;
        // R^-1 loses row l (rows below move up one lane)
        for (int jj = l; jj < q - 1; ++jj) { if (lane <= jj + 1) Rent(s, jj, lane) = Rent(s, jj + 1, lane); }
        if (lane <= q) Rent(s, q - 1, lane) = 0.0;
        {
          const bool mv = row && lane >= l && lane < q - 1;
          const double* src = mv ? Ril + NF : Ril;
          for (int j = 0; j < q; ++j) {
            const double tv = src[j];
            __syncwarp();
            if (mv) Ril[j] = tv;
          }
        }
        const double un = __shfl_down_sync(WBC_FULL, ul, 1);
        const int an = __shfl_down_sync(WBC_FULL, actl, 1);
        if (lane >= l && lane < q - 1) { ul = un; actl = an; }
        __syncwarp();
        // Givens rotations restoring the triangle; same rotations on the columns of W and of R^-1
        for (int k = l; k < q - 1; ++k) {
          const double a = Rent(s, k, k), b = Rent(s, k, k + 1);   // R[k][k], R[k+1][k]
          const double r2 = a * a + b * b;
          __syncwarp();
          if (r2 > 0.0) {
            const double irr = frsqrt(r2);
            const double c = a * irr, sn = b * irr;
            if (row && lane >= k) {                        // rows k, k+1 are zero left of column k
              const double r0 = Rent(s, lane, k), r1 = Rent(s, lane, k + 1);
              Rent(s, lane, k) = c * r0 + sn * r1; Rent(s, lane, k + 1) = -sn * r0 + c * r1;
            }
            const double w0 = Wl[k], w1 = Wl[k + 1];
            Wl[k] = c * w0 + sn * w1; Wl[k + 1] = -sn * w0 + c * w1;
            if (lane < q - 1) {                            // only the rows that stay active: an idle row keeps its zeros left of the diagonal
              const double i0 = Ril[k], i1 = Ril[k + 1]; Ril[k] = c * i0 + sn * i1; Ril[k + 1] = -sn * i0 + c * i1;
            }
          }
          __syncwarp();
        }
        --q;
      }
    }
    if (fail) { minslack = -shfl(violl, wlane); break; }
  }
  if (lane < q) { s.u[lane] = ul; s.act[lane] = actl; }
  if (Yg) {
    // x = H^-1 Y' C (y - y0)   (exact: y - y0 = Y x and H = Y' C Y); the original Y is read back from the record
    s.Rp[lane] = s.cw[lane] * (yl - Wl[NF]);              // R is free now: 32 doubles of scratch
    __syncwarp();
    double gk = 0.0;
    const double* ev = &s.Rp[0];
    for (int r = 0; r < YROWS; ++r) gk = fma(Yg[r * YS + li], ev[r], gk);
    const double bl = tri_fwd_lane<N>(s, lane, gk);
    const double xl = tri_bwd_lane<N>(s, lane, bl);
    if (row) s.x[lane] = xl;
    if (lane >= N && lane < NF) s.x[lane] = 0.0;
  }
  __syncwarp();
  q_out = q;
  return iters;
}

// ------------------------------------------------------------------------------ phase 4
// Coefficients of the functional  sum_v rho_v z_v  in the reduced variables (free lanes) or its
// value at z0 (lane 31) are accumulated by the caller with zent(); this stores one result.
WBC_DEV void put_y(WarpSmem& s, int row, int ycol, double val) { if (ycol >= 0) s.Y[row][ycol] = val; }

// Rows 0-29 of Y for all controllers: a_b, per-leg rows (contact force of a stance leg, task acceleration J_s vd of a
// swing leg), joint torques tau = M_j vd + h_j - L' f. Variables: 0-5 a_b, 6+3k+i = f_k,i (stance) or a_k,i (swing).
WBC_DEV void build_common_rows(WarpSmem& s, int lane, int ycol, unsigned cmask, unsigned long long rowmap, double* vdmap = nullptr) {
  double zb[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    zb[i] = zent(s, lane, i, rowmap); put_y(s, i, ycol, zb[i]);
    if (vdmap && ycol >= 0) vdmap[i * YS + ycol] = zb[i];
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const bool stance = (cmask >> k) & 1;
    double zl[3], ak[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) zl[i] = zent(s, lane, 6 + 3 * k + i, rowmap);
    const V3 rh = ld3(s.rho[k]);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double val;
      if (stance) {
        val = zl[i];                                       // the contact force itself
        double a = (lane == 31) ? s.AK[k][i][6] : 0.0;     // a_k = AK[:,6] - AK[:,0:6] a_b
#pragma unroll
        for (int r = 0; r < 6; ++r) a = fma(-s.AK[k][i][r], zb[r], a);
        ak[i] = a;
      } else {
        // row i of J_k = [-skew(rho) | 1 | L_k]
        val = zb[3 + i];
#pragma unroll
        for (int c = 0; c < 3; ++c) val = fma(-skew_ent(rh, i, c), zb[c], val);
#pragma unroll
        for (int c = 0; c < 3; ++c) val = fma(s.L[k][i][c], zl[c], val);
        ak[i] = zl[i];
      }
      put_y(s, 6 + 3 * k + i, ycol, val);
      if (vdmap && ycol >= 0) vdmap[(6 + 3 * k + i) * YS + ycol] = ak[i];
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int kk = 3 * k + j;
      double val = (lane == 31) ? s.hj[kk] : 0.0;
#pragma unroll
      for (int r = 0; r < 6; ++r) val = fma(s.Mb[6 + kk][r], zb[r], val);
#pragma unroll
      for (int i = 0; i < 3; ++i) val = fma(s.Mleg[k][sym3(i < j ? i : j, i < j ? j : i)], ak[i], val);
      if (stance) {
#pragma unroll
        for (int i = 0; i < 3; ++i) val = fma(-s.L[k][i][j], zl[i], val);
      }
      put_y(s, 18 + kk, ycol, val);
    }
  }
}

// ------------------------------------------------------------------------------ PC controller
// pc_controller.py:43-255 / mptc_controller.py:30-57 in the reduced formulation of DESIGN.md 7:
//   X = M^-1 J',  Lambda = (J X)^-1,  s1 = Lambda xd~,  w = v - X s1,
//   g0 = X'(b(v) - C w) - xdd_nom + Jdot w,          (C w by polarisation of the bias b)
//   cost 1/2 |W^1/2 (Lambda (J vd + g0) + Kp x~ + Kd xd~)|^2,   passivity row  s1'(J vd + g0) + xd~'Kp x~ <= 0.
// Meeting point of the warps of a CTA ahead of a pass through the (large, out-of-line) dynamics code: warps that enter it
// together share its instruction fetches. Defined by the kernel translation unit; a no-op elsewhere (host emulator).
#ifndef WBC_CTA_MEET
#define WBC_CTA_MEET(id, threads)
#endif

struct PcSmem {
  double Lam[16][17];                        // J M^-1 J' -> its Cholesky factor -> Lambda (odd row stride: a row per lane is conflict free)
  double s1[16], g0[16], kx[16], xt[16], xdt[16], wt[16];
  double vi[18], w[18], vw[18], vmw[18];     // v (internal order), w, v + w, v - w
  double tg[18];                             // gravity term of the state pass (controller sign): b(v) = h - tg
  double bvw[18], bw[18];                    // bias at v + w and at v - w
  double Sb[6][6];                           // Schur complement of the leg blocks in M -> its Cholesky factor
  double Dinv[4][6];                         // inverses of the 3x3 leg blocks (symmetric, sym3 indexing)
  int rowidx[16];                            // task row r -> row of Y
  double kpxx;                               // xd~' Kp x~
  int sync_all, sync_pc;                     // threads of this CTA that reach the dynamics passes (0: no CTA-level meeting points)
};

WBC_DEV double sym3get(const double* d, int i, int j) { return d[sym3(i < j ? i : j, i < j ? j : i)]; }

// Task-space errors of row `lane` (shared by CLF and PC): base rpy / position rows 0-5, swing-foot rows.
struct TaskRow { bool on; int type, foot, comp; double xt, xdt, xddn, jdv; };
WBC_DEV TaskRow task_row(const WarpSmem& s, const BodyTask& bt, int row, int foot, int comp) {
  const double* tr = s.traj;
  TaskRow t; t.on = true; t.foot = foot; t.comp = comp; t.jdv = 0.0;
  if (row < 3) {
    t.type = 0;
    t.xt = bt.rpy[row] - tr[9 + row];
    t.xdt = s.v[row] - (bt.N[row][0] * tr[12] + bt.N[row][1] * tr[13] + bt.N[row][2] * tr[14]);
    t.xddn = bt.N[row][0] * tr[15] + bt.N[row][1] * tr[16] + bt.N[row][2] * tr[17];
  } else if (row < 6) {
    const int i = row - 3;
    t.type = 1; t.xt = s.q[4 + i] - tr[i]; t.xdt = s.v[3 + i] - tr[3 + i]; t.xddn = tr[6 + i];
  } else {
    t.type = 2;
    t.xt = s.q[4 + comp] + s.rho[foot][comp] - tr[18 + 3 * foot + comp];
    t.xdt = s.vf[foot][comp] - tr[30 + 3 * foot + comp];
    t.xddn = tr[42 + 3 * foot + comp];
    t.jdv = s.Jdv[foot][comp];
  }
  return t;
}

WBC_DEV int swing_foot(unsigned cmask, int slot) { return stance_foot(~cmask & 15u, slot); }

WBC_DEV void pc_precompute(WarpSmem& s, PcSmem& pc, const wbc_model& md, const wbc_params& pr, const BodyTask& bt,
                           int lane, unsigned cmask, int m, int& status, double& Vout, double& errout) {
  double (*X)[17] = reinterpret_cast<double (*)[17]>(&s.Y[0][0]);       // 18 x 16 scratch (row stride 17) in the Y region (Y is built later)
  // 15 x 15 scratch (L^-1) right after X: 18 * 17 + 225 = 531 of the 544 doubles of Y + cw + ct
  static_assert(offsetof(WarpSmem, ct) + sizeof(double) * YROWS - offsetof(WarpSmem, Y) >= (18 * 17 + 225) * sizeof(double), "PC scratch");
  double (*T)[15] = reinterpret_cast<double (*)[15]>(&s.Y[0][0] + 18 * 17);
  const bool on = lane < m;
  const int slot = lane >= 6 ? (lane - 6) / 3 : 0, ri = lane >= 6 ? (lane - 6) % 3 : 0;
  const int rk = (on && lane >= 6) ? swing_foot(cmask, slot) : -1;
  TaskRow t; t.on = false; t.xt = t.xdt = t.xddn = 0.0;
  double kp = 0.0, kd = 0.0, wt = 0.0;
  if (on) {
    t = task_row(s, bt, lane, rk < 0 ? 0 : rk, ri);
    kp = t.type == 0 ? pr.pc_kp_body_rpy : (t.type == 1 ? pr.pc_kp_body_p : pr.pc_kp_foot);
    kd = t.type == 0 ? pr.pc_kd_body_rpy : (t.type == 1 ? pr.pc_kd_body_p : pr.pc_kd_foot);
    wt = t.type == 2 ? pr.pc_w_foot : pr.pc_w_body;
  }
  if (lane < 16) {
    pc.xt[lane] = t.xt; pc.xdt[lane] = t.xdt; pc.wt[lane] = wt; pc.kx[lane] = kp * t.xt + kd * t.xdt;
    pc.rowidx[lane] = lane < 6 ? lane : (rk >= 0 ? 6 + 3 * rk + ri : 0);
  }
  if (lane < 18) pc.vi[lane] = lane < 6 ? s.v[lane] : s.v[md.v_index[lane - 6]];
  const double kpxx = warp_sum(t.xdt * kp * t.xt);
  Vout = 0.5 * warp_sum(kp * t.xt * t.xt);
  errout = warp_sum(t.xt * t.xt);
  if (lane == 0) pc.kpxx = kpxx;
  // ---- inverses of the leg blocks (closed form, SPD 3x3)
  if (lane < 4) {
    const double* d = s.Mleg[lane];
    const double a = d[0], b = d[1], c = d[2], e = d[3], f = d[4], g = d[5];     // [[a b c],[b e f],[c f g]]
    const double c00 = e * g - f * f, c01 = c * f - b * g, c02 = b * f - c * e;
    const double det = a * c00 + b * c01 + c * c02, id = frcp(det);
    pc.Dinv[lane][0] = c00 * id; pc.Dinv[lane][1] = c01 * id; pc.Dinv[lane][2] = c02 * id;
    pc.Dinv[lane][3] = (a * g - c * c) * id; pc.Dinv[lane][4] = (b * c - a * f) * id; pc.Dinv[lane][5] = (a * e - b * b) * id;
  }
  __syncwarp();
  // ---- Schur complement S = Mbb - sum_k Mbk Dk^-1 Mkb, entry (i, j) by lane 6 i + j (lanes 0-31 cover 32 of 36; rest below)
  for (int e = lane; e < 36; e += 32) {
    const int i = e / 6, j = e % 6;
    double acc = s.Mb[j][i];
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) acc = fma(-s.Mb[6 + 3 * k + a][i] * sym3get(pc.Dinv[k], a, b), s.Mb[6 + 3 * k + b][j], acc);
    pc.Sb[i][j] = acc;
  }
  __syncwarp();
  for (int j = 0; j < 6; ++j) {                     // Cholesky of Sb (lower), lanes = rows
    const double dj = pc.Sb[j][j];
    if (!(dj > 1e-300)) status |= WBC_ST_NOTPD;
    const double inv = frsqrt(dj > 1e-300 ? dj : 1.0);
    __syncwarp();
    if (lane < 6 && lane >= j) pc.Sb[lane][j] *= inv;
    __syncwarp();
    if (lane < 6 && lane > j)
      for (int k = j + 1; k <= lane; ++k) pc.Sb[lane][k] = fma(-pc.Sb[lane][j], pc.Sb[k][j], pc.Sb[lane][k]);
    __syncwarp();
  }
  // ---- X = M^-1 J' : lane r solves for task row r
  if (on) {
    double cb[6], cl[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int i = 0; i < 6; ++i) cb[i] = 0.0;
    if (lane < 6) {
#pragma unroll
      for (int i = 0; i < 6; ++i) cb[i] = (i == lane) ? 1.0 : 0.0;
    } else {
      const V3 rh = ld3(s.rho[rk]);
#pragma unroll
      for (int i = 0; i < 3; ++i) { cb[i] = -skew_ent(rh, ri, i); cb[3 + i] = (i == ri) ? 1.0 : 0.0; cl[i] = s.L[rk][ri][i]; }
      double tl[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) tl[a] = sym3get(pc.Dinv[rk], a, 0) * cl[0] + sym3get(pc.Dinv[rk], a, 1) * cl[1] + sym3get(pc.Dinv[rk], a, 2) * cl[2];
#pragma unroll
      for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int a = 0; a < 3; ++a) cb[i] = fma(-s.Mb[6 + 3 * rk + a][i], tl[a], cb[i]);
    }
    double xb[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {                   // L y = cb
      double acc = cb[i];
#pragma unroll
      for (int k = 0; k < 6; ++k) if (k < i) acc = fma(-pc.Sb[i][k], xb[k], acc);
      xb[i] = acc * frcp(pc.Sb[i][i]);
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {                  // L' x = y
      double acc = xb[i];
#pragma unroll
      for (int k = 0; k < 6; ++k) if (k > i) acc = fma(-pc.Sb[k][i], xb[k], acc);
      xb[i] = acc * frcp(pc.Sb[i][i]);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) X[i][lane] = xb[i];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      double c3[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        double acc = (k == rk) ? cl[a] : 0.0;
#pragma unroll
        for (int i = 0; i < 6; ++i) acc = fma(-s.Mb[6 + 3 * k + a][i], xb[i], acc);
        c3[a] = acc;
      }
#pragma unroll
      for (int a = 0; a < 3; ++a)
        X[6 + 3 * k + a][lane] = sym3get(pc.Dinv[k], a, 0) * c3[0] + sym3get(pc.Dinv[k], a, 1) * c3[1] + sym3get(pc.Dinv[k], a, 2) * c3[2];
    }
  }
  __syncwarp();
  // ---- J M^-1 J' (row r by lane r)
  if (on) {
    const V3 rh = rk >= 0 ? ld3(s.rho[rk]) : mk(0, 0, 0);
    for (int c = 0; c < m; ++c) {
      double val;
      if (lane < 6) val = X[lane][c];
      else {
        val = X[3 + ri][c];
#pragma unroll
        for (int i = 0; i < 3; ++i) val = fma(-skew_ent(rh, ri, i), X[i][c], val);
#pragma unroll
        for (int a = 0; a < 3; ++a) val = fma(s.L[rk][ri][a], X[6 + 3 * rk + a][c], val);
      }
      pc.Lam[lane][c] = val;
    }
  }
  __syncwarp();
  // ---- Lambda = (J M^-1 J')^-1 via Cholesky (lanes = rows), T = L^-1 (lane = column), Lambda = T'T
  for (int j = 0; j < m; ++j) {
    const double dj = pc.Lam[j][j];
    if (!(dj > 1e-300)) status |= WBC_ST_RANKDEF;   // J rank deficient (singular swing leg), pc_controller.py:160 would fail too
    const double inv = frsqrt(dj > 1e-300 ? dj : 1.0);
    __syncwarp();
    if (on && lane >= j) pc.Lam[lane][j] *= inv;
    __syncwarp();
    if (on && lane > j)
      for (int k = j + 1; k <= lane; ++k) pc.Lam[lane][k] = fma(-pc.Lam[lane][j], pc.Lam[k][j], pc.Lam[lane][k]);
    __syncwarp();
  }
  if (on) {
    for (int i = 0; i < m; ++i) {
      double acc = (i == lane) ? 1.0 : 0.0;
      for (int k = lane; k < i; ++k) acc = fma(-pc.Lam[i][k], T[k][lane], acc);
      T[i][lane] = (i >= lane) ? acc * frcp(pc.Lam[i][i]) : 0.0;
    }
  }
  __syncwarp();
  if (on) {
    for (int c = 0; c < m; ++c) {
      double acc = 0.0;
      for (int k = (lane > c ? lane : c); k < m; ++k) acc = fma(T[k][lane], T[k][c], acc);
      pc.Lam[lane][c] = acc;                        // every lane writes its own row; reads are from T only
    }
  }
  __syncwarp();
  // ---- s1 = Lambda xd~,  w = v - X s1
  double s1 = 0.0;
  if (on) for (int c = 0; c < m; ++c) s1 = fma(pc.Lam[lane][c], pc.xdt[c], s1);
  if (lane < 16) pc.s1[lane] = s1;
  Vout += 0.5 * warp_sum(t.xdt * s1);
  __syncwarp();
  if (lane < 18) {
    double acc = pc.vi[lane];
    for (int c = 0; c < m; ++c) acc = fma(-X[lane][c], pc.s1[c], acc);
    pc.w[lane] = acc; pc.vw[lane] = pc.vi[lane] + acc; pc.vmw[lane] = pc.vi[lane] - acc;
  }
  __syncwarp();
  // ---- C w by polarisation of the bias (a homogeneous quadratic form b(v) = B(v, v)): C w = B(v, w) = 1/4 (b(v + w) - b(v - w))
  //      (CalcCoriolisMatrix, basic_controller.py:117-132) - two bias-only passes; b(v) itself is the state pass' h minus its
  //      gravity term. The passes run through ONE copy of the dynamics code (a rolled loop): the PC reduce kernel is bound by
  //      instruction fetch, inlined copies cost more in instruction-cache misses than the loop does in branches.
  int st2 = 0;
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    const double* vin = pass == 0 ? pc.vw : pc.vmw;
    double* bout = pass == 0 ? pc.bvw : pc.bw;
    WBC_CTA_MEET(2, pc.sync_pc);
    dynamics_pc_pass(s, md, lane, st2, vin, bout, true);
  }
  // ---- g0 = X'(b(v) - C w) - xdd_nom + Jdot w
  if (on) {
    double acc = -t.xddn;
    for (int i = 0; i < 18; ++i) {
      const double bvi = (i < 6 ? s.hb[i] : s.hj[i - 6]) - pc.tg[i];
      acc = fma(X[i][lane], bvi - 0.25 * (pc.bvw[i] - pc.bw[i]), acc);
    }
    if (rk >= 0) {
      // Jdot row: [-skew(pdot_f - pdot_b) | 0 | Ld]   (CalcFrameJacobianDot, basic_controller.py:198-220)
      const V3 dv = mk(s.vf[rk][0] - s.v[3], s.vf[rk][1] - s.v[4], s.vf[rk][2] - s.v[5]);
#pragma unroll
      for (int i = 0; i < 3; ++i) acc = fma(-skew_ent(dv, ri, i), pc.w[i], acc);
#pragma unroll
      for (int a = 0; a < 3; ++a) acc = fma(s.Ld[rk][ri][a], pc.w[6 + 3 * rk + a], acc);
    }
    pc.g0[lane] = acc;
  }
  __syncwarp();
}

// Replaces the task rows of Y by the weighted task-force rows and adds the passivity row 30 (column `ycol` per lane).
WBC_DEV void pc_rows(WarpSmem& s, const PcSmem& pc, int lane, int ycol, int m) {
  if (ycol < 0) return;
  double yt[15];
#pragma unroll
  for (int r = 0; r < 15; ++r) yt[r] = (r < m) ? s.Y[pc.rowidx[r]][ycol] + (lane == 31 ? pc.g0[r] : 0.0) : 0.0;
  double row30 = (lane == 31) ? pc.kpxx : 0.0;
#pragma unroll
  for (int r = 0; r < 15; ++r) if (r < m) row30 = fma(pc.s1[r], yt[r], row30);
  s.Y[30][ycol] = row30;
#pragma unroll 1
  for (int r = 0; r < m; ++r) {
    {
      double acc = (lane == 31) ? pc.kx[r] : 0.0;
#pragma unroll
      for (int c = 0; c < 15; ++c) if (c < m) acc = fma(pc.Lam[r][c], yt[c], acc);
      s.Y[pc.rowidx[r]][ycol] = sqrt(pc.wt[r]) * acc;
    }
  }
}

// ------------------------------------------------------------------------------ the step
// One control step of instance `inst` (DoSetControlTorques -> ControlLaw,
// basic_controller.py:286-320). KIND selects the cost / extra rows.
// One instance's input rows inside the CTA-level staging block of the reduce kernels.
struct StagedInputs { const double* q; const double* v; const double* traj; const uint8_t* contact; };

// What the solve half needs from the reduce half besides [Y | cw | ct]: registers in the fused kernels, the `misc` words of
// the hand-over record in the split path.
struct StepCarry {
  int status; unsigned cmask; int nf, nextra; bool ok, pc_ok;
  double extra_bound, err, Vl, PFl, csum, Vpc;
};

// Phases 0-4 + cost rows: state -> reduced problem [Y | cw | ct] in s (and the joint-acceleration maps in `vdmap`, if given).
template <int KIND>
WBC_DEV void reduce_instance(WarpSmem& s, const wbc_model& md, const wbc_params& pr, const Derived& dv, const StepArgs& a,
                             long long inst, int lane, StepCarry& c, PcSmem* pcs = nullptr, double* vdmap = nullptr,
                             const StagedInputs* in = nullptr) {
  int status = 0;
  unsigned cmask = 0;
  // ---- phase 0: input rows into the warp's block - from the CTA-level staging block where the kernel could bulk-copy the
  //      array (always v and traj, whose rows are multiples of 16 bytes; q and contact only for 4-instance CTAs), with
  //      coalesced per-lane loads otherwise (the trajectory row by cp.async, awaited after phase 1)
  if (in && in->q) { for (int i = lane; i < WBC_NQ; i += 32) s.q[i] = in->q[i]; }
  else { for (int i = lane; i < WBC_NQ; i += 32) s.q[i] = a.q[inst * WBC_NQ + i]; }
  if (in && in->v) { for (int i = lane; i < WBC_NV; i += 32) s.v[i] = in->v[i]; }
  else { for (int i = lane; i < WBC_NV; i += 32) s.v[i] = a.v[inst * WBC_NV + i]; }
  if (in && in->traj) { for (int i = lane; i < WBC_NTRAJ; i += 32) s.traj[i] = in->traj[i]; }
  else { for (int i = lane; i < WBC_NTRAJ; i += 32) async_copy8(&s.traj[i], a.traj + inst * WBC_NTRAJ + i); }
  {
    const uint8_t* cptr = (in && in->contact) ? in->contact : a.contact + inst * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) cmask |= (cptr[k] ? 1u : 0u) << k;
  }
  const int nc = __popc(cmask);
  __syncwarp();
  // ---- phase 1
  if (KIND == WBC_CTRL_PC) {
    WBC_CTA_MEET(1, pcs->sync_all);
    dynamics_pc_pass(s, md, lane, status, nullptr, nullptr, false, pcs->tg);
  } else dynamics_phase<DYN_STEP>(s, md, lane, status, nullptr);
  async_wait_all();
  __syncwarp();
  {
    // every input value this instance reads (q 19, v 18, traj 54) is in the warp's block now: one vote flags a NaN / inf.
    // The instance runs on as before and its outputs are zeroed in phase 7 like any other failure.
    bool nonfin = lane < WBC_NQ && !isfinite(s.q[lane]);
    nonfin |= lane < WBC_NV && !isfinite(s.v[lane]);
    nonfin |= !isfinite(s.traj[lane]) || (lane < WBC_NTRAJ - 32 && !isfinite(s.traj[32 + lane]));
    if (__any_sync(WBC_FULL, nonfin)) status |= WBC_ST_NONFINITE;
  }
  BodyTask bt;
  body_task(s, lane, status, bt);
  // ---- PC: operational-space quantities (uses the A region as scratch, so it runs before the equalities are built)
  const int mtask = 6 + 3 * (4 - nc);
  double Vpc = 0.0, errpc = 0.0;
  bool pc_ok = true;
  if (KIND == WBC_CTRL_PC) {
    if (nc == 0) { status |= WBC_ST_UNSUPPORTED; pc_ok = false; }   // reference PC raises on full flight (SURVEY E.5c)
    else pc_precompute(s, *pcs, md, pr, bt, lane, cmask, mtask, status, Vpc, errpc);
  }
  // ---- phases 2,3
  const int ndelta = (KIND == WBC_CTRL_CLF) ? 1 : 0;
  const int n = 18 + ndelta, m = 6;
  build_base_system(s, lane, cmask, pr.contact_damping, status);
  unsigned long long rowmap;
  const unsigned used = gauss_jordan(s, lane, m, n, status, rowmap);
  const unsigned freemask = ~used & ((n >= 32) ? 0xffffffffu : ((1u << n) - 1u));
  const int nf = __popc(freemask);
  const bool isfree = (freemask >> lane) & 1u;
  const int widx = __popc(freemask & ((1u << lane) - 1u));
  const int ycol = lane == 31 ? NF : (isfree ? widx : -1);
  constexpr int NA = (KIND == WBC_CTRL_CLF) ? NF : NF - 1;   // active reduced dimension: the loops of phases 5-6 run to NA
  const bool ok = nf <= NA && pc_ok;
  double err = 0.0;
  int nextra = 0;
  double extra_bound = 0.0, Vl = 0.0, PFl = 0.0, csum = 0.0;
  if (ok) {
    // ---- phase 4
    {
      double* y0 = &s.Y[0][0];                                       // 16-byte aligned: pairs go out as one 128-bit store
#pragma unroll
      for (int e = lane; e < YROWS * YS / 2; e += 32) { y0[2 * e] = 0.0; y0[2 * e + 1] = 0.0; }
    }
    s.cw[lane] = 0.0; s.ct[lane] = 0.0;
    __syncwarp();
    build_common_rows(s, lane, ycol, cmask, rowmap, vdmap);
    // ---- costs
    const double* tr = s.traj;
    if (KIND == WBC_CTRL_ID) {
      // inverse_dynamics_controller.py:187-197 task-space PD
      double rdd[3], add[3];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        rdd[i] = tr[15 + i] - pr.id_kp_body_rpy * (bt.rpy[i] - tr[9 + i]) - pr.id_kd_body_rpy * (bt.rpyd[i] - tr[12 + i]);
        add[i] = tr[6 + i] - pr.id_kp_body_p * (s.q[4 + i] - tr[i]) - pr.id_kd_body_p * (s.v[3 + i] - tr[3 + i]);
        err += (bt.rpy[i] - tr[9 + i]) * (bt.rpy[i] - tr[9 + i]) + (s.q[4 + i] - tr[i]) * (s.q[4 + i] - tr[i]);
      }
      if (lane < 3) { s.cw[lane] = pr.id_w_body; s.ct[lane] = bt.N[lane][0] * rdd[0] + bt.N[lane][1] * rdd[1] + bt.N[lane][2] * rdd[2]; }
      else if (lane < 6) { s.cw[lane] = pr.id_w_body; s.ct[lane] = add[lane - 3]; }
      else if (lane < 18) {
        const int k = (lane - 6) / 3, i = (lane - 6) % 3;
        if ((cmask >> k) & 1) { s.cw[lane] = pr.reg_f; s.ct[lane] = 0.0; }
        else {
          const double pfoot = s.q[4 + i] + s.rho[k][i];
          const double as = tr[42 + 3 * k + i] - pr.id_kp_foot * (pfoot - tr[18 + 3 * k + i]) - pr.id_kd_foot * (s.vf[k][i] - tr[30 + 3 * k + i]);
          s.cw[lane] = pr.id_w_foot; s.ct[lane] = as - s.Jdv[k][i];
        }
      } else if (lane < 30) { s.cw[lane] = pr.reg_tau; s.ct[lane] = 0.0; }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (!((cmask >> k) & 1)) {
#pragma unroll
          for (int i = 0; i < 3; ++i) { const double e = s.q[4 + i] + s.rho[k][i] - tr[18 + 3 * k + i]; err += e * e; }
        }
    }
    if (KIND == WBC_CTRL_CLF) {
      // clf_controller.py:137-209. Lane r < 18 owns task row r (base rows 0-5, swing-foot rows 6-17).
      double xt = 0.0, xdt = 0.0, xddn = 0.0, jdv = 0.0, kap = 0.0;
      bool taskrow = false;
      int type = 0;
      if (lane < 3) {
        taskrow = true; type = 0;
        xt = bt.rpy[lane] - tr[9 + lane];
        xdt = s.v[lane] - (bt.N[lane][0] * tr[12] + bt.N[lane][1] * tr[13] + bt.N[lane][2] * tr[14]);
        xddn = bt.N[lane][0] * tr[15] + bt.N[lane][1] * tr[16] + bt.N[lane][2] * tr[17];
      } else if (lane < 6) {
        const int i = lane - 3;
        taskrow = true; type = 1;
        xt = s.q[4 + i] - tr[i]; xdt = s.v[3 + i] - tr[3 + i]; xddn = tr[6 + i];
      } else if (lane < 18) {
        const int k = (lane - 6) / 3, i = (lane - 6) % 3;
        if (!((cmask >> k) & 1)) {
          taskrow = true; type = 2;
          xt = s.q[4 + i] + s.rho[k][i] - tr[18 + 3 * k + i]; xdt = s.vf[k][i] - tr[30 + 3 * k + i]; xddn = tr[42 + 3 * k + i];
          jdv = s.Jdv[k][i];
        } else { s.cw[lane] = pr.reg_f; s.ct[lane] = 0.0; }
      } else if (lane < 30) { s.cw[lane] = pr.reg_tau; s.ct[lane] = 0.0; }
      if (taskrow) {
        const double p11 = dv.clf_p[type][0], p12 = dv.clf_p[type][1], p22 = dv.clf_p[type][2];
        kap = p12 * xt + p22 * xdt;                      // (G' P eta)_r
        // 1/2 (y + Jdv - xdd_des)^2 + 2 kap y  ==  1/2 (y - t)^2 + const,  t = xdd_des - Jdv - 2 kap
        s.cw[lane] = 1.0;
        s.ct[lane] = xddn - kap / pr.clf_r - jdv - 2.0 * kap;
        Vl = p11 * xt * xt + 2.0 * p12 * xt * xdt + p22 * xdt * xdt;
        PFl = (p11 * xt + p12 * xdt) * xdt;
        csum = kap * (jdv - xddn);
        err = xt * xt;
      }
      s.y[lane] = kap;                                   // scratch: kappa per task row (0 elsewhere)
      Vl = warp_sum(Vl); PFl = warp_sum(PFl); csum = warp_sum(csum); err = warp_sum(err);
      __syncwarp();
      // extra rows: 30 = 2 kappa' J vd - delta  (Vdot constraint, :27-45), 31 = delta
      const int cdel = 18;                               // delta's column: never a pivot (all-zero column of A)
      if (ycol >= 0) {
        double acc = 0.0;
        for (int r = 0; r < 18; ++r) acc = fma(2.0 * s.y[r], s.Y[r][ycol], acc);
        const double isdel = (lane == cdel) ? 1.0 : 0.0;
        s.Y[30][ycol] = acc - isdel;
        s.Y[31][ycol] = isdel;
      }
      if (lane == 31) { s.cw[31] = 2.0 * pr.clf_w_delta; s.ct[31] = 0.0; }   // AddCost(w delta'delta) -> Q = 2w
      nextra = 1;
      extra_bound = -dv.clf_gamma[nc < 4 ? 1 : 0] * Vl - 2.0 * PFl - 2.0 * csum;
    }
    if (KIND == WBC_CTRL_PC) {
      pc_rows(s, *pcs, lane, ycol, mtask);
      if (lane < 6 || (lane < 18 && !((cmask >> ((lane - 6) / 3)) & 1))) { s.cw[lane] = 1.0; s.ct[lane] = 0.0; }
      else if (lane < 18) { s.cw[lane] = pr.reg_f; s.ct[lane] = 0.0; }
      else if (lane < 30) { s.cw[lane] = pr.reg_tau; s.ct[lane] = 0.0; }
      nextra = (a.kind == WBC_CTRL_PC) ? 1 : 0;   // MPTC (mptc_controller.py:125-310): same cost, no passivity row
      extra_bound = 0.0;
      err = errpc;
    }
    __syncwarp();
  }
  c.status = status; c.cmask = cmask; c.nf = nf; c.nextra = nextra; c.ok = ok; c.pc_ok = pc_ok;
  c.extra_bound = extra_bound; c.err = err; c.Vl = Vl; c.PFl = PFl; c.csum = csum; c.Vpc = Vpc;
}

// Phases 5-7: reduced problem in s ([Y | cw | ct], bulk-copied from the hand-over record) -> torques, metrics, status.
// `vdmap` are the 18 acceleration rows the reduce half stored (null unless vd is requested), `yrec` the record itself.
template <int KIND, class SM>
WBC_DEV void solve_instance(SM& s, const wbc_model& md, const wbc_params& pr, const StepArgs& a, long long inst, int lane,
                            const StepCarry& c, const double* vdmap = nullptr, const double* yrec = nullptr) {
  constexpr int NA = (KIND == WBC_CTRL_CLF) ? NF : NF - 1;
  int status = c.status;
  const unsigned cmask = c.cmask;
  const int nc = __popc(cmask), nf = c.nf, nextra = c.nextra;
  const double extra_bound = c.extra_bound, err = c.err, Vl = c.Vl, PFl = c.PFl, csum = c.csum, Vpc = c.Vpc;
  if (c.ok) {
    // ---- phase 5
    const TriPairs tp = tri_pairs<NA>(lane);
    reduced_hessian<NA>(s, lane, nf, pr.reg_tau != 0.0, KIND != WBC_CTRL_ID, tp);
    cholesky_factor<NA>(s, lane, status, tp);
    // ---- phase 6
    IneqSet S;
    S.cmask = cmask; S.mu = pr.mu; S.nfric = 4 * nc; S.nextra = nextra; S.ntl = pr.torque_limits ? 24 : 0;
    S.effort = md.effort; S.extra_bound[0] = extra_bound; S.extra_bound[1] = 0.0;
    int qact = 0; double minslack = 0.0;
    int iters = 0;
    if (!(status & WBC_ST_NOTPD)) {
      iters = gi_solve_ws<NA>(s, lane, S, pr.max_iter, status, qact, minslack, (SM::kVd && a.vd != nullptr) ? yrec : nullptr);
    }
    // ---- phase 7: y = Y x + y0 is current in s.y. Any status bit (unfinished active-set iterate, substituted orientation,
    //      rank-deficient problem) zeroes the torques: nothing that is not the optimum of the reference QP leaves as tau
    //      (the reference asserts there, inverse_dynamics_controller.py:224); status is warp uniform. A non-finite tau, f or vd
    //      (a finite state whose dynamics overflow) is flagged here, so it cannot leave either.
    const bool want_vd = SM::kVd && a.vd && lane < 18;
    double vdv = 0.0;
    if (want_vd) {
      // accelerations as affine maps of w (rows stored by the reduce half: a_b, then the joints in internal order)
      const double* mrow = vdmap + lane * YS;
      vdv = mrow[NF];
      for (int w = 0; w < nf; ++w) vdv = fma(mrow[w], s.x[w], vdv);
    }
    const bool nonfin = (lane < 12 && !(isfinite(s.y[18 + lane]) && isfinite(s.y[6 + lane]))) || !isfinite(vdv);
    if (__any_sync(WBC_FULL, nonfin)) status |= WBC_ST_NONFINITE;
    const bool failed = status != 0;
    const double res = minslack < 0.0 ? -minslack : 0.0;
    if (lane < 12) {
      a.tau[inst * WBC_NU + md.act_index[lane]] = failed ? 0.0 : s.y[18 + lane];
      if (a.f) a.f[inst * 12 + lane] = (!failed && ((cmask >> (lane / 3)) & 1)) ? s.y[6 + lane] : 0.0;
    }
    if (want_vd) a.vd[inst * WBC_NV + (lane < 6 ? lane : md.v_index[lane - 6])] = failed ? 0.0 : vdv;
    if (a.lam) {
      // multipliers of the active rows in the fixed layout of wbc.h (R is dead after the solve: scratch for the row)
      double* lrow = &s.Rp[0];
      __syncwarp();
      lrow[lane] = 0.0;
      if (lane < WBC_NLAM - 32) lrow[32 + lane] = 0.0;
      __syncwarp();
      if (!failed && lane < qact) {
        const int id = s.act[lane];
        int slot;
        if (id < S.nfric) slot = 4 * stance_foot(cmask, id >> 2) + (id & 3);
        else if (id < S.nfric + S.nextra) slot = 16 + (id - S.nfric);
        else { const int e = id - S.nfric - S.nextra; slot = 18 + md.act_index[e % 12] + (e < 12 ? 0 : 12); }
        lrow[slot] = s.u[lane];
      }
      __syncwarp();
      a.lam[inst * WBC_NLAM + lane] = lrow[lane];
      if (lane < WBC_NLAM - 32) a.lam[inst * WBC_NLAM + 32 + lane] = lrow[32 + lane];
    }
    // reference objective 1/2 x'P0x + q0'x (constants dropped, E.5b): rows with a reference cost
    double obj = 0.0;
    {
      const bool refrow = lane < 6 || (lane < 18 && !((cmask >> ((lane - 6) / 3)) & 1)) || (KIND == WBC_CTRL_CLF && lane == 31);
      if (refrow) { const double yy = s.y[lane], t = s.ct[lane], w = s.cw[lane]; obj = 0.5 * w * yy * yy - w * t * yy; }
    }
    obj = warp_sum(obj);
    if (lane == 0) {
      double* mt = a.metrics + inst * WBC_NMETRIC;
      double delta = 0.0;
      if (KIND == WBC_CTRL_ID) { mt[0] = 0.0; mt[1] = err; mt[2] = res; mt[3] = 0.0; }
      if (KIND == WBC_CTRL_CLF) {
        // V, err, (res unused by the reference CLF), Vdot = 2 eta'PF eta + 2 eta'PG (J vd + Jdv - xdd_nom)  (:230-232)
        delta = s.y[31];
        mt[0] = Vl; mt[1] = err; mt[2] = res; mt[3] = 2.0 * PFl + s.y[30] + delta + 2.0 * csum;
      }
      if (KIND == WBC_CTRL_PC) {
        // V = 1/2 xd~'Lambda xd~ + 1/2 x~'Kp x~, Vdot = value of the passivity row  (pc_controller.py:244-253)
        mt[0] = Vpc; mt[1] = err; mt[2] = res; mt[3] = s.y[30];
      }
      if (a.qp_info) { double* qi = a.qp_info + inst * 4; qi[0] = obj; qi[1] = res; qi[2] = delta; qi[3] = (double)iters; }
    }
  } else {
    if (c.pc_ok) status |= WBC_ST_RANKDEF;
    if (lane < 12) { a.tau[inst * WBC_NU + lane] = 0.0; if (a.f) a.f[inst * 12 + lane] = 0.0; }
    if (a.vd && lane < 18) a.vd[inst * WBC_NV + lane] = 0.0;
    if (a.lam) { a.lam[inst * WBC_NLAM + lane] = 0.0; if (lane < WBC_NLAM - 32) a.lam[inst * WBC_NLAM + 32 + lane] = 0.0; }
    if (lane < 4) a.metrics[inst * WBC_NMETRIC + lane] = 0.0;
    if (a.qp_info && lane < 4) a.qp_info[inst * 4 + lane] = 0.0;
  }
  if (lane == 0) a.status[inst] = status;
  __syncwarp();
}


// ---------------------------------------------------------------- dynamics parity entry
// CalcDynamics + CalcFramePositionQuantities x4 for instance `inst`, written in Drake order.
WBC_DEV void dynamics_instance(WarpSmem& s, const wbc_model& md, const double* q, const double* v, const DynOut& o,
                               long long inst, int lane) {
  int status = 0;
  for (int i = lane; i < WBC_NQ; i += 32) s.q[i] = q[inst * WBC_NQ + i];
  for (int i = lane; i < WBC_NV; i += 32) s.v[i] = v[inst * WBC_NV + i];
  __syncwarp();
  double* taug = &s.A[0][0];  // scratch: 18 doubles
  dynamics_phase<DYN_PARITY>(s, md, lane, status, taug);
  // internal -> Drake index
  auto didx = [&](int c) { return c < 6 ? c : md.v_index[c - 6]; };
  if (o.M) {
    double* M = o.M + inst * 324;
    for (int e = lane; e < 324; e += 32) {
      const int r = e / 18, c = e % 18;
      double val;
      if (r < 6) val = s.Mb[c][r];
      else if (c < 6) val = s.Mb[r][c];
      else if ((r - 6) / 3 == (c - 6) / 3) { const int i = (r - 6) % 3, j = (c - 6) % 3; val = s.Mleg[(r - 6) / 3][sym3(i < j ? i : j, i < j ? j : i)]; }
      else val = 0.0;
      M[didx(r) * 18 + didx(c)] = val;
    }
  }
  if (lane < 18) {
    const double cv = lane < 6 ? s.hb[lane] : s.hj[lane - 6];
    if (o.Cv) o.Cv[inst * 18 + didx(lane)] = cv;
    if (o.taug) o.taug[inst * 18 + didx(lane)] = taug[lane];
  }
  if (o.Jfeet) {
    double* J = o.Jfeet + inst * 216;
    for (int e = lane; e < 216; e += 32) {
      const int k = e / 54, i = (e % 54) / 18, c = e % 18;
      const V3 rh = ld3(s.rho[k]);
      double val = 0.0;
      if (c < 3) val = -skew_ent(rh, i, c);
      else if (c < 6) val = (c - 3 == i) ? 1.0 : 0.0;
      else if ((c - 6) / 3 == k) val = s.L[k][i][(c - 6) % 3];
      J[k * 54 + i * 18 + didx(c)] = val;
    }
  }
  if (lane < 12) {
    if (o.Jdv) o.Jdv[inst * 12 + lane] = s.Jdv[lane / 3][lane % 3];
    if (o.pfeet) o.pfeet[inst * 12 + lane] = s.q[4 + lane % 3] + s.rho[lane / 3][lane % 3];
  }
  __syncwarp();
}

// ---------------------------------------------------------------- Coriolis parity entry
// CalcCoriolisMatrix (basic_controller.py:117-132): C = 1/2 d(Cv)/dv, exact by polarisation since Cv is a homogeneous
// quadratic form in v: C e_j = 1/2 (b(v + e_j) - b(v) - b(e_j)). CalcFrameJacobianDot x4 (:198-220): analytic Jdot.
WBC_DEV void coriolis_instance(WarpSmem& s, PcSmem& pc, const wbc_model& md, const double* q, const double* v, double* Cout,
                               double* Jdout, long long inst, int lane) {
  int status = 0;
  for (int i = lane; i < WBC_NQ; i += 32) s.q[i] = q[inst * WBC_NQ + i];
  for (int i = lane; i < WBC_NV; i += 32) s.v[i] = v[inst * WBC_NV + i];
  __syncwarp();
  dynamics_phase<DYN_STEP_JD>(s, md, lane, status, nullptr);
  auto didx = [&](int c) { return c < 6 ? c : md.v_index[c - 6]; };
  if (lane < 18) pc.vi[lane] = lane < 6 ? s.v[lane] : s.v[md.v_index[lane - 6]];
  __syncwarp();
  dynamics_phase<DYN_BIAS>(s, md, lane, status, nullptr, pc.vi, pc.tg);     // (tg doubles as the b(v) scratch of this debug entry)
  if (Cout) {
    for (int j = 0; j < 18; ++j) {
      if (lane < 18) { pc.w[lane] = (lane == j) ? 1.0 : 0.0; pc.vw[lane] = pc.vi[lane] + ((lane == j) ? 1.0 : 0.0); }
      __syncwarp();
      dynamics_phase<DYN_BIAS>(s, md, lane, status, nullptr, pc.vw, pc.bvw);
      dynamics_phase<DYN_BIAS>(s, md, lane, status, nullptr, pc.w, pc.bw);
      if (lane < 18) Cout[inst * 324 + didx(lane) * 18 + didx(j)] = 0.5 * (pc.bvw[lane] - pc.tg[lane] - pc.bw[lane]);
      __syncwarp();
    }
  }
  if (Jdout) {
    double* J = Jdout + inst * 216;
    for (int e = lane; e < 216; e += 32) {
      const int k = e / 54, i = (e % 54) / 18, c = e % 18;
      const V3 dv = mk(s.vf[k][0] - s.v[3], s.vf[k][1] - s.v[4], s.vf[k][2] - s.v[5]);
      double val = 0.0;
      if (c < 3) val = -skew_ent(dv, i, c);
      else if (c >= 6 && (c - 6) / 3 == k) val = s.Ld[k][i][(c - 6) % 3];
      J[k * 54 + i * 18 + didx(c)] = val;
    }
  }
  __syncwarp();
}

// BasicController.ControlLaw (basic_controller.py:322-352): u = S tau, tau = -Kp (q - q_nom) - Kd v on the joint rows,
// clipped to +-clip. One thread per (instance, joint k in internal order).
WBC_DEV void pd_element(const wbc_model& md, const wbc_params& pr, const double* q, const double* v, double* tau,
                        long long inst, int k) {
  const int vi = md.v_index[k];
  const double e = q[inst * WBC_NQ + vi + 1] - pr.pd_q_nom[vi - 6];
  double u = -pr.pd_kp * e - pr.pd_kd * v[inst * WBC_NV + vi];
  u = u < -pr.pd_clip ? -pr.pd_clip : (u > pr.pd_clip ? pr.pd_clip : u);   // comparisons keep a NaN (np.clip does; fmin / fmax drop it)
  tau[inst * WBC_NU + md.act_index[k]] = u;
}

// ---------------------------------------------------------------- per-robot controller parameters (wbc_step_params)
// One parameter set: the gains and weights with the constants derived from them on the host (derive_constants), one 16-byte
// aligned record so that a reduce CTA stages it with the vector loop of the model constants.
struct alignas(16) ParamRec {
  wbc_params pr;
  Derived dv;
};

// Device inputs of the parameter-aware kernels: K records and the set of each robot (index [N], NULL: set 0).
struct ParamArgs {
  const ParamRec* set; const int32_t* index; int n_sets;
};

// The record robot `inst` is controlled with. An index outside [0, n_sets) sets WBC_ST_BADPARAMS in `status` (the robot's
// outputs are then zeroed like those of any other failure) and returns record 0, so that every read stays in bounds.
WBC_DEV const ParamRec& param_record(const ParamArgs& p, long long inst, int& status) {
  const int k = p.index ? p.index[inst] : 0;
  const bool bad = !(k >= 0 && k < p.n_sets);
  if (bad) status |= WBC_ST_BADPARAMS;
  return p.set[bad ? 0 : k];
}

// pd_element with the robot's own gains. A bad set index gives tau = 0; thread k = 0 of the robot writes its status word
// (WBC_ST_BADPARAMS or 0) when `status` is given.
WBC_DEV void pd_params_element(const wbc_model& md, const ParamArgs& p, const double* q, const double* v, double* tau, int32_t* status,
                               long long inst, int k) {
  int st = 0;
  const ParamRec& r = param_record(p, inst, st);
  if (st) tau[inst * WBC_NU + md.act_index[k]] = 0.0;
  else pd_element(md, r.pr, q, v, tau, inst, k);
  if (status && k == 0) status[inst] = st;
}

}  // namespace wbc
