// wbc_loop.cuh — imperfect sensing and actuation in the ground-plant loop (include/wbc.h, wbc_loop): the controller of robot i
// reads a noisy copy of its state, and its torque command reaches the plant `delay` control steps late, scaled by its motor
// strength. The semantics are stated once in include/wbc.h and restated in numpy by oracle/sensing.py.
//
// Two kernels, one thread per robot, in the style of wbcroll::integrate_kernel: observe (before the controller) and actuate
// (after it). The device functions also compile on the host (tests/emu/emu_loop.cpp), which defines WBC_DEV and sincospi.
#pragma once
#include <stdint.h>
#include <math.h>
#include "wbc.h"

#ifndef WBC_DEV
#define WBC_DEV __device__ __forceinline__
#endif

namespace wbcloop {

// Device view of a wbc_loop. hist / tick may be NULL for observe only (tick 0); actuate always gets both.
struct LoopArgs {
  const double* noise; const int32_t* delay; const double* strength; const int32_t* stream;
  unsigned long long seed; double* hist; long long* tick;
};

constexpr int NOISE_DRAWS = 18;     // Philox blocks per robot and step: 36 normals

// Philox4x32-10 (Salmon et al. 2011), the function of cuRAND's curand_Philox4x32_10: ctr = (x, y, z, w), key = (k0, k1).
WBC_DEV void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}

// Two standard normals from one Philox block (Box-Muller on two 53-bit uniforms in (0, 1)).
WBC_DEV void normal_pair(const uint32_t w[4], double& z0, double& z1) {
  const uint64_t a = ((((uint64_t)w[1]) << 32) | w[0]) >> 11, b = ((((uint64_t)w[3]) << 32) | w[2]) >> 11;
  const double ua = (double)a * 0x1p-53 + 0x1p-54, ub = (double)b * 0x1p-53 + 0x1p-54;
  const double r = sqrt(-2.0 * log(ua));
  double s, c;
  sincospi(2.0 * ub, &s, &c);
  z0 = r * c;
  z1 = r * s;
}

// The 36 normals of robot `stream` at step c.
WBC_DEV void normals(unsigned long long seed, uint32_t stream, long long c, double z[2 * NOISE_DRAWS]) {
#pragma unroll
  for (int j = 0; j < NOISE_DRAWS; ++j) {
    uint32_t w[4] = {(uint32_t)j, stream, (uint32_t)(unsigned long long)c, (uint32_t)((unsigned long long)c >> 32)};
    philox4x32_10(w, (uint32_t)seed, (uint32_t)(seed >> 32));
    normal_pair(w, z[2 * j], z[2 * j + 1]);
  }
}

WBC_DEV bool nonneg_finite(double x) { return x >= 0.0 && x <= 1.7976931348623157e308; }

// Whether robot i's profile is usable at step c: delay in [0, 15], every sigma and the strength finite and >= 0, c >= 0.
WBC_DEV bool profile_ok(const LoopArgs& a, long long i, long long c) {
  bool ok = c >= 0;
  if (a.delay) ok = ok && a.delay[i] >= 0 && a.delay[i] < WBC_LOOP_HIST;
  if (a.strength) ok = ok && nonneg_finite(a.strength[i]);
  if (a.noise) {
#pragma unroll
    for (int k = 0; k < 6; ++k) ok = ok && nonneg_finite(a.noise[i * 6 + k]);
  }
  return ok;
}

// What the controller of robot i sees at step tick[i]: q_obs [19], v_obs [18] from the true q, v (row i of each).
WBC_DEV void observe_instance(const LoopArgs& a, long long i, const double* __restrict__ q, const double* __restrict__ v,
                              double* __restrict__ qo, double* __restrict__ vo) {
  const double* qi = q + i * WBC_NQ;
  const double* vi = v + i * WBC_NV;
  double* qoi = qo + i * WBC_NQ;
  double* voi = vo + i * WBC_NV;
  const long long c = a.tick ? a.tick[i] : 0;
  double sg[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (a.noise && profile_ok(a, i, c)) {
#pragma unroll
    for (int k = 0; k < 6; ++k) sg[k] = a.noise[i * 6 + k];
  }
  double z[2 * NOISE_DRAWS];
  const bool any = sg[0] != 0.0 || sg[1] != 0.0 || sg[2] != 0.0 || sg[3] != 0.0 || sg[4] != 0.0 || sg[5] != 0.0;
  if (any) normals(a.seed, a.stream ? (uint32_t)a.stream[i] : (uint32_t)i, c, z);
  // orientation: normalize(dq (x) q), dq the rotation by the vector sigma z[0:3] (world frame)
  if (sg[0] != 0.0) {
    const double dx = sg[0] * z[0], dy = sg[0] * z[1], dz = sg[0] * z[2];
    const double th = sqrt(dx * dx + dy * dy + dz * dz);
    const double cw = cos(0.5 * th), sk = th > 0.0 ? sin(0.5 * th) / th : 0.0;
    const double ex = sk * dx, ey = sk * dy, ez = sk * dz;
    const double qw = qi[0], qx = qi[1], qy = qi[2], qz = qi[3];
    const double nw = cw * qw - ex * qx - ey * qy - ez * qz;
    const double nx = cw * qx + ex * qw + ey * qz - ez * qy;
    const double ny = cw * qy - ex * qz + ey * qw + ez * qx;
    const double nz = cw * qz + ex * qy - ey * qx + ez * qw;
    const double inv = 1.0 / sqrt(nw * nw + nx * nx + ny * ny + nz * nz);
    qoi[0] = nw * inv; qoi[1] = nx * inv; qoi[2] = ny * inv; qoi[3] = nz * inv;
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) qoi[k] = qi[k];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) qoi[4 + k] = sg[1] != 0.0 ? qi[4 + k] + sg[1] * z[3 + k] : qi[4 + k];
#pragma unroll
  for (int k = 0; k < WBC_NU; ++k) qoi[7 + k] = sg[2] != 0.0 ? qi[7 + k] + sg[2] * z[6 + k] : qi[7 + k];
#pragma unroll
  for (int k = 0; k < 3; ++k) voi[k] = sg[3] != 0.0 ? vi[k] + sg[3] * z[18 + k] : vi[k];
#pragma unroll
  for (int k = 0; k < 3; ++k) voi[3 + k] = sg[4] != 0.0 ? vi[3 + k] + sg[4] * z[21 + k] : vi[3 + k];
#pragma unroll
  for (int k = 0; k < WBC_NU; ++k) voi[6 + k] = sg[5] != 0.0 ? vi[6 + k] + sg[5] * z[24 + k] : vi[6 + k];
}

// Robot i's command tau [12] of step tick[i] enters its ring; `applied` [12] receives strength x the command of step
// max(c - d, 0); tick advances. A bad profile: applied = 0, WBC_ST_BADLOOP in status[i], hist and tick unchanged.
WBC_DEV void actuate_instance(const LoopArgs& a, long long i, const double* __restrict__ tau, double* __restrict__ applied,
                              int32_t* __restrict__ status) {
  const long long c = a.tick[i];
  double* out = applied + i * WBC_NU;
  if (!profile_ok(a, i, c)) {
#pragma unroll
    for (int k = 0; k < WBC_NU; ++k) out[k] = 0.0;
    if (status) status[i] |= WBC_ST_BADLOOP;
    return;
  }
  const int d = a.delay ? a.delay[i] : 0;
  const double s = a.strength ? a.strength[i] : 1.0;
  double* h = a.hist + i * (WBC_LOOP_HIST * WBC_NU);
  const int w = (int)(c & (WBC_LOOP_HIST - 1)), r = (int)((c > d ? c - d : 0) & (WBC_LOOP_HIST - 1));
  double t[WBC_NU];
#pragma unroll
  for (int k = 0; k < WBC_NU; ++k) { t[k] = tau[i * WBC_NU + k]; h[w * WBC_NU + k] = t[k]; }
  if (r == w) {
#pragma unroll
    for (int k = 0; k < WBC_NU; ++k) out[k] = s * t[k];
  } else {
#pragma unroll
    for (int k = 0; k < WBC_NU; ++k) out[k] = s * h[r * WBC_NU + k];
  }
  a.tick[i] = c + 1;
}

#ifdef __CUDACC__
__global__ void __launch_bounds__(256) observe_kernel(const LoopArgs a, long long n, const double* __restrict__ q,
                                                      const double* __restrict__ v, double* __restrict__ q_obs,
                                                      double* __restrict__ v_obs) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) observe_instance(a, i, q, v, q_obs, v_obs);
}

__global__ void __launch_bounds__(256) actuate_kernel(const LoopArgs a, long long n, const double* __restrict__ tau,
                                                      double* __restrict__ applied, int32_t* __restrict__ status) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) actuate_instance(a, i, tau, applied, status);
}
#endif

}  // namespace wbcloop
