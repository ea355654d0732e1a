// wbc_traj.cuh — trunk-trajectory sampler on the device (SURVEY.md 8 f1).
//
// Turns a TOWR spline solution (cubic Hermite node splines + per-foot phase durations) into the controller input
// traj[54] / contact[4] (+ planned forces) for N (plan, time) pairs per launch, i.e. what
//   towr/trunk_mpc.cpp:19-68        publish_trunk_state (GetPoint of base_linear, base_angular, ee_motion, ee_force;
//                                   IsContactPhase) and
//   planners/towr.py:92-148         TowrTrunkPlanner.SetTrunkOutputs (stand for wait_time, then NEAREST stored 1 kHz sample)
// do one sample at a time on the host. Restated arithmetic: towr/src/polynomial.cc:49-63,98-104 (cubic Hermite),
// towr/src/spline.cc:49-90 (segment lookup, "previous polynomial at junctions", eps 1e-10),
// towr/src/phase_durations.cc:120-124 (contact flag).
//
// HBM-bound: 12 B in (t, plan index), 436 (+96) B out per instance; the spline tables (tens of KB per plan) stay in
// L1/L2. See sample_kernel for the thread mapping.
#pragma once
#include <stdint.h>
#include "wbc.h"

namespace wbctraj {

constexpr int NSPLINE = 10;          // 0 base linear, 1 base angular, 2-5 foot motion LF RF LH RH, 6-9 foot force

// Device-resident tables of a set of plans (built by wbc_plan_create).
struct PlanTables {
  int n_plans;
  const int* poly_off;        // [n_plans][NSPLINE + 1] -> first polynomial of spline s in tend / coef (last = end)
  const int* phase_off;       // [n_plans][4 + 1]       -> first phase of foot k in phase_tend
  const int* grid_off;        // [n_plans + 1]          -> first stored timestamp of the plan (0 entries = continuous)
  const unsigned char* contact_start;   // [n_plans][4]
  const double* tend;         // running sum of the polynomial durations inside each spline (spline.cc:55-58)
  const double* coef;         // [poly][3][4]: A B C D of each dimension (polynomial.cc:98-104)
  const double* phase_tend;   // running sum of the phase durations of each foot
  const double* grid_ts;      // timestamps of the stored samples (trunk_mpc.cpp:168-174)
  const double* wait_time;    // [n_plans] planners/towr.py:35
  const double* standing;     // [n_plans][54] SimpleStanding (planners/simple.py:39-85) used while t < wait_time
};

// CubicHermitePolynomial::UpdateCoeff for every (polynomial, dimension): nodes[(poly + spline index)][6] = p, v.
__global__ void hermite_coeff_kernel(int n_poly_total, const int* __restrict__ node_of_poly, const double* __restrict__ nodes,
                                     const double* __restrict__ dur, double* __restrict__ coef) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_poly_total * 3) return;
  const int p = idx / 3, d = idx - 3 * p;
  const double* n0 = nodes + (size_t)node_of_poly[p] * 6;
  const double* n1 = n0 + 6;
  const double T = dur[p], p0 = n0[d], v0 = n0[3 + d], p1 = n1[d], v1 = n1[3 + d];
  double* c = coef + (size_t)idx * 4;
  c[0] = p0;
  c[1] = v0;
  c[2] = -(3.0 * (p0 - p1) + T * (2.0 * v0 + v1)) / (T * T);
  c[3] = (2.0 * (p0 - p1) + T * (v0 + v1)) / (T * T * T);
}

// Spline::GetSegmentID on the running sums: first i with tend[i] >= t - 1e-10 (clamped to the last segment).
__device__ __forceinline__ int segment_of(const double* __restrict__ tend, int n, double t) {
  const double key = t - 1e-10;
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(tend + mid) >= key) hi = mid; else lo = mid + 1;
  }
  return lo;
}

// One 32-byte coefficient record {A, B, C, D} with a single 256-bit load (sm_100: LDG.256): one sector, one request,
// instead of two 16-byte halves of the same sector.
struct Coef4 { double a, b, c, d; };
__device__ __forceinline__ Coef4 load_coef(const double* __restrict__ rec) {
  Coef4 r;
  asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.a), "=d"(r.b), "=d"(r.c), "=d"(r.d) : "l"(rec));
  return r;
}

// Two stages per chunk of IPW instances (one warp per chunk):
//   A  planner time logic (wait / nearest stored sample) once per instance, then the 10 spline segment lookups and the 4 contact
//      phase lookups - 14 dependent binary searches - spread over the 32 / IPW lanes that share an instance; (polynomial index,
//      local time) of every spline go to shared memory;
//   B  lane = output element: consecutive lanes write consecutive doubles of traj (coalesced), each evaluating one cubic
//      (or its first / second derivative) from the staged segment info and a 32-byte coefficient record.
// IPW = 32 (lane = instance, all searches serial) is the throughput shape for large batches; small batches are latency bound on
// the search chains of a few warps, so they run with IPW = 8 or 2 (4 or 1 searches per lane, 4x / 16x the warps).
constexpr int SAMPLE_WARPS = 4;
struct SampleSmem {
  double tl[32][NSPLINE];
  double t[32];
  int poly[32][NSPLINE];
  int plan[32];
  unsigned char standing[32];
  unsigned char cb[32][4];
};

template <int IPW>
__global__ void __launch_bounds__(SAMPLE_WARPS * 32) sample_kernel(PlanTables pt, long long n, const int* __restrict__ plan_index,
                                                                   const double* __restrict__ tin, double* __restrict__ traj,
                                                                   unsigned char* __restrict__ contact, double* __restrict__ fplan,
                                                                   double* __restrict__ t_eval_out, int* __restrict__ status) {
  constexpr int G = 32 / IPW;            // lanes per instance in stage A
  __shared__ SampleSmem smem[SAMPLE_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int il = lane & (IPW - 1), g = lane / IPW;
  SampleSmem& sm = smem[warp];
  const long long n_chunks = (n + IPW - 1) / IPW;
  for (long long chunk = (long long)blockIdx.x * SAMPLE_WARPS + warp; chunk < n_chunks; chunk += (long long)gridDim.x * SAMPLE_WARPS) {
    const long long i0 = chunk * IPW;
    const int cnt = (int)((n - i0) < IPW ? (n - i0) : IPW);
    __syncwarp();
    // ---------------------------------------------------------------- stage A1: time logic, one lane per instance
    if (g == 0 && il < cnt) {
      const long long inst = i0 + il;
      int pl = plan_index ? plan_index[inst] : 0;
      int st = 0;
      if (pl < 0 || pl >= pt.n_plans) { pl = 0; st |= WBC_TRAJ_BADPLAN; }
      double t = tin[inst];
      if (isnan(t)) { t = 0.0; st |= WBC_TRAJ_CLAMPED; }              // a NaN would fail every comparison below (wbc.h)
      // planner semantics (planners/towr.py:96-110): stand while t < wait_time, then the nearest stored sample
      const int g0 = __ldg(pt.grid_off + pl), gn = __ldg(pt.grid_off + pl + 1) - g0;
      bool standing = false;
      if (gn > 0) {
        const double wait = __ldg(pt.wait_time + pl);
        if (t < wait) standing = true;
        else {
          const double tq = t - wait;
          const double* ts = pt.grid_ts + g0;
          // np.abs(ts - tq).argmin(): ts is increasing, so the minimum is next to the insertion point; first minimum wins
          int lo = 0, hi = gn - 1;
          while (lo < hi) { const int mid = (lo + hi) >> 1; if (__ldg(ts + mid) >= tq) hi = mid; else lo = mid + 1; }
          int best = lo;
          if (lo > 0 && fabs(__ldg(ts + lo - 1) - tq) <= fabs(__ldg(ts + lo) - tq)) best = lo - 1;
          t = __ldg(ts + best);
        }
      }
      if (!standing) {
        const int* po = pt.poly_off + pl * (NSPLINE + 1);
        const double t_total = __ldg(pt.tend + __ldg(po + 1) - 1);      // Spline::GetTotalTime of the base spline
        if (!(t >= 0.0)) { t = 0.0; st |= WBC_TRAJ_CLAMPED; }           // the reference asserts t >= 0 (spline.cc:52) ...
        if (t > t_total + 1e-10) { t = t_total; st |= WBC_TRAJ_CLAMPED; }   // ... and runs off the end (spline.cc:65)
      }
      if (status) status[inst] = st;
      if (t_eval_out) t_eval_out[inst] = standing ? -1.0 : t;
      sm.plan[il] = pl;
      sm.standing[il] = standing ? 1 : 0;
      sm.t[il] = t;
    }
    __syncwarp();
    // ---------------------------------------------------------------- stage A2: the 14 lookups of an instance over its G lanes
    if (il < cnt && !sm.standing[il]) {
      const int pl = sm.plan[il];
      const double t = sm.t[il];
      const int* po = pt.poly_off + pl * (NSPLINE + 1);
      const int ns = fplan ? NSPLINE : 6;
      for (int s = g; s < NSPLINE + 4; s += G) {
        if (s < NSPLINE) {
          if (s >= ns) continue;
          const int p0 = __ldg(po + s), np_ = __ldg(po + s + 1) - p0;
          const int i = segment_of(pt.tend + p0, np_, t);
          sm.poly[il][s] = p0 + i;
          sm.tl[il][s] = t - (i > 0 ? __ldg(pt.tend + p0 + i - 1) : 0.0);
        } else {                                                     // contact flags (phase_durations.cc:120-124)
          const int k = s - NSPLINE;
          const int* fo = pt.phase_off + pl * 5;
          const int f0 = __ldg(fo + k);
          const int ph = segment_of(pt.phase_tend + f0, __ldg(fo + k + 1) - f0, t);
          const bool c0 = __ldg(pt.contact_start + pl * 4 + k) != 0;
          sm.cb[il][k] = ((ph & 1) ? !c0 : c0) ? 1 : 0;
        }
      }
    }
    __syncwarp();
    if (g == 0 && il < cnt)                                          // 4 flags as one aligned 32-bit store
      reinterpret_cast<unsigned*>(contact)[i0 + il] = sm.standing[il] ? 0x01010101u : *reinterpret_cast<const unsigned*>(sm.cb[il]);
    // ---------------------------------------------------------------- stage B
    // lane = (instance, spline, dimension): one coefficient record gives position, velocity and acceleration; the three
    // stores of neighbouring lanes fill whole 24-byte groups of the row, which L2 merges into full sectors
    double* out = traj + i0 * WBC_NTRAJ;
    for (int idx = lane; idx < cnt * 18; idx += 32) {
      const int bi = idx / 18, r = idx - bi * 18, s = r / 3, dim = r - 3 * s;
      const int e0 = s < 2 ? 9 * s + dim : 18 + 3 * (s - 2) + dim, stride = s < 2 ? 3 : 12;
      double p, v, a;
      if (sm.standing[bi]) {
        const double* st = pt.standing + sm.plan[bi] * WBC_NTRAJ + e0;
        p = __ldg(st); v = __ldg(st + stride); a = __ldg(st + 2 * stride);
      } else {
        const double tl = sm.tl[bi][s];
        const Coef4 c = load_coef(pt.coef + ((size_t)sm.poly[bi][s] * 3 + dim) * 4);
        p = fma(fma(fma(c.d, tl, c.c), tl, c.b), tl, c.a);
        v = fma(fma(3.0 * c.d, tl, 2.0 * c.c), tl, c.b);
        a = fma(6.0 * c.d, tl, 2.0 * c.c);
      }
      double* o = out + bi * WBC_NTRAJ + e0;
      o[0] = p; o[stride] = v; o[2 * stride] = a;
    }
    if (fplan) {
      double* fo = fplan + i0 * 12;
      for (int idx = lane; idx < cnt * 12; idx += 32) {
        const int bi = idx / 12, r = idx - bi * 12, s = 6 + r / 3, dim = r % 3;
        double val = 0.0;
        if (!sm.standing[bi]) {
          const double tl = sm.tl[bi][s];
          const Coef4 c = load_coef(pt.coef + ((size_t)sm.poly[bi][s] * 3 + dim) * 4);
          val = fma(fma(fma(c.d, tl, c.c), tl, c.b), tl, c.a);
        }
        fo[idx] = val;
      }
    }
  }
}

}  // namespace wbctraj
