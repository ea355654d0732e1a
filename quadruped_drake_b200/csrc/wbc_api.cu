// wbc_api.cu — C ABI (include/wbc.h) and kernel launches of the batched whole-body controller.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <cmath>
#include <deque>
#include <memory>
#include <string>

// named barrier `id` over `threads` threads of the CTA (a multiple of 32; skipped when at most one warp takes part)
#ifndef WBC_PC_MEET
#define WBC_PC_MEET 1
#endif
#if WBC_PC_MEET
#define WBC_CTA_MEET(id, threads)                                                                    \
  do {                                                                                               \
    const int nt_ = (threads);                                                                       \
    if (nt_ > 32) asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nt_) : "memory");                   \
  } while (0)
#endif
#include "wbc_device.cuh"
#include "wbc_wire.cuh"
#include "wbc_traj.cuh"
#include "wbc_rollout.cuh"
#include "wbc_plant.cuh"
#include "wbc_loop.cuh"
#include "wbc_monitor.cuh"
#include "wbc_motor.cuh"
#include "wbc_estimator.cuh"
#include <vector>

namespace {

// Warps (= instances) per CTA of the reduce / dynamics kernels. One warp per CTA puts the per-warp block at a compile-time
// shared-memory address, which frees the registers that held its base (spill 536 -> 44 B; 4-warp CTAs measured 3-8 % slower
// on device-resident buffers). The 4-warp shape is kept for page-locked HOST buffers (zero-copy path of wbc_step_host): there
// the CTA stages all four input arrays of its 4 consecutive instances with one bulk copy each - few large requests, which is
// what the host link wants (e2e 25.3 vs 22.3 M steps/s at 4096).
constexpr int WARPS = 1;         // device-resident buffers
#ifndef WBC_WARPS_HOST
#define WBC_WARPS_HOST 4
#endif
constexpr int WARPS_HOST = WBC_WARPS_HOST;    // host-mapped buffers (ID / CLF)
#ifndef WBC_WARPS_PC
#define WBC_WARPS_PC 6
#endif
constexpr int WARPS_PC = WBC_WARPS_PC;        // PC / MPTC reduce kernel
#ifndef WBC_PC_MIN_WARPS
#define WBC_PC_MIN_WARPS 12      // resident warps per SM the PC reduce kernel is compiled for (168 registers)
#endif
#ifndef WBC_MIN_WARPS
#define WBC_MIN_WARPS 16         // resident warps per SM the reduce kernels are compiled for (128 registers)
#endif

struct alignas(16) DevConst { wbc_model md; wbc_params pr; wbc::Derived dv; };

// CTA-level input staging of the reduce kernels: the rows of the CTA's W consecutive instances are contiguous in the caller's
// arrays, so an array whose W rows are a multiple of 16 bytes arrives with ONE bulk copy instead of 8-byte loads per lane
// (v: 144 B and traj: 432 B rows always; q: 152 B and contact: 4 B rows only for W = 4).
template <int W>
struct alignas(16) InStage {
  alignas(16) double q[W * WBC_NQ];
  alignas(16) double v[W * WBC_NV];
  alignas(16) double traj[W * WBC_NTRAJ];
  alignas(16) uint8_t contact[W * 4];
  alignas(16) unsigned long long mbar;
  static constexpr bool BULK_Q = (W * WBC_NQ * 8) % 16 == 0, BULK_C = (W * 4) % 16 == 0;
};
static_assert((WBC_NV * 8) % 16 == 0 && (WBC_NTRAJ * 8) % 16 == 0, "v / traj rows must be multiples of 16 bytes");

template <int W>
struct SmemLayoutT {
  DevConst dc;
  InStage<W> in;
  wbc::WarpSmem w[W];
};
template <int W>
struct SmemLayoutPCT {     // PC controller / Coriolis entry: extra operational-space workspace per warp
  DevConst dc;
  InStage<W> in;
  wbc::WarpSmem w[W];
  wbc::PcSmem pc[W];
};
using SmemLayout = SmemLayoutT<WARPS>;
using SmemLayoutPC = SmemLayoutPCT<WARPS>;

// A constant table into shared memory once per CTA (lane-divergent table lookups stay on chip), 16 bytes per thread and trip
template <typename T>
__device__ __forceinline__ const T& stage16(T* sm_dst, const T* g) {
  static_assert(sizeof(T) % 16 == 0, "staged with 16-byte vectors");
  const int nvec = sizeof(T) / 16;
  const uint4* src = reinterpret_cast<const uint4*>(g);
  uint4* dst = reinterpret_cast<uint4*>(sm_dst);
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) dst[i] = src[i];
  __syncthreads();
  return *sm_dst;
}
// model + gains
template <typename L>
__device__ __forceinline__ const DevConst& stage_consts(L* sm, const DevConst* g) { return stage16(&sm->dc, g); }

// ---------------------------------------------------------------------------------------------------------------------
// Split path (ID / CLF): the step is launched as two kernels with their own register / occupancy budgets.
//   wbc_reduce_kernel  phases 0-4 (dynamics, equality elimination, reduced rows): register hungry (128 regs, 16 warps / SM);
//                      leaves [Y | cw | ct] + 16 carry words per instance in a hand-over record (4224 B, device scratch).
//   wbc_solve_kernel   phases 5-7 (reduced Hessian, Cholesky, Goldfarb-Idnani, outputs): 72 registers and 7.8 KB of shared
//                      memory per warp -> 28 warps / SM, so the dependent-instruction latency of the active-set iterations is
//                      hidden by 1.75x more resident instances than the fused kernel could hold.
// The 4 KB block moves shared -> global and global -> shared with one bulk asynchronous copy each (TMA 1-D), issued by one
// lane; the solve warp waits on an mbarrier.
#ifndef WBC_SOLVE_WARPS
#define WBC_SOLVE_WARPS 1      // one warp per CTA: the shared-memory block sits at a compile-time address, so no per-warp base
#endif                         // (thread index -> warp -> offset) has to be kept live or re-derived under the 72-register budget
#ifndef WBC_SOLVE_CTAS
#define WBC_SOLVE_CTAS (21 / WBC_SOLVE_WARPS)
#endif
constexpr int SOLVE_WARPS = WBC_SOLVE_WARPS;
template <bool VD> struct SmemLayoutSolveT { wbc::SolveSmemT<VD> w[SOLVE_WARPS]; };
static_assert(sizeof(wbc::SolveSmem) % 16 == 0 && sizeof(wbc::SolveSmemVd) % 16 == 0, "SolveSmem must keep 16-byte alignment per warp");
static_assert(offsetof(wbc::WarpSmem, Y) % 16 == 0 && sizeof(wbc::WarpSmem) % 16 == 0 && sizeof(DevConst) % 16 == 0, "bulk copy alignment");
static_assert(offsetof(wbc::WarpSmem, cw) == offsetof(wbc::WarpSmem, Y) + sizeof(double) * wbc::YROWS * wbc::YS &&
              offsetof(wbc::WarpSmem, ct) == offsetof(wbc::WarpSmem, cw) + sizeof(double) * wbc::YROWS, "[Y | cw | ct] must be contiguous");
static_assert(offsetof(wbc::SolveSmem, cw) == sizeof(double) * wbc::YROWS * wbc::YS &&
              offsetof(wbc::SolveSmem, ct) == offsetof(wbc::SolveSmem, cw) + sizeof(double) * wbc::YROWS, "[Y | cw | ct] must be contiguous");
constexpr unsigned REC_Y_BYTES = wbc::REC_Y * sizeof(double);

// Programmatic dependent launch: the solve kernel is launched with the programmatic-stream-serialization attribute, so its
// CTAs become resident while the last reduce CTAs are still running (they have all started by then) and wait here; this
// hides the launch latency and CTA ramp of the second kernel. Both instructions are no-ops in an ordinary launch.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
// Lane index the compiler cannot re-derive from the special register: under the register caps of the step kernels it
// otherwise rematerialises every lane-dependent shared-memory address with an S2R (a slow special-register read) + IMAD
// pair at each use instead of keeping one register live (WBC_OPAQUE_LANE=0 restores the plain form for A/B runs).
#ifndef WBC_OPAQUE_LANE
#define WBC_OPAQUE_LANE 1
#endif
__device__ __forceinline__ int lane_index() {
  int lane = (int)(threadIdx.x & 31);
#if WBC_OPAQUE_LANE
  asm volatile("" : "+r"(lane));
#endif
  return lane;
}
// shared -> global bulk copy of `bytes` (multiple of 16), issued by the calling thread; returns once the source may be reused
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, unsigned bytes) {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes of the warp -> visible to the copy engine
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_addr(ssrc)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// global -> shared bulk copy completing on an mbarrier (armed here by the issuing thread)
__device__ __forceinline__ void bulk_load(void* sdst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  const unsigned b = smem_addr(bar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(sdst)),
               "l"(gsrc), "r"(bytes), "r"(b)
               : "memory");
}
__device__ __forceinline__ void bulk_load_on(void* sdst, const void* gsrc, unsigned bytes, unsigned bar_smem) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(sdst)),
               "l"(gsrc), "r"(bytes), "r"(bar_smem)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  const unsigned b = smem_addr(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(b), "r"(parity)
      : "memory");
}

// Hand-over record of one instance: [Y | cw | ct] by one bulk copy + the carry words (called by one lane).
__device__ __forceinline__ void store_record(double* r, const wbc::StepCarry& c, const wbc::WarpSmem& s) {
  double2* m = reinterpret_cast<double2*>(r + wbc::REC_Y);
  m[0] = make_double2((double)c.status, (double)c.cmask);
  m[1] = make_double2((double)c.nf, (double)c.nextra);
  m[2] = make_double2(c.ok ? 1.0 : 0.0, c.pc_ok ? 1.0 : 0.0);
  m[3] = make_double2(c.extra_bound, c.err);
  m[4] = make_double2(c.Vl, c.PFl);
  m[5] = make_double2(c.csum, c.Vpc);
  if (c.ok) bulk_store(r, &s.Y[0][0], REC_Y_BYTES);
}

// Issues the CTA's four input bulk copies (thread 0) - call before stage_consts so that they fly during the constant staging -
// and, after the CTA barrier inside stage_consts, waits for them. Returns false when this CTA must use the per-lane path
// (tail CTA with fewer than WARPS instances, or buffers that are not 16-byte aligned: `bulk_ok` from the host).
template <int W>
__device__ __forceinline__ bool stage_inputs_issue(InStage<W>& in, const wbc::StepArgs& a, bool bulk_ok) {
  constexpr bool BQ = InStage<W>::BULK_Q, BC = InStage<W>::BULK_C;
  const long long first = (long long)blockIdx.x * W;
  const bool full = bulk_ok && first + W <= a.n;
  if (full && threadIdx.x == 0) {
    const unsigned b = smem_addr(&in.mbar);
    const unsigned bytes = W * (WBC_NV + WBC_NTRAJ) * 8 + (BQ ? W * WBC_NQ * 8 : 0) + (BC ? W * 4 : 0);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
    if (BQ) bulk_load_on(in.q, a.q + first * WBC_NQ, W * WBC_NQ * 8, b);
    bulk_load_on(in.v, a.v + first * WBC_NV, W * WBC_NV * 8, b);
    bulk_load_on(in.traj, a.traj + first * WBC_NTRAJ, W * WBC_NTRAJ * 8, b);
    if (BC) bulk_load_on(in.contact, a.contact + first * 4, W * 4, b);
  }
  return full;
}
template <int W>
__device__ __forceinline__ wbc::StagedInputs staged_rows(const InStage<W>& in, int warp) {
  return wbc::StagedInputs{InStage<W>::BULK_Q ? in.q + warp * WBC_NQ : nullptr, in.v + warp * WBC_NV, in.traj + warp * WBC_NTRAJ,
                           InStage<W>::BULK_C ? in.contact + warp * 4 : nullptr};
}

template <int KIND, int W>
__global__ void __launch_bounds__(W * 32, WBC_MIN_WARPS / W) wbc_reduce_kernel(const DevConst* __restrict__ gdc, wbc::StepArgs a,
                                                                            double* __restrict__ rec, double* __restrict__ vdmap, int bulk_ok) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutT<W>* sm = reinterpret_cast<SmemLayoutT<W>*>(smem_raw);
  pdl_launch_dependents();
  const bool staged = stage_inputs_issue(sm->in, a, bulk_ok != 0);
  const DevConst& dc = stage_consts(sm, gdc);   // (reading the tables through L1 instead of staging them measured neutral)
  const int warp = W == 1 ? 0 : (int)(threadIdx.x >> 5), lane = lane_index();
  const long long inst = (long long)blockIdx.x * W + warp;
  if (inst >= a.n) return;
  wbc::WarpSmem& s = sm->w[warp];
  wbc::StepCarry c;
  const wbc::StagedInputs in = staged_rows(sm->in, warp);
  if (staged) mbar_wait(&sm->in.mbar, 0);
  wbc::reduce_instance<KIND>(s, dc.md, dc.pr, dc.dv, a, inst, lane, c, nullptr, vdmap ? vdmap + inst * wbc::VDMAP_DOUBLES : nullptr,
                             staged ? &in : nullptr);
  __syncwarp();
  if (lane == 0) store_record(rec + inst * wbc::REC_DOUBLES, c, s);
}

// VD: the accelerations are requested (rollout, debug outputs) - the Cholesky factor is kept for the recovery of w, which
// costs 1.3 KB more shared memory per warp (24 instead of 28 resident warps).
template <int KIND, bool VD>
__global__ void __launch_bounds__(SOLVE_WARPS * 32, VD ? (24 / SOLVE_WARPS) : WBC_SOLVE_CTAS) wbc_solve_kernel(
    const DevConst* __restrict__ gdc, wbc::StepArgs a, const double* __restrict__ rec, const double* __restrict__ vdmap) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutSolveT<VD>* sm = reinterpret_cast<SmemLayoutSolveT<VD>*>(smem_raw);
  const int warp = SOLVE_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5), lane = lane_index();
  const long long inst = (long long)blockIdx.x * SOLVE_WARPS + warp;
  if (inst >= a.n) return;
  wbc::SolveSmemT<VD>& s = sm->w[warp];
  const double* r = rec + inst * wbc::REC_DOUBLES;
  const double2* m = reinterpret_cast<const double2*>(r + wbc::REC_Y);
  pdl_wait();                      // the records of the reduce kernel are complete and visible from here on
  const double2 m2 = m[2];
  const bool ok = m2.x != 0.0;
  if (ok && lane == 0) bulk_load(&s.Y[0][0], r, REC_Y_BYTES, &s.mbar);
  const double2 m0 = m[0], m1 = m[1], m3 = m[3], m4 = m[4], m5 = m[5];
  wbc::StepCarry c;
  c.status = (int)m0.x; c.cmask = (unsigned)m0.y; c.nf = (int)m1.x; c.nextra = (int)m1.y;
  c.ok = ok; c.pc_ok = m2.y != 0.0; c.extra_bound = m3.x; c.err = m3.y; c.Vl = m4.x; c.PFl = m4.y; c.csum = m5.x; c.Vpc = m5.y;
  __syncwarp();                    // the barrier is initialised before any lane polls it
  if (ok) mbar_wait(&s.mbar, 0);
  wbc::solve_instance<KIND, wbc::SolveSmemT<VD>>(s, gdc->md, gdc->pr, a, inst, lane, c, vdmap ? vdmap + inst * wbc::VDMAP_DOUBLES : nullptr, r);
}

// PC / MPTC reduce half: same hand-over, extra operational-space workspace per warp (168 registers, 12 warps / SM).
template <int W>
__global__ void __launch_bounds__(W * 32, WBC_PC_MIN_WARPS / W) wbc_reduce_pc_kernel(const DevConst* __restrict__ gdc, wbc::StepArgs a,
                                                                    double* __restrict__ rec, double* __restrict__ vdmap, int bulk_ok) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutPCT<W>* sm = reinterpret_cast<SmemLayoutPCT<W>*>(smem_raw);
  pdl_launch_dependents();
  const bool staged = stage_inputs_issue(sm->in, a, bulk_ok != 0);
  const DevConst& dc = stage_consts(sm, gdc);
  const int warp = W == 1 ? 0 : (int)(threadIdx.x >> 5), lane = lane_index();
  const long long inst = (long long)blockIdx.x * W + warp;
  if (inst >= a.n) return;
  wbc::WarpSmem& s = sm->w[warp];
  wbc::StepCarry c;
  const wbc::StagedInputs in = staged_rows(sm->in, warp);
  if (staged) mbar_wait(&sm->in.mbar, 0);
  {
    // meeting points of the CTA's warps ahead of the dynamics passes (wbc_device.cuh: WBC_CTA_MEET): every warp with an instance
    // takes the state pass, every warp whose instance has a stance foot takes the two polarisation passes
    const long long first = (long long)blockIdx.x * W;
    const int n_act = (int)((a.n - first) < W ? (a.n - first) : W);
    int n_pc = 0;
    for (int w = 0; w < n_act; ++w) {
      const uint8_t* cp = (staged && in.contact) ? sm->in.contact + w * 4 : a.contact + (first + w) * 4;
      n_pc += (cp[0] | cp[1] | cp[2] | cp[3]) ? 1 : 0;
    }
    sm->pc[warp].sync_all = 32 * n_act;
    sm->pc[warp].sync_pc = 32 * n_pc;
  }
  wbc::reduce_instance<WBC_CTRL_PC>(s, dc.md, dc.pr, dc.dv, a, inst, lane, c, &sm->pc[warp], vdmap ? vdmap + inst * wbc::VDMAP_DOUBLES : nullptr,
                                    staged ? &in : nullptr);
  __syncwarp();
  if (lane == 0) store_record(rec + inst * wbc::REC_DOUBLES, c, s);
}

__global__ void __launch_bounds__(WARPS * 32, 12 / WARPS) wbc_coriolis_kernel(const DevConst* __restrict__ gdc, const double* q,
                                                                     const double* v, double* Cout, double* Jdout, long long n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutPC* sm = reinterpret_cast<SmemLayoutPC*>(smem_raw);
  const DevConst& dc = stage_consts(sm, gdc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long inst = (long long)blockIdx.x * WARPS + warp;
  if (inst < n) wbc::coriolis_instance(sm->w[warp], sm->pc[warp], dc.md, q, v, Cout, Jdout, inst, lane);
}

__global__ void __launch_bounds__(WARPS * 32) wbc_dynamics_kernel(const DevConst* __restrict__ gdc, const double* q,
                                                                   const double* v, wbc::DynOut o, long long n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayout* sm = reinterpret_cast<SmemLayout*>(smem_raw);
  const DevConst& dc = stage_consts(sm, gdc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long inst = (long long)blockIdx.x * WARPS + warp;
  if (inst < n) wbc::dynamics_instance(sm->w[warp], dc.md, q, v, o, inst, lane);
}

// One time step of the simulated robot on the ground (wbc_plant.cuh), one single-warp CTA per robot.
struct SmemLayoutPlant { DevConst dc; wbc::WarpSmem w; wbcplant::PlantSmem p; };
#ifndef WBC_PLANT_CTAS
#define WBC_PLANT_CTAS 16     // 128 registers: 22.2 M robot-steps/s at 4096 robots against 19.2 M at 8 CTAs (202 registers)
#endif
__global__ void __launch_bounds__(32, WBC_PLANT_CTAS) wbc_plant_kernel(const DevConst* __restrict__ gdc, wbcplant::PlantArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutPlant* sm = reinterpret_cast<SmemLayoutPlant*>(smem_raw);
  const DevConst& dc = stage_consts(sm, gdc);
  const int lane = lane_index();
  const long long inst = blockIdx.x;
  if (inst < a.n) wbcplant::plant_step_instance(sm->w, sm->p, dc.md, a, inst, lane);
}

// The same step for perturbed robots (wbc_plant_step_perturbed): the CTA stages its robot's variant record (1936 B) instead of
// the handle's constants, and the step adds the variant's friction and the robot's push.
struct SmemLayoutPlantVariant { wbcplant::PlantVariant pv; wbc::WarpSmem w; wbcplant::PlantSmem p; };
__global__ void __launch_bounds__(32, WBC_PLANT_CTAS) wbc_plant_variant_kernel(wbcplant::PerturbArgs pa, wbcplant::PlantArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutPlantVariant* sm = reinterpret_cast<SmemLayoutPlantVariant*>(smem_raw);
  const long long inst = blockIdx.x;
  const int k = inst < a.n ? wbcplant::plant_variant(pa, inst) : 0;
  const wbcplant::PlantVariant& pv = stage16(&sm->pv, pa.set + (k < 0 ? 0 : k));   // a bad index is frozen: any record will do
  const int lane = lane_index();
  if (inst < a.n)
    wbcplant::plant_step_instance<true>(sm->w, sm->p, pv.md, a, inst, lane, wbcplant::plant_perturb(pa, a, inst, k, pv.mu));
}

// The perturbed step on each robot's terrain (wbc_plant_step_terrain): staged like the variant kernel; lanes 0-3 read their
// foot's terrain record and grid corners from global memory into the small terrain block of this layout.
struct SmemLayoutPlantTerrain { wbcplant::PlantVariant pv; wbc::WarpSmem w; wbcplant::PlantSmem p; wbcplant::TerrainSmem t; };
__global__ void __launch_bounds__(32, WBC_PLANT_CTAS) wbc_plant_terrain_kernel(wbcplant::PerturbArgs pa, wbcplant::TerrainArgs ta,
                                                                                wbcplant::PlantArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutPlantTerrain* sm = reinterpret_cast<SmemLayoutPlantTerrain*>(smem_raw);
  const long long inst = blockIdx.x;
  const int k = inst < a.n ? wbcplant::plant_variant(pa, inst) : 0;
  const wbcplant::PlantVariant& pv = stage16(&sm->pv, pa.set + (k < 0 ? 0 : k));
  const int lane = lane_index();
  if (inst < a.n)
    wbcplant::plant_step_instance<true, true>(sm->w, sm->p, pv.md, a, inst, lane, wbcplant::plant_perturb(pa, a, inst, k, pv.mu), &sm->t, ta);
}

__global__ void wbc_pd_kernel(const DevConst* __restrict__ gdc, const double* q, const double* v, double* tau, long long n) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n * WBC_NU) wbc::pd_element(gdc->md, gdc->pr, q, v, tau, t / WBC_NU, (int)(t % WBC_NU));
}

// ---------------------------------------------------------------------------------------------------------------------
// Per-robot controller parameters (wbc_step_params): twins of the step kernels above that take each robot's wbc_params and
// derived constants from its record of a parameter set (wbc::ParamRec) instead of the handle's DevConst. The model stays the
// handle's. They run the same device functions; a reduce CTA stages the model and one record per warp, which at W = 1 is the
// byte count of DevConst, so shared memory and occupancy match the plain kernels.
struct alignas(16) ModelConst { wbc_model md; };   // the model at the head of DevConst, rounded up to 16 bytes
static_assert(offsetof(DevConst, md) == 0 && sizeof(ModelConst) <= sizeof(DevConst) && sizeof(wbc::ParamRec) % 16 == 0,
              "the model is staged from the head of DevConst; records are staged with 16-byte vectors");

template <int W>
struct SmemLayoutParamsT {
  ModelConst mc;
  wbc::ParamRec prm[W];
  InStage<W> in;
  wbc::WarpSmem w[W];
};
template <int W>
struct SmemLayoutPCParamsT {
  ModelConst mc;
  wbc::ParamRec prm[W];
  InStage<W> in;
  wbc::WarpSmem w[W];
  wbc::PcSmem pc[W];
};
static_assert(sizeof(SmemLayoutParamsT<WARPS>) == sizeof(SmemLayoutT<WARPS>), "single-warp CTAs stage as many bytes as the plain kernel");

// Stages the model and the records of the CTA's W robots (record 0 for a slot past the end) with 16-byte vectors and one CTA
// barrier at the end; returns the status bits of the calling warp's robot (WBC_ST_BADPARAMS for an index out of range).
template <int W, typename L>
__device__ __forceinline__ int stage_params(L* sm, const DevConst* gdc, const wbc::ParamArgs& p, long long n, int warp) {
  constexpr int NM = (int)(sizeof(ModelConst) / 16), NR = (int)(sizeof(wbc::ParamRec) / 16);
  const uint4* gm = reinterpret_cast<const uint4*>(gdc);
  uint4* dm = reinterpret_cast<uint4*>(&sm->mc);
  for (int i = threadIdx.x; i < NM; i += blockDim.x) dm[i] = gm[i];
  const long long first = (long long)blockIdx.x * W;
  int mine = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    int st = 0;
    const wbc::ParamRec& r = first + w < n ? wbc::param_record(p, first + w, st) : p.set[0];
    if (w == warp) mine = st;
    const uint4* src = reinterpret_cast<const uint4*>(&r);
    uint4* dst = reinterpret_cast<uint4*>(&sm->prm[w]);
    for (int i = threadIdx.x; i < NR; i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  return mine;
}

template <int KIND, int W>
__global__ void __launch_bounds__(W * 32, WBC_MIN_WARPS / W) wbc_reduce_params_kernel(const DevConst* __restrict__ gdc, wbc::ParamArgs p,
                                                                                   wbc::StepArgs a, double* __restrict__ rec,
                                                                                   double* __restrict__ vdmap, int bulk_ok) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutParamsT<W>* sm = reinterpret_cast<SmemLayoutParamsT<W>*>(smem_raw);
  pdl_launch_dependents();
  const bool staged = stage_inputs_issue(sm->in, a, bulk_ok != 0);
  const int warp = W == 1 ? 0 : (int)(threadIdx.x >> 5), lane = lane_index();
  const int pstatus = stage_params<W>(sm, gdc, p, a.n, warp);
  const long long inst = (long long)blockIdx.x * W + warp;
  if (inst >= a.n) return;
  wbc::WarpSmem& s = sm->w[warp];
  const wbc::ParamRec& pr = sm->prm[warp];
  wbc::StepCarry c;
  const wbc::StagedInputs in = staged_rows(sm->in, warp);
  if (staged) mbar_wait(&sm->in.mbar, 0);
  wbc::reduce_instance<KIND>(s, sm->mc.md, pr.pr, pr.dv, a, inst, lane, c, nullptr, vdmap ? vdmap + inst * wbc::VDMAP_DOUBLES : nullptr,
                             staged ? &in : nullptr);
  c.status |= pstatus;
  __syncwarp();
  if (lane == 0) store_record(rec + inst * wbc::REC_DOUBLES, c, s);
}

template <int KIND, bool VD>
__global__ void __launch_bounds__(SOLVE_WARPS * 32, VD ? (24 / SOLVE_WARPS) : WBC_SOLVE_CTAS) wbc_solve_params_kernel(
    const DevConst* __restrict__ gdc, wbc::ParamArgs p, wbc::StepArgs a, const double* __restrict__ rec, const double* __restrict__ vdmap) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutSolveT<VD>* sm = reinterpret_cast<SmemLayoutSolveT<VD>*>(smem_raw);
  const int warp = SOLVE_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5), lane = lane_index();
  const long long inst = (long long)blockIdx.x * SOLVE_WARPS + warp;
  if (inst >= a.n) return;
  wbc::SolveSmemT<VD>& s = sm->w[warp];
  const double* r = rec + inst * wbc::REC_DOUBLES;
  const double2* m = reinterpret_cast<const double2*>(r + wbc::REC_Y);
  int pstatus = 0;                 // (the reduce kernel has set the same bit in the record's status word)
  const wbc::ParamRec& pr = wbc::param_record(p, inst, pstatus);
  pdl_wait();
  const double2 m2 = m[2];
  const bool ok = m2.x != 0.0;
  if (ok && lane == 0) bulk_load(&s.Y[0][0], r, REC_Y_BYTES, &s.mbar);
  const double2 m0 = m[0], m1 = m[1], m3 = m[3], m4 = m[4], m5 = m[5];
  wbc::StepCarry c;
  c.status = (int)m0.x | pstatus; c.cmask = (unsigned)m0.y; c.nf = (int)m1.x; c.nextra = (int)m1.y;
  c.ok = ok; c.pc_ok = m2.y != 0.0; c.extra_bound = m3.x; c.err = m3.y; c.Vl = m4.x; c.PFl = m4.y; c.csum = m5.x; c.Vpc = m5.y;
  __syncwarp();
  if (ok) mbar_wait(&s.mbar, 0);
  wbc::solve_instance<KIND, wbc::SolveSmemT<VD>>(s, gdc->md, pr.pr, a, inst, lane, c, vdmap ? vdmap + inst * wbc::VDMAP_DOUBLES : nullptr, r);
}

template <int W>
__global__ void __launch_bounds__(W * 32, WBC_PC_MIN_WARPS / W) wbc_reduce_pc_params_kernel(const DevConst* __restrict__ gdc, wbc::ParamArgs p,
                                                                                          wbc::StepArgs a, double* __restrict__ rec,
                                                                                          double* __restrict__ vdmap, int bulk_ok) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemLayoutPCParamsT<W>* sm = reinterpret_cast<SmemLayoutPCParamsT<W>*>(smem_raw);
  pdl_launch_dependents();
  const bool staged = stage_inputs_issue(sm->in, a, bulk_ok != 0);
  const int warp = W == 1 ? 0 : (int)(threadIdx.x >> 5), lane = lane_index();
  const int pstatus = stage_params<W>(sm, gdc, p, a.n, warp);
  const long long inst = (long long)blockIdx.x * W + warp;
  if (inst >= a.n) return;
  wbc::WarpSmem& s = sm->w[warp];
  const wbc::ParamRec& pr = sm->prm[warp];
  wbc::StepCarry c;
  const wbc::StagedInputs in = staged_rows(sm->in, warp);
  if (staged) mbar_wait(&sm->in.mbar, 0);
  {
    // the meeting points of wbc_reduce_pc_kernel
    const long long first = (long long)blockIdx.x * W;
    const int n_act = (int)((a.n - first) < W ? (a.n - first) : W);
    int n_pc = 0;
    for (int w = 0; w < n_act; ++w) {
      const uint8_t* cp = (staged && in.contact) ? sm->in.contact + w * 4 : a.contact + (first + w) * 4;
      n_pc += (cp[0] | cp[1] | cp[2] | cp[3]) ? 1 : 0;
    }
    sm->pc[warp].sync_all = 32 * n_act;
    sm->pc[warp].sync_pc = 32 * n_pc;
  }
  wbc::reduce_instance<WBC_CTRL_PC>(s, sm->mc.md, pr.pr, pr.dv, a, inst, lane, c, &sm->pc[warp], vdmap ? vdmap + inst * wbc::VDMAP_DOUBLES : nullptr,
                                    staged ? &in : nullptr);
  c.status |= pstatus;
  __syncwarp();
  if (lane == 0) store_record(rec + inst * wbc::REC_DOUBLES, c, s);
}

__global__ void wbc_pd_params_kernel(const DevConst* __restrict__ gdc, wbc::ParamArgs p, const double* q, const double* v, double* tau,
                                     int32_t* status, long long n) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n * WBC_NU) wbc::pd_params_element(gdc->md, p, q, v, tau, status, t / WBC_NU, (int)(t % WBC_NU));
}

// Register-resident DFMA loop: 8 independent chains per thread, 2 flop per FMA.
__global__ void fp64_peak_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------------------ resource owners
// Every device resource of the library is held by one of these and released in its destructor, on whatever device is
// current then (the owners of a handle or a plan select theirs first).

// Device array that only grows: reserve(n) reallocates, without keeping the contents, when n exceeds the capacity.
template <typename T>
struct DevArray {
  T* p = nullptr;
  size_t cap = 0;
  DevArray() = default;
  DevArray(const DevArray&) = delete;
  DevArray& operator=(const DevArray&) = delete;
  ~DevArray() { if (p) cudaFree(p); }
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    const cudaError_t e = cudaMalloc(&p, n * sizeof(T));
    if (e == cudaSuccess) cap = n;
    return e;
  }
};

// A stream, event, graph or graph exec; created through &v.
template <typename R, cudaError_t (*Destroy)(R)>
struct Owned {
  R v = nullptr;
  Owned() = default;
  Owned(const Owned&) = delete;
  Owned& operator=(const Owned&) = delete;
  ~Owned() { if (v) Destroy(v); }
  operator R() const { return v; }
};
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;
using Event = Owned<cudaEvent_t, cudaEventDestroy>;
using Graph = Owned<cudaGraph_t, cudaGraphDestroy>;
using GraphExec = Owned<cudaGraphExec_t, cudaGraphExecDestroy>;

// Instances per reduce / solve launch pair of the split path: bounds the hand-over scratch (4224 B per instance) at 1.1 GB
// while each kernel still runs for milliseconds, so the drain at the kernel boundaries stays below ~1 % of the step.
constexpr int64_t SPLIT_CHUNK = 262144;

// Hand-over scratch of the split step (reduce -> solve) for one stream lane, and the ordering of its users: the stream of
// the last step that used it.
struct Slot {
  DevArray<double> rec, vdmap;
  cudaStream_t last_stream = nullptr;
  bool used = false;
  // Records (and the accelerations of the vd outputs) for min(n, SPLIT_CHUNK) instances. Never grows inside a stream
  // capture: callers that capture reserve first.
  cudaError_t reserve(int64_t n, bool with_vd) {
    const int64_t m = std::min(n, SPLIT_CHUNK);
    cudaError_t e = rec.reserve(m * wbc::REC_DOUBLES);
    if (e == cudaSuccess && with_vd) e = vdmap.reserve(m * wbc::VDMAP_DOUBLES);
    return e;
  }
};

// Device rows of wbc_step_host and wbc_step_plan_host, for n instances.
struct Staging {
  DevArray<double> q, v, traj, tau, metrics, vd, f, info, lam;
  DevArray<uint8_t> contact;
  DevArray<int32_t> status;
  DevArray<int32_t> index;             // parameter-set index of wbc_step_params_host (reserved by that entry only)
  cudaError_t reserve(int64_t n) {
    cudaError_t e = q.reserve(n * WBC_NQ);
    if (e == cudaSuccess) e = v.reserve(n * WBC_NV);
    if (e == cudaSuccess) e = traj.reserve(n * WBC_NTRAJ);
    if (e == cudaSuccess) e = contact.reserve(n * 4);
    if (e == cudaSuccess) e = tau.reserve(n * WBC_NU);
    if (e == cudaSuccess) e = metrics.reserve(n * WBC_NMETRIC);
    if (e == cudaSuccess) e = status.reserve(n);
    if (e == cudaSuccess) e = vd.reserve(n * WBC_NV);
    if (e == cudaSuccess) e = f.reserve(n * 12);
    if (e == cudaSuccess) e = info.reserve(n * 4);
    if (e == cudaSuccess) e = lam.reserve(n * WBC_NLAM);
    return e;
  }
};

// Scratch of wbc_rollout and wbc_step_plan_host, for n instances: the sampled targets, the outputs the caller does not
// keep, and the step counter of the metrics log.
struct RolloutScratch {
  DevArray<double> traj, vd, metrics, tau, t;
  DevArray<uint8_t> contact;
  DevArray<int32_t> status;
  DevArray<int> counter;
  cudaError_t reserve(int64_t n) {
    cudaError_t e = counter.reserve(1);
    if (e == cudaSuccess) e = traj.reserve(n * WBC_NTRAJ);
    if (e == cudaSuccess) e = vd.reserve(n * WBC_NV);
    if (e == cudaSuccess) e = metrics.reserve(n * WBC_NMETRIC);
    if (e == cudaSuccess) e = tau.reserve(n * WBC_NU);
    if (e == cudaSuccess) e = t.reserve(n);
    if (e == cudaSuccess) e = contact.reserve(n * 4);
    if (e == cudaSuccess) e = status.reserve(n);
    return e;
  }
};

// Scratch of the loop entries (wbc_rollout_loop, wbc_loop_observe), reserved by them only: the observed state, the applied
// torque and the loop state of a call that brings none.
struct LoopScratch {
  DevArray<double> q_obs, v_obs, applied, hist;
  DevArray<long long> tick;
  cudaError_t reserve(int64_t n, bool own_state) {
    cudaError_t e = q_obs.reserve(n * WBC_NQ);
    if (e == cudaSuccess) e = v_obs.reserve(n * WBC_NV);
    if (e == cudaSuccess) e = applied.reserve(n * WBC_NU);
    if (e == cudaSuccess && own_state) e = hist.reserve(n * WBC_LOOP_HIST * WBC_NU);
    if (e == cudaSuccess && own_state) e = tick.reserve(n);
    return e;
  }
};

// Scratch of the monitor entries (wbc_rollout_monitor), reserved by them only: the plant's per-step status word, and its ground
// forces when the caller keeps none.
struct MonScratch {
  DevArray<int32_t> word;
  DevArray<double> f;
  cudaError_t reserve(int64_t n, bool own_f) {
    cudaError_t e = word.reserve(n);
    if (e == cudaSuccess && own_f) e = f.reserve(n * 12);
    return e;
  }
};

// Scratch of the motor entries (wbc_rollout_motor), reserved by them only: the plant input, and the motor state of a call that
// brings none.
struct MotorScratch {
  DevArray<double> plant, tau_m;
  DevArray<long long> count;
  cudaError_t reserve(int64_t n, bool own_state) {
    cudaError_t e = plant.reserve(n * WBC_NU);
    if (e == cudaSuccess && own_state) e = tau_m.reserve(n * WBC_NU);
    if (e == cudaSuccess && own_state) e = count.reserve(n);
    return e;
  }
};

// Scratch of the estimator entries (wbc_rollout_estimator), reserved by them only: the filter state of a call that brings none.
struct EstScratch {
  DevArray<double> x, P, v_prev;
  DevArray<long long> count;
  cudaError_t reserve(int64_t n) {
    cudaError_t e = x.reserve(n * wbcest::NX);
    if (e == cudaSuccess) e = P.reserve(n * wbcest::NX * wbcest::NX);
    if (e == cudaSuccess) e = v_prev.reserve(n * 3);
    if (e == cudaSuccess) e = count.reserve(n);
    return e;
  }
};

}  // namespace

constexpr int WBC_NSLOT = 4;
struct wbc_handle {
  int device = 0;
  DevArray<DevConst> d_const;
  wbc_model model;
  wbc_params params;
  DevArray<wbcplant::PlantVariant> d_nominal;   // the handle's model as the one variant of a perturbed step without a set
  DevArray<wbc::ParamRec> d_params;            // the handle's params as the one record of a parameter step without a set
  std::string err;
  int64_t launches = 0;
  int sm_count = 148;
  DevArray<int> d_tau_map;             // message slot (velocity order) -> actuator index, for wbc_lcm_encode_robot_state
  // internal streams: lane 0 serves the host entries, lanes 0-1 the host pipelines, lanes 1.. chunks 1.. of a device step
  // (its chunk 0 runs on the caller's stream); slot[i] is the hand-over scratch of the chain on lane i
  Stream lane[WBC_NSLOT];
  Slot slot[WBC_NSLOT];
  Event order_ev, join_ev;
  Event prof_ev[3];                    // wbc_profile_step: before reduce / between / after solve
  Staging stage;
  RolloutScratch ro;
  LoopScratch loop;
  MonScratch mon;
  MotorScratch motor;
  EstScratch est;
  ~wbc_handle() { cudaSetDevice(device); }   // the members are released after this, on the handle's device
};

#define WBC_CUDA(h, call)                                                                       \
  do {                                                                                          \
    cudaError_t e_ = (call);                                                                    \
    if (e_ != cudaSuccess) {                                                                    \
      (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                            \
      return WBC_ERR_CUDA;                                                                      \
    }                                                                                           \
  } while (0)

static int fail_arg(wbc_handle* h, const char* msg) {
  if (h) h->err = msg;
  return WBC_ERR_ARG;
}

extern "C" int wbc_default_params(wbc_params* p) {
  if (!p) return WBC_ERR_ARG;
  memset(p, 0, sizeof(*p));
  p->id_kp_body_p = 500; p->id_kd_body_p = 50; p->id_kp_body_rpy = 500; p->id_kd_body_rpy = 50;
  p->id_kp_foot = 100; p->id_kd_foot = 20; p->id_w_body = 10; p->id_w_foot = 1;
  p->clf_q_body_p = 5000; p->clf_q_body_pd = 200; p->clf_q_body_rpy = 5000; p->clf_q_body_rpyd = 200;
  p->clf_q_foot_p = 200; p->clf_q_foot_pd = 20; p->clf_r = 1; p->clf_w_delta = 1000;
  p->pc_kp_body_p = 100; p->pc_kd_body_p = 10; p->pc_kp_body_rpy = 100; p->pc_kd_body_rpy = 10;
  p->pc_kp_foot = 200; p->pc_kd_foot = 20; p->pc_w_body = 10; p->pc_w_foot = 1;
  p->mu = 0.7; p->contact_damping = 100; p->reg_f = 1e-6; p->reg_tau = 0; p->reg_vd = 0;
  p->torque_limits = 0; p->max_iter = 200;
  p->pd_kp = 30; p->pd_kd = 1.5; p->pd_clip = 150;
  for (int l = 0; l < 4; ++l) { p->pd_q_nom[3 * l] = 0.0; p->pd_q_nom[3 * l + 1] = -0.8; p->pd_q_nom[3 * l + 2] = 1.6; }   // basic_controller.py:335-340
  return WBC_OK;
}

static int set_smem_attr(wbc_handle* h) {
  const int bytes = (int)sizeof(SmemLayout);
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_kernel<WBC_CTRL_ID, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_kernel<WBC_CTRL_CLF, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_kernel<WBC_CTRL_ID, WARPS_HOST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutT<WARPS_HOST>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_kernel<WBC_CTRL_CLF, WARPS_HOST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutT<WARPS_HOST>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_pc_kernel<WARPS_PC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutPCT<WARPS_PC>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_kernel<WBC_CTRL_ID, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<false>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_kernel<WBC_CTRL_CLF, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<false>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_kernel<WBC_CTRL_PC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<false>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_kernel<WBC_CTRL_ID, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<true>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_kernel<WBC_CTRL_CLF, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<true>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_kernel<WBC_CTRL_PC, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<true>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_coriolis_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutPC)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_dynamics_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_plant_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutPlant)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_plant_variant_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutPlantVariant)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_plant_terrain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutPlantTerrain)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_params_kernel<WBC_CTRL_ID, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutParamsT<WARPS>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_params_kernel<WBC_CTRL_CLF, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutParamsT<WARPS>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_params_kernel<WBC_CTRL_ID, WARPS_HOST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutParamsT<WARPS_HOST>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_params_kernel<WBC_CTRL_CLF, WARPS_HOST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutParamsT<WARPS_HOST>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_reduce_pc_params_kernel<WARPS_PC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutPCParamsT<WARPS_PC>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_params_kernel<WBC_CTRL_ID, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<false>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_params_kernel<WBC_CTRL_CLF, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<false>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_params_kernel<WBC_CTRL_PC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<false>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_params_kernel<WBC_CTRL_ID, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<true>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_params_kernel<WBC_CTRL_CLF, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<true>)));
  WBC_CUDA(h, cudaFuncSetAttribute(wbc_solve_params_kernel<WBC_CTRL_PC, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemLayoutSolveT<true>)));
  return WBC_OK;
}

extern "C" int wbc_create(const wbc_model* model, const wbc_params* params, int device, wbc_handle** out) {
  if (!model || !out) return WBC_ERR_ARG;
  wbc_handle* h = new (std::nothrow) wbc_handle();
  *out = h;                            // handed back even when creation fails part-way, so that wbc_last_error works
  if (!h) return WBC_ERR_NOMEM;
  h->device = device;
  if (params) h->params = *params; else wbc_default_params(&h->params);
  if (h->params.reg_vd != 0.0) return fail_arg(h, "reg_vd is not supported yet (must be 0)");
  if (!(h->params.reg_f > 0.0)) return fail_arg(h, "reg_f must be > 0 (tie-break that makes the QP strictly convex)");
  for (int k = 0; k < WBC_NU; ++k) {
    if (model->v_index[k] < 6 || model->v_index[k] >= WBC_NV || model->act_index[k] < 0 || model->act_index[k] >= WBC_NU)
      return fail_arg(h, "wbc_model: v_index/act_index out of range");
  }
  WBC_CUDA(h, cudaSetDevice(device));
  DevConst hc;
  hc.md = *model; hc.pr = h->params;
  wbc::derive_constants(h->params, hc.dv);
  WBC_CUDA(h, h->d_const.reserve(1));
  WBC_CUDA(h, cudaMemcpy(h->d_const.p, &hc, sizeof(DevConst), cudaMemcpyHostToDevice));
  h->model = *model;
  wbcplant::PlantVariant nominal{*model, 0.0};
  WBC_CUDA(h, h->d_nominal.reserve(1));
  WBC_CUDA(h, cudaMemcpy(h->d_nominal.p, &nominal, sizeof(nominal), cudaMemcpyHostToDevice));
  const wbc::ParamRec own{hc.pr, hc.dv};
  WBC_CUDA(h, h->d_params.reserve(1));
  WBC_CUDA(h, cudaMemcpy(h->d_params.p, &own, sizeof(own), cudaMemcpyHostToDevice));
  // the streams and events: created here, not on first use, so that a step never calls a resource-creating API while some
  // other stream of the process is being captured
  for (Stream& s : h->lane) WBC_CUDA(h, cudaStreamCreateWithFlags(&s.v, cudaStreamNonBlocking));
  WBC_CUDA(h, cudaEventCreateWithFlags(&h->order_ev.v, cudaEventDisableTiming));
  WBC_CUDA(h, cudaEventCreateWithFlags(&h->join_ev.v, cudaEventDisableTiming));
  for (Event& e : h->prof_ev) WBC_CUDA(h, cudaEventCreate(&e.v));
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) h->sm_count = prop.multiProcessorCount;
  int tmap[WBC_NU];
  for (int k = 0; k < WBC_NU; ++k) tmap[model->v_index[k] - 6] = model->act_index[k];
  WBC_CUDA(h, h->d_tau_map.reserve(WBC_NU));
  WBC_CUDA(h, cudaMemcpy(h->d_tau_map.p, tmap, sizeof(tmap), cudaMemcpyHostToDevice));
  return set_smem_attr(h);
}

extern "C" int wbc_destroy(wbc_handle* h) {
  delete h;
  return WBC_OK;
}

extern "C" const char* wbc_last_error(const wbc_handle* h) { return h ? h->err.c_str() : "null handle"; }
extern "C" int64_t wbc_launch_count(const wbc_handle* h) { return h ? h->launches : 0; }

extern "C" int wbc_dynamics(wbc_handle* h, int64_t n, const double* q, const double* v, double* M, double* Cv,
                            double* taug, double* Jfeet, double* Jdv, double* pfeet, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!q || !v))) return fail_arg(h, "wbc_dynamics: null input");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbc::DynOut o{M, Cv, taug, Jfeet, Jdv, pfeet};
  const unsigned grid = (unsigned)((n + WARPS - 1) / WARPS);
  wbc_dynamics_kernel<<<grid, WARPS * 32, sizeof(SmemLayout), (cudaStream_t)stream>>>(h->d_const.p, q, v, o, n);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_coriolis(wbc_handle* h, int64_t n, const double* q, const double* v, double* Cm, double* Jd, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!q || !v))) return fail_arg(h, "wbc_coriolis: null input");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  const unsigned grid = (unsigned)((n + WARPS - 1) / WARPS);
  wbc_coriolis_kernel<<<grid, WARPS * 32, sizeof(SmemLayoutPC), (cudaStream_t)stream>>>(h->d_const.p, q, v, Cm, Jd, n);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

#define WBC_SCRATCH_CHECK(h, s)                                                                  \
  do {                                                                                           \
    if ((s).err != cudaSuccess) { (h)->err = std::string("host-buffer entry: ") + cudaGetErrorString((s).err); return WBC_ERR_CUDA; } \
  } while (0)

namespace {
// Device copies of the host arrays of one host-buffer entry, on the stream `st`. Each array is recorded once, with its
// element count: in() uploads it, out() downloads it in finish(), inout() does both. A null host array stays null. The
// device memory is freed when the scope ends (early error returns included).
struct DevScratch {
  struct Copy { DevArray<unsigned char> dev; void* back = nullptr; size_t bytes = 0; };
  cudaStream_t st;
  std::deque<Copy> copies;             // (a deque never moves its elements)
  cudaError_t err = cudaSuccess;
  explicit DevScratch(cudaStream_t s) : st(s) {}
  template <typename T> T* in(const T* host, size_t count) { return add(host, (T*)nullptr, count); }
  template <typename T> T* out(T* host, size_t count) { return add((const T*)nullptr, host, count); }
  template <typename T> T* inout(T* host, size_t count) { return add((const T*)host, host, count); }
  // After the launch: downloads every out / inout array, waits for the stream and reports the first error.
  int finish(wbc_handle* h) {
    for (const Copy& c : copies)
      if (c.back && err == cudaSuccess) err = cudaMemcpyAsync(c.back, c.dev.p, c.bytes, cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);
    WBC_SCRATCH_CHECK(h, *this);
    return WBC_OK;
  }

 private:
  template <typename T> T* add(const T* up, T* back, size_t count) {
    if ((!up && !back) || err != cudaSuccess) return nullptr;
    Copy& c = copies.emplace_back();
    c.back = back; c.bytes = count * sizeof(T);
    err = c.dev.reserve(c.bytes > 0 ? c.bytes : 1);
    if (err == cudaSuccess && up) err = cudaMemcpyAsync(c.dev.p, up, c.bytes, cudaMemcpyHostToDevice, st);
    return err == cudaSuccess ? reinterpret_cast<T*>(c.dev.p) : nullptr;
  }
};
}  // namespace

extern "C" int wbc_coriolis_host(wbc_handle* h, int64_t n, const double* q, const double* v, double* Cm, double* Jd) {
  if (!h) return WBC_ERR_ARG;
  if (n <= 0) return n == 0 ? WBC_OK : fail_arg(h, "wbc_coriolis_host: n < 0");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const double* dq = s.in(q, N * WBC_NQ); const double* dv = s.in(v, N * WBC_NV);
  double* dC = s.out(Cm, N * 324); double* dJ = s.out(Jd, N * 216);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_coriolis(h, n, dq, dv, dC, dJ, s.st);
  return rc ? rc : s.finish(h);
}

extern "C" int wbc_step_pd(wbc_handle* h, int64_t n, const double* q, const double* v, double* tau, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!q || !v || !tau))) return fail_arg(h, "wbc_step_pd: null buffer");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  const long long total = (long long)n * WBC_NU;
  wbc_pd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->d_const.p, q, v, tau, n);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// ------------------------------------------------------------------------------ launch schedule
// Which kernels a step entry point issues, by batch size. The thresholds were measured on B200 (profiles/README.md); an
// experiment with them is a local edit built as a variant (tools/sweep_variants.sh).

// Programmatic dependent launch of the solve kernel (its CTAs become resident while the last reduce CTAs run): +1.5 % at 4096
// instances, neutral above; never inside a stream capture, and not for chains below 4096 instances that run beside other
// chains of the same step (chunked issue): there the early-resident solve CTAs take the slots the other chunk's reduce CTAs
// need (-22 % at 2 x 2048). A lone chain gains at every size (+3-4 % at 64 - 1024).
static bool use_pdl(int64_t m, bool beside_others) { return !beside_others || m >= 4096; }

// wbc_step: small batches go through as chunks of about 2048 instances, independent reduce -> solve chains on as many streams
// (the caller's and internal ones, joined by events): the solve kernel of one chunk overlaps the reduce kernel and the
// ramp-down of the others. Measured against one chain: +5.5 % at 4096 instances (2 chunks; 3: +4.5 %, 4: +2.5 %), +7.7 % at
// 8192 (4 chunks; 2: +4.1 %), +2.6 % at 16384, +1 % at 65536, -2 % at 2048. Never inside a stream capture.
constexpr int64_t CHUNKED_STEP_MIN = 4096, CHUNKED_STEP_MAX = 65536;
constexpr int device_step_chunks(int64_t n) { return n >= 7168 ? 4 : n >= 5120 ? 3 : 2; }
static_assert(device_step_chunks(CHUNKED_STEP_MAX) <= WBC_NSLOT, "every chunk needs its own stream and hand-over slot");

// wbc_step_host on page-locked buffers: reading the inputs over the host link from the SMs (zero-copy, ~32 GB/s) wins up to
// ~48 k instances per call (no staging copies, no extra API calls); above that the inputs go through the copy engine
// (~55 GB/s) in a chunked two-stream pipeline. Page-locked outputs are written straight to host memory in both modes.
//  * below 24576 instances the reduce kernel reads its inputs over the host link (zero-copy), two halves from 4096 on:
//    the solve kernel of one half overlaps the link-bound reduce kernel of the other (e2e +4.6 % at 4096, +3.8 % at
//    16384; three or more chunks lose);
//  * above, the inputs go through the copy engine into device staging and the single-warp reduce CTAs read resident
//    inputs: e2e +5 % at 32768, +16 % at 65536, +10 % at 2^17 - 2^20.
// PC / MPTC are compute bound at a third of the rate: the zero-copy reads hide under the reduce kernel up to 131072
// instances (e2e 22.3 M steps/s against 20.0 M staged at 65536)
static bool stage_pinned_inputs(int kind, int64_t n) { return n >= (kind == WBC_CTRL_PC || kind == WBC_CTRL_MPTC ? 131072 : 24576); }
// staged: four chunks below 98304 instances, then chunks of n / 8 clamped to [16384, 32768] instances
static int pinned_chunks(int64_t n, bool staged) {
  if (!staged) return n >= 4096 ? 2 : 1;
  if (n < 98304) return 4;
  const int64_t per = std::clamp<int64_t>(n / 8, 16384, 32768);
  return (int)((n + per - 1) / per);
}

// wbc_step_host on pageable buffers: chunked two-stream pipeline, the upload of chunk c + 1 overlaps the kernel of chunk c,
// the download of chunk c the kernel of chunk c + 1 (separate copy engines); small batches go through in one piece.
// chunk = n / 8 clamped to [8192, 65536] instances: short pipeline fill, copies long enough for the copy engines
static int pageable_chunks(int64_t n) {
  if (n < 32768) return n >= 2048 ? 2 : 1;
  const int64_t per = std::clamp<int64_t>(n / 8, 8192, 65536);
  return (int)std::min<int64_t>((n + per - 1) / per, 64);
}

// wbc_sample_trajectory, instances per warp: 32 (lane = instance) is the throughput shape; small batches are latency bound on
// the 14 dependent binary searches per instance, so they spread them over 4 or 16 lanes per instance (rollout of 4096 robots:
// 45.2 / 48.7 / 49.7 M robot-steps/s with 32 / 8 / 2)
static int sample_ipw(int64_t n) { return n >= 32768 ? 32 : n >= 8192 ? 8 : 2; }

// ------------------------------------------------------------------------------ step issue
// How the chains of one step are issued; the entry point decides, launch_split follows.
struct Issue {
  bool host_mapped = false;     // the reduce kernel reads page-locked host memory: 4-warp CTAs, every array staged per CTA
  bool beside_others = false;   // the chain runs beside other chains of the same step (chunked issue)
  bool profile = false;         // wbc_profile_step: events before the reduce kernel, between the kernels, after the solve kernel
};

// The instances from `o` on of a per-instance array with `width` elements per instance; a null array stays null.
template <typename T>
static T* rows_at(T* p, int64_t o, int width) { return p ? p + o * width : nullptr; }
// ... of every array of `io`
static wbc_io io_at(const wbc_io& io, int64_t o) {
  auto at = [o](auto* p, int width) { return rows_at(p, o, width); };
  return wbc_io{at(io.q, WBC_NQ), at(io.v, WBC_NV), at(io.traj, WBC_NTRAJ), at(io.contact, 4), at(io.tau, WBC_NU),
                at(io.metrics, WBC_NMETRIC), at(io.status, 1), at(io.vd, WBC_NV), at(io.f, 12), at(io.qp_info, 4), at(io.lam, WBC_NLAM)};
}
// ... of the set indices of a parameter step
static wbc::ParamArgs params_at(const wbc::ParamArgs& p, int64_t o) { return wbc::ParamArgs{p.set, rows_at(p.index, o, 1), p.n_sets}; }
static wbc::StepArgs step_args(const wbc_io& io, int64_t m, int kind) {
  return wbc::StepArgs{io.q, io.v, io.traj, io.contact, io.tau, io.metrics, io.status, io.vd, io.f, io.qp_info, io.lam, (long long)m, kind};
}

// Splits [0, n) into k chunks of a multiple of 4 instances, the last one shorter, and calls f(c, offset, count) for each
// non-empty one; stops at the first error f returns. The rounding keeps the CTA-level bulk copies of 4-warp reduce CTAs
// on 16-byte boundaries.
template <typename F>
static int for_each_chunk(int64_t n, int k, F f) {
  const int64_t per = ((n + k - 1) / k + 3) & ~(int64_t)3;
  for (int c = 0; c < k && c * per < n; ++c) {
    const int rc = f(c, c * per, std::min(per, n - c * per));
    if (rc) return rc;
  }
  return WBC_OK;
}

// Device aliases of page-locked host buffers (wbc_host_alloc / cudaHostRegister): when every non-null pointer is page-locked,
// replaces each by the address the kernels read and write it through and returns true; otherwise changes nothing and
// returns false.
template <typename... T>
static bool to_device_aliases(T*&... p) {
  const void* host[] = {p...};
  void* dev[sizeof...(T)] = {};
  for (size_t i = 0; i < sizeof...(T); ++i) {
    if (!host[i]) continue;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host[i]) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
      cudaGetLastError();
      return false;
    }
    dev[i] = at.devicePointer;
  }
  size_t i = 0;
  ((p = static_cast<T*>(dev[i++])), ...);
  return true;
}

// Streams to[0 .. k) wait for everything submitted to `from` so far: the fork of chunk streams from the caller's stream and
// the join of a chunk stream back into it, through an event of the handle (created with it, so never inside a capture).
static int streams_wait(wbc_handle* h, cudaEvent_t ev, cudaStream_t from, const cudaStream_t* to, int k) {
  WBC_CUDA(h, cudaEventRecord(ev, from));
  for (int i = 0; i < k; ++i) WBC_CUDA(h, cudaStreamWaitEvent(to[i], ev, 0));
  return WBC_OK;
}

static bool capturing(cudaStream_t st) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cap);
  return cap != cudaStreamCaptureStatusNone;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// The hand-over scratch of a slot belongs to one step at a time. A step on another stream than the slot's previous user is
// ordered behind everything submitted to that stream so far (event dependency; never inside a stream capture, where the
// caller owns the ordering).
static int order_slot(wbc_handle* h, Slot& s, cudaStream_t st) {
  if (s.used && s.last_stream != st && !capturing(st)) {
    if (cudaEventRecord(h->order_ev, s.last_stream) == cudaSuccess) WBC_CUDA(h, cudaStreamWaitEvent(st, h->order_ev, 0));
    else cudaGetLastError();      // the previous stream no longer exists: its work has completed
  }
  s.used = true;
  s.last_stream = st;
  return WBC_OK;
}

// pa != nullptr: the parameter-aware kernels with these per-robot parameters (the index array is sliced with the chunk).
template <int KIND>
static int launch_split(wbc_handle* h, int kind, int64_t n, const wbc_io& io, cudaStream_t st, int slot, Issue is,
                        const wbc::ParamArgs* pa) {
  Slot& sl = h->slot[slot];
  WBC_CUDA(h, sl.reserve(n, io.vd != nullptr));
  const int rc = order_slot(h, sl, st);
  if (rc) return rc;
  const DevConst* dc = h->d_const.p;
  double* rec = sl.rec.p;
  double* vdmap = io.vd ? sl.vdmap.p : nullptr;
  for (int64_t o = 0; o < n; o += SPLIT_CHUNK) {
    const int64_t m = (n - o) < SPLIT_CHUNK ? (n - o) : SPLIT_CHUNK;
    const wbc::StepArgs a = step_args(io_at(io, o), m, kind);
    const wbc::ParamArgs p = pa ? params_at(*pa, o) : wbc::ParamArgs{};
    // bulk input staging needs 16-byte aligned rows at the CTA boundaries (chunk offsets are multiples of 4)
    const bool al_vt = aligned16(a.v) && aligned16(a.traj), al_qc = aligned16(a.q) && aligned16(a.contact);
    if (is.profile) cudaEventRecord(h->prof_ev[0], st);
    if (is.host_mapped || KIND == WBC_CTRL_PC) {   // zero-copy call of wbc_step_host: 4-warp CTAs, every array staged per CTA
                                                   // (PC / MPTC too: 20.0 vs 19.7 M steps/s with single-warp CTAs)
      constexpr int W = (KIND == WBC_CTRL_PC) ? WARPS_PC : WARPS_HOST;
      const unsigned grid = (unsigned)((m + W - 1) / W);
      const int bulk_ok = al_vt && al_qc;
      if constexpr (KIND == WBC_CTRL_PC) {
        if (pa) wbc_reduce_pc_params_kernel<W><<<grid, W * 32, sizeof(SmemLayoutPCParamsT<W>), st>>>(dc, p, a, rec, vdmap, bulk_ok);
        else wbc_reduce_pc_kernel<W><<<grid, W * 32, sizeof(SmemLayoutPCT<W>), st>>>(dc, a, rec, vdmap, bulk_ok);
      } else if (pa) {
        wbc_reduce_params_kernel<KIND, W><<<grid, W * 32, sizeof(SmemLayoutParamsT<W>), st>>>(dc, p, a, rec, vdmap, bulk_ok);
      } else {
        wbc_reduce_kernel<KIND, W><<<grid, W * 32, sizeof(SmemLayoutT<W>), st>>>(dc, a, rec, vdmap, bulk_ok);
      }
    } else {
      constexpr int W = WARPS;
      const unsigned grid = (unsigned)((m + W - 1) / W);
      const int bulk_ok = al_vt;
      if constexpr (KIND != WBC_CTRL_PC) {
        if (pa) wbc_reduce_params_kernel<KIND, W><<<grid, W * 32, sizeof(SmemLayoutParamsT<W>), st>>>(dc, p, a, rec, vdmap, bulk_ok);
        else wbc_reduce_kernel<KIND, W><<<grid, W * 32, sizeof(SmemLayoutT<W>), st>>>(dc, a, rec, vdmap, bulk_ok);
      }
    }
    if (is.profile) cudaEventRecord(h->prof_ev[1], st);
    const unsigned sgrid = (unsigned)((m + SOLVE_WARPS - 1) / SOLVE_WARPS);
    const bool pdl = use_pdl(m, is.beside_others) && !capturing(st);
    const bool with_vd = io.vd != nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(sgrid); cfg.blockDim = dim3(SOLVE_WARPS * 32); cfg.stream = st;
    cfg.dynamicSmemBytes = with_vd ? sizeof(SmemLayoutSolveT<true>) : sizeof(SmemLayoutSolveT<false>);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    const double* crec = rec;
    const double* cvd = vdmap;
    if (pa && with_vd) WBC_CUDA(h, cudaLaunchKernelEx(&cfg, wbc_solve_params_kernel<KIND, true>, dc, p, a, crec, cvd));
    else if (pa) WBC_CUDA(h, cudaLaunchKernelEx(&cfg, wbc_solve_params_kernel<KIND, false>, dc, p, a, crec, cvd));
    else if (with_vd) WBC_CUDA(h, cudaLaunchKernelEx(&cfg, wbc_solve_kernel<KIND, true>, dc, a, crec, cvd));
    else WBC_CUDA(h, cudaLaunchKernelEx(&cfg, wbc_solve_kernel<KIND, false>, dc, a, crec, cvd));
    if (is.profile) cudaEventRecord(h->prof_ev[2], st);
    h->launches += 2;
  }
  return WBC_OK;
}

// One control step = reduce kernel (per controller kind) + solve kernel, stream ordered; `slot` selects the hand-over scratch
// (the host pipelines run two streams side by side); pa: per-robot parameters (nullptr: the handle's).
static int step_launch(wbc_handle* h, int kind, int64_t n, const wbc_io& io, cudaStream_t st, int slot, Issue is,
                       const wbc::ParamArgs* pa = nullptr) {
  int rc = WBC_OK;
  switch (kind) {
    case WBC_CTRL_ID: rc = launch_split<WBC_CTRL_ID>(h, kind, n, io, st, slot, is, pa); break;
    case WBC_CTRL_CLF: rc = launch_split<WBC_CTRL_CLF>(h, kind, n, io, st, slot, is, pa); break;
    case WBC_CTRL_PC:
    case WBC_CTRL_MPTC: rc = launch_split<WBC_CTRL_PC>(h, kind, n, io, st, slot, is, pa); break;   // MPTC: a.kind drops the passivity row
    default: return fail_arg(h, "wbc_step: unknown controller kind");
  }
  if (rc) return rc;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// The PD law on device rows; with pa, each robot's gains (and its status word when io.status is given).
static int pd_launch(wbc_handle* h, int64_t n, const wbc_io& io, const wbc::ParamArgs* pa, cudaStream_t st) {
  if (!pa) return wbc_step_pd(h, n, io.q, io.v, io.tau, st);
  if (n < 0 || (n > 0 && (!io.q || !io.v || !io.tau))) return fail_arg(h, "wbc_step_params: q, v and tau are required");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  const long long total = (long long)n * WBC_NU;
  wbc_pd_params_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(h->d_const.p, *pa, io.q, io.v, io.tau, io.status, n);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// wbc_step on device buffers; `profile` (wbc_profile_step) issues one chain with events around its two kernels; pa:
// per-robot parameters (wbc_step_params), nullptr for the handle's.
static int device_step(wbc_handle* h, int kind, int64_t n, const wbc_io* io, cudaStream_t st, bool profile,
                       const wbc::ParamArgs* pa = nullptr) {
  if (!h) return WBC_ERR_ARG;
  if (!io || n < 0) return fail_arg(h, "wbc_step: bad arguments");
  if (n == 0) return WBC_OK;
  if (kind == WBC_CTRL_PD) return pd_launch(h, n, *io, pa, st);
  if (!io->q || !io->v || !io->traj || !io->contact || !io->tau || !io->metrics || !io->status)
    return fail_arg(h, "wbc_step: q, v, traj, contact, tau, metrics and status are required");
  WBC_CUDA(h, cudaSetDevice(h->device));
  if (profile || n < CHUNKED_STEP_MIN || n > CHUNKED_STEP_MAX || capturing(st))
    return step_launch(h, kind, n, *io, st, 0, Issue{false, false, profile}, pa);
  const int k = device_step_chunks(n);
  cudaStream_t lanes[WBC_NSLOT] = {st};
  for (int c = 1; c < k; ++c) lanes[c] = h->lane[c];
  const int rc = streams_wait(h, h->order_ev, st, lanes + 1, k - 1);
  if (rc) return rc;
  return for_each_chunk(n, k, [&](int c, int64_t o, int64_t m) {
    const wbc::ParamArgs p = pa ? params_at(*pa, o) : wbc::ParamArgs{};
    int r = step_launch(h, kind, m, io_at(*io, o), lanes[c], c, Issue{false, true}, pa ? &p : nullptr);
    if (!r && c) r = streams_wait(h, h->join_ev, lanes[c], &st, 1);
    return r;
  });
}

extern "C" int wbc_step(wbc_handle* h, int kind, int64_t n, const wbc_io* io, void* stream) {
  return device_step(h, kind, n, io, (cudaStream_t)stream, false);
}

#define WBC_STEP_WRAPPER(name, kind)                                                                               \
  extern "C" int name(wbc_handle* h, int64_t n, const double* q, const double* v, const double* traj,              \
                      const uint8_t* contact, double* tau, double* metrics, int32_t* status, void* stream) {       \
    wbc_io io{q, v, traj, contact, tau, metrics, status, nullptr, nullptr, nullptr};                               \
    return wbc_step(h, kind, n, &io, stream);                                                                      \
  }
WBC_STEP_WRAPPER(wbc_step_id, WBC_CTRL_ID)
WBC_STEP_WRAPPER(wbc_step_clf, WBC_CTRL_CLF)
WBC_STEP_WRAPPER(wbc_step_pc, WBC_CTRL_PC)
WBC_STEP_WRAPPER(wbc_step_mptc, WBC_CTRL_MPTC)

// Enqueues one host-buffer step on the handle's two internal streams without waiting for it; `wait` must follow before the
// outputs are read or the next step is enqueued on this handle (wbc_step_host = enqueue + wait; wbc_multi_step_host enqueues on
// every device first and waits afterwards, so the devices run side by side from one host thread).
static int step_host_wait(wbc_handle* h) {
  WBC_CUDA(h, cudaSetDevice(h->device));
  WBC_CUDA(h, cudaStreamSynchronize(h->lane[0]));
  WBC_CUDA(h, cudaStreamSynchronize(h->lane[1]));
  return WBC_OK;
}

// pa: per-robot parameters whose index array is a host array (wbc_step_params_host), nullptr for the handle's. The index is one
// more input: read by the kernels with the others (zero-copy) or copied with them.
static int step_host_enqueue(wbc_handle* h, int kind, int64_t n, const wbc_io* io, const wbc::ParamArgs* pa = nullptr) {
  if (!h) return WBC_ERR_ARG;
  if (!io || n < 0) return fail_arg(h, "wbc_step_host: bad arguments");
  if (n == 0) return WBC_OK;
  const bool pd = kind == WBC_CTRL_PD;
  if (!io->q || !io->v || !io->tau || (!pd && (!io->traj || !io->contact || !io->metrics || !io->status)))
    return fail_arg(h, "wbc_step_host: q, v, traj, contact, tau, metrics and status are required");
  WBC_CUDA(h, cudaSetDevice(h->device));
  const Staging& sg = h->stage;
  // Zero-copy path: when every buffer is page-locked host memory (wbc_host_alloc / cudaHostRegister) the kernel reads
  // its 732 B of inputs and writes its 132 B of outputs per instance straight over the host link - one launch, no
  // staging copies, the transfers of one warp overlap the arithmetic of the others.
  wbc_io hio = *io;
  const int32_t* hidx = pa ? pa->index : nullptr;    // the index array as the kernels read it
  if (to_device_aliases(hio.q, hio.v, hio.traj, hio.contact, hio.tau, hio.metrics, hio.status, hio.vd, hio.f, hio.qp_info, hio.lam, hidx)) {
    // The batch goes through in chunks alternating between the two internal streams (each with its own hand-over scratch); the
    // outputs are written straight to host memory by the solve kernel in every mode. PD takes the chunk count of the staged
    // mode but reads its inputs over the link at every size.
    const bool stage_in = stage_pinned_inputs(kind, n), staged = stage_in && !pd;
    const int k = pinned_chunks(n, stage_in);
    if (staged) {
      WBC_CUDA(h, h->stage.reserve(n));
      hio.q = sg.q.p; hio.v = sg.v.p; hio.traj = sg.traj.p; hio.contact = sg.contact.p;
      if (hidx) {
        WBC_CUDA(h, h->stage.index.reserve(n));
        hidx = sg.index.p;
      }
    }
    const wbc::ParamArgs dpa = pa ? wbc::ParamArgs{pa->set, hidx, pa->n_sets} : wbc::ParamArgs{};
    return for_each_chunk(n, k, [&](int c, int64_t o, int64_t m) {
      const cudaStream_t st = h->lane[c & 1];
      const wbc_io s = io_at(*io, o), d = io_at(hio, o);
      const wbc::ParamArgs sp = pa ? params_at(*pa, o) : wbc::ParamArgs{}, dp = pa ? params_at(dpa, o) : wbc::ParamArgs{};
      if (staged) {
        WBC_CUDA(h, cudaMemcpyAsync((void*)d.q, s.q, m * WBC_NQ * sizeof(double), cudaMemcpyHostToDevice, st));
        WBC_CUDA(h, cudaMemcpyAsync((void*)d.v, s.v, m * WBC_NV * sizeof(double), cudaMemcpyHostToDevice, st));
        WBC_CUDA(h, cudaMemcpyAsync((void*)d.traj, s.traj, m * WBC_NTRAJ * sizeof(double), cudaMemcpyHostToDevice, st));
        WBC_CUDA(h, cudaMemcpyAsync((void*)d.contact, s.contact, m * 4, cudaMemcpyHostToDevice, st));
        if (dp.index) WBC_CUDA(h, cudaMemcpyAsync((void*)dp.index, sp.index, m * sizeof(int32_t), cudaMemcpyHostToDevice, st));
      }
      return pd ? pd_launch(h, m, d, pa ? &dp : nullptr, st) : step_launch(h, kind, m, d, st, c & 1, Issue{!staged, k > 1}, pa ? &dp : nullptr);
    });
  }
  WBC_CUDA(h, h->stage.reserve(n));
  // pageable buffers: the device staging rows, with the optional outputs the caller asked for
  const wbc_io dev{sg.q.p, sg.v.p, sg.traj.p, sg.contact.p, sg.tau.p, sg.metrics.p, sg.status.p, io->vd ? sg.vd.p : nullptr,
                   io->f ? sg.f.p : nullptr, io->qp_info ? sg.info.p : nullptr, io->lam ? sg.lam.p : nullptr};
  const int k = pageable_chunks(n);
  if (pa && pa->index) WBC_CUDA(h, h->stage.index.reserve(n));
  const wbc::ParamArgs dpa = pa ? wbc::ParamArgs{pa->set, pa->index ? sg.index.p : nullptr, pa->n_sets} : wbc::ParamArgs{};
  return for_each_chunk(n, k, [&](int c, int64_t o, int64_t m) {
    const cudaStream_t st = h->lane[c & 1];
    const wbc_io s = io_at(*io, o), d = io_at(dev, o);
    const wbc::ParamArgs sp = pa ? params_at(*pa, o) : wbc::ParamArgs{}, dp = pa ? params_at(dpa, o) : wbc::ParamArgs{};
    WBC_CUDA(h, cudaMemcpyAsync((void*)d.q, s.q, m * WBC_NQ * sizeof(double), cudaMemcpyHostToDevice, st));
    WBC_CUDA(h, cudaMemcpyAsync((void*)d.v, s.v, m * WBC_NV * sizeof(double), cudaMemcpyHostToDevice, st));
    if (dp.index) WBC_CUDA(h, cudaMemcpyAsync((void*)dp.index, sp.index, m * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (!pd) {
      WBC_CUDA(h, cudaMemcpyAsync((void*)d.traj, s.traj, m * WBC_NTRAJ * sizeof(double), cudaMemcpyHostToDevice, st));
      WBC_CUDA(h, cudaMemcpyAsync((void*)d.contact, s.contact, m * 4, cudaMemcpyHostToDevice, st));
    }
    // (the PD law with parameters writes status only where the caller asked for it)
    const wbc_io dpd = pa && !s.status ? wbc_io{d.q, d.v, nullptr, nullptr, d.tau} : d;
    const int r = pd ? pd_launch(h, m, dpd, pa ? &dp : nullptr, st) : step_launch(h, kind, m, d, st, c & 1, Issue{false, k > 1}, pa ? &dp : nullptr);
    if (r) return r;
    if (pd && pa && s.status) WBC_CUDA(h, cudaMemcpyAsync(s.status, d.status, m * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    WBC_CUDA(h, cudaMemcpyAsync(s.tau, d.tau, m * WBC_NU * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (!pd) {
      WBC_CUDA(h, cudaMemcpyAsync(s.metrics, d.metrics, m * WBC_NMETRIC * sizeof(double), cudaMemcpyDeviceToHost, st));
      WBC_CUDA(h, cudaMemcpyAsync(s.status, d.status, m * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      if (s.vd) WBC_CUDA(h, cudaMemcpyAsync(s.vd, d.vd, m * WBC_NV * sizeof(double), cudaMemcpyDeviceToHost, st));
      if (s.f) WBC_CUDA(h, cudaMemcpyAsync(s.f, d.f, m * 12 * sizeof(double), cudaMemcpyDeviceToHost, st));
      if (s.qp_info) WBC_CUDA(h, cudaMemcpyAsync(s.qp_info, d.qp_info, m * 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
      if (s.lam) WBC_CUDA(h, cudaMemcpyAsync(s.lam, d.lam, m * WBC_NLAM * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    return WBC_OK;
  });
}

extern "C" int wbc_step_host(wbc_handle* h, int kind, int64_t n, const wbc_io* io) {
  const int rc = step_host_enqueue(h, kind, n, io);
  if (rc || !h || n <= 0) return rc;
  return step_host_wait(h);
}

// ------------------------------------------------------------------------------ per-robot controller parameters
// A set keeps the number of the device its records live on, not its handle: it may be destroyed after the handle.
struct wbc_param_set {
  int device = 0;
  int32_t n_sets = 0;
  DevArray<wbc::ParamRec> table;
  ~wbc_param_set() { cudaSetDevice(device); }   // the table is freed after this, on the set's device
};

extern "C" int wbc_param_set_destroy(wbc_param_set* s) {
  delete s;
  return WBC_OK;
}

static bool finite_all(const double* x, size_t n) {
  for (size_t i = 0; i < n; ++i)
    if (!std::isfinite(x[i])) return false;
  return true;
}

// Why a parameter set cannot be used, or nullptr: the checks of wbc_create, and what derive_constants and the step assume.
static const char* params_problem(const wbc_params& p) {
  static_assert(offsetof(wbc_params, torque_limits) % sizeof(double) == 0 && offsetof(wbc_params, pd_kp) % sizeof(double) == 0,
                "the doubles of wbc_params surround its two integers");
  const double* d = reinterpret_cast<const double*>(&p);
  if (!finite_all(d, offsetof(wbc_params, torque_limits) / sizeof(double)) || !finite_all(&p.pd_kp, 3 + WBC_NU))
    return "wbc_param_set_create: non-finite parameter";
  if (p.reg_vd != 0.0) return "wbc_param_set_create: reg_vd is not supported yet (must be 0)";
  if (!(p.reg_f > 0.0)) return "wbc_param_set_create: reg_f must be > 0 (tie-break that makes the QP strictly convex)";
  if (p.max_iter < 1) return "wbc_param_set_create: max_iter must be >= 1";
  if (p.torque_limits != 0 && p.torque_limits != 1) return "wbc_param_set_create: torque_limits must be 0 or 1";
  if (!(p.mu >= 0.0)) return "wbc_param_set_create: mu must be >= 0";
  if (!(p.clf_r > 0.0)) return "wbc_param_set_create: clf_r must be > 0";
  const double clf_w[] = {p.clf_q_body_p, p.clf_q_body_pd, p.clf_q_body_rpy, p.clf_q_body_rpyd, p.clf_q_foot_p, p.clf_q_foot_pd, p.clf_w_delta};
  for (double w : clf_w)
    if (!(w >= 0.0)) return "wbc_param_set_create: the CLF weights clf_q_* and clf_w_delta must be >= 0";
  return nullptr;
}

extern "C" int wbc_param_set_create(wbc_handle* h, int32_t n_sets, const wbc_params* params, wbc_param_set** out) {
  if (!h) return WBC_ERR_ARG;
  if (!out || !params || n_sets < 1) return fail_arg(h, "wbc_param_set_create: params and n_sets >= 1 are required");
  *out = nullptr;
  std::vector<wbc::ParamRec> rec((size_t)n_sets);
  for (int32_t k = 0; k < n_sets; ++k) {
    if (const char* why = params_problem(params[k])) return fail_arg(h, why);
    rec[k].pr = params[k];
    wbc::derive_constants(params[k], rec[k].dv);
  }
  WBC_CUDA(h, cudaSetDevice(h->device));
  std::unique_ptr<wbc_param_set> ps(new (std::nothrow) wbc_param_set());
  if (!ps) return WBC_ERR_NOMEM;
  ps->device = h->device;
  ps->n_sets = n_sets;
  WBC_CUDA(h, ps->table.reserve(rec.size()));
  WBC_CUDA(h, cudaMemcpy(ps->table.p, rec.data(), rec.size() * sizeof(rec[0]), cudaMemcpyHostToDevice));
  *out = ps.release();
  return WBC_OK;
}

// The kernel arguments of per-robot parameters with the index array `index` (as the kernels read it).
static int ctrl_args(wbc_handle* h, const wbc_ctrl_params* p, const int32_t* index, wbc::ParamArgs* pa) {
  const wbc_param_set* set = p ? p->set : nullptr;
  if (set && set->device != h->device) return fail_arg(h, "wbc_ctrl_params: the set lives on another device than the handle");
  *pa = wbc::ParamArgs{set ? set->table.p : h->d_params.p, index, set ? set->n_sets : 1};
  return WBC_OK;
}

extern "C" int wbc_step_params(wbc_handle* h, int kind, int64_t n, const wbc_io* io, const wbc_ctrl_params* p, void* stream) {
  if (!h) return WBC_ERR_ARG;
  wbc::ParamArgs pa;
  const int rc = ctrl_args(h, p, p ? p->index : nullptr, &pa);
  return rc ? rc : device_step(h, kind, n, io, (cudaStream_t)stream, false, &pa);
}

extern "C" int wbc_step_params_host(wbc_handle* h, int kind, int64_t n, const wbc_io* io, const wbc_ctrl_params* p) {
  if (!h) return WBC_ERR_ARG;
  wbc::ParamArgs pa;
  int rc = ctrl_args(h, p, p ? p->index : nullptr, &pa);
  if (!rc) rc = step_host_enqueue(h, kind, n, io, &pa);
  if (rc || n <= 0) return rc;
  return step_host_wait(h);
}

// ------------------------------------------------------------------------------ all GPUs of the box from one call
// north star: "instances shard trivially across the 8 GPUs of one box, with no NCCL beyond an optional host gather". One
// handle per device; a call splits [0, n) into contiguous equal shards (SURVEY 8e), enqueues each shard on its device and
// waits for all of them: the outputs land in the caller's (page-locked or pageable) host arrays, which IS the host gather.
struct wbc_multi {
  std::vector<std::unique_ptr<wbc_handle>> h;
  std::string err;
};

extern "C" int wbc_multi_destroy(wbc_multi* m) {
  delete m;
  return WBC_OK;
}

extern "C" int wbc_multi_create(const wbc_model* model, const wbc_params* params, int n_devices, const int* devices, wbc_multi** out) {
  if (!model || !out || n_devices <= 0) return WBC_ERR_ARG;
  *out = nullptr;
  wbc_multi* m = new (std::nothrow) wbc_multi();
  if (!m) return WBC_ERR_NOMEM;
  for (int i = 0; i < n_devices; ++i) {
    wbc_handle* h = nullptr;
    const int rc = wbc_create(model, params, devices ? devices[i] : i, &h);
    if (h) m->h.emplace_back(h);
    if (rc) { m->err = h ? h->err : "wbc_create failed"; *out = m; return rc; }
  }
  *out = m;
  return WBC_OK;
}

extern "C" const char* wbc_multi_last_error(const wbc_multi* m) { return m ? m->err.c_str() : "null handle"; }
extern "C" int wbc_multi_device_count(const wbc_multi* m) { return m ? (int)m->h.size() : 0; }
extern "C" int64_t wbc_multi_launch_count(const wbc_multi* m) {
  int64_t s = 0;
  if (m) for (const auto& h : m->h) s += h->launches;
  return s;
}

// Shard r of n over w devices: contiguous, sizes differ by at most one (the same rule as quadruped_drake_b200/sharding.py).
static void shard_of(int64_t n, int r, int w, int64_t* lo, int64_t* hi) {
  const int64_t base = n / w, rem = n % w;
  *lo = r * base + (r < rem ? r : rem);
  *hi = *lo + base + (r < rem ? 1 : 0);
}

extern "C" int wbc_multi_step_host(wbc_multi* m, int kind, int64_t n, const wbc_io* io) {
  if (!m) return WBC_ERR_ARG;
  if (!io || n < 0) { m->err = "wbc_multi_step_host: bad arguments"; return WBC_ERR_ARG; }
  const int w = (int)m->h.size();
  int rc = WBC_OK;
  int enq = 0;
  for (int r = 0; r < w && rc == WBC_OK; ++r) {
    int64_t lo, hi;
    shard_of(n, r, w, &lo, &hi);
    if (hi <= lo) { ++enq; continue; }
    const wbc_io sio = io_at(*io, lo);
    rc = step_host_enqueue(m->h[r].get(), kind, hi - lo, &sio);
    if (rc) m->err = m->h[r]->err;
    ++enq;
  }
  for (int r = 0; r < enq && r < w; ++r) {                 // always drain what was enqueued, even after an error
    const int rw = step_host_wait(m->h[r].get());
    if (rw && rc == WBC_OK) { rc = rw; m->err = m->h[r]->err; }
  }
  return rc;
}

extern "C" int wbc_dynamics_host(wbc_handle* h, int64_t n, const double* q, const double* v, double* M, double* Cv,
                                 double* taug, double* Jfeet, double* Jdv, double* pfeet) {
  if (!h) return WBC_ERR_ARG;
  if (n <= 0) return n == 0 ? WBC_OK : fail_arg(h, "wbc_dynamics_host: n < 0");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const double* dq = s.in(q, N * WBC_NQ); const double* dv = s.in(v, N * WBC_NV);
  double* dM = s.out(M, N * 324); double* dCv = s.out(Cv, N * 18); double* dtg = s.out(taug, N * 18);
  double* dJ = s.out(Jfeet, N * 216); double* dJdv = s.out(Jdv, N * 12); double* dp = s.out(pfeet, N * 12);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_dynamics(h, n, dq, dv, dM, dCv, dtg, dJ, dJdv, dp, s.st);
  return rc ? rc : s.finish(h);
}

extern "C" int wbc_time_step(wbc_handle* h, int kind, int64_t n, const wbc_io* io, int reps, void* stream,
                             double* ms_per_launch) {
  if (!h) return WBC_ERR_ARG;
  if (!ms_per_launch || reps <= 0) return fail_arg(h, "wbc_time_step: bad arguments");
  WBC_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  Event e0, e1;
  WBC_CUDA(h, cudaEventCreate(&e0.v));
  WBC_CUDA(h, cudaEventCreate(&e1.v));
  WBC_CUDA(h, cudaEventRecord(e0, st));
  for (int r = 0; r < reps; ++r) {
    const int rc = wbc_step(h, kind, n, io, stream);
    if (rc) return rc;
  }
  WBC_CUDA(h, cudaEventRecord(e1, st));
  WBC_CUDA(h, cudaEventSynchronize(e1));
  float ms = 0.f;
  WBC_CUDA(h, cudaEventElapsedTime(&ms, e0, e1));
  *ms_per_launch = (double)ms / reps;
  return WBC_OK;
}

// Per-kernel share of one control step: CUDA events before the reduce kernel, between the two kernels and after the solve
// kernel, averaged over `reps` steps (n <= 262144 so that the step is one launch pair). Measurement aid for bench.py.
extern "C" int wbc_profile_step(wbc_handle* h, int kind, int64_t n, const wbc_io* io, int reps, void* stream, double* ms_reduce,
                                double* ms_solve) {
  if (!h) return WBC_ERR_ARG;
  if (!ms_reduce || !ms_solve || reps <= 0 || n <= 0 || n > SPLIT_CHUNK || kind == WBC_CTRL_PD) return fail_arg(h, "wbc_profile_step: bad arguments");
  WBC_CUDA(h, cudaSetDevice(h->device));
  double r = 0.0, s = 0.0;
  for (int k = 0; k < reps; ++k) {
    const int rc = device_step(h, kind, n, io, (cudaStream_t)stream, true);
    if (rc) return rc;
    WBC_CUDA(h, cudaEventSynchronize(h->prof_ev[2]));
    float a = 0.f, b = 0.f;
    WBC_CUDA(h, cudaEventElapsedTime(&a, h->prof_ev[0], h->prof_ev[1]));
    WBC_CUDA(h, cudaEventElapsedTime(&b, h->prof_ev[1], h->prof_ev[2]));
    r += a; s += b;
  }
  *ms_reduce = r / reps; *ms_solve = s / reps;
  return WBC_OK;
}

// ------------------------------------------------------------------------------ LCM wire codecs (wbc_wire.cuh)
static unsigned wire_grid(const wbc_handle* h, int64_t n, int tile) {
  const int64_t tiles = (n + tile - 1) / tile, cap = (int64_t)h->sm_count * 8;     // grid-stride over tiles
  return (unsigned)(tiles < cap ? tiles : cap);
}

extern "C" int wbc_lcm_decode_trunk_state(wbc_handle* h, int64_t n, const uint8_t* msgs, double* timestamp, uint8_t* finished,
                                          double* traj, uint8_t* contact, double* f_plan, int32_t* status, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!msgs || !traj || !contact))) return fail_arg(h, "wbc_lcm_decode_trunk_state: msgs, traj and contact are required");
  if (!aligned16(msgs)) return fail_arg(h, "wbc_lcm_decode_trunk_state: msgs must be 16-byte aligned");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcwire::decode_trunk_kernel<<<wire_grid(h, n, wbcwire::TILE), wbcwire::THREADS, 0, (cudaStream_t)stream>>>(
      msgs, n, timestamp, finished, traj, contact, f_plan, status);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_lcm_encode_trunk_state(wbc_handle* h, int64_t n, const double* timestamp, const uint8_t* finished,
                                          const double* traj, const uint8_t* contact, const double* f_plan, uint8_t* msgs,
                                          void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!msgs || !traj || !contact))) return fail_arg(h, "wbc_lcm_encode_trunk_state: msgs, traj and contact are required");
  if (!aligned16(msgs)) return fail_arg(h, "wbc_lcm_encode_trunk_state: msgs must be 16-byte aligned");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcwire::encode_trunk_kernel<<<wire_grid(h, n, wbcwire::TILE), wbcwire::THREADS, 0, (cudaStream_t)stream>>>(
      msgs, n, timestamp, finished, traj, contact, f_plan);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_lcm_decode_robot_state(wbc_handle* h, int64_t n, const uint8_t* msgs, double* q, double* v, double* tau,
                                          int32_t* status, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!msgs || !q || !v))) return fail_arg(h, "wbc_lcm_decode_robot_state: msgs, q and v are required");
  if (!aligned16(msgs)) return fail_arg(h, "wbc_lcm_decode_robot_state: msgs must be 16-byte aligned");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcwire::decode_robot_kernel<<<wire_grid(h, n, wbcwire::RTILE), wbcwire::THREADS, 0, (cudaStream_t)stream>>>(msgs, n, q, v, tau, status);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_lcm_encode_robot_state(wbc_handle* h, int64_t n, const double* q, const double* v, const double* tau,
                                          int tau_in_actuator_order, uint8_t* msgs, int32_t* status, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!msgs || !tau))) return fail_arg(h, "wbc_lcm_encode_robot_state: msgs and tau are required");
  if (!aligned16(msgs)) return fail_arg(h, "wbc_lcm_encode_robot_state: msgs must be 16-byte aligned");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcwire::encode_robot_kernel<<<wire_grid(h, n, wbcwire::RTILE), wbcwire::THREADS, 0, (cudaStream_t)stream>>>(
      msgs, n, q, v, tau, tau_in_actuator_order ? h->d_tau_map.p : nullptr, status);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_lcm_decode_trunk_state_host(wbc_handle* h, int64_t n, const uint8_t* msgs, double* timestamp, uint8_t* finished,
                                               double* traj, uint8_t* contact, double* f_plan, int32_t* status) {
  if (!h) return WBC_ERR_ARG;
  if (n <= 0) return n == 0 ? WBC_OK : fail_arg(h, "wbc_lcm_decode_trunk_state_host: n < 0");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  uint8_t* dm = s.in(msgs, N * WBC_LCM_TRUNK_STATE_BYTES);
  double* dts = s.out(timestamp, N); uint8_t* dfin = s.out(finished, N);
  double* dtr = s.out(traj, N * WBC_NTRAJ); uint8_t* dc = s.out(contact, N * 4);
  double* dfp = s.out(f_plan, N * 12); int32_t* dst = s.out(status, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_lcm_decode_trunk_state(h, n, dm, dts, dfin, dtr, dc, dfp, dst, s.st);
  return rc ? rc : s.finish(h);
}

extern "C" int wbc_lcm_encode_trunk_state_host(wbc_handle* h, int64_t n, const double* timestamp, const uint8_t* finished,
                                               const double* traj, const uint8_t* contact, const double* f_plan, uint8_t* msgs) {
  if (!h) return WBC_ERR_ARG;
  if (n <= 0) return n == 0 ? WBC_OK : fail_arg(h, "wbc_lcm_encode_trunk_state_host: n < 0");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const double* dts = s.in(timestamp, N); const uint8_t* dfin = s.in(finished, N);
  const double* dtr = s.in(traj, N * WBC_NTRAJ); const uint8_t* dc = s.in(contact, N * 4);
  const double* dfp = s.in(f_plan, N * 12);
  uint8_t* dm = s.out(msgs, N * WBC_LCM_TRUNK_STATE_BYTES);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_lcm_encode_trunk_state(h, n, dts, dfin, dtr, dc, dfp, dm, s.st);
  return rc ? rc : s.finish(h);
}

extern "C" int wbc_lcm_decode_robot_state_host(wbc_handle* h, int64_t n, const uint8_t* msgs, double* q, double* v, double* tau,
                                               int32_t* status) {
  if (!h) return WBC_ERR_ARG;
  if (n <= 0) return n == 0 ? WBC_OK : fail_arg(h, "wbc_lcm_decode_robot_state_host: n < 0");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  uint8_t* dm = s.in(msgs, N * WBC_LCM_ROBOT_STATE_BYTES);
  double* dq = s.out(q, N * WBC_NQ); double* dv = s.out(v, N * WBC_NV); double* dt = s.out(tau, N * WBC_NU);
  int32_t* dst = s.out(status, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_lcm_decode_robot_state(h, n, dm, dq, dv, dt, dst, s.st);
  return rc ? rc : s.finish(h);
}

extern "C" int wbc_lcm_encode_robot_state_host(wbc_handle* h, int64_t n, const double* q, const double* v, const double* tau,
                                               int tau_in_actuator_order, uint8_t* msgs, int32_t* status) {
  if (!h) return WBC_ERR_ARG;
  if (n <= 0) return n == 0 ? WBC_OK : fail_arg(h, "wbc_lcm_encode_robot_state_host: n < 0");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const double* dq = s.in(q, N * WBC_NQ); const double* dv = s.in(v, N * WBC_NV); const double* dt = s.in(tau, N * WBC_NU);
  uint8_t* dm = s.out(msgs, N * WBC_LCM_ROBOT_STATE_BYTES); int32_t* dst = s.out(status, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_lcm_encode_robot_state(h, n, dq, dv, dt, tau_in_actuator_order, dm, dst, s.st);
  return rc ? rc : s.finish(h);
}

// ------------------------------------------------------------------------------ trajectory sampler (wbc_traj.cuh)
// A plan keeps the number of the device its tables live on, not its handle: it may be destroyed after the handle.
struct wbc_plan {
  int device = 0;
  wbctraj::PlanTables t{};
  std::deque<DevArray<unsigned char>> bufs;
  ~wbc_plan() { cudaSetDevice(device); }   // the tables are freed after this, on the plan's device
};

extern "C" int wbc_plan_destroy(wbc_plan* p) {
  delete p;
  return WBC_OK;
}

extern "C" int wbc_plan_create(wbc_handle* h, int32_t n_plans, const wbc_plan_desc* plans, wbc_plan** out) {
  if (!h) return WBC_ERR_ARG;
  if (!out || !plans || n_plans <= 0) return fail_arg(h, "wbc_plan_create: bad arguments");
  *out = nullptr;
  using wbctraj::NSPLINE;
  // ---- flatten on the host: offsets, running sums of the durations (in the reference's summation order), nodes
  std::vector<int> poly_off, phase_off, grid_off, node_of_poly;
  std::vector<unsigned char> cstart;
  std::vector<double> tend, dur, nodes, phase_tend, grid_ts, wait, standing;
  grid_off.push_back(0);
  for (int p = 0; p < n_plans; ++p) {
    const wbc_plan_desc& d = plans[p];
    const wbc_spline_desc* sp[NSPLINE] = {&d.base_linear, &d.base_angular, &d.ee_motion[0], &d.ee_motion[1], &d.ee_motion[2],
                                          &d.ee_motion[3], &d.ee_force[0], &d.ee_force[1], &d.ee_force[2], &d.ee_force[3]};
    for (int s = 0; s < NSPLINE; ++s) {
      if (sp[s]->n_poly <= 0 || !sp[s]->durations || !sp[s]->nodes) return fail_arg(h, "wbc_plan_create: empty spline");
      poly_off.push_back((int)tend.size());
      double acc = 0.0;
      const int node0 = (int)(nodes.size() / 6);
      for (int i = 0; i < sp[s]->n_poly; ++i) {
        if (!(sp[s]->durations[i] > 0.0)) return fail_arg(h, "wbc_plan_create: polynomial duration must be > 0");
        acc += sp[s]->durations[i];
        tend.push_back(acc);
        dur.push_back(sp[s]->durations[i]);
        node_of_poly.push_back(node0 + i);
      }
      nodes.insert(nodes.end(), sp[s]->nodes, sp[s]->nodes + (size_t)(sp[s]->n_poly + 1) * 6);
    }
    poly_off.push_back((int)tend.size());
    for (int k = 0; k < WBC_NLEG; ++k) {
      if (d.n_phase[k] <= 0 || !d.phase_durations[k]) return fail_arg(h, "wbc_plan_create: empty phase list");
      phase_off.push_back((int)phase_tend.size());
      double acc = 0.0;
      for (int i = 0; i < d.n_phase[k]; ++i) { acc += d.phase_durations[k][i]; phase_tend.push_back(acc); }
      cstart.push_back(d.contact_at_start[k] ? 1 : 0);
    }
    phase_off.push_back((int)phase_tend.size());
    if (d.n_grid < 0 || (d.n_grid > 0 && !d.grid_timestamps)) return fail_arg(h, "wbc_plan_create: bad sample grid");
    for (int i = 0; i < d.n_grid; ++i) {
      if (i > 0 && !(d.grid_timestamps[i] > d.grid_timestamps[i - 1])) return fail_arg(h, "wbc_plan_create: grid timestamps must increase");
      grid_ts.push_back(d.grid_timestamps[i]);
    }
    grid_off.push_back((int)grid_ts.size());
    wait.push_back(d.wait_time);
    standing.insert(standing.end(), d.standing, d.standing + WBC_NTRAJ);
  }
  if (grid_ts.empty()) grid_ts.push_back(0.0);
  WBC_CUDA(h, cudaSetDevice(h->device));
  std::unique_ptr<wbc_plan> pl(new (std::nothrow) wbc_plan());
  if (!pl) return WBC_ERR_NOMEM;
  pl->device = h->device;
  cudaError_t err = cudaSuccess;
  auto up = [&](const void* src, size_t bytes) -> void* {
    if (err != cudaSuccess) return nullptr;
    DevArray<unsigned char>& d = pl->bufs.emplace_back();
    err = d.reserve(bytes ? bytes : 1);
    if (err == cudaSuccess && src) err = cudaMemcpy(d.p, src, bytes, cudaMemcpyHostToDevice);
    return err == cudaSuccess ? d.p : nullptr;
  };
  const int n_poly_total = (int)tend.size();
  pl->t.n_plans = n_plans;
  pl->t.poly_off = (const int*)up(poly_off.data(), poly_off.size() * sizeof(int));
  pl->t.phase_off = (const int*)up(phase_off.data(), phase_off.size() * sizeof(int));
  pl->t.grid_off = (const int*)up(grid_off.data(), grid_off.size() * sizeof(int));
  pl->t.contact_start = (const unsigned char*)up(cstart.data(), cstart.size());
  pl->t.tend = (const double*)up(tend.data(), tend.size() * sizeof(double));
  pl->t.phase_tend = (const double*)up(phase_tend.data(), phase_tend.size() * sizeof(double));
  pl->t.grid_ts = (const double*)up(grid_ts.data(), grid_ts.size() * sizeof(double));
  pl->t.wait_time = (const double*)up(wait.data(), wait.size() * sizeof(double));
  pl->t.standing = (const double*)up(standing.data(), standing.size() * sizeof(double));
  double* d_coef = (double*)up(nullptr, (size_t)n_poly_total * 12 * sizeof(double));
  pl->t.coef = d_coef;
  const int* d_node_of = (const int*)up(node_of_poly.data(), node_of_poly.size() * sizeof(int));
  const double* d_nodes = (const double*)up(nodes.data(), nodes.size() * sizeof(double));
  const double* d_dur = (const double*)up(dur.data(), dur.size() * sizeof(double));
  if (err == cudaSuccess) {
    wbctraj::hermite_coeff_kernel<<<(n_poly_total * 3 + 255) / 256, 256, 0, h->lane[0]>>>(n_poly_total, d_node_of, d_nodes, d_dur, d_coef);
    h->launches++;
    err = cudaGetLastError();
    if (err == cudaSuccess) err = cudaStreamSynchronize(h->lane[0]);
  }
  if (err != cudaSuccess) {
    h->err = std::string("wbc_plan_create: ") + cudaGetErrorString(err);
    return WBC_ERR_CUDA;
  }
  *out = pl.release();
  return WBC_OK;
}

extern "C" int wbc_sample_trajectory(wbc_handle* h, const wbc_plan* plan, int64_t n, const int32_t* plan_index, const double* t,
                                     double* traj, uint8_t* contact, double* f_plan, double* t_eval, int32_t* status, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (!plan || n < 0 || (n > 0 && (!t || !traj || !contact))) return fail_arg(h, "wbc_sample_trajectory: plan, t, traj and contact are required");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  if (reinterpret_cast<uintptr_t>(contact) & 3u) return fail_arg(h, "wbc_sample_trajectory: contact must be 4-byte aligned");
  const int ipw = sample_ipw(n);
  const long long chunks = (n + ipw - 1) / ipw, blocks = (chunks + wbctraj::SAMPLE_WARPS - 1) / wbctraj::SAMPLE_WARPS, cap = (long long)h->sm_count * 16;
  const unsigned grid = (unsigned)(blocks < cap ? blocks : cap);
  cudaStream_t sst = (cudaStream_t)stream;
  if (ipw == 32) wbctraj::sample_kernel<32><<<grid, wbctraj::SAMPLE_WARPS * 32, 0, sst>>>(plan->t, n, plan_index, t, traj, contact, f_plan, t_eval, status);
  else if (ipw == 8) wbctraj::sample_kernel<8><<<grid, wbctraj::SAMPLE_WARPS * 32, 0, sst>>>(plan->t, n, plan_index, t, traj, contact, f_plan, t_eval, status);
  else wbctraj::sample_kernel<2><<<grid, wbctraj::SAMPLE_WARPS * 32, 0, sst>>>(plan->t, n, plan_index, t, traj, contact, f_plan, t_eval, status);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_sample_trajectory_host(wbc_handle* h, const wbc_plan* plan, int64_t n, const int32_t* plan_index, const double* t,
                                          double* traj, uint8_t* contact, double* f_plan, double* t_eval, int32_t* status) {
  if (!h) return WBC_ERR_ARG;
  if (!plan || n < 0) return fail_arg(h, "wbc_sample_trajectory_host: plan and n >= 0 are required");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const int32_t* dpi = s.in(plan_index, N); const double* dt = s.in(t, N);
  double* dtr = s.out(traj, N * WBC_NTRAJ); uint8_t* dc = s.out(contact, N * 4); double* dfp = s.out(f_plan, N * 12);
  double* dte = s.out(t_eval, N); int32_t* dst = s.out(status, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_sample_trajectory(h, plan, n, dpi, dt, dtr, dc, dfp, dte, dst, s.st);
  return rc ? rc : s.finish(h);
}

// Control step whose trunk targets come from a device-resident plan: the host sends q, v and the plan time only (300 B + 8 B
// per instance instead of 732 B - the 54-double trajectory row is 59 % of the step's input bytes), wbc_sample_trajectory fills
// traj / contact in device scratch and the step kernels read them from there. Page-locked buffers are read / written by the
// kernels directly (zero-copy), pageable ones are staged.
extern "C" int wbc_step_plan_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, const double* q, const double* v,
                                  const double* t, const int32_t* plan_index, double* tau, double* metrics, int32_t* status) {
  if (!h) return WBC_ERR_ARG;
  if (!plan || n < 0 || kind == WBC_CTRL_PD) return fail_arg(h, "wbc_step_plan_host: plan and a QP controller kind are required");
  if (n > 0 && (!q || !v || !t || !tau || !metrics || !status)) return fail_arg(h, "wbc_step_plan_host: q, v, t, tau, metrics and status are required");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  WBC_CUDA(h, h->ro.reserve(n));
  const RolloutScratch& ro = h->ro;
  const Staging& sg = h->stage;
  const cudaStream_t st = h->lane[0];
  int rc;
  if (to_device_aliases(q, v, t, plan_index, tau, metrics, status)) {   // from here on the kernels' aliases of the host arrays
    rc = wbc_sample_trajectory(h, plan, n, plan_index, t, ro.traj.p, ro.contact.p, nullptr, nullptr, nullptr, st);
    if (rc) return rc;
    // the step itself as in the zero-copy mode of wbc_step_host: two halves on the two internal streams. q and v are 304 B per
    // instance, which the reduce CTAs pull over the link without slowing down at any batch size (57.3 M steps/s at 65536,
    // 60.8 M at 2^20; copy-engine staging of q and v: 51.5 / 60.6 M)
    const int k = pinned_chunks(n, false);
    const cudaStream_t lanes[2] = {st, h->lane[1]};
    if (k > 1) {
      rc = streams_wait(h, h->order_ev, st, lanes + 1, 1);   // the sampled rows
      if (rc) return rc;
    }
    const wbc_io zio{q, v, ro.traj.p, ro.contact.p, tau, metrics, status};
    rc = for_each_chunk(n, k, [&](int c, int64_t o, int64_t m) {
      return step_launch(h, kind, m, io_at(zio, o), lanes[c & 1], c & 1, Issue{true, k > 1});
    });
    if (rc) return rc;
    return step_host_wait(h);
  }
  WBC_CUDA(h, h->stage.reserve(n));
  DevScratch s(st);
  const int32_t* dpi = s.in(plan_index, (size_t)n);
  WBC_SCRATCH_CHECK(h, s);
  WBC_CUDA(h, cudaMemcpyAsync(sg.q.p, q, n * WBC_NQ * sizeof(double), cudaMemcpyHostToDevice, st));
  WBC_CUDA(h, cudaMemcpyAsync(sg.v.p, v, n * WBC_NV * sizeof(double), cudaMemcpyHostToDevice, st));
  WBC_CUDA(h, cudaMemcpyAsync(ro.t.p, t, n * sizeof(double), cudaMemcpyHostToDevice, st));
  rc = wbc_sample_trajectory(h, plan, n, dpi, ro.t.p, ro.traj.p, ro.contact.p, nullptr, nullptr, nullptr, st);
  if (rc) return rc;
  const wbc_io io{sg.q.p, sg.v.p, ro.traj.p, ro.contact.p, sg.tau.p, sg.metrics.p, sg.status.p};
  rc = step_launch(h, kind, n, io, st, 0, Issue{});
  if (rc) return rc;
  WBC_CUDA(h, cudaMemcpyAsync(tau, sg.tau.p, n * WBC_NU * sizeof(double), cudaMemcpyDeviceToHost, st));
  WBC_CUDA(h, cudaMemcpyAsync(metrics, sg.metrics.p, n * WBC_NMETRIC * sizeof(double), cudaMemcpyDeviceToHost, st));
  WBC_CUDA(h, cudaMemcpyAsync(status, sg.status.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  WBC_CUDA(h, cudaStreamSynchronize(st));
  return WBC_OK;
}

// ------------------------------------------------------------------------------ closed-loop rollout (wbc_rollout.cuh)
extern "C" int wbc_integrate(wbc_handle* h, int64_t n, double dt, double* q, double* v, const double* vd, double* t, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!q || !v || !vd))) return fail_arg(h, "wbc_integrate: q, v and vd are required");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcroll::integrate_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, dt, q, v, vd, t, nullptr, nullptr, nullptr,
                                                                                          nullptr, nullptr, nullptr);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_default_plant_opts(wbc_plant_opts* o) {
  if (!o) return WBC_ERR_ARG;
  o->mu = 1.0; o->erp = 0.2; o->iters = 30; o->reserved = 0;      // simulate.py:44-46: static = dynamic friction 1.0
  return WBC_OK;
}

// pa == nullptr: the unperturbed plant kernel; otherwise the variant kernel with these perturbations, or with ta != nullptr the
// terrain kernel.
static int plant_launch(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbcplant::PerturbArgs* pa,
                        const wbcplant::TerrainArgs* ta, double* q,
                        double* v, const double* tau, double* t, const int32_t* ctrl_status, int32_t* status_or, double* f_contact,
                        const double* metrics, double* err_max, double* metrics_log, const int* counter, cudaStream_t st) {
  wbc_plant_opts o;
  if (opts) o = *opts; else wbc_default_plant_opts(&o);
  if (!(o.mu >= 0.0) || !(o.erp >= 0.0 && o.erp <= 1.0) || o.iters < 1 || o.iters > 1000) return fail_arg(h, "wbc_plant_step: bad options");
  const wbcplant::PlantArgs a{q, v, tau, t, ctrl_status, status_or, f_contact, metrics, err_max, metrics_log, counter, (long long)n, dt,
                              o.mu, o.erp, o.iters};
  if (pa && ta) wbc_plant_terrain_kernel<<<(unsigned)n, 32, sizeof(SmemLayoutPlantTerrain), st>>>(*pa, *ta, a);
  else if (pa) wbc_plant_variant_kernel<<<(unsigned)n, 32, sizeof(SmemLayoutPlantVariant), st>>>(*pa, a);
  else wbc_plant_kernel<<<(unsigned)n, 32, sizeof(SmemLayoutPlant), st>>>(h->d_const.p, a);
  h->launches++;
  return WBC_OK;
}

// ------------------------------------------------------------------------------ perturbed robots (wbc_plant.cuh)
// A set keeps the number of the device its table lives on, not its handle: it may be destroyed after the handle.
struct wbc_plant_set {
  int device = 0;
  int32_t n_variants = 0;
  bool own_mu = false;
  DevArray<wbcplant::PlantVariant> table;
  ~wbc_plant_set() { cudaSetDevice(device); }   // the table is freed after this, on the set's device
};

extern "C" int wbc_plant_set_destroy(wbc_plant_set* s) {
  delete s;
  return WBC_OK;
}

extern "C" int wbc_plant_set_create(wbc_handle* h, int32_t n_variants, const wbc_model* models, const double* mu, wbc_plant_set** out) {
  if (!h) return WBC_ERR_ARG;
  if (!out || !models || n_variants <= 0) return fail_arg(h, "wbc_plant_set_create: models and n_variants > 0 are required");
  *out = nullptr;
  std::vector<wbcplant::PlantVariant> rec((size_t)n_variants);
  for (int32_t k = 0; k < n_variants; ++k) {
    const wbc_model& m = models[k];
    if (memcmp(m.v_index, h->model.v_index, sizeof(m.v_index)) || memcmp(m.act_index, h->model.act_index, sizeof(m.act_index)))
      return fail_arg(h, "wbc_plant_set_create: every model must have the handle's v_index and act_index");
    static_assert(offsetof(wbc_model, mass) == 0 && offsetof(wbc_model, v_index) % sizeof(double) == 0, "the doubles of wbc_model come first");
    if (!finite_all(reinterpret_cast<const double*>(&m), offsetof(wbc_model, v_index) / sizeof(double)))
      return fail_arg(h, "wbc_plant_set_create: non-finite model value");
    for (int b = 0; b < WBC_NBODY; ++b) {
      const double* I = m.inertia_com[b];      // xx yy zz xy xz yz
      const double m2 = I[0] * I[1] - I[3] * I[3];
      const double det = I[0] * (I[1] * I[2] - I[5] * I[5]) - I[3] * (I[3] * I[2] - I[5] * I[4]) + I[4] * (I[3] * I[5] - I[1] * I[4]);
      if (!(m.mass[b] > 0.0)) return fail_arg(h, "wbc_plant_set_create: every body mass must be > 0");
      if (!(I[0] > 0.0 && m2 > 0.0 && det > 0.0)) return fail_arg(h, "wbc_plant_set_create: every inertia_com must be positive definite");
    }
    if (mu && !(std::isfinite(mu[k]) && mu[k] >= 0.0)) return fail_arg(h, "wbc_plant_set_create: every mu must be finite and >= 0");
    rec[k].md = m;
    rec[k].mu = mu ? mu[k] : 0.0;
  }
  WBC_CUDA(h, cudaSetDevice(h->device));
  std::unique_ptr<wbc_plant_set> ps(new (std::nothrow) wbc_plant_set());
  if (!ps) return WBC_ERR_NOMEM;
  ps->device = h->device;
  ps->n_variants = n_variants;
  ps->own_mu = mu != nullptr;
  WBC_CUDA(h, ps->table.reserve(rec.size()));
  WBC_CUDA(h, cudaMemcpy(ps->table.p, rec.data(), rec.size() * sizeof(rec[0]), cudaMemcpyHostToDevice));
  *out = ps.release();
  return WBC_OK;
}

// The kernel arguments of a perturbation whose variant / push arrays are already on the device.
static int perturb_args(wbc_handle* h, const wbc_plant_perturb* p, const int32_t* variant, const double* push, bool has_t,
                        wbcplant::PerturbArgs* pa) {
  const wbc_plant_set* set = p ? p->set : nullptr;
  if (set && set->device != h->device) return fail_arg(h, "wbc_plant_perturb: the set lives on another device than the handle");
  if (push && !has_t) return fail_arg(h, "wbc_plant_perturb: pushes need the robots' times t");
  *pa = wbcplant::PerturbArgs{set ? set->table.p : h->d_nominal.p, variant, push, set ? set->n_variants : 1, set && set->own_mu ? 1 : 0};
  return WBC_OK;
}

extern "C" int wbc_plant_step(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, double* q, double* v, const double* tau,
                              double* t, const int32_t* ctrl_status, int32_t* status_or, double* f_contact, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || !(dt > 0.0) || (n > 0 && (!q || !v || !tau))) return fail_arg(h, "wbc_plant_step: q, v, tau and dt > 0 are required");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  const int rc = plant_launch(h, n, dt, opts, nullptr, nullptr, q, v, tau, t, ctrl_status, status_or, f_contact, nullptr, nullptr, nullptr, nullptr,
                              (cudaStream_t)stream);
  if (rc) return rc;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_plant_step_perturbed(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbc_plant_perturb* perturb,
                                        double* q, double* v, const double* tau, double* t, const int32_t* ctrl_status, int32_t* status_or,
                                        double* f_contact, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || !(dt > 0.0) || (n > 0 && (!q || !v || !tau))) return fail_arg(h, "wbc_plant_step_perturbed: q, v, tau and dt > 0 are required");
  wbcplant::PerturbArgs pa;
  int rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, t != nullptr, &pa);
  if (rc || n == 0) return rc;
  WBC_CUDA(h, cudaSetDevice(h->device));
  rc = plant_launch(h, n, dt, opts, &pa, nullptr, q, v, tau, t, ctrl_status, status_or, f_contact, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
  if (rc) return rc;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// ------------------------------------------------------------------------------ uneven ground (wbc_plant.cuh)
// A set keeps the number of the device its records live on, not its handle: it may be destroyed after the handle.
struct wbc_terrain_set {
  int device = 0;
  int32_t n_terrains = 0;
  DevArray<wbcplant::TerrainRec> table;
  DevArray<double> heights;       // every grid, concatenated (TerrainRec::off)
  ~wbc_terrain_set() { cudaSetDevice(device); }   // the arrays are freed after this, on the set's device
};

extern "C" int wbc_terrain_set_destroy(wbc_terrain_set* s) {
  delete s;
  return WBC_OK;
}

extern "C" int wbc_terrain_set_create(wbc_handle* h, int32_t n_terrains, const wbc_terrain_desc* terrains, wbc_terrain_set** out) {
  if (!h) return WBC_ERR_ARG;
  if (!out || !terrains || n_terrains <= 0) return fail_arg(h, "wbc_terrain_set_create: terrains and n_terrains > 0 are required");
  *out = nullptr;
  std::vector<wbcplant::TerrainRec> rec((size_t)n_terrains);
  std::vector<double> heights;
  for (int32_t k = 0; k < n_terrains; ++k) {
    const wbc_terrain_desc& d = terrains[k];
    const double vals[] = {d.z0, d.sx, d.sy, d.x0, d.y0, d.dx, d.dy};
    if (!finite_all(vals, 7)) return fail_arg(h, "wbc_terrain_set_create: non-finite terrain value");
    const bool grid = d.nx != 0 || d.ny != 0;
    if (grid && !(d.nx >= 2 && d.ny >= 2)) return fail_arg(h, "wbc_terrain_set_create: nx and ny must both be 0 or both >= 2");
    if (grid && !(d.dx > 0.0 && d.dy > 0.0)) return fail_arg(h, "wbc_terrain_set_create: a grid needs dx > 0 and dy > 0");
    if (grid && !d.heights) return fail_arg(h, "wbc_terrain_set_create: a grid needs heights");
    const size_t cells = grid ? (size_t)d.nx * (size_t)d.ny : 0;
    if (grid && !finite_all(d.heights, cells)) return fail_arg(h, "wbc_terrain_set_create: non-finite height");
    rec[k] = wbcplant::terrain_record(d, (long long)heights.size());
    if (grid) heights.insert(heights.end(), d.heights, d.heights + cells);
  }
  WBC_CUDA(h, cudaSetDevice(h->device));
  std::unique_ptr<wbc_terrain_set> ts(new (std::nothrow) wbc_terrain_set());
  if (!ts) return WBC_ERR_NOMEM;
  ts->device = h->device;
  ts->n_terrains = n_terrains;
  WBC_CUDA(h, ts->table.reserve(rec.size()));
  WBC_CUDA(h, cudaMemcpy(ts->table.p, rec.data(), rec.size() * sizeof(rec[0]), cudaMemcpyHostToDevice));
  if (!heights.empty()) {
    WBC_CUDA(h, ts->heights.reserve(heights.size()));
    WBC_CUDA(h, cudaMemcpy(ts->heights.p, heights.data(), heights.size() * sizeof(double), cudaMemcpyHostToDevice));
  }
  *out = ts.release();
  return WBC_OK;
}

// The kernel arguments of a terrain whose index array is already on the device.
static int terrain_args(wbc_handle* h, const wbc_plant_terrain* p, wbcplant::TerrainArgs* ta) {
  const wbc_terrain_set* set = p ? p->set : nullptr;
  if (set && set->device != h->device) return fail_arg(h, "wbc_plant_terrain: the set lives on another device than the handle");
  *ta = wbcplant::TerrainArgs{set ? set->table.p : nullptr, set ? set->heights.p : nullptr, p ? p->index : nullptr, set ? set->n_terrains : 1};
  return WBC_OK;
}

extern "C" int wbc_plant_step_terrain(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbc_plant_perturb* perturb,
                                      const wbc_plant_terrain* terrain, double* q, double* v, const double* tau, double* t,
                                      const int32_t* ctrl_status, int32_t* status_or, double* f_contact, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || !(dt > 0.0) || (n > 0 && (!q || !v || !tau))) return fail_arg(h, "wbc_plant_step_terrain: q, v, tau and dt > 0 are required");
  wbcplant::PerturbArgs pa;
  wbcplant::TerrainArgs ta;
  int rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, t != nullptr, &pa);
  if (!rc) rc = terrain_args(h, terrain, &ta);
  if (rc || n == 0) return rc;
  WBC_CUDA(h, cudaSetDevice(h->device));
  rc = plant_launch(h, n, dt, opts, &pa, &ta, q, v, tau, t, ctrl_status, status_or, f_contact, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
  if (rc) return rc;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// Which plant a host entry runs (params: the rollout with per-robot controller parameters, on any plant; loop: the same with
// sensing and actuation, on the ground plant; monitor: the loop with the rollout monitor; motor: the monitor entry with the
// actuator model).
enum class PlantEntry { plain, perturbed, terrain, params, loop, monitor, motor, estimator };

// Host buffers of the three plant steps.
static int plant_step_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, PlantEntry entry, const wbc_plant_perturb* perturb,
                           const wbc_plant_terrain* terrain, double* q, double* v, const double* tau, double* t, const int32_t* ctrl_status,
                           int32_t* status_or, double* f_contact, const char* what) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || !(dt > 0.0)) return fail_arg(h, what);
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  double* dq = s.inout(q, N * WBC_NQ); double* dv = s.inout(v, N * WBC_NV); const double* dtau = s.in(tau, N * WBC_NU);
  double* dt_ = s.inout(t, N); const int32_t* dcs = s.in(ctrl_status, N); int32_t* dso = s.inout(status_or, N);
  double* df = s.out(f_contact, N * 12);
  wbc_plant_perturb dp{};
  if (perturb) dp = wbc_plant_perturb{perturb->set, s.in(perturb->variant, N), s.in(perturb->push, N * 8)};
  wbc_plant_terrain dtr{};
  if (terrain) dtr = wbc_plant_terrain{terrain->set, s.in(terrain->index, N)};
  WBC_SCRATCH_CHECK(h, s);
  const int rc =
      entry == PlantEntry::terrain ? wbc_plant_step_terrain(h, n, dt, opts, perturb ? &dp : nullptr, terrain ? &dtr : nullptr, dq, dv, dtau,
                                                            dt_, dcs, dso, df, s.st)
      : entry == PlantEntry::perturbed ? wbc_plant_step_perturbed(h, n, dt, opts, perturb ? &dp : nullptr, dq, dv, dtau, dt_, dcs, dso, df, s.st)
                                       : wbc_plant_step(h, n, dt, opts, dq, dv, dtau, dt_, dcs, dso, df, s.st);
  return rc ? rc : s.finish(h);
}

extern "C" int wbc_plant_step_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, double* q, double* v, const double* tau,
                                   double* t, const int32_t* ctrl_status, int32_t* status_or, double* f_contact) {
  return plant_step_host(h, n, dt, opts, PlantEntry::plain, nullptr, nullptr, q, v, tau, t, ctrl_status, status_or, f_contact,
                         "wbc_plant_step_host: n >= 0 and dt > 0 are required");
}

extern "C" int wbc_plant_step_perturbed_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbc_plant_perturb* perturb,
                                             double* q, double* v, const double* tau, double* t, const int32_t* ctrl_status,
                                             int32_t* status_or, double* f_contact) {
  return plant_step_host(h, n, dt, opts, PlantEntry::perturbed, perturb, nullptr, q, v, tau, t, ctrl_status, status_or, f_contact,
                         "wbc_plant_step_perturbed_host: n >= 0 and dt > 0 are required");
}

extern "C" int wbc_plant_step_terrain_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbc_plant_perturb* perturb,
                                           const wbc_plant_terrain* terrain, double* q, double* v, const double* tau, double* t,
                                           const int32_t* ctrl_status, int32_t* status_or, double* f_contact) {
  return plant_step_host(h, n, dt, opts, PlantEntry::terrain, perturb, terrain, q, v, tau, t, ctrl_status, status_or, f_contact,
                         "wbc_plant_step_terrain_host: n >= 0 and dt > 0 are required");
}

// The rollout loop of wbc_rollout_ex, wbc_rollout_perturbed, wbc_rollout_terrain, wbc_rollout_params and wbc_rollout_loop;
// pa != nullptr: the plant step runs the variant kernel, or with ta != nullptr the terrain kernel; cp != nullptr: the controller
// step runs with these per-robot parameters; lp != nullptr (ground plant): the controller reads the observed state and the plant
// applies the actuated torque (wbc_loop.cuh), with the loop state in the handle's scratch when lp->hist is null; mp != nullptr
// (ground plant): the monitor runs after the plant (wbc_monitor.cuh) on the plant's per-step status word, which it folds into
// io->status_or; mt != nullptr (ground plant): the motor (wbc_motor.cuh) turns the applied torque into the plant input, with its
// state in the handle's scratch when mt->tau_m is null, and the monitor sees the motor torque tau_m; ep != nullptr (with a loop):
// the estimator (wbc_estimator.cuh) replaces the observed base position and linear velocity in place, with its state in the
// handle's scratch when ep->x is null, and ORs its status bit into the plant's status word.
static int rollout_run(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt, const wbc_rollout_io* io,
                       const wbc_rollout_opts* opts, const wbcplant::PerturbArgs* pa, const wbcplant::TerrainArgs* ta, cudaStream_t st,
                       const wbc::ParamArgs* cp = nullptr, const wbcloop::LoopArgs* lp = nullptr, const wbcmon::MonArgs* mp = nullptr,
                       const wbcmotor::MotorArgs* mt = nullptr, const wbcest::EstArgs* ep = nullptr) {
  const bool plant = opts && opts->plant != 0;
  const int use_graph = opts ? opts->use_graph : 1;
  if (kind == WBC_CTRL_PD && !plant) return fail_arg(h, "wbc_rollout: the PD law returns no accelerations to integrate (use the ground plant)");
  if (n > 0 && (!io->q || !io->v || !io->t)) return fail_arg(h, "wbc_rollout: q, v and t are required");
  if (n == 0 || n_steps == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  WBC_CUDA(h, h->ro.reserve(n));
  WBC_CUDA(h, h->slot[0].reserve(n, !plant));   // before the capture below: a step grows no scratch while being captured
  const RolloutScratch& ro = h->ro;
  double* tau = io->tau ? io->tau : ro.tau.p;
  double* metrics = io->metrics ? io->metrics : ro.metrics.p;
  wbcloop::LoopArgs la{};
  if (lp) {
    la = *lp;
    WBC_CUDA(h, h->loop.reserve(n, !la.hist));
    if (!la.hist) {                                // a fresh history: tick 0 (no slot of hist is read before it is written)
      la.hist = h->loop.hist.p;
      la.tick = h->loop.tick.p;
      WBC_CUDA(h, cudaMemsetAsync(la.tick, 0, n * sizeof(long long), st));
    }
  }
  wbcmotor::MotorArgs ma{};
  if (mt) {
    ma = *mt;
    WBC_CUDA(h, h->motor.reserve(n, !ma.tau_m));
    if (!ma.tau_m) {                               // a fresh motor state: count 0 (no tau_m is read before it is written)
      ma.tau_m = h->motor.tau_m.p;
      ma.count = h->motor.count.p;
      WBC_CUDA(h, cudaMemsetAsync(ma.tau_m, 0, n * WBC_NU * sizeof(double), st));
      WBC_CUDA(h, cudaMemsetAsync(ma.count, 0, n * sizeof(long long), st));
    }
  }
  wbcest::EstArgs ea{};
  if (ep) {
    ea = *ep;
    ea.seed = la.seed; ea.stream = la.stream; ea.tick = la.tick;
    if (!ea.x) {                                   // a fresh filter state: count 0 (the first step primes it)
      WBC_CUDA(h, h->est.reserve(n));
      ea.x = h->est.x.p; ea.P = h->est.P.p; ea.v_prev = h->est.v_prev.p; ea.count = h->est.count.p;
      WBC_CUDA(h, cudaMemsetAsync(ea.count, 0, n * sizeof(long long), st));
    }
  }
  const unsigned loop_grid = (unsigned)((n + 255) / 256);
  // with a monitor the plant ORs each step's status into a word of its own, and writes its forces somewhere in any case
  int32_t* plant_status_or = io->status_or;
  double* f_contact = opts ? opts->f_contact : nullptr;
  if (mp) {
    WBC_CUDA(h, h->mon.reserve(n, !f_contact));
    plant_status_or = h->mon.word.p;
    if (!f_contact) f_contact = h->mon.f.p;
    WBC_CUDA(h, cudaMemsetAsync(plant_status_or, 0, n * sizeof(int32_t), st));
  }
  WBC_CUDA(h, cudaMemsetAsync(ro.counter.p, 0, sizeof(int), st));
  if (io->status_or) WBC_CUDA(h, cudaMemsetAsync(io->status_or, 0, n * sizeof(int32_t), st));
  if (io->err_max) WBC_CUDA(h, cudaMemsetAsync(io->err_max, 0, n * sizeof(double), st));
  if (kind == WBC_CTRL_PD) {                       // the PD law has no QP: no status / metrics of its own
    WBC_CUDA(h, cudaMemsetAsync(ro.status.p, 0, n * sizeof(int32_t), st));
    WBC_CUDA(h, cudaMemsetAsync(metrics, 0, n * WBC_NMETRIC * sizeof(double), st));
  }
  // with the ground plant the controller's accelerations are not needed: the step runs without the vd outputs
  // with a loop the controller reads the observed state and the plant applies the actuated torque
  wbc_io sio{lp ? h->loop.q_obs.p : io->q, lp ? h->loop.v_obs.p : io->v, ro.traj.p, ro.contact.p, tau, metrics, ro.status.p,
             plant ? nullptr : ro.vd.p, nullptr, nullptr};
  const double* applied = lp ? h->loop.applied.p : tau;
  const double* plant_tau = mt ? h->motor.plant.p : applied;      // with a motor the plant gets its input, the monitor its torque
  const double* mon_tau = mt ? ma.tau_m : applied;
  auto one_step = [&]() -> int {
    int r = wbc_sample_trajectory(h, plan, n, io->plan_index, io->t, ro.traj.p, ro.contact.p, nullptr, nullptr, nullptr, st);
    if (r) return r;
    if (lp) {
      wbcloop::observe_kernel<<<loop_grid, 256, 0, st>>>(la, n, io->q, io->v, h->loop.q_obs.p, h->loop.v_obs.p);
      h->launches++;
    }
    if (ep) {
      wbcest::estimate_kernel<<<(unsigned)((n + 3) / 4), wbcest::EST_BLOCK, 0, st>>>(ea, n, io->q, io->v, h->loop.q_obs.p, h->loop.v_obs.p,
                                                                                  ro.contact.p, plant_status_or);
      h->launches++;
    }
    r = device_step(h, kind, n, &sio, st, false, cp);
    if (r) return r;
    if (lp) {
      wbcloop::actuate_kernel<<<loop_grid, 256, 0, st>>>(la, n, tau, h->loop.applied.p, ro.status.p);
      h->launches++;
    }
    if (mt) {
      wbcmotor::motor_kernel<<<(unsigned)((n + 15) / 16), wbcmotor::MOTOR_BLOCK, 0, st>>>(ma, n, io->v, applied, h->motor.plant.p,
                                                                                         ro.status.p);
      h->launches++;
    }
    if (plant) {
      r = plant_launch(h, n, dt, &opts->plant_opts, pa, ta, io->q, io->v, plant_tau, io->t, ro.status.p, plant_status_or, f_contact, metrics,
                       io->err_max, io->metrics_log, ro.counter.p, st);
      if (r) return r;
      if (mp) {
        wbcmon::monitor_kernel<<<loop_grid, 256, 0, st>>>(*mp, n, io->q, io->v, ro.traj.p, ro.contact.p, mon_tau, f_contact, nullptr,
                                                          plant_status_or, io->status_or);
        h->launches++;
      }
    } else {
      wbcroll::integrate_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, dt, io->q, io->v, ro.vd.p, io->t, ro.status.p, io->status_or,
                                                                           metrics, io->err_max, io->metrics_log, ro.counter.p);
      h->launches++;
    }
    if (io->metrics_log) { wbcroll::bump_counter_kernel<<<1, 1, 0, st>>>(ro.counter.p); h->launches++; }
    return WBC_OK;
  };
  if (use_graph && n_steps > 1 && st != nullptr && st != cudaStreamLegacy) {   // the legacy default stream cannot be captured
    // capture one control step (3-4 kernels) once, replay it n_steps times: one graph launch per step instead of 3-4 kernel launches
    Graph graph;
    GraphExec exec;
    const int64_t launches0 = h->launches;
    WBC_CUDA(h, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    const int rc = one_step();
    cudaError_t e = cudaStreamEndCapture(st, &graph.v);
    const int64_t per_step = h->launches - launches0;
    if (rc) return rc;
    if (e != cudaSuccess) { h->err = std::string("wbc_rollout: graph capture: ") + cudaGetErrorString(e); return WBC_ERR_CUDA; }
    e = cudaGraphInstantiate(&exec.v, graph, 0);
    if (e != cudaSuccess) { h->err = std::string("wbc_rollout: graph instantiate: ") + cudaGetErrorString(e); return WBC_ERR_CUDA; }
    h->launches = launches0;
    for (int k = 0; k < n_steps && e == cudaSuccess; ++k) { e = cudaGraphLaunch(exec, st); h->launches += per_step; }
    // the exec graph must outlive its launches: wait for the stream before it is destroyed
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { h->err = std::string("wbc_rollout: graph launch: ") + cudaGetErrorString(e); return WBC_ERR_CUDA; }
  } else {
    for (int k = 0; k < n_steps; ++k) {
      const int rc = one_step();
      if (rc) return rc;
    }
  }
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

extern "C" int wbc_rollout_ex(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                              const wbc_rollout_io* io, const wbc_rollout_opts* opts, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || n < 0 || n_steps < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_rollout: bad arguments");
  return rollout_run(h, kind, plan, n, n_steps, dt, io, opts, nullptr, nullptr, (cudaStream_t)stream);
}

extern "C" int wbc_rollout_perturbed(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                     const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || !opts || n < 0 || n_steps < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_rollout_perturbed: bad arguments");
  if (opts->plant == 0) return fail_arg(h, "wbc_rollout_perturbed: perturbations act on the ground plant (opts->plant = 1)");
  wbcplant::PerturbArgs pa;
  const int rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, io->t != nullptr, &pa);
  return rc ? rc : rollout_run(h, kind, plan, n, n_steps, dt, io, opts, &pa, nullptr, (cudaStream_t)stream);
}

extern "C" int wbc_rollout_terrain(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                   const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                   const wbc_plant_terrain* terrain, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || !opts || n < 0 || n_steps < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_rollout_terrain: bad arguments");
  if (opts->plant == 0) return fail_arg(h, "wbc_rollout_terrain: terrain is ground for the ground plant (opts->plant = 1)");
  wbcplant::PerturbArgs pa;
  wbcplant::TerrainArgs ta;
  int rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, io->t != nullptr, &pa);
  if (!rc) rc = terrain_args(h, terrain, &ta);
  return rc ? rc : rollout_run(h, kind, plan, n, n_steps, dt, io, opts, &pa, &ta, (cudaStream_t)stream);
}

extern "C" int wbc_rollout(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                           const wbc_rollout_io* io, int use_graph, void* stream) {
  wbc_rollout_opts o{};
  o.use_graph = use_graph; o.plant = 0; o.f_contact = nullptr;
  wbc_default_plant_opts(&o.plant_opts);
  return wbc_rollout_ex(h, kind, plan, n, n_steps, dt, io, &o, stream);
}

extern "C" int wbc_rollout_params(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                  const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                  const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || n < 0 || n_steps < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_rollout_params: bad arguments");
  const bool ground = perturb || terrain;
  if (ground && !(opts && opts->plant != 0))
    return fail_arg(h, "wbc_rollout_params: perturbations and terrain act on the ground plant (opts->plant = 1)");
  wbc::ParamArgs cp;
  wbcplant::PerturbArgs pa;
  wbcplant::TerrainArgs ta;
  int rc = ctrl_args(h, ctrl, ctrl ? ctrl->index : nullptr, &cp);
  if (!rc && ground) rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, io->t != nullptr, &pa);
  if (!rc && terrain) rc = terrain_args(h, terrain, &ta);
  return rc ? rc : rollout_run(h, kind, plan, n, n_steps, dt, io, opts, ground ? &pa : nullptr, terrain ? &ta : nullptr, (cudaStream_t)stream, &cp);
}

// ------------------------------------------------------------------------------ sensing and actuation (wbc_loop.cuh)
// The kernel arguments of a loop whose arrays are already on the device (hist / tick may both be null).
static int loop_args(wbc_handle* h, const wbc_loop* l, wbcloop::LoopArgs* la) {
  if (l && !l->hist != !l->tick) return fail_arg(h, "wbc_loop: hist and tick are given together or not at all");
  *la = l ? wbcloop::LoopArgs{l->noise, l->delay, l->strength, l->stream, (unsigned long long)l->seed, l->hist, (long long*)l->tick}
          : wbcloop::LoopArgs{};
  return WBC_OK;
}

extern "C" int wbc_rollout_loop(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop, void* stream) {
  if (!loop) return wbc_rollout_params(h, kind, plan, n, n_steps, dt, io, opts, perturb, terrain, ctrl, stream);
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || n < 0 || n_steps < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_rollout_loop: bad arguments");
  if (!(opts && opts->plant == 1))
    return fail_arg(h, "wbc_rollout_loop: sensing and actuation close the loop around the ground plant (opts->plant = 1)");
  wbc::ParamArgs cp;
  wbcplant::PerturbArgs pa;
  wbcplant::TerrainArgs ta;
  wbcloop::LoopArgs la;
  int rc = loop_args(h, loop, &la);
  if (!rc) rc = ctrl_args(h, ctrl, ctrl ? ctrl->index : nullptr, &cp);
  if (!rc && (perturb || terrain))
    rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, io->t != nullptr, &pa);
  if (!rc && terrain) rc = terrain_args(h, terrain, &ta);
  return rc ? rc : rollout_run(h, kind, plan, n, n_steps, dt, io, opts, (perturb || terrain) ? &pa : nullptr, terrain ? &ta : nullptr,
                               (cudaStream_t)stream, &cp, &la);
}

extern "C" int wbc_loop_observe(wbc_handle* h, int64_t n, const wbc_loop* loop, const double* q, const double* v, double* q_obs,
                                double* v_obs, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!q || !v || !q_obs || !v_obs))) return fail_arg(h, "wbc_loop_observe: q, v, q_obs and v_obs are required");
  wbcloop::LoopArgs la;
  const int rc = loop_args(h, loop, &la);
  if (rc || n == 0) return rc;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcloop::observe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(la, n, q, v, q_obs, v_obs);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// Device copies of a host wbc_loop's arrays; hist and tick are copied in and out.
static wbc_loop loop_to_device(DevScratch& s, const wbc_loop& l, size_t N) {
  return wbc_loop{s.in(l.noise, N * 6), s.in(l.delay, N), s.in(l.strength, N), s.in(l.stream, N), l.seed,
                  s.inout(l.hist, N * WBC_LOOP_HIST * WBC_NU), s.inout(l.tick, N)};
}

extern "C" int wbc_loop_observe_host(wbc_handle* h, int64_t n, const wbc_loop* loop, const double* q, const double* v, double* q_obs,
                                     double* v_obs) {
  if (!h) return WBC_ERR_ARG;
  if (n < 0 || (n > 0 && (!q || !v || !q_obs || !v_obs))) return fail_arg(h, "wbc_loop_observe_host: q, v, q_obs and v_obs are required");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const double* dq = s.in(q, N * WBC_NQ); const double* dv = s.in(v, N * WBC_NV);
  double* dqo = s.out(q_obs, N * WBC_NQ); double* dvo = s.out(v_obs, N * WBC_NV);
  wbc_loop dl{};
  if (loop) dl = loop_to_device(s, *loop, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_loop_observe(h, n, loop ? &dl : nullptr, dq, dv, dqo, dvo, s.st);
  return rc ? rc : s.finish(h);
}

// ------------------------------------------------------------------------------ rollout monitor (wbc_monitor.cuh)
// The kernel arguments of a monitor whose arrays are already on the device.
static int mon_args(wbc_handle* h, const wbc_monitor* m, int64_t n, double dt, wbcmon::MonArgs* ma) {
  if (!(m->pos_max >= 0.0) || !(m->ang_max >= 0.0)) return fail_arg(h, "wbc_monitor: pos_max and ang_max must be >= 0 (+inf: no bound)");
  if (n > 0 && (!m->stats || !m->steps || !m->fail_step || !m->fail_why))
    return fail_arg(h, "wbc_monitor: stats, steps, fail_step and fail_why are required");
  *ma = wbcmon::MonArgs{m->pos_max, m->ang_max, dt, m->stats, (long long*)m->steps, (long long*)m->fail_step, m->fail_why, m->why, {}, {}, {}};
  for (int j = 0; j < WBC_NU; ++j) {
    ma->v_index[j] = h->model.v_index[j];
    ma->act_index[j] = h->model.act_index[j];
    ma->effort[j] = h->model.effort[j];
  }
  return WBC_OK;
}

extern "C" int wbc_rollout_monitor(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                   const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                   const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                                   const wbc_monitor* mon, void* stream) {
  if (!mon) return wbc_rollout_loop(h, kind, plan, n, n_steps, dt, io, opts, perturb, terrain, ctrl, loop, stream);
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || n < 0 || n_steps < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_rollout_monitor: bad arguments");
  if (!(opts && opts->plant == 1)) return fail_arg(h, "wbc_rollout_monitor: the monitor watches the ground plant (opts->plant = 1)");
  wbc::ParamArgs cp;
  wbcplant::PerturbArgs pa;
  wbcplant::TerrainArgs ta;
  wbcloop::LoopArgs la;
  wbcmon::MonArgs ma;
  int rc = mon_args(h, mon, n, dt, &ma);
  if (!rc && loop) rc = loop_args(h, loop, &la);
  if (!rc) rc = ctrl_args(h, ctrl, ctrl ? ctrl->index : nullptr, &cp);
  if (!rc && (perturb || terrain))
    rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, io->t != nullptr, &pa);
  if (!rc && terrain) rc = terrain_args(h, terrain, &ta);
  return rc ? rc : rollout_run(h, kind, plan, n, n_steps, dt, io, opts, (perturb || terrain) ? &pa : nullptr, terrain ? &ta : nullptr,
                               (cudaStream_t)stream, &cp, loop ? &la : nullptr, &ma);
}

extern "C" int wbc_monitor_step(wbc_handle* h, int64_t n, double dt, const wbc_monitor* mon, const double* q, const double* v,
                                const double* traj, const uint8_t* contact, const double* tau_applied, const double* f_contact,
                                const int32_t* status, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (!mon || n < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_monitor_step: mon, n >= 0 and dt > 0 are required");
  if (n > 0 && (!q || !v || !traj || !contact || !tau_applied || !f_contact))
    return fail_arg(h, "wbc_monitor_step: q, v, traj, contact, tau_applied and f_contact are required");
  wbcmon::MonArgs ma;
  const int rc = mon_args(h, mon, n, dt, &ma);
  if (rc || n == 0) return rc;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcmon::monitor_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ma, n, q, v, traj, contact, tau_applied, f_contact,
                                                                                        status, nullptr, nullptr);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// Device copies of a host wbc_monitor's arrays; the state is copied in and out, why out.
static wbc_monitor monitor_to_device(DevScratch& s, const wbc_monitor& m, size_t N) {
  return wbc_monitor{m.pos_max, m.ang_max, s.inout(m.stats, N * WBC_MON_NSTAT), s.inout(m.steps, N), s.inout(m.fail_step, N),
                     s.inout(m.fail_why, N), s.out(m.why, N)};
}

extern "C" int wbc_monitor_step_host(wbc_handle* h, int64_t n, double dt, const wbc_monitor* mon, const double* q, const double* v,
                                     const double* traj, const uint8_t* contact, const double* tau_applied, const double* f_contact,
                                     const int32_t* status) {
  if (!h) return WBC_ERR_ARG;
  if (!mon || n <= 0) return n == 0 && mon ? WBC_OK : fail_arg(h, "wbc_monitor_step_host: mon and n >= 0 are required");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const double* dq = s.in(q, N * WBC_NQ); const double* dv = s.in(v, N * WBC_NV); const double* dtr = s.in(traj, N * WBC_NTRAJ);
  const uint8_t* dc = s.in(contact, N * 4); const double* dtau = s.in(tau_applied, N * WBC_NU); const double* df = s.in(f_contact, N * 12);
  const int32_t* dst = s.in(status, N);
  const wbc_monitor dm = monitor_to_device(s, *mon, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_monitor_step(h, n, dt, &dm, dq, dv, dtr, dc, dtau, df, dst, s.st);
  return rc ? rc : s.finish(h);
}

// ------------------------------------------------------------------------------ actuator model (wbc_motor.cuh)
// A set keeps the number of the device its records live on, not its handle: it may be destroyed after the handle.
struct wbc_motor_set {
  int device = 0;
  int32_t n_sets = 0;
  DevArray<wbc_motor_desc> table;
  ~wbc_motor_set() { cudaSetDevice(device); }   // the table is freed after this, on the set's device
};

extern "C" int wbc_motor_set_destroy(wbc_motor_set* s) {
  delete s;
  return WBC_OK;
}

extern "C" int wbc_motor_set_create(wbc_handle* h, int32_t n_sets, const wbc_motor_desc* descs, wbc_motor_set** out) {
  if (!h) return WBC_ERR_ARG;
  if (!out || !descs || n_sets < 1) return fail_arg(h, "wbc_motor_set_create: descs and n_sets >= 1 are required");
  *out = nullptr;
  for (int32_t k = 0; k < n_sets; ++k)
    if (const char* why = wbcmotor::desc_problem(descs[k])) return fail_arg(h, why);
  WBC_CUDA(h, cudaSetDevice(h->device));
  std::unique_ptr<wbc_motor_set> ms(new (std::nothrow) wbc_motor_set());
  if (!ms) return WBC_ERR_NOMEM;
  ms->device = h->device;
  ms->n_sets = n_sets;
  WBC_CUDA(h, ms->table.reserve((size_t)n_sets));
  WBC_CUDA(h, cudaMemcpy(ms->table.p, descs, (size_t)n_sets * sizeof(wbc_motor_desc), cudaMemcpyHostToDevice));
  *out = ms.release();
  return WBC_OK;
}

// The kernel arguments of a motor whose arrays are already on the device (tau_m / count may both be null).
static int motor_args(wbc_handle* h, const wbc_plant_motor* m, double dt, wbcmotor::MotorArgs* ma) {
  if (!m->tau_m != !m->count) return fail_arg(h, "wbc_plant_motor: tau_m and count are given together or not at all");
  const wbc_motor_set* set = m->set;
  if (set && set->device != h->device) return fail_arg(h, "wbc_plant_motor: the set lives on another device than the handle");
  *ma = wbcmotor::MotorArgs{set ? set->table.p : nullptr, m->index, set ? set->n_sets : 1, m->tau_m, (long long*)m->count, dt, {}, {}, {}};
  for (int j = 0; j < WBC_NU; ++j) {
    ma->v_index[j] = h->model.v_index[j];
    ma->act_index[j] = h->model.act_index[j];
    ma->effort[j] = h->model.effort[j];
  }
  return WBC_OK;
}

extern "C" int wbc_rollout_motor(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                 const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                 const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                                 const wbc_monitor* mon, const wbc_plant_motor* motor, void* stream) {
  if (!motor) return wbc_rollout_monitor(h, kind, plan, n, n_steps, dt, io, opts, perturb, terrain, ctrl, loop, mon, stream);
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || n < 0 || n_steps < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_rollout_motor: bad arguments");
  if (!(opts && opts->plant == 1)) return fail_arg(h, "wbc_rollout_motor: the motors drive the ground plant (opts->plant = 1)");
  wbc::ParamArgs cp;
  wbcplant::PerturbArgs pa;
  wbcplant::TerrainArgs ta;
  wbcloop::LoopArgs la;
  wbcmon::MonArgs ma;
  wbcmotor::MotorArgs mt;
  int rc = motor_args(h, motor, dt, &mt);
  if (!rc && mon) rc = mon_args(h, mon, n, dt, &ma);
  if (!rc && loop) rc = loop_args(h, loop, &la);
  if (!rc) rc = ctrl_args(h, ctrl, ctrl ? ctrl->index : nullptr, &cp);
  if (!rc && (perturb || terrain))
    rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, io->t != nullptr, &pa);
  if (!rc && terrain) rc = terrain_args(h, terrain, &ta);
  return rc ? rc : rollout_run(h, kind, plan, n, n_steps, dt, io, opts, (perturb || terrain) ? &pa : nullptr, terrain ? &ta : nullptr,
                               (cudaStream_t)stream, &cp, loop ? &la : nullptr, mon ? &ma : nullptr, &mt);
}

extern "C" int wbc_motor_apply(wbc_handle* h, int64_t n, double dt, const wbc_plant_motor* motor, const double* v, const double* tau_in,
                               double* tau_plant, int32_t* status, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (!motor || n < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_motor_apply: motor, n >= 0 and dt > 0 are required");
  if (n > 0 && (!v || !tau_in || !tau_plant || !motor->tau_m || !motor->count))
    return fail_arg(h, "wbc_motor_apply: v, tau_in, tau_plant and the motor state tau_m, count are required");
  wbcmotor::MotorArgs mt;
  const int rc = motor_args(h, motor, dt, &mt);
  if (rc || n == 0) return rc;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcmotor::motor_kernel<<<(unsigned)((n + 15) / 16), wbcmotor::MOTOR_BLOCK, 0, (cudaStream_t)stream>>>(mt, n, v, tau_in, tau_plant, status);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// Device copies of a host wbc_plant_motor's arrays; tau_m and count are copied in and out.
static wbc_plant_motor motor_to_device(DevScratch& s, const wbc_plant_motor& m, size_t N) {
  return wbc_plant_motor{m.set, s.in(m.index, N), s.inout(m.tau_m, N * WBC_NU), s.inout(m.count, N)};
}

extern "C" int wbc_motor_apply_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_motor* motor, const double* v,
                                    const double* tau_in, double* tau_plant, int32_t* status) {
  if (!h) return WBC_ERR_ARG;
  if (!motor || n <= 0) return n == 0 && motor ? WBC_OK : fail_arg(h, "wbc_motor_apply_host: motor and n >= 0 are required");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const double* dv = s.in(v, N * WBC_NV); const double* dti = s.in(tau_in, N * WBC_NU);
  double* dtp = s.out(tau_plant, N * WBC_NU); int32_t* dst = s.inout(status, N);
  const wbc_plant_motor dm = motor_to_device(s, *motor, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_motor_apply(h, n, dt, &dm, dv, dti, dtp, dst, s.st);
  return rc ? rc : s.finish(h);
}

// ------------------------------------------------------------------------------ state estimator (wbc_estimator.cuh)
// A set keeps the number of the device its records live on, not its handle: it may be destroyed after the handle.
struct wbc_estimator_set {
  int device = 0;
  int32_t n_sets = 0;
  DevArray<wbc_estimator_desc> table;
  ~wbc_estimator_set() { cudaSetDevice(device); }   // the table is freed after this, on the set's device
};

extern "C" int wbc_estimator_set_destroy(wbc_estimator_set* s) {
  delete s;
  return WBC_OK;
}

extern "C" int wbc_estimator_set_create(wbc_handle* h, int32_t n_sets, const wbc_estimator_desc* descs, wbc_estimator_set** out) {
  if (!h) return WBC_ERR_ARG;
  if (!out || !descs || n_sets < 1) return fail_arg(h, "wbc_estimator_set_create: descs and n_sets >= 1 are required");
  *out = nullptr;
  for (int32_t k = 0; k < n_sets; ++k)
    if (const char* why = wbcest::desc_problem(descs[k])) return fail_arg(h, why);
  WBC_CUDA(h, cudaSetDevice(h->device));
  std::unique_ptr<wbc_estimator_set> es(new (std::nothrow) wbc_estimator_set());
  if (!es) return WBC_ERR_NOMEM;
  es->device = h->device;
  es->n_sets = n_sets;
  WBC_CUDA(h, es->table.reserve((size_t)n_sets));
  WBC_CUDA(h, cudaMemcpy(es->table.p, descs, (size_t)n_sets * sizeof(wbc_estimator_desc), cudaMemcpyHostToDevice));
  *out = es.release();
  return WBC_OK;
}

// The kernel arguments of an estimator whose arrays are already on the device (x / P / v_prev / count may all be null); the
// loop's seed, stream and tick are filled in by the caller.
static int est_args(wbc_handle* h, const wbc_estimator* e, double dt, wbcest::EstArgs* ea) {
  const int given = (e->x != nullptr) + (e->P != nullptr) + (e->v_prev != nullptr) + (e->count != nullptr);
  if (given != 0 && given != 4) return fail_arg(h, "wbc_estimator: x, P, v_prev and count are given together or not at all");
  const wbc_estimator_set* set = e->set;
  if (!set) return fail_arg(h, "wbc_estimator: a set is required");
  if (set->device != h->device) return fail_arg(h, "wbc_estimator: the set lives on another device than the handle");
  *ea = wbcest::EstArgs{};
  ea->set = set->table.p; ea->index = e->index; ea->n_sets = set->n_sets; ea->accel_noise = e->accel_noise;
  ea->x = e->x; ea->P = e->P; ea->v_prev = e->v_prev; ea->count = (long long*)e->count; ea->stats = e->stats;
  ea->dt = dt;
  const wbc_model& m = h->model;
  for (int c = 0; c < 3; ++c) ea->gravity[c] = m.gravity[c];
  for (int k = 0; k < WBC_NU; ++k) {
    ea->v_index[k] = m.v_index[k];
    for (int c = 0; c < 3; ++c) { ea->joint_xyz[k][c] = m.joint_xyz[k][c]; ea->joint_axis[k][c] = m.joint_axis[k][c]; }
  }
  for (int l = 0; l < WBC_NLEG; ++l)
    for (int c = 0; c < 3; ++c) ea->foot_xyz[l][c] = m.foot_xyz[l][c];
  return WBC_OK;
}

extern "C" int wbc_rollout_estimator(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                     const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                     const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                                     const wbc_monitor* mon, const wbc_plant_motor* motor, const wbc_estimator* est, void* stream) {
  if (!est) return wbc_rollout_motor(h, kind, plan, n, n_steps, dt, io, opts, perturb, terrain, ctrl, loop, mon, motor, stream);
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || n < 0 || n_steps < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_rollout_estimator: bad arguments");
  if (!(opts && opts->plant == 1)) return fail_arg(h, "wbc_rollout_estimator: the estimator runs in the ground-plant loop (opts->plant = 1)");
  if (!loop) return fail_arg(h, "wbc_rollout_estimator: the estimator needs a loop (its observed state, seed, streams and ticks)");
  wbc::ParamArgs cp;
  wbcplant::PerturbArgs pa;
  wbcplant::TerrainArgs ta;
  wbcloop::LoopArgs la;
  wbcmon::MonArgs ma;
  wbcmotor::MotorArgs mt;
  wbcest::EstArgs ea;
  int rc = est_args(h, est, dt, &ea);
  if (!rc && motor) rc = motor_args(h, motor, dt, &mt);
  if (!rc && mon) rc = mon_args(h, mon, n, dt, &ma);
  if (!rc) rc = loop_args(h, loop, &la);
  if (!rc) rc = ctrl_args(h, ctrl, ctrl ? ctrl->index : nullptr, &cp);
  if (!rc && (perturb || terrain))
    rc = perturb_args(h, perturb, perturb ? perturb->variant : nullptr, perturb ? perturb->push : nullptr, io->t != nullptr, &pa);
  if (!rc && terrain) rc = terrain_args(h, terrain, &ta);
  return rc ? rc : rollout_run(h, kind, plan, n, n_steps, dt, io, opts, (perturb || terrain) ? &pa : nullptr, terrain ? &ta : nullptr,
                               (cudaStream_t)stream, &cp, &la, mon ? &ma : nullptr, motor ? &mt : nullptr, &ea);
}

extern "C" int wbc_estimator_step(wbc_handle* h, int64_t n, double dt, const wbc_estimator* est, const wbc_loop* loop, const double* q,
                                  const double* v, double* q_obs, double* v_obs, const uint8_t* contact, int32_t* status_or, void* stream) {
  if (!h) return WBC_ERR_ARG;
  if (!est || n < 0 || !(dt > 0.0)) return fail_arg(h, "wbc_estimator_step: est, n >= 0 and dt > 0 are required");
  if (n > 0 && (!q || !v || !q_obs || !v_obs || !contact || !est->x))
    return fail_arg(h, "wbc_estimator_step: q, v, q_obs, v_obs, contact and the filter state x, P, v_prev, count are required");
  wbcest::EstArgs ea;
  int rc = est_args(h, est, dt, &ea);
  wbcloop::LoopArgs la;
  if (!rc) rc = loop_args(h, loop, &la);
  if (rc || n == 0) return rc;
  ea.seed = la.seed; ea.stream = la.stream; ea.tick = la.tick;
  WBC_CUDA(h, cudaSetDevice(h->device));
  wbcest::estimate_kernel<<<(unsigned)((n + 3) / 4), wbcest::EST_BLOCK, 0, (cudaStream_t)stream>>>(ea, n, q, v, q_obs, v_obs, contact,
                                                                                                   status_or);
  h->launches++;
  WBC_CUDA(h, cudaGetLastError());
  return WBC_OK;
}

// Device copies of a host wbc_estimator's arrays; the filter state and the statistics are copied in and out.
static wbc_estimator est_to_device(DevScratch& s, const wbc_estimator& e, size_t N) {
  return wbc_estimator{e.set, s.in(e.index, N), s.in(e.accel_noise, N), s.inout(e.x, N * wbcest::NX),
                       s.inout(e.P, N * wbcest::NX * wbcest::NX), s.inout(e.v_prev, N * 3), s.inout(e.count, N), s.inout(e.stats, N * 4)};
}

extern "C" int wbc_estimator_step_host(wbc_handle* h, int64_t n, double dt, const wbc_estimator* est, const wbc_loop* loop,
                                       const double* q, const double* v, double* q_obs, double* v_obs, const uint8_t* contact,
                                       int32_t* status_or) {
  if (!h) return WBC_ERR_ARG;
  if (!est || n <= 0) return n == 0 && est ? WBC_OK : fail_arg(h, "wbc_estimator_step_host: est and n >= 0 are required");
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  const double* dq = s.in(q, N * WBC_NQ); const double* dv = s.in(v, N * WBC_NV);
  double* dqo = s.inout(q_obs, N * WBC_NQ); double* dvo = s.inout(v_obs, N * WBC_NV);
  const uint8_t* dc = s.in(contact, N * WBC_NLEG); int32_t* dst = s.inout(status_or, N);
  const wbc_estimator de = est_to_device(s, *est, N);
  wbc_loop dl{};
  if (loop) dl = loop_to_device(s, *loop, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc = wbc_estimator_step(h, n, dt, &de, loop ? &dl : nullptr, dq, dv, dqo, dvo, dc, dst, s.st);
  return rc ? rc : s.finish(h);
}

// Host buffers of the eight rollouts.
static int rollout_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt, const wbc_rollout_io* io,
                        const wbc_rollout_opts* opts, PlantEntry entry, const wbc_plant_perturb* perturb, const wbc_plant_terrain* terrain,
                        const wbc_ctrl_params* ctrl = nullptr, const wbc_loop* loop = nullptr, const wbc_monitor* mon = nullptr,
                        const wbc_plant_motor* motor = nullptr, const wbc_estimator* est = nullptr) {
  if (!h) return WBC_ERR_ARG;
  if (!plan || !io || n < 0 || n_steps < 0) return fail_arg(h, "wbc_rollout_host: bad arguments");
  if (n == 0) return WBC_OK;
  WBC_CUDA(h, cudaSetDevice(h->device));
  DevScratch s(h->lane[0]);
  const size_t N = (size_t)n;
  wbc_rollout_io d{};
  d.q = s.inout(io->q, N * WBC_NQ); d.v = s.inout(io->v, N * WBC_NV); d.t = s.inout(io->t, N);
  d.plan_index = s.in(io->plan_index, N);
  d.tau = s.out(io->tau, N * WBC_NU); d.metrics = s.out(io->metrics, N * WBC_NMETRIC);
  d.status_or = s.out(io->status_or, N); d.err_max = s.out(io->err_max, N);
  d.metrics_log = s.out(io->metrics_log, N * WBC_NMETRIC * (size_t)n_steps);
  wbc_rollout_opts o{};
  if (opts) o = *opts; else { o.use_graph = 1; wbc_default_plant_opts(&o.plant_opts); }
  o.f_contact = s.out(o.f_contact, N * 12);
  wbc_plant_perturb dp{};
  if (perturb) dp = wbc_plant_perturb{perturb->set, s.in(perturb->variant, N), s.in(perturb->push, N * 8)};
  wbc_plant_terrain dtr{};
  if (terrain) dtr = wbc_plant_terrain{terrain->set, s.in(terrain->index, N)};
  wbc_ctrl_params dcp{};
  if (ctrl) dcp = wbc_ctrl_params{ctrl->set, s.in(ctrl->index, N)};
  wbc_loop dl{};
  if (loop) dl = loop_to_device(s, *loop, N);
  wbc_monitor dm{};
  if (mon) dm = monitor_to_device(s, *mon, N);
  wbc_plant_motor dmt{};
  if (motor) dmt = motor_to_device(s, *motor, N);
  wbc_estimator de{};
  if (est) de = est_to_device(s, *est, N);
  WBC_SCRATCH_CHECK(h, s);
  const int rc =
      entry == PlantEntry::estimator
          ? wbc_rollout_estimator(h, kind, plan, n, n_steps, dt, &d, opts ? &o : nullptr, perturb ? &dp : nullptr, terrain ? &dtr : nullptr,
                                  ctrl ? &dcp : nullptr, loop ? &dl : nullptr, mon ? &dm : nullptr, motor ? &dmt : nullptr,
                                  est ? &de : nullptr, s.st)
      : entry == PlantEntry::motor ? wbc_rollout_motor(h, kind, plan, n, n_steps, dt, &d, opts ? &o : nullptr, perturb ? &dp : nullptr,
                                                     terrain ? &dtr : nullptr, ctrl ? &dcp : nullptr, loop ? &dl : nullptr,
                                                     mon ? &dm : nullptr, motor ? &dmt : nullptr, s.st)
      : entry == PlantEntry::monitor ? wbc_rollout_monitor(h, kind, plan, n, n_steps, dt, &d, opts ? &o : nullptr, perturb ? &dp : nullptr,
                                                         terrain ? &dtr : nullptr, ctrl ? &dcp : nullptr, loop ? &dl : nullptr,
                                                         mon ? &dm : nullptr, s.st)
      : entry == PlantEntry::loop ? wbc_rollout_loop(h, kind, plan, n, n_steps, dt, &d, opts ? &o : nullptr, perturb ? &dp : nullptr,
                                                   terrain ? &dtr : nullptr, ctrl ? &dcp : nullptr, loop ? &dl : nullptr, s.st)
      : entry == PlantEntry::params ? wbc_rollout_params(h, kind, plan, n, n_steps, dt, &d, opts ? &o : nullptr, perturb ? &dp : nullptr,
                                                       terrain ? &dtr : nullptr, ctrl ? &dcp : nullptr, s.st)
      : entry == PlantEntry::terrain ? wbc_rollout_terrain(h, kind, plan, n, n_steps, dt, &d, opts ? &o : nullptr, perturb ? &dp : nullptr,
                                                         terrain ? &dtr : nullptr, s.st)
      : entry == PlantEntry::perturbed ? wbc_rollout_perturbed(h, kind, plan, n, n_steps, dt, &d, opts ? &o : nullptr, perturb ? &dp : nullptr, s.st)
                                       : wbc_rollout_ex(h, kind, plan, n, n_steps, dt, &d, &o, s.st);
  return rc ? rc : s.finish(h);
}

extern "C" int wbc_rollout_ex_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                   const wbc_rollout_io* io, const wbc_rollout_opts* opts) {
  return rollout_host(h, kind, plan, n, n_steps, dt, io, opts, PlantEntry::plain, nullptr, nullptr);
}

extern "C" int wbc_rollout_perturbed_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                          const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb) {
  return rollout_host(h, kind, plan, n, n_steps, dt, io, opts, PlantEntry::perturbed, perturb, nullptr);
}

extern "C" int wbc_rollout_terrain_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                        const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                        const wbc_plant_terrain* terrain) {
  return rollout_host(h, kind, plan, n, n_steps, dt, io, opts, PlantEntry::terrain, perturb, terrain);
}

extern "C" int wbc_rollout_params_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                       const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                       const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl) {
  return rollout_host(h, kind, plan, n, n_steps, dt, io, opts, PlantEntry::params, perturb, terrain, ctrl);
}

extern "C" int wbc_rollout_loop_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                     const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                     const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop) {
  return rollout_host(h, kind, plan, n, n_steps, dt, io, opts, PlantEntry::loop, perturb, terrain, ctrl, loop);
}

extern "C" int wbc_rollout_monitor_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                        const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                        const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                                        const wbc_monitor* mon) {
  return rollout_host(h, kind, plan, n, n_steps, dt, io, opts, PlantEntry::monitor, perturb, terrain, ctrl, loop, mon);
}

extern "C" int wbc_rollout_motor_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                      const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                      const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                                      const wbc_monitor* mon, const wbc_plant_motor* motor) {
  return rollout_host(h, kind, plan, n, n_steps, dt, io, opts, PlantEntry::motor, perturb, terrain, ctrl, loop, mon, motor);
}

extern "C" int wbc_rollout_estimator_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                          const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                                          const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                                          const wbc_monitor* mon, const wbc_plant_motor* motor, const wbc_estimator* est) {
  return rollout_host(h, kind, plan, n, n_steps, dt, io, opts, PlantEntry::estimator, perturb, terrain, ctrl, loop, mon, motor, est);
}

extern "C" int wbc_rollout_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                                const wbc_rollout_io* io, int use_graph) {
  wbc_rollout_opts o{};
  o.use_graph = use_graph; o.plant = 0; o.f_contact = nullptr;
  wbc_default_plant_opts(&o.plant_opts);
  return wbc_rollout_ex_host(h, kind, plan, n, n_steps, dt, io, &o);
}

extern "C" void* wbc_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
  return p;
}
extern "C" void wbc_host_free(void* p) { if (p) cudaFreeHost(p); }

extern "C" int wbc_measure_fp64_peak(int device, double* tflops) {
  if (!tflops) return WBC_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return WBC_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return WBC_ERR_CUDA;
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 15;
  DevArray<double> out;
  if (out.reserve((size_t)blocks * threads) != cudaSuccess) return WBC_ERR_CUDA;
  Event e0, e1;
  cudaEventCreate(&e0.v); cudaEventCreate(&e1.v);
  fp64_peak_kernel<<<blocks, threads>>>(out.p, 1024);  // warm-up
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    fp64_peak_kernel<<<blocks, threads>>>(out.p, iters);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) return WBC_ERR_CUDA;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double fl = 2.0 * 8.0 * (double)iters * blocks * threads;
    const double tf = fl / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  *tflops = best;
  return WBC_OK;
}
