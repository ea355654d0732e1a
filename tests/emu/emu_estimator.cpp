// Host harness around the state estimator of csrc/wbc_estimator.cuh (see cuda_emu.h): what one warp of estimate_kernel does per
// robot, run on the host with one thread per lane, and the record check of wbc_estimator_set_create. Exports emu_estimator_step,
// emu_leg_kinematics and emu_estimator_desc_problem for tests/test_estimator.py. TEST INFRASTRUCTURE ONLY.
#include "cuda_emu.h"
// CUDA's sincospi(x) is sin / cos of pi x; the host restatement rounds pi x first (a few ulp, inside the tests' bars)
static inline void sincospi(double x, double* s, double* c) { sincos(M_PI * x, s, c); }
#include "../../quadruped_drake_b200/csrc/wbc_estimator.cuh"
#include <vector>

thread_local int emu_lane;
thread_local EmuWarp* emu_warp;

namespace {
wbcest::EstArgs args(const wbc_model* md, double dt, const wbc_estimator_desc* records, int n_sets, const int32_t* index,
                     const double* accel_noise, double* x, double* P, double* v_prev, int64_t* count, double* stats, uint64_t seed,
                     const int32_t* stream, const int64_t* tick) {
  wbcest::EstArgs a{};
  a.set = records; a.index = index; a.n_sets = n_sets; a.accel_noise = accel_noise;
  a.x = x; a.P = P; a.v_prev = v_prev; a.count = (long long*)count; a.stats = stats; a.dt = dt;
  a.seed = seed; a.stream = stream; a.tick = (const long long*)tick;
  for (int c = 0; c < 3; ++c) a.gravity[c] = md->gravity[c];
  for (int k = 0; k < WBC_NU; ++k) {
    a.v_index[k] = md->v_index[k];
    for (int c = 0; c < 3; ++c) { a.joint_xyz[k][c] = md->joint_xyz[k][c]; a.joint_axis[k][c] = md->joint_axis[k][c]; }
  }
  for (int l = 0; l < WBC_NLEG; ++l)
    for (int c = 0; c < 3; ++c) a.foot_xyz[l][c] = md->foot_xyz[l][c];
  return a;
}

struct Lane {
  EmuWarp* warp; int lane; wbcest::EstSmem* sm; const wbcest::EstArgs* a; long long n;
  const double *q, *v; double *q_obs, *v_obs; const uint8_t* contact; int32_t* status_or;
};
void* lane_main(void* p) {
  Lane* j = (Lane*)p;
  emu_lane = j->lane;
  emu_warp = j->warp;
  for (long long i = 0; i < j->n; ++i) {
    wbcest::estimate_robot(*j->a, i, j->lane, *j->sm, j->q, j->v, j->q_obs, j->v_obs, j->contact, j->status_or);
    __syncwarp();                      // the next robot reuses the warp's shared memory (on the device each robot has its own)
  }
  return nullptr;
}
}  // namespace

// One estimator step of n robots: the handle's model, records [n_sets], index [n] or NULL, accel_noise [n] or NULL, the state
// x [n][18], P [n][18][18], v_prev [n][3], count [n], stats [n][4] or NULL; the loop's seed, stream [n] or NULL, tick [n] or NULL;
// q [n][19], v [n][18], q_obs / v_obs (in/out), contact [n][4], status_or [n] or NULL (ORed).
extern "C" void emu_estimator_step(const wbc_model* md, long long n, double dt, const wbc_estimator_desc* records, int n_sets,
                                   const int32_t* index, const double* accel_noise, double* x, double* P, double* v_prev, int64_t* count,
                                   double* stats, uint64_t seed, const int32_t* stream, const int64_t* tick, const double* q,
                                   const double* v, double* q_obs, double* v_obs, const uint8_t* contact, int32_t* status_or) {
  const wbcest::EstArgs a = args(md, dt, records, n_sets, index, accel_noise, x, P, v_prev, count, stats, seed, stream, tick);
  EmuWarp warp;
  pthread_barrier_init(&warp.bar, nullptr, 32);
  wbcest::EstSmem* sm = new wbcest::EstSmem();
  std::vector<Lane> lanes(32);
  std::vector<pthread_t> th(32);
  for (int l = 0; l < 32; ++l) {
    lanes[l] = Lane{&warp, l, sm, &a, n, q, v, q_obs, v_obs, contact, status_or};
    pthread_create(&th[l], nullptr, lane_main, &lanes[l]);
  }
  for (int l = 0; l < 32; ++l) pthread_join(th[l], nullptr);
  pthread_barrier_destroy(&warp.bar);
  delete sm;
}

// Foot `leg` of the model at q [19], v [18]: r [3] (base axes, relative to the base origin) and J thetadot [3].
extern "C" void emu_leg_kinematics(const wbc_model* md, const double* q, const double* v, int leg, double* r, double* jv) {
  const wbcest::EstArgs a = args(md, 1.0, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr);
  wbcest::leg_kinematics(a, q, v, leg, r, jv);
}

// The reason wbc_estimator_set_create rejects the record, or NULL.
extern "C" const char* emu_estimator_desc_problem(const wbc_estimator_desc* d) { return wbcest::desc_problem(*d); }
