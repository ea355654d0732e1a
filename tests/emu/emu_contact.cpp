// Host harness around the contact detector of csrc/wbc_contact.cuh (see cuda_emu.h): what one warp of contact_detect_kernel does
// per robot and what contact_record_kernel does per element, run on the host with one thread per lane, and the record check of
// wbc_contact_set_create. Exports emu_contact_step, emu_contact_record and emu_contact_desc_problem for tests/test_contact.py.
// TEST INFRASTRUCTURE ONLY.
#include "cuda_emu.h"
#include "../../quadruped_drake_b200/csrc/wbc_contact.cuh"
#include <vector>

thread_local int emu_lane;
thread_local EmuWarp* emu_warp;

namespace {
wbccontact::ContactArgs args(double dt, const wbc_contact_desc* records, int n_sets, const int32_t* index, double* q_prev,
                             double* v_prev, double* tau_prev, double* f_true, double* f_hat, uint8_t* flag, int64_t* count,
                             double* stats) {
  return wbccontact::ContactArgs{records, index, n_sets, q_prev, v_prev, tau_prev, f_true, f_hat, flag, (long long*)count, stats, dt};
}

struct Lane {
  EmuWarp* warp; int lane; wbc::WarpSmem* sm; const wbccontact::ContactArgs* a; const wbc_model* md; long long n;
  const double *q, *v; const uint8_t* plan; uint8_t *detected, *ctrl; int32_t* status_or;
};
void* lane_main(void* p) {
  Lane* j = (Lane*)p;
  emu_lane = j->lane;
  emu_warp = j->warp;
  for (long long i = 0; i < j->n; ++i) {
    wbccontact::detect_robot(*j->a, *j->md, i, j->lane, *j->sm, j->q, j->v, j->plan, j->detected, j->ctrl, j->status_or);
    __syncwarp();                      // the next robot reuses the warp's shared memory (on the device each robot has its own)
  }
  return nullptr;
}
}  // namespace

// One detector step of n robots: the handle's model, records [n_sets], index [n] or NULL, the state q_prev [n][19], v_prev [n][18],
// tau_prev [n][12], f_true [n][12], f_hat [n][12], flag [n][4], count [n], stats [n][6] or NULL; q [n][19], v [n][18], the plan's
// flags [n][4] -> detected [n][4], ctrl [n][4] (plan AND detected) or NULL, status_or [n] or NULL (ORed).
extern "C" void emu_contact_step(const wbc_model* md, long long n, double dt, const wbc_contact_desc* records, int n_sets,
                                 const int32_t* index, double* q_prev, double* v_prev, double* tau_prev, double* f_true, double* f_hat,
                                 uint8_t* flag, int64_t* count, double* stats, const double* q, const double* v, const uint8_t* plan,
                                 uint8_t* detected, uint8_t* ctrl, int32_t* status_or) {
  const wbccontact::ContactArgs a = args(dt, records, n_sets, index, q_prev, v_prev, tau_prev, f_true, f_hat, flag, count, stats);
  EmuWarp warp;
  pthread_barrier_init(&warp.bar, nullptr, 32);
  wbc::WarpSmem* sm = new wbc::WarpSmem();
  std::vector<Lane> lanes(32);
  std::vector<pthread_t> th(32);
  for (int l = 0; l < 32; ++l) {
    lanes[l] = Lane{&warp, l, sm, &a, md, n, q, v, plan, detected, ctrl, status_or};
    pthread_create(&th[l], nullptr, lane_main, &lanes[l]);
  }
  for (int l = 0; l < 32; ++l) pthread_join(th[l], nullptr);
  pthread_barrier_destroy(&warp.bar);
  delete sm;
}

// The record step of n robots: tau_meas [n][12] and f_contact [n][12] into tau_prev and f_true (robots with a bad index untouched).
extern "C" void emu_contact_record(long long n, int n_sets, const int32_t* index, double* tau_prev, double* f_true, const double* tau_meas,
                                   const double* f_contact) {
  const wbccontact::ContactArgs a = args(1.0, nullptr, n_sets, index, nullptr, nullptr, tau_prev, f_true, nullptr, nullptr, nullptr,
                                         nullptr);
  for (long long t = 0; t < n * WBC_NU; ++t) wbccontact::record_element(a, t, tau_meas, f_contact);
}

// The reason wbc_contact_set_create rejects the record, or NULL.
extern "C" const char* emu_contact_desc_problem(const wbc_contact_desc* d) { return wbccontact::desc_problem(*d); }
