// Host harness around the monitor of csrc/wbc_monitor.cuh: what monitor_kernel does per robot, run on the host. Exports
// emu_monitor_step for tests/test_rollout_monitor.py. TEST INFRASTRUCTURE ONLY.
#include "cuda_emu.h"
#include "../../quadruped_drake_b200/csrc/wbc_monitor.cuh"

thread_local int emu_lane;
thread_local EmuWarp* emu_warp;

// One monitored step of n robots; the model's v_index / act_index / effort [12] and the state arrays as in wbc_monitor.
extern "C" void emu_monitor_step(long long n, double dt, double pos_max, double ang_max, const int32_t* v_index, const int32_t* act_index,
                                 const double* effort, double* stats, int64_t* steps, int64_t* fail_step, int32_t* fail_why, int32_t* why,
                                 const double* q, const double* v, const double* traj, const uint8_t* contact, const double* tau,
                                 const double* f, const int32_t* status) {
  wbcmon::MonArgs a{pos_max, ang_max, dt, stats, (long long*)steps, (long long*)fail_step, fail_why, why, {}, {}, {}};
  for (int j = 0; j < WBC_NU; ++j) { a.v_index[j] = v_index[j]; a.act_index[j] = act_index[j]; a.effort[j] = effort[j]; }
  for (long long i = 0; i < n; ++i) wbcmon::monitor_instance(a, i, q, v, traj, contact, tau, f, status ? status[i] : 0);
}
