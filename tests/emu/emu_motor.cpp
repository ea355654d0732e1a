// Host harness around the actuator model of csrc/wbc_motor.cuh: what one 16-lane group of motor_kernel does per robot (lane 0's
// record and count, the 12 joint lanes, lane 0's bookkeeping), run on the host, and the record check of wbc_motor_set_create.
// Exports emu_motor_apply and emu_motor_desc_problem for tests/test_motor.py. TEST INFRASTRUCTURE ONLY.
#include "cuda_emu.h"
#include "../../quadruped_drake_b200/csrc/wbc_motor.cuh"

thread_local int emu_lane;
thread_local EmuWarp* emu_warp;

// One motor step of n robots: records [n_sets] (NULL: the one record of `effort`), index [n] or NULL, the state tau_m [n][12] and
// count [n], the model's v_index / act_index / effort [12]; v [n][18], tau_in [n][12] -> tau_plant [n][12], status [n] (ORed).
extern "C" void emu_motor_apply(long long n, double dt, const wbc_motor_desc* records, int n_sets, const int32_t* index, double* tau_m,
                                int64_t* count, const int32_t* v_index, const int32_t* act_index, const double* effort, const double* v,
                                const double* tau_in, double* tau_plant, int32_t* status) {
  wbcmotor::MotorArgs a{records, index, records ? n_sets : 1, tau_m, (long long*)count, dt, {}, {}, {}};
  for (int j = 0; j < WBC_NU; ++j) { a.v_index[j] = v_index[j]; a.act_index[j] = act_index[j]; a.effort[j] = effort[j]; }
  for (long long i = 0; i < n; ++i) {
    const int r = wbcmotor::motor_record(a, i);
    const long long c = r >= 0 ? a.count[i] : 0;
    for (int k = 0; k < WBC_NU; ++k) wbcmotor::motor_joint(a, i, k, r, c, v, tau_in, tau_plant);
    wbcmotor::motor_finish(a, i, r, c, status);
  }
}

// The reason wbc_motor_set_create rejects the record, or NULL.
extern "C" const char* emu_motor_desc_problem(const wbc_motor_desc* d) { return wbcmotor::desc_problem(*d); }
