// Host harness around the sensing and actuation functions of csrc/wbc_loop.cuh: what observe_kernel and actuate_kernel do per
// robot, one thread per robot, run on the host. Exports emu_philox, emu_normals, emu_observe and emu_actuate for
// tests/test_sensing_loop.py. TEST INFRASTRUCTURE ONLY.
#include "cuda_emu.h"
// CUDA's sincospi(x) is sin / cos of pi x; the host restatement rounds pi x first (a few ulp, inside the tests' bars)
static inline void sincospi(double x, double* s, double* c) { sincos(M_PI * x, s, c); }
#include "../../quadruped_drake_b200/csrc/wbc_loop.cuh"

thread_local int emu_lane;
thread_local EmuWarp* emu_warp;

namespace {
wbcloop::LoopArgs args(const double* noise, const int32_t* delay, const double* strength, const int32_t* stream, uint64_t seed,
                       double* hist, int64_t* tick) {
  return wbcloop::LoopArgs{noise, delay, strength, stream, (unsigned long long)seed, hist, (long long*)tick};
}
}  // namespace

// ctr [n][4], key [n][2] -> out [n][4]
extern "C" void emu_philox(long long n, const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
  for (long long i = 0; i < n; ++i) {
    uint32_t c[4] = {ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3]};
    wbcloop::philox4x32_10(c, key[2 * i], key[2 * i + 1]);
    for (int k = 0; k < 4; ++k) out[4 * i + k] = c[k];
  }
}

// the 36 normals of (seed, stream, c) -> z [36]
extern "C" void emu_normals(uint64_t seed, uint32_t stream, long long c, double* z) { wbcloop::normals(seed, stream, c, z); }

extern "C" void emu_observe(long long n, const double* noise, const int32_t* delay, const double* strength, const int32_t* stream,
                            uint64_t seed, int64_t* tick, const double* q, const double* v, double* q_obs, double* v_obs) {
  const wbcloop::LoopArgs a = args(noise, delay, strength, stream, seed, nullptr, tick);
  for (long long i = 0; i < n; ++i) wbcloop::observe_instance(a, i, q, v, q_obs, v_obs);
}

extern "C" void emu_actuate(long long n, const int32_t* delay, const double* strength, const double* noise, double* hist, int64_t* tick,
                            const double* tau, double* applied, int32_t* status) {
  const wbcloop::LoopArgs a = args(noise, delay, strength, nullptr, 0, hist, tick);
  for (long long i = 0; i < n; ++i) wbcloop::actuate_instance(a, i, tau, applied, status);
}
