// Host harness around the terrain plant step of csrc/wbc_plant.cuh (see cuda_emu.h): what wbc_plant_terrain_kernel does per
// robot, with the variant and terrain records read in place instead of staged. Exports emu_plant_step_terrain for
// tests/test_plant_terrain.py. TEST INFRASTRUCTURE ONLY.
#include "cuda_emu.h"
#include "../../quadruped_drake_b200/csrc/wbc_device.cuh"
#include "../../quadruped_drake_b200/csrc/wbc_plant.cuh"
#include <vector>

thread_local int emu_lane;
thread_local EmuWarp* emu_warp;

namespace {
struct Lane {
  EmuWarp* warp; int lane; wbc::WarpSmem* sm; wbcplant::PlantSmem* psm; wbcplant::TerrainSmem* tsm; wbcplant::PlantArgs a;
  wbcplant::PerturbArgs pa; wbcplant::TerrainArgs ta;
};
void* lane_main(void* p) {
  Lane* j = (Lane*)p;
  emu_lane = j->lane;
  emu_warp = j->warp;
  for (long long i = 0; i < j->a.n; ++i) {
    const int k = wbcplant::plant_variant(j->pa, i);
    const wbcplant::PlantVariant& pv = j->pa.set[k < 0 ? 0 : k];
    wbcplant::plant_step_instance<true, true>(*j->sm, *j->psm, pv.md, j->a, i, j->lane, wbcplant::plant_perturb(j->pa, j->a, i, k, pv.mu),
                                              j->tsm, j->ta);
  }
  return nullptr;
}
}  // namespace

// models [K] with their friction mu [K] (NULL: the call's mu for every variant), variant [N] (NULL: 0), push [N][8] or NULL,
// t [N] (advanced by dt; required with pushes); terrains [T] as in wbc_terrain_set_create (NULL: flat ground, one terrain),
// terrain [N] (NULL: 0). The descriptors are not validated here.
extern "C" int emu_plant_step_terrain(const wbc_model* models, const double* mu, int n_variants, const int32_t* variant,
                                      const double* push, const wbc_terrain_desc* terrains, int n_terrains, const int32_t* terrain,
                                      double* t, long long n, double dt, double call_mu, double erp, int iters, double* q, double* v,
                                      const double* tau, double* f_contact, int32_t* status_or) {
  std::vector<wbcplant::PlantVariant> set(n_variants);
  for (int k = 0; k < n_variants; ++k) set[k] = wbcplant::PlantVariant{models[k], mu ? mu[k] : 0.0};
  std::vector<wbcplant::TerrainRec> trs;
  std::vector<double> heights;
  for (int k = 0; terrains && k < n_terrains; ++k) {
    trs.push_back(wbcplant::terrain_record(terrains[k], (long long)heights.size()));
    if (terrains[k].nx > 0) heights.insert(heights.end(), terrains[k].heights, terrains[k].heights + (size_t)terrains[k].nx * terrains[k].ny);
  }
  EmuWarp warp;
  pthread_barrier_init(&warp.bar, nullptr, 32);
  wbc::WarpSmem* sm = new wbc::WarpSmem();
  memset(sm, 0, sizeof(*sm));
  wbcplant::PlantSmem* psm = new wbcplant::PlantSmem();
  memset(psm, 0, sizeof(*psm));
  wbcplant::TerrainSmem* tsm = new wbcplant::TerrainSmem();
  memset(tsm, 0, sizeof(*tsm));
  const wbcplant::PlantArgs a{q, v, tau, t, nullptr, status_or, f_contact, nullptr, nullptr, nullptr, nullptr, n, dt, call_mu, erp, iters};
  const wbcplant::PerturbArgs pa{set.data(), variant, push, n_variants, mu ? 1 : 0};
  const wbcplant::TerrainArgs ta{terrains ? trs.data() : nullptr, heights.data(), terrain, terrains ? n_terrains : 1};
  std::vector<Lane> lanes(32);
  std::vector<pthread_t> th(32);
  for (int l = 0; l < 32; ++l) {
    lanes[l] = Lane{&warp, l, sm, psm, tsm, a, pa, ta};
    pthread_create(&th[l], nullptr, lane_main, &lanes[l]);
  }
  for (int l = 0; l < 32; ++l) pthread_join(th[l], nullptr);
  pthread_barrier_destroy(&warp.bar);
  delete sm;
  delete psm;
  delete tsm;
  return 0;
}
