// Host harness around the parameter-aware step of csrc/wbc_device.cuh (see cuda_emu.h): what wbc_reduce_params_kernel,
// wbc_solve_params_kernel and wbc_pd_params_kernel do per robot - the record selection of param_record, reduce on the robot's
// record, hand-over, solve on the same record - with the records read in place instead of staged. Exports emu_step_params for
// tests/test_param_sets.py. TEST INFRASTRUCTURE ONLY.
#include "cuda_emu.h"
#include "../../quadruped_drake_b200/csrc/wbc_device.cuh"
#include <vector>

thread_local int emu_lane;
thread_local EmuWarp* emu_warp;

namespace {
struct Lane {
  EmuWarp* warp; int lane; wbc::WarpSmem* sm; wbc::SolveSmemVd* ssm; wbc::PcSmem* pcs; double* rec; double* vdmap;
  const wbc_model* md; wbc::ParamArgs p; wbc::StepArgs a;
};
template <int KIND> void step(Lane* j, long long i) {
  int pstatus = 0;
  const wbc::ParamRec& r = wbc::param_record(j->p, i, pstatus);
  wbc::StepCarry c;
  double* vd = j->a.vd ? j->vdmap : nullptr;
  wbc::reduce_instance<KIND>(*j->sm, *j->md, r.pr, r.dv, j->a, i, j->lane, c, KIND == WBC_CTRL_PC ? j->pcs : nullptr, vd);
  c.status |= pstatus;
  __syncwarp();
  if (j->lane == 0) memcpy(j->rec, &j->sm->Y[0][0], sizeof(double) * wbc::REC_Y);
  __syncwarp();
  if (j->lane == 0) memcpy(&j->ssm->Y[0][0], j->rec, sizeof(double) * wbc::REC_Y);
  __syncwarp();
  int sstatus = 0;                 // the solve kernel selects the record again from the index
  const wbc::ParamRec& rs = wbc::param_record(j->p, i, sstatus);
  c.status |= sstatus;
  wbc::solve_instance<KIND, wbc::SolveSmemVd>(*j->ssm, *j->md, rs.pr, j->a, i, j->lane, c, vd, j->rec);
  __syncwarp();
}
void* lane_main(void* p) {
  Lane* j = (Lane*)p;
  emu_lane = j->lane;
  emu_warp = j->warp;
  for (long long i = 0; i < j->a.n; ++i) {
    if (j->a.kind == WBC_CTRL_ID) step<WBC_CTRL_ID>(j, i);
    else if (j->a.kind == WBC_CTRL_CLF) step<WBC_CTRL_CLF>(j, i);
    else step<WBC_CTRL_PC>(j, i);
  }
  return nullptr;
}
}  // namespace

// params [K] (derived constants computed here, as wbc_param_set_create does), index [N] (NULL: set 0). WBC_CTRL_PD uses q, v,
// tau and status of io only.
extern "C" int emu_step_params(const wbc_model* md, const wbc_params* params, int n_sets, const int32_t* index, int kind, long long n,
                               const wbc_io* io) {
  std::vector<wbc::ParamRec> set(n_sets);
  for (int k = 0; k < n_sets; ++k) {
    set[k].pr = params[k];
    wbc::derive_constants(params[k], set[k].dv);
  }
  const wbc::ParamArgs p{set.data(), index, n_sets};
  if (kind == WBC_CTRL_PD) {
    for (long long t = 0; t < n * WBC_NU; ++t) wbc::pd_params_element(*md, p, io->q, io->v, io->tau, io->status, t / WBC_NU, (int)(t % WBC_NU));
    return 0;
  }
  const wbc::StepArgs a{io->q, io->v, io->traj, io->contact, io->tau, io->metrics, io->status, io->vd, io->f, io->qp_info, io->lam, n, kind};
  EmuWarp warp;
  pthread_barrier_init(&warp.bar, nullptr, 32);
  wbc::WarpSmem* sm = new wbc::WarpSmem();
  memset(sm, 0, sizeof(*sm));
  wbc::PcSmem* pcs = new wbc::PcSmem();
  memset(pcs, 0, sizeof(*pcs));
  wbc::SolveSmemVd* ssm = new wbc::SolveSmemVd();
  memset(ssm, 0, sizeof(*ssm));
  std::vector<double> rec(wbc::REC_DOUBLES), vdmap(wbc::VDMAP_DOUBLES);
  std::vector<Lane> lanes(32);
  std::vector<pthread_t> th(32);
  for (int l = 0; l < 32; ++l) {
    lanes[l] = Lane{&warp, l, sm, ssm, pcs, rec.data(), vdmap.data(), md, p, a};
    pthread_create(&th[l], nullptr, lane_main, &lanes[l]);
  }
  for (int l = 0; l < 32; ++l) pthread_join(th[l], nullptr);
  pthread_barrier_destroy(&warp.bar);
  delete sm;
  delete pcs;
  delete ssm;
  return 0;
}
