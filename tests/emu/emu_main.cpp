// Host harness around csrc/wbc_device.cuh (see cuda_emu.h). Exports two C functions used by
// tests/test_emulator.py. TEST INFRASTRUCTURE ONLY.
#include "cuda_emu.h"
#include "../../quadruped_drake_b200/csrc/wbc_device.cuh"
#include "../../quadruped_drake_b200/csrc/wbc_plant.cuh"
#include <vector>

thread_local int emu_lane;
thread_local EmuWarp* emu_warp;

namespace {
struct Job {
  EmuWarp* warp; int lane; wbc::WarpSmem* sm; wbc::SolveSmemVd* ssm; wbc::SolveSmem* ssm0; double* rec; double* vdmap; wbc::PcSmem* pcs; double* Cout; double* Jdout; const wbc_model* md; const wbc_params* pr; wbc::Derived dv;
  wbc::StepArgs args; wbc::DynOut dyn; const double* q; const double* v; long long n; int mode;
  wbcplant::PlantSmem* psm; wbcplant::PlantArgs pargs;
};
template <int KIND> void split_step(Job* j, long long i) {
  wbc::StepCarry c;
  double* vd = j->args.vd ? j->vdmap : nullptr;
  wbc::reduce_instance<KIND>(*j->sm, *j->md, *j->pr, j->dv, j->args, i, j->lane, c, KIND == WBC_CTRL_PC ? j->pcs : nullptr, vd);
  __syncwarp();
  if (j->lane == 0) memcpy(j->rec, &j->sm->Y[0][0], sizeof(double) * wbc::REC_Y);
  __syncwarp();
  // the solve kernel variant launch_split picks: with vd, L kept beside R^-1 (SolveSmemVd) and the x recovery from the
  // record; without, R^-1 overlaid on L (SolveSmem), no acceleration maps and no record read-back
  if (vd) {
    if (j->lane == 0) memcpy(&j->ssm->Y[0][0], j->rec, sizeof(double) * wbc::REC_Y);
    __syncwarp();
    wbc::solve_instance<KIND, wbc::SolveSmemVd>(*j->ssm, *j->md, *j->pr, j->args, i, j->lane, c, vd, j->rec);
  } else {
    if (j->lane == 0) memcpy(&j->ssm0->Y[0][0], j->rec, sizeof(double) * wbc::REC_Y);
    __syncwarp();
    wbc::solve_instance<KIND, wbc::SolveSmem>(*j->ssm0, *j->md, *j->pr, j->args, i, j->lane, c);
  }
  __syncwarp();
}
void* lane_main(void* p) {
  Job* j = (Job*)p;
  emu_lane = j->lane;
  emu_warp = j->warp;
  for (long long i = 0; i < j->n; ++i) {
    if (j->mode == 0) {
      // reduce on the full block, hand-over record (what the reduce / solve kernels do with bulk copies), solve on the compact block
      if (j->args.kind == WBC_CTRL_ID) split_step<WBC_CTRL_ID>(j, i);
      else if (j->args.kind == WBC_CTRL_CLF) split_step<WBC_CTRL_CLF>(j, i);
      else split_step<WBC_CTRL_PC>(j, i);
    } else if (j->mode == 1) {
      wbc::dynamics_instance(*j->sm, *j->md, j->q, j->v, j->dyn, i, j->lane);
    } else if (j->mode == 2) {
      wbc::coriolis_instance(*j->sm, *j->pcs, *j->md, j->q, j->v, j->Cout, j->Jdout, i, j->lane);
    } else {
      wbcplant::plant_step_instance(*j->sm, *j->psm, *j->md, j->pargs, i, j->lane);
    }
  }
  return nullptr;
}
int run(Job proto) {
  EmuWarp warp;
  pthread_barrier_init(&warp.bar, nullptr, 32);
  wbc::WarpSmem* sm = new wbc::WarpSmem();
  memset(sm, 0, sizeof(*sm));
  wbc::PcSmem* pcs = new wbc::PcSmem();
  memset(pcs, 0, sizeof(*pcs));
  wbc::SolveSmemVd* ssm = new wbc::SolveSmemVd();
  memset(ssm, 0, sizeof(*ssm));
  wbc::SolveSmem* ssm0 = new wbc::SolveSmem();
  memset(ssm0, 0, sizeof(*ssm0));
  wbcplant::PlantSmem* psm = new wbcplant::PlantSmem();
  memset(psm, 0, sizeof(*psm));
  std::vector<double> rec(wbc::REC_DOUBLES), vdmap(wbc::VDMAP_DOUBLES);
  std::vector<Job> jobs(32, proto);
  std::vector<pthread_t> th(32);
  for (int l = 0; l < 32; ++l) {
    jobs[l].warp = &warp; jobs[l].lane = l; jobs[l].sm = sm; jobs[l].pcs = pcs; jobs[l].ssm = ssm; jobs[l].ssm0 = ssm0; jobs[l].psm = psm; jobs[l].rec = rec.data(); jobs[l].vdmap = vdmap.data();
    pthread_create(&th[l], nullptr, lane_main, &jobs[l]);
  }
  for (int l = 0; l < 32; ++l) pthread_join(th[l], nullptr);
  pthread_barrier_destroy(&warp.bar);
  delete sm;
  delete pcs;
  delete ssm;
  delete ssm0;
  delete psm;
  return 0;
}
}  // namespace

extern "C" int emu_step(const wbc_model* md, const wbc_params* pr, int kind, long long n, const wbc_io* io) {
  Job j{};
  wbc::derive_constants(*pr, j.dv);
  j.md = md; j.pr = pr; j.n = n; j.mode = 0;
  j.args.q = io->q; j.args.v = io->v; j.args.traj = io->traj; j.args.contact = io->contact;
  j.args.tau = io->tau; j.args.metrics = io->metrics; j.args.status = io->status;
  j.args.vd = io->vd; j.args.f = io->f; j.args.qp_info = io->qp_info; j.args.lam = io->lam; j.args.n = n; j.args.kind = kind;
  return run(j);
}
extern "C" int emu_dynamics(const wbc_model* md, long long n, const double* q, const double* v, double* M, double* Cv,
                            double* taug, double* Jfeet, double* Jdv, double* pfeet) {
  Job j{};
  j.md = md; j.n = n; j.mode = 1; j.q = q; j.v = v;
  j.dyn.M = M; j.dyn.Cv = Cv; j.dyn.taug = taug; j.dyn.Jfeet = Jfeet; j.dyn.Jdv = Jdv; j.dyn.pfeet = pfeet;
  return run(j);
}
extern "C" int emu_coriolis(const wbc_model* md, long long n, const double* q, const double* v, double* Cm, double* Jd) {
  Job j{};
  j.md = md; j.n = n; j.mode = 2; j.q = q; j.v = v; j.Cout = Cm; j.Jdout = Jd;
  return run(j);
}
extern "C" int emu_plant_step(const wbc_model* md, long long n, double dt, double mu, double erp, int iters, double* q, double* v,
                              const double* tau, double* f_contact, int32_t* status_or) {
  Job j{};
  j.md = md; j.n = n; j.mode = 3;
  j.pargs = wbcplant::PlantArgs{q, v, tau, nullptr, nullptr, status_or, f_contact, nullptr, nullptr, nullptr, nullptr, n, dt, mu, erp, iters};
  return run(j);
}
extern "C" int emu_smem_bytes() { return (int)sizeof(wbc::WarpSmem); }
