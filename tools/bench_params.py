#!/usr/bin/env python
"""Cost of per-robot controller parameters, and two gain studies they make possible in one run.

Cost: the device step (torch tensors, synthetic "mixed" states) of ID and PC at 4096 and 65536 instances through wbc_step
against wbc_step_params with N distinct parameter sets (every robot its own record), and the ground-plant rollout of the ID
and PC controllers (standing plan, 4096 robots x 100 steps, 65536 x 20) through wbc_rollout_ex against wbc_rollout_params. Three
rounds alternate the two entries; a step figure is the mean over 200 steps (CUDA events) after 20 warm-up steps, a rollout
figure the mean of 3 timed rollouts after one warm-up.

--study: 6 s of standing robots on the ground plant, 64 per cell with jittered joints; prints the fraction of each cell still
standing at the end, by the criterion of tools/bench_terrain.py (no status bit, base within 5 cm of its start, tilt below
0.3 rad).
  1. the PD law over a pd_kp x pd_kd grid, at dt = 1e-3 and 5e-3;
  2. ID over a scale of its body gains (id_kp_body_*, id_kd_body_*) x a horizontal push impulse at t = 1 s over 0.1 s,
     the push of tools/bench_perturbed.py (at 5 cm above the base origin), dt = 5e-3.
Each table is one rollout of all its cells.

The card name and its power limit are printed beside the numbers."""
import argparse
import ctypes as C
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from bench_perturbed import card  # noqa: E402


def distinct_sets(ctl, n, rng):
    """n parameter sets that differ in every record (gains x 1 +- 1e-3), for the cost measurement."""
    from quadruped_drake_b200.capi import WbcParams
    from quadruped_drake_b200.controller import ParamSet
    recs = (WbcParams * n)()
    scale = 1.0 + rng.uniform(-1e-3, 1e-3, n)
    for i in range(n):
        C.memmove(C.byref(recs[i]), C.byref(ctl.params), C.sizeof(WbcParams))
        for f in ("id_kp_body_p", "pc_kp_body_p"):
            setattr(recs[i], f, getattr(ctl.params, f) * scale[i])
    return ParamSet(ctl, recs)


def cost(rounds):
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.rollout import Q0_MINI_CHEETAH as Q0, rollout
    from quadruped_drake_b200.synth import generate
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(0)
    for n in (4096, 65536):
        ps = distinct_sets(ctl, n, rng)
        idx = torch.arange(n, dtype=torch.int32, device="cuda")
        q, v, traj, contact = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in generate(ctl.model, n, 1, "mixed", ctl.fk))
        for kind in ("id", "pc"):
            def steps(per_robot, reps):
                kw = dict(param_set=ps, param_index=idx) if per_robot else {}
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    ctl.step(kind, q, v, traj, contact, **kw)
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / reps
            for rnd in range(rounds):
                for per_robot in (False, True):
                    steps(per_robot, 20)
                    ms = steps(per_robot, 200)
                    print("step  %-2s %6d  %-10s round %d  %.2f M steps/s" % (kind, n, "params" if per_robot else "wbc_step", rnd, n / ms / 1e3),
                          flush=True)
        bh = Q0[6] - ctl.dynamics(Q0[None], np.zeros((1, 18)))["p_feet"][0, :, 2].min()
        s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh))
        k = 100 if n == 4096 else 20
        q0 = np.tile(Q0, (n, 1)); q0[:, 6] = bh

        def once(kind, per_robot):
            kw = dict(param_set=ps, param_index=idx) if per_robot else {}
            qt, vt, tt = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rollout(ctl, s, kind, qt, vt, tt, k, 5e-3, plant=True, **kw)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)

        with torch.cuda.stream(torch.cuda.Stream()):
            for kind in ("id", "pc"):
                for rnd in range(rounds):
                    for per_robot in (False, True):
                        once(kind, per_robot)
                        ms = float(np.mean([once(kind, per_robot) for _ in range(3)]))
                        print("rollout %-2s %6d x %3d  %-10s round %d  %.2f M robot-steps/s"
                              % (kind, n, k, "params" if per_robot else "wbc_rollout_ex", rnd, n * k / (ms * 1e-3) / 1e6), flush=True)
        s.close(); ps.close()
    ctl.close()


def standing(ctl, kind, sets, set_of_cell, per_cell, dt, rng, push=None):
    """Fraction of per_cell robots of each cell standing after 6 s; cell c runs with sets[set_of_cell[c]] and push row push[c]."""
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.rollout import Q0_MINI_CHEETAH as Q0, rollout
    q = Q0.copy()
    q[6] -= ctl.dynamics(q[None], np.zeros((1, 18)))["p_feet"][0, :, 2].min()
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=float(q[6])))
    cells = len(set_of_cell)
    n = cells * per_cell
    q0 = np.tile(q, (n, 1))
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    cell = np.repeat(np.arange(cells), per_cell)
    ps = ParamSet(ctl, sets)
    idx = torch.from_numpy(np.asarray(set_of_cell, np.int32)[cell]).cuda()
    kw = {} if push is None else dict(push=torch.from_numpy(np.ascontiguousarray(push[cell])).cuda())
    qt, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    with torch.cuda.stream(torch.cuda.Stream()):
        r = rollout(ctl, s, kind, qt, v, t, int(round(6.0 / dt)), dt, plant=True, param_set=ps, param_index=idx, **kw)
    torch.cuda.synchronize()
    qf, st = qt.cpu().numpy(), r.status_or.cpu().numpy()
    dotq = np.abs((q0[:, 0:4] * qf[:, 0:4]).sum(axis=1)) / np.linalg.norm(qf[:, 0:4], axis=1)
    tilt = 2 * np.arccos(np.clip(dotq, -1, 1))
    up = (st == 0) & (np.linalg.norm(qf[:, 4:7] - q0[:, 4:7], axis=1) < 0.05) & (tilt < 0.3)
    ps.close(); s.close()
    return np.array([up[cell == c].mean() for c in range(cells)])


def study(per_cell=64):
    from quadruped_drake_b200.capi import DEFAULT_PARAMS
    from quadruped_drake_b200.controller import BatchedController
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(1)
    kps, kds = [10.0, 20.0, 30.0, 60.0, 120.0], [0.3, 0.75, 1.5, 3.0, 6.0]
    sets = [dict(pd_kp=kp, pd_kd=kd) for kp in kps for kd in kds]
    for dt in (1e-3, 5e-3):
        up = standing(ctl, "pd", sets, list(range(len(sets))), per_cell, dt, rng).reshape(len(kps), len(kds))
        print("PD: fraction standing after 6 s at dt = %g (rows: pd_kp, columns: pd_kd; %d robots per cell)" % (dt, per_cell))
        print("%8s " % "" + "".join("%7.2f" % kd for kd in kds))
        for i, kp in enumerate(kps):
            print("%8.1f " % kp + "".join("%7.2f" % x for x in up[i]))
    scales, impulses = [0.25, 0.5, 1.0, 2.0, 4.0], [0.0, 5.0, 10.0, 15.0, 20.0]
    gains = ["id_kp_body_p", "id_kd_body_p", "id_kp_body_rpy", "id_kd_body_rpy"]
    sets = [{g: DEFAULT_PARAMS[g] * s for g in gains} for s in scales]
    set_of_cell, push = [], []
    for i in range(len(scales)):
        for j in impulses:
            set_of_cell.append(i)
            push.append([j / 0.1, 0, 0, 0, 0, 0.05, 1.0, 1.1])
    up = standing(ctl, "id", sets, set_of_cell, per_cell, 5e-3, rng, np.array(push)).reshape(len(scales), len(impulses))
    print("ID: fraction standing after 6 s (rows: body-gain scale, columns: push impulse N s over 0.1 s at t = 1 s; dt = 5e-3; %d robots "
          "per cell)" % per_cell)
    print("%8s " % "" + "".join("%7.1f" % j for j in impulses))
    for i, sc in enumerate(scales):
        print("%8.2f " % sc + "".join("%7.2f" % x for x in up[i]))
    ctl.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--study", action="store_true", help="also run the PD gain grid and the ID gain x push grid")
    a = ap.parse_args()
    print(card())
    cost(a.rounds)
    if a.study:
        study()
    print(card())


if __name__ == "__main__":
    main()
