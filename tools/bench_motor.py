#!/usr/bin/env python
"""Cost of the actuator model in the ground-plant loop, and three studies with it.

Cost: the ground-plant rollout of the ID and PC controllers (standing plan, 4096 robots x 100 steps, 65536 x 20) with the full
configuration of tools/bench_monitor.py - two plant variants, pushes, two terrains, N distinct parameter sets, distinct loop
profiles and a monitor - through wbc_rollout_monitor, and through wbc_rollout_motor with the ideal motor (one record) and with
16 distinct records (lag, envelope, friction) spread over the robots. Three rounds alternate the three; a figure is the mean of
3 timed rollouts after one warm-up (CUDA events).

--study:
  1. peak torque (0.3-1.5 x the URDF effort) x push impulse (0-20 N s at t = 1 s over 0.1 s): ID at dt = 5e-3, 64 jittered
     standing robots per cell, 6 s, with the monitor's three verdicts per cell - the end-state standing fraction of the tools (no
     status bit, base within 5 cm of its start, tilt below 0.3 rad) / the fraction that never failed (bounds 5 cm and 0.3 rad, no
     status bit at any step) / the median time to failure ("-" while more than half never failed).
  2. the QP's torque_limits 0 vs 1 (through a parameter set) with motors at peak = effort, over the push impulse: the same
     verdicts. Does a controller that knows its torque limits survive a push better than one that does not?
  3. motor lag (0, 2, 5, 10, 20 ms) x controller (ID, CLF, PC, PD) at dt = 1e-3, peak = effort, 3 s: the end-state standing
     fraction / never failed, and the median peak |tau| over effort.

The card name and its power limit are printed beside the numbers."""
import argparse
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from bench_loop import NOISE, standing_q0  # noqa: E402
from bench_params import distinct_sets  # noqa: E402
from bench_perturbed import card  # noqa: E402

IMPULSES = [0.0, 5.0, 10.0, 15.0, 20.0]


def distinct_motors(ctl, k, rng):
    from quadruped_drake_b200.rollout import MotorSet, motor_desc
    return MotorSet(ctl, [motor_desc(ctl.model, float(rng.uniform(0.6, 1.2)), speed_knee=rng.uniform(5, 15, 12),
                                     speed_free=rng.uniform(25, 40, 12), lag=rng.uniform(0, 4e-3, 12), damping=rng.uniform(0, 0.02, 12),
                                     coulomb=rng.uniform(0, 0.2, 12), coulomb_speed=0.1) for _ in range(k)])


def cost(rounds):
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import Loop, Monitor, Motor, MotorSet, PlantSet, Terrain, TerrainSet, motor_desc, rollout
    from quadruped_drake_b200.urdf import load_description
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(0)
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    plants = PlantSet(ctl, [flatten(d), flatten(with_payload(d, 1.2, (0.04, -0.02, 0.05)))], [1.0, 0.6])
    terrains = TerrainSet(ctl, [Terrain(), Terrain(slope=(np.tan(np.radians(5.0)), 0.0))])
    ideal = MotorSet(ctl, [motor_desc(ctl.model, np.inf)])
    motors = distinct_motors(ctl, 16, rng)
    q = standing_q0(ctl)
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=float(q[6])))
    for n in (4096, 65536):
        ps = distinct_sets(ctl, n, rng)
        T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
        push = np.zeros((n, 8))
        push[:, 0] = 50.0; push[:, 5] = 0.05; push[:, 6], push[:, 7] = 0.05, 0.1
        kw = dict(plant_set=plants, terrain_set=terrains, param_set=ps, param_index=torch.arange(n, dtype=torch.int32, device="cuda"),
                  variant=T((np.arange(n) % 2).astype(np.int32)), push=T(push), terrain=T((np.arange(n) // 2 % 2).astype(np.int32)),
                  loop=Loop(noise=T(NOISE * rng.uniform(0.5, 2.0, (n, 1))), delay=T(rng.integers(0, 3, n).astype(np.int32)),
                            strength=T(rng.uniform(0.8, 1.2, n)), stream=T(rng.integers(-2**31, 2**31, n).astype(np.int32)), seed=2026))
        modes = {"wbc_rollout_monitor": None, "ideal motor": (ideal, None),
                 "16 records": (motors, T(rng.integers(0, 16, n).astype(np.int32)))}
        k = 100 if n == 4096 else 20
        q0 = np.tile(q, (n, 1))

        def once(kind, mode):
            qt, vt, tt = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
            mo = None if modes[mode] is None else Motor(*modes[mode])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = rollout(ctl, s, kind, qt, vt, tt, k, 5e-3, plant=True, monitor=Monitor(), motor=mo, **kw)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), float((r.status_or.cpu().numpy() == 0).mean())

        with torch.cuda.stream(torch.cuda.Stream()):
            for kind in ("id", "pc"):
                ms = {m: [] for m in modes}
                for rnd in range(rounds):
                    for mode in modes:
                        once(kind, mode)
                        runs = [once(kind, mode) for _ in range(3)]
                        ms[mode].append(float(np.mean([x[0] for x in runs])))
                        print("rollout %-2s %6d x %3d  %-19s round %d  %8.2f ms  %.3f ms/step  status 0: %.2f"
                              % (kind, n, k, mode, rnd, ms[mode][-1], ms[mode][-1] / k, runs[-1][1]), flush=True)
                a = np.mean(ms["wbc_rollout_monitor"])
                for mode in list(modes)[1:]:
                    b = np.mean(ms[mode])
                    print("  %-2s %6d %-12s: %.3f -> %.3f ms/step, motor %+.1f %% (%+.1f us per step)"
                          % (kind, n, mode, a / k, b / k, 100.0 * (b / a - 1.0), 1e3 * (b - a) / k), flush=True)
        ps.close()
    motors.close(); ideal.close(); s.close(); terrains.close(); plants.close(); ctl.close()


def run_cells(ctl, kind, cells, per_cell, dt, seconds, rng):
    """per_cell jittered standing robots per cell (cells[c] = dict(peak, lag, push or None, params or None)) under the loop's
    noise profile, with a monitor and motors -> (the tools' end-state verdict [n], the rollout result, cell of each robot)."""
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import ParamSet
    from quadruped_drake_b200.rollout import Loop, Monitor, Motor, MotorSet, motor_desc, rollout
    q = standing_q0(ctl)
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=float(q[6])))
    n = len(cells) * per_cell
    cell = np.repeat(np.arange(len(cells)), per_cell)
    q0 = np.tile(q, (n, 1))
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    ms = MotorSet(ctl, [motor_desc(ctl.model, c.get("peak", 1.0), lag=c.get("lag", 0.0)) for c in cells])
    kw = dict(loop=Loop(noise=NOISE, seed=11), motor=Motor(ms, T(cell.astype(np.int32))))
    if any(c.get("push") is not None for c in cells):
        kw["push"] = T(np.array([[c["push"] / 0.1, 0, 0, 0, 0, 0.05, 1.0, 1.1] for c in cells])[cell])
    pset = None
    if any(c.get("params") is not None for c in cells):
        pset = ParamSet(ctl, [c.get("params") or {} for c in cells])
        kw.update(param_set=pset, param_index=T(cell.astype(np.int32)))
    qt, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    with torch.cuda.stream(torch.cuda.Stream()):
        r = rollout(ctl, s, kind, qt, v, t, int(round(seconds / dt)), dt, plant=True, monitor=Monitor(), **kw)
    torch.cuda.synchronize()
    qf, st = qt.cpu().numpy(), r.status_or.cpu().numpy()
    dotq = np.abs((q0[:, 0:4] * qf[:, 0:4]).sum(axis=1)) / np.linalg.norm(qf[:, 0:4], axis=1)
    tilt = 2 * np.arccos(np.clip(dotq, -1, 1))
    up = (st == 0) & (np.linalg.norm(qf[:, 4:7] - q0[:, 4:7], axis=1) < 0.05) & (tilt < 0.3)
    if pset is not None:
        pset.close()
    ms.close(); s.close()
    return up, r, cell


def verdicts(up, r, cell, c, dt):
    m = r.monitor
    never = (m.fail_step == 0).cpu().numpy()[cell == c]
    med = np.median(m.fail_time(0.0, dt).cpu().numpy()[cell == c])
    return "  %4.2f/%4.2f/%5s" % (up[cell == c].mean(), never.mean(), "-" if np.isinf(med) else "%.2f" % med)


def study(per_cell=64):
    from quadruped_drake_b200.controller import BatchedController
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(1)
    dt = 5e-3
    print("noise profile (std) of every study: orientation %g rad, base position %g m, joints %g rad, angular velocity %g rad/s, "
          "linear velocity %g m/s, joint velocities %g rad/s; no delay" % tuple(NOISE))
    peaks = [0.3, 0.5, 0.7, 1.0, 1.5]
    cells = [dict(peak=p, push=j) for j in IMPULSES for p in peaks]
    up, r, cell = run_cells(ctl, "id", cells, per_cell, dt, 6.0, rng)
    print("1. ID at dt = 5e-3, peak torque x push (rows: impulse N s over 0.1 s at t = 1 s, columns: peak / effort; %d robots per "
          "cell). Each cell: end-state standing / never failed / median time to failure (s)" % per_cell)
    print("%8s " % "" + "".join("%17.1f" % p for p in peaks))
    for i, j in enumerate(IMPULSES):
        print("%8.1f " % j + "".join(verdicts(up, r, cell, c, dt) for c in range(i * len(peaks), (i + 1) * len(peaks))))
    sat = r.monitor.sat_max.cpu().numpy()
    print("   median SAT_MAX per column at 0 N s: " + " ".join("%.2f" % np.median(sat[cell == c]) for c in range(len(peaks))))
    cells = [dict(peak=1.0, push=j, params={"torque_limits": tl}) for j in IMPULSES for tl in (0, 1)]
    up, r, cell = run_cells(ctl, "id", cells, per_cell, dt, 6.0, rng)
    print("2. ID at dt = 5e-3, motors at peak = effort: QP torque_limits 0 vs 1 over the push (%d robots per cell)" % per_cell)
    print("%8s %17s %17s" % ("", "torque_limits 0", "torque_limits 1"))
    for i, j in enumerate(IMPULSES):
        print("%8.1f " % j + "".join(verdicts(up, r, cell, c, dt) for c in (2 * i, 2 * i + 1)))
    lags = [0.0, 2e-3, 5e-3, 10e-3, 20e-3]
    print("3. controller x motor lag at dt = 1e-3, peak = effort, 3 s (%d robots per cell). Each cell: end-state standing / never "
          "failed / median SAT_MAX" % per_cell)
    print("%8s " % "" + "".join("%13.0f ms" % (1e3 * x) for x in lags))
    for kind in ("id", "clf", "pc", "pd"):
        up, r, cell = run_cells(ctl, kind, [dict(peak=1.0, lag=x) for x in lags], per_cell, 1e-3, 3.0, rng)
        never = (r.monitor.fail_step == 0).cpu().numpy()
        sat = r.monitor.sat_max.cpu().numpy()
        print("%8s " % kind + "".join("  %4.2f/%4.2f/%5.2f" % (up[cell == c].mean(), never[cell == c].mean(), np.median(sat[cell == c]))
                                      for c in range(len(lags))))
    ctl.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--study", action="store_true", help="also run the three studies")
    ap.add_argument("--no-cost", action="store_true", help="skip the cost measurement")
    a = ap.parse_args()
    print(card())
    if not a.no_cost:
        cost(a.rounds)
    if a.study:
        study()
    print(card())


if __name__ == "__main__":
    main()
