#!/usr/bin/env python
"""Cost of the rollout monitor in the ground-plant loop, and what it adds to the push x delay study of tools/bench_loop.py.

Cost: the ground-plant rollout of the ID and PC controllers (standing plan, 4096 robots x 100 steps, 65536 x 20) with the full
configuration of the cost run of tools/bench_loop.py - two plant variants, pushes, two terrains, N distinct parameter sets and
distinct loop profiles (noise, delay 0-2, strength, streams) - through wbc_rollout_loop without and with a monitor (the same
work plus one launch per step). Three rounds alternate the two; a figure is the mean of 3 timed rollouts after one warm-up
(CUDA events).

--study: the push x delay study (study 2 of tools/bench_loop.py: ID at dt = 5e-3 with the noise profile, a horizontal push
impulse at t = 1 s over 0.1 s, 64 robots per cell, 6 s) with a monitor. Per cell: the end-state standing fraction of the tools
(no status bit, base within 5 cm of its start, tilt below 0.3 rad), the fraction that never failed (monitor bounds 5 cm and
0.3 rad, no status bit at any step) and the median time to failure (over every robot of the cell; "-" while more than half never
failed). Then study 1 of tools/bench_loop.py (ID, CLF, PC and PD x delay, dt = 1e-3, the noise profile) with a monitor: per
controller and delay, the medians over the cell of RMS position error, mean absolute joint power (WORK_ABS / 6 s) and the peak
torque over the effort limit (SAT_MAX).

The card name and its power limit are printed beside the numbers."""
import argparse
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from bench_loop import DELAYS, NOISE, standing_q0  # noqa: E402
from bench_params import distinct_sets  # noqa: E402
from bench_perturbed import card  # noqa: E402


def cost(rounds):
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import Loop, Monitor, PlantSet, Terrain, TerrainSet, rollout
    from quadruped_drake_b200.urdf import load_description
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(0)
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    plants = PlantSet(ctl, [flatten(d), flatten(with_payload(d, 1.2, (0.04, -0.02, 0.05)))], [1.0, 0.6])
    terrains = TerrainSet(ctl, [Terrain(), Terrain(slope=(np.tan(np.radians(5.0)), 0.0))])
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
        k = 100 if n == 4096 else 20
        q0 = np.tile(q, (n, 1))

        def once(kind, monitor):
            qt, vt, tt = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
            mon = Monitor() if monitor else None
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = rollout(ctl, s, kind, qt, vt, tt, k, 5e-3, plant=True, monitor=mon, **kw)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), float((r.status_or.cpu().numpy() == 0).mean())

        with torch.cuda.stream(torch.cuda.Stream()):
            for kind in ("id", "pc"):
                ms = {False: [], True: []}
                for rnd in range(rounds):
                    for monitor in (False, True):
                        once(kind, monitor)
                        runs = [once(kind, monitor) for _ in range(3)]
                        ms[monitor].append(float(np.mean([x[0] for x in runs])))
                        print("rollout %-2s %6d x %3d  %-15s round %d  %8.2f ms  %.3f ms/step  status 0: %.2f"
                              % (kind, n, k, "monitor" if monitor else "wbc_rollout_loop", rnd, ms[monitor][-1], ms[monitor][-1] / k,
                                 runs[-1][1]), flush=True)
                a, b = np.mean(ms[False]), np.mean(ms[True])
                print("  %-2s %6d: %.3f -> %.3f ms/step, monitor %+.1f %% (%+.1f us per step)"
                      % (kind, n, a / k, b / k, 100.0 * (b / a - 1.0), 1e3 * (b - a) / k), flush=True)
        ps.close()
    s.close(); terrains.close(); plants.close(); ctl.close()


def monitored(ctl, kind, cells, per_cell, dt, rng):
    """6 s of per_cell jittered standing robots per cell (cells[c] = dict(noise, delay, strength, push or None)) with a monitor
    -> (the tools' end-state verdict [n], the rollout result, cell of each robot)."""
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.rollout import Loop, Monitor, rollout
    q = standing_q0(ctl)
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=float(q[6])))
    n = len(cells) * per_cell
    cell = np.repeat(np.arange(len(cells)), per_cell)
    q0 = np.tile(q, (n, 1))
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    pick = lambda key, dtype: np.array([c[key] for c in cells], dtype)[cell]  # noqa: E731
    loop = Loop(noise=T(pick("noise", np.float64)), delay=T(pick("delay", np.int32)), strength=T(pick("strength", np.float64)), seed=11)
    kw = {}
    if any(c.get("push") is not None for c in cells):
        kw["push"] = T(np.array([c.get("push") if c.get("push") is not None else np.zeros(8) for c in cells])[cell])
    qt, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    with torch.cuda.stream(torch.cuda.Stream()):
        r = rollout(ctl, s, kind, qt, v, t, int(round(6.0 / dt)), dt, plant=True, loop=loop, monitor=Monitor(), **kw)
    torch.cuda.synchronize()
    qf, st = qt.cpu().numpy(), r.status_or.cpu().numpy()
    dotq = np.abs((q0[:, 0:4] * qf[:, 0:4]).sum(axis=1)) / np.linalg.norm(qf[:, 0:4], axis=1)
    tilt = 2 * np.arccos(np.clip(dotq, -1, 1))
    up = (st == 0) & (np.linalg.norm(qf[:, 4:7] - q0[:, 4:7], axis=1) < 0.05) & (tilt < 0.3)
    s.close()
    return up, r, cell


def study(per_cell=64):
    from quadruped_drake_b200.controller import BatchedController
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(1)
    print("noise profile (std): orientation %g rad, base position %g m, joints %g rad, angular velocity %g rad/s, linear velocity "
          "%g m/s, joint velocities %g rad/s" % tuple(NOISE))
    impulses, dt = [0.0, 5.0, 10.0, 15.0, 20.0], 5e-3
    cells = [dict(noise=NOISE, delay=d, strength=1.0, push=[j / 0.1, 0, 0, 0, 0, 0.05, 1.0, 1.1]) for j in impulses for d in DELAYS]
    up, r, cell = monitored(ctl, "id", cells, per_cell, dt, rng)
    m = r.monitor
    never = (m.fail_step == 0).cpu().numpy()
    tf = m.fail_time(0.0, dt).cpu().numpy()
    print("ID, push x delay at dt = 5e-3 with the noise profile (rows: push impulse N s over 0.1 s at t = 1 s, columns: delay in "
          "steps; %d robots per cell). Each cell: end-state standing fraction / fraction never failed / median time to failure (s)"
          % per_cell)
    print("%8s " % "" + "".join("%17d" % d for d in DELAYS))
    for i, j in enumerate(impulses):
        line = "%8.1f " % j
        for c in range(i * len(DELAYS), (i + 1) * len(DELAYS)):
            med = np.median(tf[cell == c])
            line += "  %4.2f/%4.2f/%5s" % (up[cell == c].mean(), never[cell == c].mean(), "-" if np.isinf(med) else "%.2f" % med)
        print(line)
    print("robots standing at the end that failed at some step: %d of %d" % (int((up & ~never).sum()), len(up)))
    print("ID, CLF, PC, PD x delay at dt = 1e-3 with the noise profile (%d robots per cell): medians of RMS position error (mm) / "
          "mean |joint power| (W) / peak |tau| / effort" % per_cell)
    print("%8s " % "" + "".join("%20d" % d for d in DELAYS))
    for kind in ("id", "clf", "pc", "pd"):
        up, r, cell = monitored(ctl, kind, [dict(noise=NOISE, delay=d, strength=1.0) for d in DELAYS], per_cell, 1e-3, rng)
        m = r.monitor
        rms, work, sat = (x.cpu().numpy() for x in (m.rms_pos, m.work_abs / 6.0, m.sat_max))
        print("%8s " % kind + "".join("  %5.1f/%6.1f/%5.2f" % (1e3 * np.median(rms[cell == c]), np.median(work[cell == c]),
                                                               np.median(sat[cell == c])) for c in range(len(DELAYS))))
    ctl.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--study", action="store_true", help="also run the push x delay study and the controller x delay statistics")
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
