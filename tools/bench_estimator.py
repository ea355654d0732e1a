#!/usr/bin/env python
"""Cost of the state estimator in the ground-plant loop, and three studies with it.

Cost: the ground-plant rollout of the ID and PC controllers (standing plan, 4096 robots x 100 steps, 65536 x 20) with the full
configuration of tools/bench_motor.py - two plant variants, pushes, two terrains, N distinct parameter sets, distinct loop
profiles, a monitor and 16 distinct motor records - through wbc_rollout_motor, and through wbc_rollout_estimator with one
estimator record and with 16 distinct records spread over the robots (accelerometer noise on). Three rounds alternate the three;
a figure is the mean of 3 timed rollouts after one warm-up (CUDA events).

--study (64 jittered robots per cell, dt = 5e-3 except PD at 1e-3, 6 s, loop noise profile NOISE of tools/bench_loop.py):
  1. observed against estimated base states: ID, CLF, PC and PD standing, and ID trotting to (1.5, 0); "observed" is the loop
     alone (base position and linear velocity read with the profile's noise), "estimated" adds the default filter and an
     accelerometer with 0.1 m/s^2 noise. The trot runs 1.5 s: the straight-line plan is not dynamically consistent, and longer
     trots tip over with either sensing (section 10 of DESIGN.md). Per row: the estimation RMS / max of position and velocity,
     the final |p_est - p| (drift), the monitor's RMS position error, the mean joint power int |tau thetadot| dt / T and the
     never-failed fraction.
  2. push impulse (0-20 N s at t = 1 s over 0.1 s, ID) x sensing: never failed / median time to failure.
  3. incline (0-10 degrees, oracle/terrain.incline along x, ID standing) x sensing: the mean z bias of the estimate at the end,
     never failed.

The card name and its power limit are printed beside the numbers."""
import argparse
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from bench_loop import NOISE, standing_q0  # noqa: E402
from bench_motor import IMPULSES, distinct_motors  # noqa: E402
from bench_params import distinct_sets  # noqa: E402
from bench_perturbed import card  # noqa: E402

ACCEL = 0.1


def distinct_estimators(ctl, k, rng):
    from quadruped_drake_b200.rollout import ESTIMATOR_DEFAULTS, EstimatorSet, estimator_desc
    return EstimatorSet(ctl, [estimator_desc(**{f: x * float(rng.uniform(0.5, 2.0)) for f, x in ESTIMATOR_DEFAULTS.items()
                                                 if f != "swing_scale"}) for _ in range(k)])


def cost(rounds):
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import (Estimator, EstimatorSet, Loop, Monitor, Motor, PlantSet, Terrain, TerrainSet,
                                              estimator_desc, rollout)
    from quadruped_drake_b200.urdf import load_description
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(0)
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    plants = PlantSet(ctl, [flatten(d), flatten(with_payload(d, 1.2, (0.04, -0.02, 0.05)))], [1.0, 0.6])
    terrains = TerrainSet(ctl, [Terrain(), Terrain(slope=(np.tan(np.radians(5.0)), 0.0))])
    motors = distinct_motors(ctl, 16, rng)
    one = EstimatorSet(ctl, [estimator_desc()])
    many = distinct_estimators(ctl, 16, rng)
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
                            strength=T(rng.uniform(0.8, 1.2, n)), stream=T(rng.integers(-2**31, 2**31, n).astype(np.int32)), seed=2026),
                  motor=Motor(motors, T(rng.integers(0, 16, n).astype(np.int32))))
        accel = T(np.full(n, ACCEL))
        modes = {"wbc_rollout_motor": None, "1 record": (one, None), "16 records": (many, T(rng.integers(0, 16, n).astype(np.int32)))}
        k = 100 if n == 4096 else 20
        q0 = np.tile(q, (n, 1))

        def once(kind, mode):
            qt, vt, tt = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
            es = None if modes[mode] is None else Estimator(modes[mode][0], modes[mode][1], accel)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = rollout(ctl, s, kind, qt, vt, tt, k, 5e-3, plant=True, monitor=Monitor(), estimator=es, **kw)
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
                        print("rollout %-2s %6d x %3d  %-17s round %d  %8.2f ms  %.3f ms/step  status 0: %.2f"
                              % (kind, n, k, mode, rnd, ms[mode][-1], ms[mode][-1] / k, runs[-1][1]), flush=True)
                a = np.mean(ms["wbc_rollout_motor"])
                for mode in list(modes)[1:]:
                    b = np.mean(ms[mode])
                    print("  %-2s %6d %-10s: %.3f -> %.3f ms/step, estimator %+.1f %% (%+.1f us per step)"
                          % (kind, n, mode, a / k, b / k, 100.0 * (b / a - 1.0), 1e3 * (b - a) / k), flush=True)
        ps.close()
    many.close(); one.close(); motors.close(); s.close(); terrains.close(); plants.close(); ctl.close()


def run(ctl, kind, n, estimated, rng, plan="standing", seconds=6.0, push=None, incline=None):
    """n jittered robots under the loop's noise profile, with a monitor, optionally the default estimator -> (rollout result,
    final q, the estimator state or None, dt)."""
    import torch
    from oracle.terrain import incline as incline_terrain
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.rollout import Estimator, EstimatorSet, EstimatorState, Loop, Monitor, TerrainSet, estimator_desc, rollout
    dt = 1e-3 if kind == "pd" else 5e-3
    q = standing_q0(ctl)
    if plan == "standing":
        s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", seconds, base_height=float(q[6])))
    else:
        s = pl.TrajectorySampler(ctl, pl.make_gait_plan("mini_cheetah", "trot", goal=(1.5, 0.0), base_height=float(q[6])))
    q0 = np.tile(q, (n, 1))
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    kw = dict(loop=Loop(noise=NOISE, stream=T(np.arange(n, dtype=np.int32)), seed=11), monitor=Monitor())
    if push is not None:
        kw["push"] = T(np.tile([push / 0.1, 0, 0, 0, 0, 0.05, 1.0, 1.1], (n, 1)))
    ts = es = None
    if incline is not None:
        ts = TerrainSet(ctl, [incline_terrain(incline)])
        kw["terrain_set"] = ts
    if estimated:
        es = EstimatorSet(ctl, [estimator_desc()])
        kw["estimator"] = Estimator(es, accel_noise=T(np.full(n, ACCEL)), state=EstimatorState(n, like=T(q0)))
    qt, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    with torch.cuda.stream(torch.cuda.Stream()):
        r = rollout(ctl, s, kind, qt, v, t, int(round(seconds / dt)), dt, plant=True, **kw)
    torch.cuda.synchronize()
    for x in (es, ts, s):
        if x is not None:
            x.close()
    return r, qt.cpu().numpy(), r.estimator, dt, seconds


def row(name, r, qf, est, seconds):
    m = r.monitor
    never = (m.fail_step == 0).cpu().numpy().mean()
    rms_pos = np.median(m.rms_pos.cpu().numpy())
    power = np.median(m.work_abs.cpu().numpy()) / seconds
    if est is None:
        e = "%31s" % "-"
    else:
        x, cnt, st = est.x.cpu().numpy(), est.count.cpu().numpy(), est.stats.cpu().numpy()
        good = cnt > 0
        rp, mp = np.sqrt(np.median(st[:, 0] / np.maximum(cnt, 1))), np.median(st[:, 1])
        rv, mv = np.sqrt(np.median(st[:, 2] / np.maximum(cnt, 1))), np.median(st[:, 3])
        drift = np.median(np.linalg.norm(x[good, 0:3] - qf[good, 4:7], axis=1)) if good.any() else np.nan
        e = "%5.1f/%5.1f mm %5.1f/%5.1f cm/s %5.1f mm" % (1e3 * rp, 1e3 * mp, 1e2 * rv, 1e2 * mv, 1e3 * drift)
    print("  %-30s %s   %6.1f mm  %6.1f W  %4.2f" % (name, e, 1e3 * rms_pos, power, never), flush=True)


def study(n=64):
    from quadruped_drake_b200.controller import BatchedController
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(1)
    print("loop noise profile (std): orientation %g rad, base position %g m, joints %g rad, angular velocity %g rad/s, linear "
          "velocity %g m/s, joint velocities %g rad/s; no delay; estimated rows add the default filter and %g m/s^2 accelerometer "
          "noise" % (tuple(NOISE) + (ACCEL,)))
    print("1. observed vs estimated base states, %d robots, 6 s (medians over robots). Columns: estimation RMS/max position, "
          "RMS/max velocity, final |p_est - p|; monitor RMS position error; joint power; never failed" % n)
    for kind, plan, sec in (("id", "standing", 6.0), ("clf", "standing", 6.0), ("pc", "standing", 6.0), ("pd", "standing", 6.0),
                            ("id", "trot", 1.5)):
        for estimated in (False, True):
            r, qf, est, dt, sec = run(ctl, kind, n, estimated, rng, plan, seconds=sec)
            row("%s %s %.1f s %s" % (kind, plan, sec, "estimated" if estimated else "observed"), r, qf, est, sec)
    print("2. ID standing, push impulse (N s over 0.1 s at t = 1 s) x sensing: never failed / median time to failure (s)")
    print("%8s %16s %16s" % ("", "observed", "estimated"))
    for j in IMPULSES:
        cells = []
        for estimated in (False, True):
            r, qf, est, dt, sec = run(ctl, "id", n, estimated, rng, push=j)
            med = np.median(r.monitor.fail_time(0.0, dt).cpu().numpy())
            cells.append("%10.2f/%5s" % ((r.monitor.fail_step == 0).cpu().numpy().mean(), "-" if np.isinf(med) else "%.2f" % med))
        print("%8.1f " % j + " ".join(cells), flush=True)
    print("3. ID standing on an incline (degrees, rising along x) x sensing: estimated z bias at the end (mean p_est,z - p_z) / "
          "never failed (observed, estimated)")
    for deg in (0.0, 2.0, 5.0, 10.0):
        r0, _, _, _, _ = run(ctl, "id", n, False, rng, incline=deg)
        r1, qf, est, _, _ = run(ctl, "id", n, True, rng, incline=deg)
        x, cnt = est.x.cpu().numpy(), est.count.cpu().numpy()
        bias = np.mean((x[:, 2] - qf[:, 6])[cnt > 0]) if (cnt > 0).any() else np.nan
        print("%8.1f  z bias %+7.1f mm   never failed %4.2f %4.2f" % (deg, 1e3 * bias, (r0.monitor.fail_step == 0).cpu().numpy().mean(),
                                                                     (r1.monitor.fail_step == 0).cpu().numpy().mean()), flush=True)
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
