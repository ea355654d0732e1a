#!/usr/bin/env python
"""Cost of the contact detector in the ground-plant loop, and three studies with it.

Cost: the ground-plant rollout of the ID controller (standing plan, 4096 robots x 100 steps, 65536 x 20) with the configuration
of tools/bench_estimator.py - two plant variants, pushes, two terrains, N distinct parameter sets, distinct loop profiles, a
monitor, 16 distinct motor records and the default estimator - through wbc_rollout_estimator, and through wbc_rollout_contact
with the default detector (feed = 0 and feed = estimator + controller). Rounds alternate the three; a figure is the mean of 3
timed rollouts after one warm-up (CUDA events). Robot-steps/s are N x steps / time.

--study (64 jittered robots per cell, dt = 5e-3 except PD at 1e-3, loop noise profile NOISE of tools/bench_loop.py):
  1. per controller (ID, CLF, PC, PD) on the standing and raise_foot plans, 4 s, feed = 0: the force-estimate RMS / max error
     against the plant's forces and the per-foot-step confusion counts (true stance, true swing, false stance, false swing), as
     fractions of all foot-steps.
  2. sensing-noise scale (0, 0.5, 1, 2 x NOISE) x tau_f (0, 10 ms, 50 ms), ID standing 2 s: force RMS and the false fractions.
  3. feed = 0 / estimator / estimator + controller, ID standing with the default estimator, on an incline (0, 5, 10 degrees) and
     under a push impulse (0, 10, 20 N s at t = 1 s): the estimator's RMS position / velocity error, the z bias of its estimate at
     the end, and the monitor's never-failed fraction.

No figure has a pass threshold. The card name and its power limit are printed beside the numbers."""
import argparse
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from bench_loop import NOISE, standing_q0  # noqa: E402
from bench_motor import distinct_motors  # noqa: E402
from bench_params import distinct_sets  # noqa: E402
from bench_perturbed import card  # noqa: E402


def cost(rounds):
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.capi import CONTACT_FEED_CONTROLLER, CONTACT_FEED_ESTIMATOR
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import (ContactDetector, ContactSet, Estimator, EstimatorSet, Loop, Monitor, Motor, PlantSet,
                                              Terrain, TerrainSet, contact_desc, estimator_desc, rollout)
    from quadruped_drake_b200.urdf import load_description
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(0)
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    plants = PlantSet(ctl, [flatten(d), flatten(with_payload(d, 1.2, (0.04, -0.02, 0.05)))], [1.0, 0.6])
    terrains = TerrainSet(ctl, [Terrain(), Terrain(slope=(np.tan(np.radians(5.0)), 0.0))])
    motors = distinct_motors(ctl, 16, rng)
    es, cs = EstimatorSet(ctl, [estimator_desc()]), ContactSet(ctl, [contact_desc()])
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
        modes = {"wbc_rollout_estimator": None, "detector feed 0": 0,
                 "detector feed est+ctrl": CONTACT_FEED_ESTIMATOR | CONTACT_FEED_CONTROLLER}
        k = 100 if n == 4096 else 20
        q0 = np.tile(q, (n, 1))

        def once(mode):
            qt, vt, tt = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
            det = None if modes[mode] is None else ContactDetector(cs, feed=modes[mode])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = rollout(ctl, s, "id", qt, vt, tt, k, 5e-3, plant=True, monitor=Monitor(), estimator=Estimator(es), contact=det, **kw)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), float((r.status_or.cpu().numpy() == 0).mean())

        with torch.cuda.stream(torch.cuda.Stream()):
            ms = {m: [] for m in modes}
            for rnd in range(rounds):
                for mode in modes:
                    once(mode)
                    runs = [once(mode) for _ in range(3)]
                    ms[mode].append(float(np.mean([x[0] for x in runs])))
                    print("rollout id %6d x %3d  %-23s round %d  %8.2f ms  %.3f ms/step  %.2f M robot-steps/s  status 0: %.2f"
                          % (n, k, mode, rnd, ms[mode][-1], ms[mode][-1] / k, n * k / ms[mode][-1] / 1e3, runs[-1][1]), flush=True)
            a = np.mean(ms["wbc_rollout_estimator"])
            for mode in list(modes)[1:]:
                b = np.mean(ms[mode])
                print("  id %6d %-23s: %.3f -> %.3f ms/step, %.2f -> %.2f M robot-steps/s, detector %+.1f %% (%+.1f us per step)"
                      % (n, mode, a / k, b / k, n * k / a / 1e3, n * k / b / 1e3, 100.0 * (b / a - 1.0), 1e3 * (b - a) / k), flush=True)
        ps.close()
    cs.close(); es.close(); motors.close(); s.close(); terrains.close(); plants.close(); ctl.close()


def run(ctl, kind, n, rng, plan="standing", seconds=4.0, noise=1.0, tau_f=None, feed=0, estimated=False, push=None, incline=None):
    """n jittered robots under `noise` x the loop's noise profile, with a monitor and the default detector (tau_f replaced when
    given), optionally the default estimator -> (result, final q, dt)."""
    import torch
    from oracle.terrain import incline as incline_terrain
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.rollout import (ContactDetector, ContactSet, ContactState, Estimator, EstimatorSet, EstimatorState, Loop,
                                              Monitor, TerrainSet, contact_desc, estimator_desc, rollout)
    dt = 1e-3 if kind == "pd" else 5e-3
    q = standing_q0(ctl)
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", plan, 6.0, base_height=float(q[6])))
    q0 = np.tile(q, (n, 1))
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    cs = ContactSet(ctl, [contact_desc() if tau_f is None else contact_desc(tau_f=tau_f)])
    kw = dict(loop=Loop(noise=NOISE * noise, stream=T(np.arange(n, dtype=np.int32)), seed=11), monitor=Monitor(),
              contact=ContactDetector(cs, feed=feed, state=ContactState(n, like=T(q0))))
    if push is not None:
        kw["push"] = T(np.tile([push / 0.1, 0, 0, 0, 0, 0.05, 1.0, 1.1], (n, 1)))
    ts = es = None
    if incline is not None:
        ts = TerrainSet(ctl, [incline_terrain(incline)])
        kw["terrain_set"] = ts
    if estimated:
        es = EstimatorSet(ctl, [estimator_desc()])
        kw["estimator"] = Estimator(es, state=EstimatorState(n, like=T(q0)))
    qt, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    with torch.cuda.stream(torch.cuda.Stream()):
        r = rollout(ctl, s, kind, qt, v, t, int(round(seconds / dt)), dt, plant=True, **kw)
    torch.cuda.synchronize()
    for x in (es, ts, cs, s):
        if x is not None:
            x.close()
    return r, qt.cpu().numpy(), dt


def force_row(name, r):
    st = r.contact.stats.cpu().numpy()
    steps = st[:, 2:6].sum()
    rms = np.sqrt(st[:, 0].sum() / max(steps, 1))
    frac = st[:, 2:6].sum(axis=0) / max(steps, 1)
    print("  %-28s force RMS %7.2f N  max %7.1f N   TS %.3f  TW %.3f  FS %.4f  FW %.4f   never failed %.2f"
          % (name, rms, st[:, 1].max(), *frac, (r.monitor.fail_step == 0).cpu().numpy().mean()), flush=True)


def study(n=64):
    from quadruped_drake_b200.capi import CONTACT_FEED_CONTROLLER, CONTACT_FEED_ESTIMATOR
    from quadruped_drake_b200.controller import BatchedController
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(1)
    print("loop noise profile (std): orientation %g rad, base position %g m, joints %g rad, angular velocity %g rad/s, linear "
          "velocity %g m/s, joint velocities %g rad/s; no delay; default detector (untuned)" % tuple(NOISE))
    print("1. per controller and plan, %d robots, 4 s, feed = 0: force-estimate error and the confusion fractions of all foot-steps "
          "(TS true stance, TW true swing, FS false stance, FW false swing)" % n)
    for kind in ("id", "clf", "pc", "pd"):
        for plan in ("standing", "raise_foot"):
            r, _, _ = run(ctl, kind, n, rng, plan)
            force_row("%s %s" % (kind, plan), r)
    print("2. ID standing 2 s: sensing-noise scale x tau_f")
    for scale in (0.0, 0.5, 1.0, 2.0):
        for tau_f in (0.0, 0.01, 0.05):
            r, _, _ = run(ctl, "id", n, rng, seconds=2.0, noise=scale, tau_f=tau_f)
            force_row("noise x%.1f tau_f %2.0f ms" % (scale, 1e3 * tau_f), r)
    print("3. ID standing with the default estimator, feed = 0 / estimator / estimator + controller. Columns: estimator RMS "
          "position / velocity error, z bias of the estimate at the end (mean p_est,z - p_z), never failed")
    feeds = (("feed 0", 0), ("feed est", CONTACT_FEED_ESTIMATOR), ("feed est+ctrl", CONTACT_FEED_ESTIMATOR | CONTACT_FEED_CONTROLLER))
    cases = [("incline %2.0f deg" % d, dict(incline=d)) for d in (0.0, 5.0, 10.0)] + \
        [("push %2.0f N s" % j, dict(push=j)) for j in (10.0, 20.0)]
    for cname, extra in cases:
        for fname, feed in feeds:
            r, qf, _ = run(ctl, "id", n, rng, feed=feed, estimated=True, **extra)
            e = r.estimator
            x, cnt, st = e.x.cpu().numpy(), e.count.cpu().numpy(), e.stats.cpu().numpy()
            good = cnt > 0
            rp = np.sqrt(np.median(st[:, 0] / np.maximum(cnt, 1)))
            rv = np.sqrt(np.median(st[:, 2] / np.maximum(cnt, 1)))
            bias = np.mean((x[:, 2] - qf[:, 6])[good]) if good.any() else np.nan
            print("  %-16s %-14s  %6.1f mm  %6.1f cm/s  z bias %+7.1f mm   never failed %.2f"
                  % (cname, fname, 1e3 * rp, 1e2 * rv, 1e3 * bias, (r.monitor.fail_step == 0).cpu().numpy().mean()), flush=True)
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
