#!/usr/bin/env python
"""Cost of imperfect sensing and actuation in the ground-plant loop, and three robustness studies it makes possible.

Cost: the ground-plant rollout of the ID and PC controllers (standing plan, 4096 robots x 100 steps, 65536 x 20) with every
per-robot feature on - two plant variants, pushes, two terrains and N distinct parameter sets - through wbc_rollout_params
against wbc_rollout_loop, once with a zero profile for every robot (the same controller work plus the two loop kernels) and
once with distinct profiles (noise 0.5-2 x NOISE, delay 0-2, strength 0.8-1.2, its own stream; the robots keep standing, but
the controller now works on noisy states). Three rounds alternate the three; a figure is the mean of 3 timed rollouts after
one warm-up (CUDA events). The two loop kernels alone are timed through wbc_loop_observe and a rollout difference.

--study: 6 s of standing robots on the ground plant, 64 per cell with jittered joints; prints the fraction of each cell still
standing at the end, by the criterion of tools/bench_terrain.py (no status bit, base within 5 cm of its start, tilt below
0.3 rad). The noise profile NOISE below is the "moderate" one. Each table is one rollout of all its cells.
  1. ID, CLF, PC and PD x a command delay of 0, 1, 2, 4, 8 and 15 steps, at dt = 1e-3 with NOISE;
  2. ID at dt = 5e-3: a horizontal push impulse at t = 1 s over 0.1 s (the push of tools/bench_perturbed.py) x the delay,
     with NOISE;
  3. ID at dt = 5e-3, no delay: the noise scale (0 - 8 x NOISE) x the motor strength (0.6 - 1.2).

The card name and its power limit are printed beside the numbers."""
import argparse
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from bench_params import distinct_sets  # noqa: E402
from bench_perturbed import card  # noqa: E402

# standard deviations: orientation 0.01 rad, base position 2 mm, joints 0.01 rad, angular velocity 0.05 rad/s, linear velocity
# 0.02 m/s, joint velocities 0.1 rad/s
NOISE = np.array([0.01, 0.002, 0.01, 0.05, 0.02, 0.1])
DELAYS = [0, 1, 2, 4, 8, 15]


def standing_q0(ctl):
    from quadruped_drake_b200.rollout import Q0_MINI_CHEETAH as Q0
    q = Q0.copy()
    q[6] -= ctl.dynamics(q[None], np.zeros((1, 18)))["p_feet"][0, :, 2].min()
    return q


def cost(rounds):
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import Loop, PlantSet, Terrain, TerrainSet, observe, rollout
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
                  variant=T((np.arange(n) % 2).astype(np.int32)), push=T(push), terrain=T((np.arange(n) // 2 % 2).astype(np.int32)))
        loops = {"wbc_rollout_params": None,
                 "loop, zero profile": Loop(noise=T(np.zeros((n, 6))), delay=T(np.zeros(n, np.int32)), strength=T(np.ones(n)), seed=2026),
                 "loop, distinct": Loop(noise=T(NOISE * rng.uniform(0.5, 2.0, (n, 1))), delay=T(rng.integers(0, 3, n).astype(np.int32)),
                                        strength=T(rng.uniform(0.8, 1.2, n)), stream=T(rng.integers(-2**31, 2**31, n).astype(np.int32)),
                                        seed=2026)}
        k = 100 if n == 4096 else 20
        q0 = np.tile(q, (n, 1))

        def once(kind, loop):
            qt, vt, tt = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = rollout(ctl, s, kind, qt, vt, tt, k, 5e-3, plant=True, loop=loop, **kw)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), float((r.status_or.cpu().numpy() == 0).mean())

        with torch.cuda.stream(torch.cuda.Stream()):
            for kind in ("id", "pc"):
                for rnd in range(rounds):
                    for name, loop in loops.items():
                        once(kind, loop)
                        runs = [once(kind, loop) for _ in range(3)]
                        ms = float(np.mean([x[0] for x in runs]))
                        print("rollout %-2s %6d x %3d  %-18s round %d  %8.2f ms  %.3f ms/step  status 0: %.2f"
                              % (kind, n, k, name, rnd, ms, ms / k, runs[-1][1]), flush=True)
            # the observe kernel alone, on the distinct profiles
            lp = loops["loop, distinct"]
            qt, vt = torch.from_numpy(q0).cuda(), torch.zeros((n, 18), dtype=torch.float64, device="cuda")
            for _ in range(5):
                observe(ctl, qt, vt, lp)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(200):
                observe(ctl, qt, vt, lp)
            e1.record()
            torch.cuda.synchronize()
            print("observe kernel %6d  %.1f us per launch (incl. the Python call)" % (n, e0.elapsed_time(e1) / 200 * 1e3), flush=True)
        ps.close()
    s.close(); terrains.close(); plants.close(); ctl.close()


def standing(ctl, kind, cells, per_cell, dt, rng):
    """Fraction of per_cell robots of each cell standing after 6 s; cells[c] = dict(noise (6,), delay, strength, push (8,) or
    None)."""
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.rollout import Loop, rollout
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
        r = rollout(ctl, s, kind, qt, v, t, int(round(6.0 / dt)), dt, plant=True, loop=loop, **kw)
    torch.cuda.synchronize()
    qf, st = qt.cpu().numpy(), r.status_or.cpu().numpy()
    dotq = np.abs((q0[:, 0:4] * qf[:, 0:4]).sum(axis=1)) / np.linalg.norm(qf[:, 0:4], axis=1)
    tilt = 2 * np.arccos(np.clip(dotq, -1, 1))
    up = (st == 0) & (np.linalg.norm(qf[:, 4:7] - q0[:, 4:7], axis=1) < 0.05) & (tilt < 0.3)
    s.close()
    return np.array([up[cell == c].mean() for c in range(len(cells))])


def table(title, rows, row_fmt, cols, col_fmt, up):
    print(title)
    print("%8s " % "" + "".join(col_fmt % c for c in cols))
    for i, r in enumerate(rows):
        print(row_fmt % r + "".join("%7.2f" % x for x in up[i]))


def study(per_cell=64):
    from quadruped_drake_b200.controller import BatchedController
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(1)
    print("noise profile (std): orientation %g rad, base position %g m, joints %g rad, angular velocity %g rad/s, linear velocity "
          "%g m/s, joint velocities %g rad/s" % tuple(NOISE))
    kinds = ["id", "clf", "pc", "pd"]
    up = np.array([standing(ctl, k, [dict(noise=NOISE, delay=d, strength=1.0) for d in DELAYS], per_cell, 1e-3, rng) for k in kinds])
    table("1. fraction standing after 6 s at dt = 1e-3 with the noise profile (rows: controller, columns: delay in steps; %d robots "
          "per cell)" % per_cell, kinds, "%8s ", DELAYS, "%7d", up)
    impulses = [0.0, 5.0, 10.0, 15.0, 20.0]
    cells = [dict(noise=NOISE, delay=d, strength=1.0, push=[j / 0.1, 0, 0, 0, 0, 0.05, 1.0, 1.1]) for j in impulses for d in DELAYS]
    up = standing(ctl, "id", cells, per_cell, 5e-3, rng).reshape(len(impulses), len(DELAYS))
    table("2. ID: fraction standing after 6 s at dt = 5e-3 with the noise profile (rows: push impulse N s over 0.1 s at t = 1 s, "
          "columns: delay in steps; %d robots per cell)" % per_cell, impulses, "%8.1f ", DELAYS, "%7d", up)
    scales, strengths = [0.0, 1.0, 2.0, 4.0, 8.0], [0.6, 0.7, 0.8, 0.9, 1.0, 1.1, 1.2]
    cells = [dict(noise=NOISE * sc, delay=0, strength=st) for sc in scales for st in strengths]
    up = standing(ctl, "id", cells, per_cell, 5e-3, rng).reshape(len(scales), len(strengths))
    table("3. ID: fraction standing after 6 s at dt = 5e-3, no delay (rows: noise scale x the profile, columns: motor strength; "
          "%d robots per cell)" % per_cell, scales, "%8.1f ", strengths, "%7.2f", up)
    ctl.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--study", action="store_true", help="also run the three robustness studies")
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
