#!/usr/bin/env python
"""Cost of uneven ground in the ground-plant rollout, and which inclines and steps knock standing robots over.

Throughput: the closed-loop rollout of tools/bench_perturbed.py (reference test motions, ID controller, ground plant, CUDA-graph
replay, N distinct variants, every robot pushed for the whole run) at 4096 robots x 100 steps and 65536 robots x 20 steps,
three rounds that alternate wbc_rollout_perturbed with wbc_rollout_terrain, where in addition every robot stands on its own
terrain: a gentle plane plus a 16 x 16 height field (1.5 cm bumps, 10 cm spacing). Each run is the mean of 5 timed rollouts
after 2 warm-up rollouts.

--grid: 6 s of standing robots, 64 per cell with jittered joints, the base level and every foot placed on the terrain; prints
the fraction of each cell still standing at the end (no status bit, base within 5 cm of its start position, tilt against its
start orientation below 0.3 rad). The controllers assume flat ground: their friction pyramid is about world z (mu = 0.7) and
their feet come from a flat-ground plan.
  1. controller (ID, CLF, PC, PD; dt = 1e-3) x incline along x of 0 - 25 degrees, ground friction 1.0;
  2. ID x height of a step under the two left feet (0 - 6 cm, a 1 cm ramp) x ground friction 0.5 / 1.0.

The card name and its power limit are printed beside the numbers."""
import argparse
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from bench_perturbed import card, variant_set  # noqa: E402


def terrain_set(ctl, n, rng):
    """n distinct terrains: slope up to 3 degrees in a random direction, 16 x 16 grid of +-1.5 cm bumps at 10 cm around the origin."""
    from quadruped_drake_b200.rollout import Terrain, TerrainSet
    ts = []
    for _ in range(n):
        s = np.tan(np.radians(rng.uniform(0, 3))) * np.array([np.cos(a := rng.uniform(0, 2 * np.pi)), np.sin(a)])
        ts.append(Terrain(slope=tuple(s), origin=(-0.75, -0.75), spacing=(0.1, 0.1), heights=rng.uniform(-0.015, 0.015, (16, 16))))
    return TerrainSet(ctl, ts)


def throughput(rounds):
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.rollout import Q0_MINI_CHEETAH as Q0, rollout
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(0)
    bh = Q0[6] - ctl.dynamics(Q0[None], np.zeros((1, 18)))["p_feet"][0, :, 2].mean()
    plans = [pl.make_motion_plan("mini_cheetah", m, 6.0, base_height=bh, phase=ph) for m in ("orientation", "heave", "raise_foot")
             for ph in np.linspace(0, 2 * np.pi, 8, endpoint=False)]
    s = pl.TrajectorySampler(ctl, plans)
    for nr, k in ((4096, 100), (65536, 20)):
        q0 = np.tile(Q0, (nr, 1)); q0[:, 6] = bh
        pi = torch.from_numpy(rng.integers(0, len(plans), nr).astype(np.int32)).cuda()
        ps = variant_set(ctl, nr, rng)
        ts = terrain_set(ctl, nr, rng)
        idx = torch.arange(nr, dtype=torch.int32, device="cuda")
        push = np.zeros((nr, 8))
        push[:, 0:3] = rng.uniform(-5, 5, (nr, 3)); push[:, 3:6] = rng.uniform(-0.1, 0.1, (nr, 3)); push[:, 6:8] = [-1.0, 100.0]
        push = torch.from_numpy(push).cuda()
        base = dict(plant_set=ps, variant=idx, push=push)
        kw = {False: base, True: dict(base, terrain_set=ts, terrain=idx)}

        def once(terrain):
            q, v, t = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((nr, 18)), np.zeros(nr)))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = rollout(ctl, s, "id", q, v, t, k, 5e-3, plan_index=pi, plant=True, **kw[terrain])
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), int((r.status_or != 0).sum().item())

        with torch.cuda.stream(torch.cuda.Stream()):
            for rnd in range(rounds):
                for terrain in (False, True):
                    for _ in range(2):
                        once(terrain)
                    runs = [once(terrain) for _ in range(5)]
                    ms = float(np.mean([r[0] for r in runs]))
                    print("%6d robots x %3d steps  %-9s  round %d  %.2f M robot-steps/s  (robots with a status bit: %d)"
                          % (nr, k, "terrain" if terrain else "perturbed", rnd, nr * k / (ms * 1e-3) / 1e6, runs[-1][1]), flush=True)
        ts.close(); ps.close()
    s.close(); ctl.close()


def placed(ctl, P, q, tr):
    """q with every foot moved (Newton on the foot Jacobians of oracle.dynamics, base fixed) onto terrain tr, keeping its x, y."""
    from oracle import terrain as otr
    from oracle.terrain import Terrain
    ot = Terrain(z0=tr.z0, slope=tuple(tr.slope), origin=tuple(tr.origin), spacing=tuple(tr.spacing), heights=tr.heights)
    q = q.copy()
    for _ in range(8):
        quant = [P.frame_position_quantities(q, np.zeros(18), fr) for fr in P.foot_frames]
        p = np.array([x[0] for x in quant])
        target = p.copy()
        target[:, 2] = [otr.height(ot, x, y) for x, y, _ in p]
        q[7:] += np.linalg.lstsq(np.vstack([x[1][:, 6:] for x in quant]), (target - p).reshape(-1), rcond=None)[0]
    return q


def standing_fraction(ctl, kind, terrains, mu, per_cell, dt, rng):
    """Fraction of per_cell robots per terrain still standing after 6 s."""
    import torch
    from oracle.dynamics import Plant
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.model import ROBOT_DIR
    from quadruped_drake_b200.rollout import Q0_MINI_CHEETAH as Q0, TerrainSet, rollout
    from quadruped_drake_b200.urdf import load_description
    P = Plant(load_description(ROBOT_DIR / "mini_cheetah.json"))
    q = Q0.copy()
    q[6] -= ctl.dynamics(q[None], np.zeros((1, 18)))["p_feet"][0, :, 2].min()
    bh = float(q[6])
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh))
    n = len(terrains) * per_cell
    q0 = np.repeat(np.array([placed(ctl, P, q, tr) for tr in terrains]), per_cell, axis=0)
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    ts = TerrainSet(ctl, terrains)
    index = np.repeat(np.arange(len(terrains)), per_cell).astype(np.int32)
    qt, v, t = (torch.from_numpy(x).cuda() for x in (q0.copy(), np.zeros((n, 18)), np.zeros(n)))
    with torch.cuda.stream(torch.cuda.Stream()):
        r = rollout(ctl, s, kind, qt, v, t, int(round(6.0 / dt)), dt, plant=True, mu=mu, terrain_set=ts, terrain=torch.from_numpy(index).cuda())
    torch.cuda.synchronize()
    qf, st = qt.cpu().numpy(), r.status_or.cpu().numpy()
    # tilt against the start orientation: angle of q0^-1 q
    dotq = np.abs((q0[:, 0:4] * qf[:, 0:4]).sum(axis=1)) / np.linalg.norm(qf[:, 0:4], axis=1)
    tilt = 2 * np.arccos(np.clip(dotq, -1, 1))
    up = (st == 0) & (np.linalg.norm(qf[:, 4:7] - q0[:, 4:7], axis=1) < 0.05) & (tilt < 0.3)
    ts.close(); s.close()
    return [float(up[index == i].mean()) for i in range(len(terrains))]


def grid(per_cell=64):
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.rollout import Terrain
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(1)
    degs = [0, 5, 10, 15, 20, 25]
    inclines = [Terrain(slope=(np.tan(np.radians(d)), 0.0)) for d in degs]
    print("fraction standing after 6 s on an incline along x (ground friction 1.0, dt = 1e-3, %d robots per cell)" % per_cell)
    print("controller \\ incline deg " + "".join("%7d" % d for d in degs))
    for kind in ("id", "clf", "pc", "pd"):
        fr = standing_fraction(ctl, kind, inclines, 1.0, per_cell, 1e-3, rng)
        print("%25s " % kind.upper() + "".join("%7.2f" % x for x in fr), flush=True)
    heights = [0.0, 0.01, 0.02, 0.03, 0.04, 0.05, 0.06]
    y = -0.3 + 0.01 * np.arange(61)
    steps = [Terrain(origin=(-1.0, -0.3), spacing=(2.0, 0.01), heights=np.tile(np.where(y >= 0.01 - 1e-12, h, 0.0)[:, None], (1, 2)))
             for h in heights]
    print("fraction of ID robots standing after 6 s with a step under the two left feet (dt = 5e-3, %d robots per cell)" % per_cell)
    print("friction \\ step cm " + "".join("%7d" % round(100 * h) for h in heights))
    for mu in (0.5, 1.0):
        fr = standing_fraction(ctl, "id", steps, mu, per_cell, 5e-3, rng)
        print("%18.1f " % mu + "".join("%7.2f" % x for x in fr), flush=True)
    ctl.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--grid", action="store_true", help="also run the incline and step tables")
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    print(card(), flush=True)
    throughput(a.rounds)
    if a.grid:
        grid()
