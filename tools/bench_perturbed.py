#!/usr/bin/env python
"""Cost of perturbed robots in the ground-plant rollout, and how many standing robots a payload and a push knock over.

Throughput: the closed-loop rollout of tools/bench_aux.py (reference test motions, ID controller, ground plant, CUDA-graph
replay) at 4096 robots x 100 steps and 65536 robots x 20 steps, three rounds that alternate an unperturbed run (wbc_rollout_ex)
with a perturbed one (wbc_rollout_perturbed: K = N distinct variants - its own base mass and inertia and its own friction
- and every robot pushed for the whole run). Each run is the mean of 5 timed rollouts after 2 warm-up rollouts.

--grid: 1200 steps (6 s) of standing ID robots over a grid of payload mass x horizontal push impulse (the push lasts 0.1 s and
starts at t = 1 s), 64 robots per cell with jittered joints; prints the fraction of each cell that is still standing at the end
(no status bit, base within 5 cm of the standing height, tilt below 0.3 rad).

The card name and its power limit are printed beside the numbers."""
import argparse
import subprocess
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        limit = "unknown"
    return f"{name}, power limit {limit or 'unknown'}"


def variant_set(ctl, n, rng):
    """n distinct variants of the handle's robot: base mass and inertia scaled by 1.00 - 1.15 (up to 0.5 kg of load spread over
    the base), friction 0.6 - 1.0."""
    from quadruped_drake_b200.model import WbcModelStruct
    from quadruped_drake_b200.rollout import PlantSet
    nominal = ctl.model.as_struct()
    models = []
    for k in range(n):
        m = WbcModelStruct.from_buffer_copy(nominal)
        sc = 1.0 + 0.15 * k / max(n - 1, 1)
        m.mass[0] *= sc
        for a in range(6):
            m.inertia_com[0][a] *= sc
        models.append(m)
    return PlantSet(ctl, models, rng.uniform(0.6, 1.0, n))


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
        variant = torch.arange(nr, dtype=torch.int32, device="cuda")
        push = np.zeros((nr, 8))
        push[:, 0:3] = rng.uniform(-5, 5, (nr, 3)); push[:, 3:6] = rng.uniform(-0.1, 0.1, (nr, 3)); push[:, 6:8] = [-1.0, 100.0]
        push = torch.from_numpy(push).cuda()
        kw = {False: {}, True: dict(plant_set=ps, variant=variant, push=push)}

        def once(perturbed):
            q, v, t = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((nr, 18)), np.zeros(nr)))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = rollout(ctl, s, "id", q, v, t, k, 5e-3, plan_index=pi, plant=True, **kw[perturbed])
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), int((r.status_or != 0).sum().item())

        with torch.cuda.stream(torch.cuda.Stream()):
            for rnd in range(rounds):
                for perturbed in (False, True):
                    for _ in range(2):
                        once(perturbed)
                    runs = [once(perturbed) for _ in range(5)]
                    ms = float(np.mean([r[0] for r in runs]))
                    print("%6d robots x %3d steps  %-11s  round %d  %.2f M robot-steps/s  (robots with a status bit: %d)"
                          % (nr, k, "perturbed" if perturbed else "unperturbed", rnd, nr * k / (ms * 1e-3) / 1e6, runs[-1][1]), flush=True)
        ps.close()
    s.close(); ctl.close()


def grid(per_cell=64):
    import torch
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.model import ROBOT_DIR, flatten, with_payload
    from quadruped_drake_b200.rollout import Q0_MINI_CHEETAH as Q0, PlantSet, rollout
    from quadruped_drake_b200.urdf import load_description
    ctl = BatchedController("mini_cheetah", device=0)
    rng = np.random.default_rng(1)
    masses, impulses = [0.0, 0.5, 1.0, 1.5, 2.0, 3.0], [0.0, 2.0, 4.0, 6.0, 8.0, 10.0]
    d = load_description(ROBOT_DIR / "mini_cheetah.json")
    ps = PlantSet(ctl, [flatten(d)] + [flatten(with_payload(d, m, (0.0, 0.0, 0.05))) for m in masses[1:]])
    cells = [(i, j) for i in range(len(masses)) for j in range(len(impulses))]
    n = len(cells) * per_cell
    q0 = np.tile(Q0, (n, 1)); q0[:, 7:] += rng.uniform(-0.02, 0.02, (n, 12))
    q0[:, 6] -= ctl.dynamics(q0, np.zeros((n, 18)))["p_feet"][:, :, 2].min(axis=1)
    bh = float(np.median(q0[:, 6]))
    s = pl.TrajectorySampler(ctl, pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh))
    variant = np.repeat([i for i, _ in cells], per_cell).astype(np.int32)
    push = np.zeros((n, 8))
    push[:, 0] = np.repeat([impulses[j] / 0.1 for _, j in cells], per_cell)
    push[:, 5] = 0.05                                   # at the payload's height above the base origin
    push[:, 6:8] = [1.0, 1.1]
    q, v, t = (torch.from_numpy(x).cuda() for x in (q0, np.zeros((n, 18)), np.zeros(n)))
    with torch.cuda.stream(torch.cuda.Stream()):
        r = rollout(ctl, s, "id", q, v, t, 1200, 5e-3, plant=True, plant_set=ps, variant=torch.from_numpy(variant).cuda(),
                    push=torch.from_numpy(push).cuda())
    torch.cuda.synchronize()
    qf, st = q.cpu().numpy(), r.status_or.cpu().numpy()
    x, y = qf[:, 1], qf[:, 2]
    tilt = np.arccos(np.clip(1 - 2 * (x * x + y * y), -1, 1))
    up = (st == 0) & (np.abs(qf[:, 6] - bh) < 0.05) & (tilt < 0.3)
    print("fraction standing after 6 s (rows: payload kg, columns: push impulse N s over 0.1 s at t = 1 s; %d robots per cell)" % per_cell)
    print("payload \\ impulse " + "".join("%7.1f" % p for p in impulses))
    for i, m in enumerate(masses):
        print("%17.1f " % m + "".join("%7.2f" % up[(variant == i) & (push[:, 0] == impulses[j] / 0.1)].mean() for j in range(len(impulses))))
    ps.close(); s.close(); ctl.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--grid", action="store_true", help="also run the payload x push-impulse grid")
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    print(card(), flush=True)
    throughput(a.rounds)
    if a.grid:
        grid()
