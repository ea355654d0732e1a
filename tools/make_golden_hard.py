#!/usr/bin/env python
"""Frozen deep-active-set fixture: tests/golden/hard_tail.npz (+ hard_tail.json).

The golden files of tools/make_golden.py are mostly shallow (0-12 active-set pivots); the soak reaches 17-26 pivots at
p99.9 and 28-38 at the maximum, with many drops and re-adds. This fixture freezes the deepest instances of large seeded
batches, so that a change of the pivot chain is checked against the oracle where it is most likely to go wrong.

Choosing the instances needs the kernel's pivot counts, so the tool has two stages:

  --select  (needs a GPU)  for each combination below, generate 65536 states (synth.generate, fixed seed), step them with
            every output on and keep the 16 status-0 instances with the most pivots (qp_info[:, 3]); writes
            tests/golden/hard_tail.json (combination, seed, index, pivots) and asserts every kept instance reaches
            MIN_PIVOTS.
  --solve   (CPU)  regenerates those inputs with the oracle's forward kinematics and runs the oracle controllers with the
            same parameters on a process pool; writes tests/golden/hard_tail.npz: inputs, the oracle's tau, vd, f,
            objective, metrics and ok flags, and the kernel's pivot count (information only: block-start or warm-start
            work may lower it).

Usage: python tools/make_golden_hard.py --select | --solve [--json PATH] [--jobs J]
"""
import argparse
import json
import os
import sys
from multiprocessing import get_context
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

N_BATCH = 65536
KEEP = 16
MIN_PIVOTS = 20
JSON = ROOT / "tests" / "golden" / "hard_tail.json"
NPZ = ROOT / "tests" / "golden" / "hard_tail.npz"


def combinations():
    """(name, robot, pattern, dof_order, params, kind, seed): stand for both robots x {id, clf, pc, mptc} with the torque box
    off, stand x {id, clf} with it on, and mini_cheetah ID on mixed contacts with breadth-first numbering and the box on."""
    out = []
    for robot in ("mini_cheetah", "anymal_b"):
        for kind in ("id", "clf", "pc", "mptc"):
            out.append((f"stand_{robot}_{kind}", robot, "stand", "depth_first", {}, kind))
        for kind in ("id", "clf"):
            out.append((f"stand_{robot}_{kind}_box", robot, "stand", "depth_first", {"torque_limits": 1}, kind))
    out.append(("bf_mini_cheetah_mixed_id_box", "mini_cheetah", "mixed", "breadth_first", {"torque_limits": 1}, "id"))
    return [c + (20261100 + i,) for i, c in enumerate(out)]


def select(path):
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.synth import generate
    rows, shallow = [], []
    for name, robot, pattern, dof_order, params, kind, seed in combinations():
        ctl = BatchedController(robot, device=0, dof_order=dof_order, **params)
        q, v, traj, contact = generate(ctl.model, N_BATCH, seed, pattern, ctl.fk)
        out = ctl.step(kind, q, v, traj, contact, debug=True)
        ctl.close()
        piv = out.qp_info[:, 3].astype(int)
        cand = np.flatnonzero(out.status == 0)
        order = cand[np.lexsort((cand, -piv[cand]))][:KEEP]          # most pivots first, ties by index
        rows.append(dict(name=name, robot=robot, pattern=pattern, dof_order=dof_order, params=params, kind=kind, seed=seed,
                         index=[int(i) for i in order], pivots=[int(piv[i]) for i in order],
                         batch_max=int(piv[cand].max()), batch_p999=float(np.percentile(piv[cand], 99.9))))
        print(name, "pivots of the kept instances", rows[-1]["pivots"], "batch p99.9", rows[-1]["batch_p999"], flush=True)
        if min(rows[-1]["pivots"]) < MIN_PIVOTS:
            shallow.append(name)
    Path(path).write_text(json.dumps(dict(n_batch=N_BATCH, keep=KEEP, combinations=rows), indent=1) + "\n")
    assert not shallow, f"kept instances below {MIN_PIVOTS} pivots: {shallow}"


def sparse_oracle_fk(plant, index):
    """Forward kinematics of the oracle at the rows `index` only (zeros elsewhere). synth.generate draws its noise
    independently of the feet it is given, so the rows `index` come out exactly as with the full oracle_fk."""
    def fk(q, v):
        P, V = np.zeros((len(q), 4, 3)), np.zeros((len(q), 4, 3))
        for i in index:
            for k, f in enumerate(plant.foot_frames):
                p, J, _ = plant.frame_position_quantities(q[i], v[i], f)
                P[i, k], V[i, k] = p, J @ v[i]
        return P, V
    return fk


def _solve_one(args):
    robot, dof_order, params, kind, q, v, traj, contact = args
    from oracle import controllers as oc
    from oracle.dynamics import Plant
    ctrl = {"id": oc.IDController, "clf": oc.CLFController, "pc": oc.PCController, "mptc": oc.MPTCController}[kind]
    ctl = ctrl(Plant(robot, dof_order), **params)
    try:
        o = ctl.control_law(q, v, oc.traj_to_dict(traj, contact))
    except Exception:  # noqa: BLE001  (infeasible torque box etc.: recorded as not ok)
        return np.zeros(12), np.zeros(18), np.zeros((4, 3)), np.zeros(4), 0.0, False
    ok = o.status in ("optimal", "ipm") and o.primal_res < 1e-7
    return o.tau, o.vd, o.f, o.metrics, o.objective, ok


def solve(path, jobs):
    from oracle.dynamics import Plant
    from quadruped_drake_b200 import load_robot
    from quadruped_drake_b200.synth import generate
    sel = json.loads(Path(path).read_text())
    data = {k: [] for k in ("q", "v", "traj", "contact", "combo", "batch_index", "pivots")}
    work = []
    for c, row in enumerate(sel["combinations"]):
        idx = np.asarray(row["index"])
        model = load_robot(row["robot"], dof_order=row["dof_order"])
        q, v, traj, contact = generate(model, sel["n_batch"], row["seed"], row["pattern"],
                                       sparse_oracle_fk(Plant(row["robot"], row["dof_order"]), idx))
        for i in idx:
            work.append((row["robot"], row["dof_order"], row["params"], row["kind"], q[i], v[i], traj[i], contact[i]))
        for k, x in (("q", q[idx]), ("v", v[idx]), ("traj", traj[idx]), ("contact", contact[idx])):
            data[k].append(x)
        data["combo"].append(np.full(len(idx), c, np.int32))
        data["batch_index"].append(idx.astype(np.int64))
        data["pivots"].append(np.asarray(row["pivots"], np.int32))
    with get_context("spawn").Pool(jobs) as pool:
        res = pool.map(_solve_one, work, chunksize=1)
    out = {k: np.concatenate(x) for k, x in data.items()}
    for j, key in enumerate(("tau", "vd", "f", "metrics", "objective", "ok")):
        out[key] = np.asarray([r[j] for r in res])
    rows = sel["combinations"]
    out.update(names=np.array([r["name"] for r in rows]), robots=np.array([r["robot"] for r in rows]),
               kinds=np.array([r["kind"] for r in rows]), dof_orders=np.array([r["dof_order"] for r in rows]),
               torque_limits=np.array([int(r["params"].get("torque_limits", 0)) for r in rows], np.int32),
               seeds=np.array([r["seed"] for r in rows], np.int64), n_batch=np.array(sel["n_batch"]))
    for c, r in enumerate(rows):
        print(r["name"], "oracle solved", int(out["ok"][out["combo"] == c].sum()), "/", len(r["index"]), flush=True)
    np.savez_compressed(NPZ, **out)


def main():
    ap = argparse.ArgumentParser()
    g = ap.add_mutually_exclusive_group(required=True)
    g.add_argument("--select", action="store_true")
    g.add_argument("--solve", action="store_true")
    ap.add_argument("--json", default=str(JSON), help="selection file written by --select, read by --solve")
    ap.add_argument("--jobs", type=int, default=os.cpu_count() or 1)
    args = ap.parse_args()
    select(args.json) if args.select else solve(args.json, args.jobs)


if __name__ == "__main__":
    main()
