"""Host-side model flattener: neutral robot description -> SoA link tables.

Stands in for what Drake's Parser + MultibodyPlant.Finalize() keep after reference
simulate.py:37-64: the kinematic tree is flattened once on the host into the
`wbc_model` struct of include/wbc.h (floating base + 4 legs x 3 revolute joints,
welded links merged into their parents, foot frames as fixed offsets on the shank).

DOF order (SURVEY.md Appendix E.1): Drake's velocity numbering is version dependent.
`dof_order="depth_first"` (default; modern Drake and the per-leg literals q0 /
q_nom in reference simulate.py:171-176, basic_controller.py:335-340) numbers the
joints leg by leg; `"breadth_first"` (2021-era Drake) numbers all hips, then all
thighs, then all knees. An explicit list of joint names is accepted too.
"""
from __future__ import annotations

import copy
import ctypes as C
from dataclasses import dataclass, field
from pathlib import Path

import numpy as np

from .urdf import load_description, parse_urdf, rpy_to_matrix

NQ, NV, NU, NLEG, NBODY, NTRAJ = 19, 18, 12, 4, 13, 54
ROBOT_DIR = Path(__file__).resolve().parent / "robots"


class WbcModelStruct(C.Structure):
    """ctypes mirror of `wbc_model` (include/wbc.h)."""
    _fields_ = [
        ("mass", C.c_double * NBODY),
        ("com", (C.c_double * 3) * NBODY),
        ("inertia_com", (C.c_double * 6) * NBODY),
        ("joint_xyz", (C.c_double * 3) * NU),
        ("joint_axis", (C.c_double * 3) * NU),
        ("foot_xyz", (C.c_double * 3) * NLEG),
        ("effort", C.c_double * NU),
        ("gravity", C.c_double * 3),
        ("v_index", C.c_int32 * NU),
        ("act_index", C.c_int32 * NU),
    ]


def _sym(v6):
    xx, yy, zz, xy, xz, yz = v6
    return np.array([[xx, xy, xz], [xy, yy, yz], [xz, yz, zz]], dtype=float)


def _v6(I):
    return np.array([I[0, 0], I[1, 1], I[2, 2], I[0, 1], I[0, 2], I[1, 2]])


def _merge(bodies):
    """Composite of rigid pieces [(m, c, I_com)] given in one frame -> (m, c, I about c)."""
    m = sum(b[0] for b in bodies)
    if m <= 0.0:
        return 0.0, np.zeros(3), np.zeros((3, 3))
    c = sum(b[0] * b[1] for b in bodies) / m
    I = np.zeros((3, 3))
    for mb, cb, Ib in bodies:
        d = cb - c
        I += Ib + mb * (d @ d * np.eye(3) - np.outer(d, d))
    return m, c, I


@dataclass
class RobotModel:
    """Flattened quadruped. Arrays are indexed as documented in include/wbc.h."""
    name: str
    mass: np.ndarray
    com: np.ndarray
    inertia_com: np.ndarray
    joint_xyz: np.ndarray
    joint_axis: np.ndarray
    foot_xyz: np.ndarray
    effort: np.ndarray
    v_index: np.ndarray
    act_index: np.ndarray
    joint_names: list
    base_link: str
    gravity: np.ndarray = field(default_factory=lambda: np.array([0.0, 0.0, -9.81]))

    @property
    def total_mass(self) -> float:
        return float(self.mass.sum())

    def actuation_matrix(self) -> np.ndarray:
        """B (nv x nu) of MultibodyPlant.MakeActuationMatrix (basic_controller.py:113)."""
        B = np.zeros((NV, NU))
        for k in range(NU):
            B[self.v_index[k], self.act_index[k]] = 1.0
        return B

    def as_struct(self) -> WbcModelStruct:
        s = WbcModelStruct()
        for i in range(NBODY):
            s.mass[i] = self.mass[i]
            for a in range(3):
                s.com[i][a] = self.com[i, a]
            for a in range(6):
                s.inertia_com[i][a] = self.inertia_com[i, a]
        for k in range(NU):
            for a in range(3):
                s.joint_xyz[k][a] = self.joint_xyz[k, a]
                s.joint_axis[k][a] = self.joint_axis[k, a]
            s.effort[k] = self.effort[k]
            s.v_index[k] = int(self.v_index[k])
            s.act_index[k] = int(self.act_index[k])
        for l in range(NLEG):
            for a in range(3):
                s.foot_xyz[l][a] = self.foot_xyz[l, a]
        for a in range(3):
            s.gravity[a] = self.gravity[a]
        return s

    def nominal_q(self) -> np.ndarray:
        """Standing posture: reference simulate.py:171-176 for mini_cheetah; for ANYmal the
        reference gives none (SURVEY 8d) - HAA 0, HFE +-0.4, KFE -+0.8, mirrored front/hind."""
        q = np.zeros(NQ)
        q[0] = 1.0
        if self.name == "anymal_b":
            q[6] = 0.5
            legs = [(0.0, 0.4, -0.8), (0.0, 0.4, -0.8), (0.0, -0.4, 0.8), (0.0, -0.4, 0.8)]
        else:
            q[6] = 0.3
            legs = [(0.0, -0.8, 1.6)] * 4
        for l in range(NLEG):
            for j in range(3):
                q[1 + self.v_index[3 * l + j]] = legs[l][j]
        return q


def flatten(desc: dict, dof_order="depth_first") -> RobotModel:
    links = {l["name"]: l for l in desc["links"]}
    parent_joint = {j["child"]: j for j in desc["joints"]}
    children = {}
    for j in desc["joints"]:
        children.setdefault(j["parent"], []).append(j)
    base = desc["base_link"]

    def welded_pieces(link, X_R, X_p):
        """All mass pieces rigidly attached to `link`, expressed in the frame (X_R, X_p)."""
        l = links[link]
        out = []
        if l["mass"] > 0.0:
            out.append((l["mass"], X_R @ np.array(l["com"]) + X_p, X_R @ _sym(l["inertia_com"]) @ X_R.T))
        for j in children.get(link, []):
            if j["type"] == "fixed":
                R = X_R @ rpy_to_matrix(j["rpy"])
                p = X_R @ np.array(j["xyz"]) + X_p
                out += welded_pieces(j["child"], R, p)
        return out

    mass, com, inertia = np.zeros(NBODY), np.zeros((NBODY, 3)), np.zeros((NBODY, 6))
    joint_xyz, joint_axis = np.zeros((NU, 3)), np.zeros((NU, 3))
    foot_xyz, effort = np.zeros((NLEG, 3)), np.zeros(NU)
    joint_names = [None] * NU

    m, c, I = _merge(welded_pieces(base, np.eye(3), np.zeros(3)))
    mass[0], com[0], inertia[0] = m, c, _v6(I)

    for leg, foot in enumerate(desc["foot_frames"]):
        # walk foot -> base collecting joints
        chain, link = [], foot
        while link != base:
            j = parent_joint[link]
            chain.append(j)
            link = j["parent"]
        chain.reverse()
        moving = [j for j in chain if j["type"] == "revolute"]
        if len(moving) != 3:
            raise ValueError(f"leg {foot}: expected 3 revolute joints, found {len(moving)}")
        # fixed joints between base and first revolute would need a rotated joint frame
        X_R, X_p = np.eye(3), np.zeros(3)
        jcount = -1
        for j in chain:
            R = rpy_to_matrix(j["rpy"])
            if j["type"] == "revolute":
                if not np.allclose(X_R @ R, np.eye(3), atol=1e-12):
                    raise ValueError(f"joint {j['name']}: rotated joint frames are not supported")
                jcount += 1
                k = 3 * leg + jcount
                joint_xyz[k] = X_R @ np.array(j["xyz"]) + X_p
                ax = np.array(j["axis"], dtype=float)
                joint_axis[k] = ax / np.linalg.norm(ax)
                effort[k] = j["effort"]
                joint_names[k] = j["name"]
                m, c, I = _merge(welded_pieces(j["child"], np.eye(3), np.zeros(3)))
                mass[k + 1], com[k + 1], inertia[k + 1] = m, c, _v6(I)
                X_R, X_p = np.eye(3), np.zeros(3)
            else:
                X_p = X_R @ np.array(j["xyz"]) + X_p
                X_R = X_R @ R
        foot_xyz[leg] = X_p  # accumulated fixed offset after the last revolute joint

    total = sum(l["mass"] for l in desc["links"])
    if abs(mass.sum() - total) > 1e-9 * max(total, 1.0):
        raise ValueError("flattened mass does not match the description (unreached links?)")

    if dof_order == "depth_first":
        order = list(range(NU))
    elif dof_order == "breadth_first":
        order = [3 * l + j for j in range(3) for l in range(NLEG)]
    else:
        order = [joint_names.index(n) for n in dof_order]
        if sorted(order) != list(range(NU)):
            raise ValueError("dof_order must name each of the 12 joints once")
    v_index = np.zeros(NU, dtype=np.int32)
    for pos, k in enumerate(order):
        v_index[k] = 6 + pos
    act = desc.get("actuated_joints") or joint_names
    act_index = np.array([act.index(n) for n in joint_names], dtype=np.int32)
    if sorted(act_index.tolist()) != list(range(NU)):
        raise ValueError("every leg joint must have exactly one transmission")

    return RobotModel(name=desc["name"], mass=mass, com=com, inertia_com=inertia, joint_xyz=joint_xyz,
                      joint_axis=joint_axis, foot_xyz=foot_xyz, effort=effort, v_index=v_index,
                      act_index=act_index, joint_names=joint_names, base_link=base)


def with_payload(desc: dict, mass, com, inertia=None, name="payload") -> dict:
    """Copy of a robot description with one more link welded to the base link: `mass` (kg) with its CoM at `com` (base
    coordinates, m) and `inertia` about that CoM (xx yy zz xy xz yz; None: a point mass). `flatten` merges it into body 0;
    oracle.dynamics.Plant keeps it as a separate welded body."""
    d = copy.deepcopy(desc)
    if any(l["name"] == name for l in d["links"]):
        raise ValueError(f"the description already has a link named {name!r}")
    d["links"].append({"name": name, "mass": float(mass), "com": [0.0, 0.0, 0.0],
                       "inertia_com": [float(x) for x in (inertia if inertia is not None else np.zeros(6))]})
    d["joints"].append({"name": f"{d['base_link']}_to_{name}", "type": "fixed", "parent": d["base_link"], "child": name,
                        "xyz": [float(x) for x in com], "rpy": [0.0, 0.0, 0.0], "axis": [1, 0, 0], "effort": float("inf")})
    return d


def load_robot(name_or_path="mini_cheetah", dof_order="depth_first", base_link=None, foot_frames=None) -> RobotModel:
    """`name_or_path`: a packaged robot ("mini_cheetah", "anymal_b"), a .json description or a URDF."""
    p = Path(str(name_or_path))
    if p.suffix == ".urdf":
        desc = parse_urdf(p)
        names = {l["name"] for l in desc["links"]}
        desc["base_link"] = base_link or ("body" if "body" in names else "base")
        desc["foot_frames"] = foot_frames or ["LF_FOOT", "RF_FOOT", "LH_FOOT", "RH_FOOT"]
    elif p.suffix == ".json":
        desc = load_description(p)
    else:
        desc = load_description(ROBOT_DIR / f"{name_or_path}.json")
    return flatten(desc, dof_order=dof_order)
