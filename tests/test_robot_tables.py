"""Robot tables (quadruped_drake_b200/robots/*.json -> wbc_model) cross-checked against sources the product parser
(urdf.py) did not produce: (a) an independent regex reader of the reference URDFs, when the reference tree is present
(this container), every mass / CoM / inertia / joint origin / axis / effort; (b) the SURVEY.md Appendix B table as frozen
constants (always, also on the GPU box). Oracle and kernel share the JSON, so a mis-parsed number would be invisible to
the parity tests - this file is what guards it."""
import json
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
ROBOTS = ROOT / "quadruped_drake_b200" / "robots"
REF = Path("/root/reference")
URDFS = {"mini_cheetah": "models/mini_cheetah/mini_cheetah_mesh.urdf",
         "anymal_b": "models/anymal_b_simple_description/urdf/anymal_drake.urdf"}


def _attr(tag, name, default=None):
    m = re.search(r'\b%s\s*=\s*"([^"]*)"' % name, tag)
    return m.group(1) if m else default


def _vec(text, default):
    return [float(t) for t in text.split()] if text is not None else list(default)


def regex_urdf(path):
    """Minimal independent reader: no XML library, comments stripped, elements located by regular expressions."""
    txt = re.sub(r"<!--.*?-->", "", Path(path).read_text(), flags=re.S)
    links, joints = {}, {}
    for m in re.finditer(r"<link\b([^>]*?)(/>|>(.*?)</link>)", txt, flags=re.S):
        name, body = _attr(m.group(1), "name"), m.group(3) or ""
        ine = re.search(r"<inertial>(.*?)</inertial>", body, flags=re.S)
        rec = {"mass": 0.0, "com": [0.0] * 3, "inertia": [0.0] * 6, "rpy": [0.0] * 3}
        if ine:
            blk = ine.group(1)
            rec["mass"] = float(_attr(re.search(r"<mass\b[^>]*>", blk).group(0), "value"))
            org = re.search(r"<origin\b[^>]*>", blk)
            if org:
                rec["com"] = _vec(_attr(org.group(0), "xyz"), [0, 0, 0])
                rec["rpy"] = _vec(_attr(org.group(0), "rpy"), [0, 0, 0])
            it = re.search(r"<inertia\b[^>]*>", blk).group(0)
            rec["inertia"] = [float(_attr(it, k)) for k in ("ixx", "iyy", "izz", "ixy", "ixz", "iyz")]
        links[name] = rec
    for m in re.finditer(r"<joint\b([^>]*?)>(.*?)</joint>", txt, flags=re.S):
        name, body = _attr(m.group(1), "name"), m.group(2)
        if re.search(r"<transmission", txt[max(0, m.start() - 400):m.start()]) and "<parent" not in body:
            continue                                    # <joint name=...> inside a <transmission>
        if "<parent" not in body:
            continue
        org = re.search(r"<origin\b[^>]*>", body)
        ax = re.search(r"<axis\b[^>]*>", body)
        lim = re.search(r"<limit\b[^>]*>", body)
        joints[name] = {"type": _attr(m.group(1), "type"),
                        "parent": _attr(re.search(r"<parent\b[^>]*>", body).group(0), "link"),
                        "child": _attr(re.search(r"<child\b[^>]*>", body).group(0), "link"),
                        "xyz": _vec(_attr(org.group(0), "xyz") if org else None, [0, 0, 0]),
                        "rpy": _vec(_attr(org.group(0), "rpy") if org else None, [0, 0, 0]),
                        "axis": _vec(_attr(ax.group(0), "xyz") if ax else None, [1, 0, 0]),
                        "effort": float(_attr(lim.group(0), "effort")) if lim and _attr(lim.group(0), "effort") else None}
    order = []
    for m in re.finditer(r"<transmission\b.*?</transmission>", txt, flags=re.S):
        order.append(_attr(re.search(r"<joint\b[^>]*>", m.group(0)).group(0), "name"))
    return links, joints, order


@pytest.mark.skipif(not REF.exists(), reason="reference tree not present (GPU box)")
@pytest.mark.parametrize("robot", ["mini_cheetah", "anymal_b"])
def test_json_matches_independent_urdf_reader(robot):
    desc = json.loads((ROBOTS / f"{robot}.json").read_text())
    links, joints, order = regex_urdf(REF / URDFS[robot])
    assert {l["name"] for l in desc["links"]} == set(links)
    assert {j["name"] for j in desc["joints"]} == set(joints)
    for l in desc["links"]:
        r = links[l["name"]]
        assert l["mass"] == r["mass"], l["name"]
        assert l["com"] == r["com"], l["name"]
        assert np.allclose(r["rpy"], 0.0), "inertial frames are unrotated in both reference URDFs (SURVEY A.4)"
        assert l["inertia_com"] == r["inertia"], l["name"]
    for j in desc["joints"]:
        r = joints[j["name"]]
        assert (j["parent"], j["child"]) == (r["parent"], r["child"]), j["name"]
        assert j["type"] == ("revolute" if r["type"] in ("revolute", "continuous") else r["type"]), j["name"]
        assert j["xyz"] == r["xyz"] and j["rpy"] == r["rpy"], j["name"]
        if j["type"] == "revolute":
            assert j["axis"] == r["axis"], j["name"]
            assert j["effort"] == r["effort"], j["name"]
    assert desc["actuated_joints"] == order
    assert sum(l["mass"] for l in desc["links"]) == pytest.approx(sum(r["mass"] for r in links.values()), abs=0)


# ------------------------------------------------------------------ SURVEY.md Appendix B, frozen
MC_LEGS = {"fl": (+1, +1), "fr": (+1, -1), "hl": (-1, +1), "hr": (-1, -1)}      # (sx, sy)


def test_mini_cheetah_frozen_table():
    """mini_cheetah_mesh.urdf:5-10,26-39,62-75,92-104,437-441 as listed in SURVEY Appendix B."""
    d = json.loads((ROBOTS / "mini_cheetah.json").read_text())
    L = {l["name"]: l for l in d["links"]}
    J = {j["child"]: j for j in d["joints"]}
    assert L["body"]["mass"] == 3.3 and L["body"]["com"] == [0, 0, 0]
    assert L["body"]["inertia_com"] == [0.011253, 0.036203, 0.042673, 0, 0, 0]
    for leg, (sx, sy) in MC_LEGS.items():
        ab, th, sh = L[f"abduct_{leg}"], L[f"thigh_{leg}"], L[f"shank_{leg}"]
        assert ab["mass"] == 0.54 and th["mass"] == 0.634 and sh["mass"] == 0.064
        # CoM / products of inertia are NOT mirrored left/right in this URDF (Appendix B note): same numbers on all legs
        assert ab["com"] == [0.0, 0.036, 0.0] and th["com"] == [0.0, 0.016, -0.02] and sh["com"] == [0.0, 0.0, -0.209]
        assert ab["inertia_com"] == [0.000381, 0.00056, 0.000444, 5.8e-05, 4.5e-07, 9.5e-07]
        assert th["inertia_com"] == [0.001983, 0.002103, 0.000508, 0.000245, 1.3e-05, 1.5e-06]
        assert sh["inertia_com"] == [0.000245, 0.000248, 6e-06, 0.0, 0.0, 0.0]
        assert J[f"abduct_{leg}"]["xyz"] == [sx * 0.19, sy * 0.049, 0.0] and J[f"abduct_{leg}"]["axis"] == [1.0, 0.0, 0.0]
        assert J[f"thigh_{leg}"]["xyz"] == [0.0, sy * 0.062, 0.0] and J[f"thigh_{leg}"]["axis"] == [0.0, -1.0, 0.0]
        assert J[f"shank_{leg}"]["xyz"] == [0.0, 0.0, -0.209] and J[f"shank_{leg}"]["axis"] == [0.0, -1.0, 0.0]
        assert (J[f"abduct_{leg}"]["effort"], J[f"thigh_{leg}"]["effort"], J[f"shank_{leg}"]["effort"]) == (18.0, 18.0, 26.0)
    for foot in ("LF_FOOT", "RF_FOOT", "LH_FOOT", "RH_FOOT"):
        assert J[foot]["type"] == "fixed" and J[foot]["xyz"] == [0.0, 0.0, -0.19] and L[foot]["mass"] == 0.0
    assert sum(l["mass"] for l in d["links"]) == pytest.approx(8.252, abs=1e-12)


def test_anymal_frozen_table():
    """anymal_drake.urdf:83-89,112-124,156-167,185-232 as listed in SURVEY Appendix B."""
    d = json.loads((ROBOTS / "anymal_b.json").read_text())
    L = {l["name"]: l for l in d["links"]}
    J = {j["name"]: j for j in d["joints"]}
    ap = lambda x: pytest.approx(x, rel=5e-6)   # noqa: E731  (Appendix B quotes 6 significant digits)
    assert L["base"]["mass"] == 0.0 and L["base_inertia"]["mass"] == ap(16.7935)
    for leg, (sx, sy) in {"LF": (1, 1), "RF": (1, -1), "LH": (-1, 1), "RH": (-1, -1)}.items():
        assert L[f"{leg}_HIP"]["mass"] == ap(1.42462) and L[f"{leg}_THIGH"]["mass"] == ap(1.63498)
        assert L[f"{leg}_SHANK"]["mass"] == ap(0.207204) and L[f"{leg}_ADAPTER"]["mass"] == ap(0.140171)
        assert J[f"{leg}_HAA"]["xyz"] == [sx * 0.277, sy * 0.116, 0.0] and J[f"{leg}_HAA"]["axis"] == [1.0, 0.0, 0.0]
        assert J[f"{leg}_HFE"]["xyz"] == [sx * 0.0635, sy * 0.041, 0.0] and J[f"{leg}_HFE"]["axis"] == [0.0, 1.0, 0.0]
        assert J[f"{leg}_KFE"]["xyz"] == [0.0, sy * 0.109, -0.25] and J[f"{leg}_KFE"]["axis"] == [0.0, 1.0, 0.0]
        assert all(J[f"{leg}_{j}"]["effort"] == 80.0 for j in ("HAA", "HFE", "KFE"))
        ad = J[f"{leg}_SHANK_TO_ADAPTER"]["xyz"]
        assert ad == [sx * 0.1, -sy * 0.02, 0.0]
        assert J[f"{leg}_ADAPTER_TO_FOOT"]["xyz"] == [0.0, 0.0, -0.32125]
        # CoMs ARE mirrored per leg here (Appendix B): y of the hip CoM flips with the side, x with front/hind
        for part in ("HIP", "THIGH", "SHANK"):
            assert np.allclose(L[f"{leg}_{part}"]["com"], np.array([sx, sy, 1.0]) * np.array(L[f"LF_{part}"]["com"]), atol=1e-12)
    assert sum(l["mass"] for l in d["links"]) == pytest.approx(30.4214, abs=5e-5)


def test_frozen_actuation_order_frames_and_mirroring():
    """SURVEY A.5: actuator order = <transmission> order, legs LF/fl, RF/fr, LH/hl, RH/hr x (abduction, hip, knee);
    SURVEY 7: every joint rpy is zero in both URDFs; Appendix B: anymal products of inertia are mirrored per leg."""
    mc = json.loads((ROBOTS / "mini_cheetah.json").read_text())
    by_child = {j["child"]: j["name"] for j in mc["joints"]}
    assert mc["actuated_joints"] == [by_child[f"{part}_{leg}"] for leg in MC_LEGS for part in ("abduct", "thigh", "shank")]
    an = json.loads((ROBOTS / "anymal_b.json").read_text())
    assert an["actuated_joints"] == [f"{leg}_{j}" for leg in ("LF", "RF", "LH", "RH") for j in ("HAA", "HFE", "KFE")]
    for d in (mc, an):
        assert all(j["rpy"] == [0.0, 0.0, 0.0] for j in d["joints"])
    L = {l["name"]: l for l in an["links"]}
    for leg, (sx, sy) in {"LF": (1, 1), "RF": (1, -1), "LH": (-1, 1), "RH": (-1, -1)}.items():
        for part in ("HIP", "THIGH", "SHANK"):
            # S I S with S = diag(sx, sy, 1): diagonal kept, Ixy x sx sy, Ixz x sx, Iyz x sy
            lf = np.array(L[f"LF_{part}"]["inertia_com"])
            assert np.array_equal(L[f"{leg}_{part}"]["inertia_com"], lf * np.array([1, 1, 1, sx * sy, sx, sy]))


@pytest.mark.parametrize("robot,total", [("mini_cheetah", 8.252), ("anymal_b", 30.4214)])
def test_flattened_model_conserves_mass_moments(robot, total):
    """Welding (anymal: base_inertia into base, adapter into shank) conserves mass, first and second moments: the
    flattened 13-body model and the unmerged link list give the same composite inertia about the base origin at q = 0."""
    from quadruped_drake_b200 import load_robot
    m = load_robot(robot)
    assert m.total_mass == pytest.approx(total, abs=5e-5)
    d = json.loads((ROBOTS / f"{robot}.json").read_text())
    parent = {j["child"]: j for j in d["joints"]}

    def origin(link):
        p = np.zeros(3)
        while link in parent:
            p += np.array(parent[link]["xyz"])
            link = parent[link]["parent"]
        return p
    mass = h = 0.0
    I = np.zeros((3, 3))
    for l in d["links"]:
        if l["mass"] == 0.0:
            continue
        c = origin(l["name"]) + np.array(l["com"])
        ic = l["inertia_com"]
        Ic = np.array([[ic[0], ic[3], ic[4]], [ic[3], ic[1], ic[5]], [ic[4], ic[5], ic[2]]])
        mass, h = mass + l["mass"], h + l["mass"] * c
        I += Ic + l["mass"] * (c @ c * np.eye(3) - np.outer(c, c))
    # flattened model at q = 0: body b sits at the sum of the joint origins of its chain
    fm = fh = 0.0
    fI = np.zeros((3, 3))
    for b in range(13):
        p = np.zeros(3)
        if b > 0:
            leg, j = (b - 1) // 3, (b - 1) % 3
            for jj in range(j + 1):
                p += m.joint_xyz[3 * leg + jj]
        c = p + m.com[b]
        ic = m.inertia_com[b]
        Ic = np.array([[ic[0], ic[3], ic[4]], [ic[3], ic[1], ic[5]], [ic[4], ic[5], ic[2]]])
        fm, fh = fm + m.mass[b], fh + m.mass[b] * c
        fI += Ic + m.mass[b] * (c @ c * np.eye(3) - np.outer(c, c))
    assert fm == pytest.approx(mass, abs=1e-12) and np.allclose(fh, h, atol=1e-12) and np.allclose(fI, I, atol=1e-12)
