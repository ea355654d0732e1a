"""ORACLE (test infrastructure only): the terrain of the ground plant, restated in numpy from its definition (include/wbc.h).

    h(x, y) = z0 + sx x + sy y + H(x, y)

H is the bilinear interpolant of the row-major grid heights[ny][nx] with origin (x0, y0) and spacing (dx, dy); no grid means
H = 0. Grid coordinates are clamped to the grid (a clamped direction has zero gradient), and the cell of a coordinate is
min(floor(u), nx - 2). A foot at p contacts along n = (-h_x, -h_y, 1) / |.|, with t1 = normalize(e_x - n_x n), t2 = n x t1,
R = [t1 t2 n], and its gap is phi = (p_z - h(p_x, p_y)) n_z."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


@dataclass
class Terrain:
    z0: float = 0.0
    slope: tuple = (0.0, 0.0)             # (sx, sy)
    origin: tuple = (0.0, 0.0)            # world (x, y) of heights[0, 0]
    spacing: tuple = (1.0, 1.0)           # (dx, dy)
    heights: np.ndarray | None = None     # [ny, nx] or None


def _axis(c, n):
    """Cell index, fraction and whether the coordinate was clamped, for a grid coordinate c on n samples."""
    clamped = c < 0.0 or c > n - 1
    c = min(max(c, 0.0), n - 1.0)
    i = min(int(np.floor(c)), n - 2)
    return i, c - i, clamped


def height_and_gradient(tr: Terrain, x: float, y: float):
    """h(x, y) and (h_x, h_y)."""
    sx, sy = tr.slope
    h = tr.z0 + sx * x + sy * y
    gx, gy = sx, sy
    if tr.heights is not None:
        H = np.asarray(tr.heights, float)
        ny, nx = H.shape
        dx, dy = tr.spacing
        i, fu, cu = _axis((x - tr.origin[0]) / dx, nx)
        j, fw, cw = _axis((y - tr.origin[1]) / dy, ny)
        h00, h10, h01, h11 = H[j, i], H[j, i + 1], H[j + 1, i], H[j + 1, i + 1]
        h += (1 - fu) * (1 - fw) * h00 + fu * (1 - fw) * h10 + (1 - fu) * fw * h01 + fu * fw * h11
        if not cu:
            gx += ((1 - fw) * (h10 - h00) + fw * (h11 - h01)) / dx
        if not cw:
            gy += ((1 - fu) * (h01 - h00) + fu * (h11 - h10)) / dy
    return h, np.array([gx, gy])


def height(tr, x, y):
    return height_and_gradient(tr, x, y)[0]


def gradient(tr, x, y):
    return height_and_gradient(tr, x, y)[1]


def frame(tr, x, y):
    """R = [t1 t2 n] (columns) at (x, y)."""
    g = gradient(tr, x, y)
    n = np.array([-g[0], -g[1], 1.0])
    n /= np.linalg.norm(n)
    t1 = np.array([1.0, 0.0, 0.0]) - n[0] * n
    t1 /= np.linalg.norm(t1)
    return np.column_stack([t1, np.cross(n, t1), n])


def gap(tr, p):
    """Gap of the point p along the local normal: (p_z - h(p_x, p_y)) n_z."""
    R = frame(tr, p[0], p[1])
    return (p[2] - height(tr, p[0], p[1])) * R[2, 2]


def incline(deg, direction=(1.0, 0.0), z0=0.0):
    """A plane rising at `deg` degrees along the horizontal `direction`."""
    d = np.asarray(direction, float)
    d = d / np.linalg.norm(d)
    s = np.tan(np.radians(deg))
    return Terrain(z0=z0, slope=(s * d[0], s * d[1]))


class _LocalFramePlant:
    """A plant whose foot quantities are taken in each foot's terrain frame: Jacobian rows R' J (t1, t2, n) and, as the
    height the flat-ground step reads, the gap phi along n. Everything else is the wrapped plant's."""

    def __init__(self, plant, terrain):
        self.plant, self.terrain, self.frames = plant, terrain, {}

    def __getattr__(self, name):
        return getattr(self.plant, name)

    def frame_position_quantities(self, q, v, fr):
        p, J, Jdv = self.plant.frame_position_quantities(q, v, fr)[:3]
        R = self.frames[fr] = frame(self.terrain, p[0], p[1])
        return np.array([p[0], p[1], gap(self.terrain, p)]), R.T @ J, R.T @ Jdv


def plant_step(plant, q, v, tau, dt, mu=1.0, erp=0.2, iters=30, terrain=None):
    """oracle/rollout.py:plant_step on a terrain (None: the plane z = 0, the flat step itself). Foot k contacts its terrain
    along R_k = [t1 t2 n] at its position at the start of the step: its rows become R_k' J_k (normal still row 2), its gap is
    phi_k, and its force is mapped back to world axes, f_k = R_k p_k / dt."""
    from . import rollout as ro
    if terrain is None:
        return ro.plant_step(plant, q, v, tau, dt, mu, erp, iters)
    lp = _LocalFramePlant(plant, terrain)
    qn, vn, f = ro.plant_step(lp, q, v, tau, dt, mu, erp, iters)
    return qn, vn, np.stack([lp.frames[fr] @ f[k] for k, fr in enumerate(plant.foot_frames)])
