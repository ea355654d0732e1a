// wbc_plant.cuh — one time step of the simulated robot on flat ground (SURVEY.md 8 f2: "semi-implicit integrator + flat-ground
// contact"), the other half of the closed loop of simulate.py:36-57,160-182.
//
// The reference steps a discrete MultibodyPlant(time_step = dt) with a ground half-space (static = dynamic friction 1.0,
// simulate.py:44-46) through Drake's implicit contact solver, which is third party and not restatable. This file is a
// time-stepping scheme of the same family, defined here and pinned by invariants (tests/test_gpu_rollout.py) and by the numpy
// restatement in oracle/rollout.py - NOT by Drake:
//
//   v_free = v + dt M^-1 (B tau - C v - tau_g)                          forward dynamics from the APPLIED torques
//   u      = J_c v+ = J_c v_free + A p,   A = J_c M^-1 J_c'              foot velocities as a function of the contact impulses p
//   per foot:  0 <= p_n  _|_  u_n + bias_n >= 0                          no penetration (velocity level, Signorini)
//              |p_x|, |p_y| <= mu p_n, tangential velocity driven to 0   Coulomb friction, pyramid as in the controller
//   v+ = v_free + M^-1 J_c' p,   q+ = q + dt N(q) v+                      semi-implicit (symplectic) Euler
//
// bias_n = phi / dt for an open gap phi > 0 (the foot may close the gap in this step but not pass it) and erp * phi / dt for a
// penetration (Baumgarte push-out). The complementarity problem is solved by `iters` sweeps of projected Gauss-Seidel over
// the 12 rows in the fixed order foot LF RF LH RH x (normal, x, y), from p = 0. Contact state comes from the geometry here;
// the controller keeps using the PLANNED contact flags (SURVEY E.5). The terrain step (TERRAIN below) replaces the plane z = 0 by
// each robot's own terrain: the rows of each foot are taken along its local frame instead of the world axes.
//
// One warp per robot, like the control-step kernels; the dynamics block is the same `dynamics_phase` the controllers use, and
// M^-1 is applied through M's block-arrow structure (four closed-form 3x3 leg-block inverses + a 6x6 Cholesky of the Schur
// complement), 13 right-hand sides at once with one lane each.
#pragma once
#include "wbc_device.cuh"

namespace wbcplant {
using namespace wbc;

struct alignas(16) PlantSmem {
  double X[18][13];        // M^-1 [J_c' | B tau - h]: column c < 12 contact row c, column 12 the free acceleration
  double A[12][13];        // Delassus matrix J_c M^-1 J_c' (row per lane, odd stride)
  double Sb[6][6];         // Schur complement of the leg blocks -> its Cholesky factor
  double Dinv[4][6];       // inverses of the 3x3 leg blocks (symmetric storage)
  double p[12];            // contact impulses (N s), row 3 k + i = foot k, world axis i
  double tauk[12];         // applied torque of internal joint k
};

struct PlantArgs {
  double* q; double* v; const double* tau; double* t; const int32_t* ctrl_status; int32_t* status_or; double* f_contact;
  const double* metrics; double* err_max; double* metrics_log; const int* step_counter;     // rollout bookkeeping (optional)
  long long n; double dt, mu, erp; int iters;
};

// Freeze mask: a robot whose controller reported any failure keeps its state (the reference asserts there) and stays flagged.
constexpr int PLANT_FREEZE = WBC_ST_MAXITER | WBC_ST_INFEASIBLE | WBC_ST_RANKDEF | WBC_ST_GIMBAL | WBC_ST_NOTPD | WBC_ST_BADQUAT |
                             WBC_ST_UNSUPPORTED | WBC_ST_DIVERGED | WBC_ST_NONFINITE;

// ---- perturbed robots (wbc_plant_step_perturbed): the plant simulates a variant of the robot, the controller keeps its model.
// One entry of a variant table: 1936 B = 121 x 16 B, so a CTA stages it with the 16-byte vector loop of the model constants.
struct alignas(16) PlantVariant {
  wbc_model md;   // what the plant simulates for this variant
  double mu;      // its ground friction
};
static_assert(sizeof(PlantVariant) == 1936, "variant record: wbc_model + mu, a multiple of 16 bytes");

// Device inputs of the variant kernel. variant [N] (NULL: variant 0); push [N][8]: force F (world) [0:3], point r in base
// coordinates relative to the base origin [3:6], t_on [6], t_off [7] (NULL: no pushes). own_mu == 0: every variant uses the
// call's mu instead of its own.
struct PerturbArgs {
  const PlantVariant* set; const int32_t* variant; const double* push; int n_variants; int own_mu;
};

// What the step of one robot sees: its friction, its push row while t_on <= t < t_off holds for the step's start time t (NULL
// otherwise), and whether its variant index was out of range (the robot is then frozen and flagged WBC_ST_BADVARIANT).
struct Perturb {
  double mu; const double* push; bool bad_variant;
};

// Variant of robot `inst`, or -1 when its index is out of range.
WBC_DEV int plant_variant(const PerturbArgs& pa, long long inst) {
  const int k = pa.variant ? pa.variant[inst] : 0;
  return (k >= 0 && k < pa.n_variants) ? k : -1;
}

WBC_DEV Perturb plant_perturb(const PerturbArgs& pa, const PlantArgs& a, long long inst, int k, double variant_mu) {
  const double* row = pa.push ? pa.push + inst * 8 : nullptr;
  const double t = row ? a.t[inst] : 0.0;
  return Perturb{pa.own_mu ? variant_mu : a.mu, (row && row[6] <= t && t < row[7]) ? row : nullptr, k < 0};
}

// ---- uneven ground (wbc_plant_step_terrain): per robot, a plane plus an optional height field
//
//   h(x, y) = z0 + sx x + sy y + H(x, y)
//
// H is the bilinear interpolant of the row-major grid heights[ny][nx] with origin (x0, y0) and spacing (dx, dy); nx = ny = 0
// is no grid (H = 0). Grid coordinates u = (x - x0) / dx, w = (y - y0) / dy are clamped to [0, nx - 1] x [0, ny - 1] (a clamped
// direction contributes zero gradient), and the cell is min(floor(u), nx - 2), so a point on the far edge uses the last cell.
// The interpolant is continuous: a vertical step in the heights is a ramp one cell wide. Per foot, at its position p at the
// start of the step: n = (-h_x, -h_y, 1) / |.|, t1 = normalize(e_x - n_x n), t2 = n x t1, R = [t1 t2 n], and the gap along
// the normal phi = (p_z - h(p_x, p_y)) n_z (the signed distance for a plane). The contact rows of foot k become d' J_k with
// d = t1, t2, n (normal still row 2); the impulses are solved in that frame and f_contact = R p / dt is in world axes.
// On flat ground (all zero) R = I, n_z = 1 and h = 0: every added term is a product with an exact 0 or 1, so the step gives
// the bits of the flat one.
struct alignas(16) TerrainRec {
  double z0, sx, sy;      // plane
  double x0, y0, dx, dy;  // grid origin and spacing
  double idx, idy;        // 1 / dx, 1 / dy
  int32_t nx, ny;         // grid size, 0 x 0: no grid
  long long off;          // first height of this grid in the set's concatenated heights
};

// Device inputs of the terrain kernel. set == NULL: flat ground z = 0 (one terrain); index [N] (NULL: terrain 0).
struct TerrainArgs {
  const TerrainRec* set; const double* heights; const int32_t* index; int n_terrains;
};

// Per foot k: its contact directions d[k][i] (t1, t2, n in world axes) and its gap phi[k]; per contact row r: the row's
// coefficients [-d' skew(rho) | d | d' L_k] of J_c (9 values).
struct alignas(16) TerrainSmem {
  double d[4][3][3];
  double phi[4];
  double cf[12][9];
};

// The record of one terrain descriptor (host side; heights go to the set's array at offset `off`).
inline TerrainRec terrain_record(const wbc_terrain_desc& t, long long off) {
  const bool grid = t.nx > 0;
  return TerrainRec{t.z0, t.sx, t.sy, t.x0, t.y0, t.dx, t.dy, grid ? 1.0 / t.dx : 0.0, grid ? 1.0 / t.dy : 0.0, t.nx, t.ny, off};
}

// Terrain of robot `inst`, or -1 when its index is out of range.
WBC_DEV int plant_terrain(const TerrainArgs& ta, long long inst) {
  const int k = ta.index ? ta.index[inst] : 0;
  return (k >= 0 && k < ta.n_terrains) ? k : -1;
}

// Clamped grid coordinate along one axis: cell index, fraction in the cell, and whether the direction was clamped. A NaN
// coordinate is clamped to 0 (the robot is frozen as DIVERGED later; the grid read stays in bounds).
WBC_DEV void grid_coord(double c, int n, int& cell, double& frac, bool& clamped) {
  clamped = !(c >= 0.0) || c > n - 1;
  if (!(c >= 0.0)) c = 0.0;
  if (c > n - 1) c = n - 1;
  const int i = (int)floor(c);
  cell = i < n - 2 ? i : n - 2;
  frac = c - cell;
}

// Height and gradient of terrain `tr` at (x, y).
WBC_DEV void terrain_height(const TerrainRec& tr, const double* heights, double x, double y, double& h, double& hx, double& hy) {
  h = tr.z0 + tr.sx * x + tr.sy * y;
  hx = tr.sx; hy = tr.sy;
  if (tr.nx > 0) {
    int i, j; double fu, fw; bool cu, cw;
    grid_coord((x - tr.x0) * tr.idx, tr.nx, i, fu, cu);
    grid_coord((y - tr.y0) * tr.idy, tr.ny, j, fw, cw);
    const double* g = heights + tr.off + (long long)j * tr.nx + i;
    const double h00 = g[0], h10 = g[1], h01 = g[tr.nx], h11 = g[tr.nx + 1];
    const double lo = h00 + fu * (h10 - h00), hi = h01 + fu * (h11 - h01);
    h += lo + fw * (hi - lo);
    if (!cu) hx += ((1.0 - fw) * (h10 - h00) + fw * (h11 - h01)) * tr.idx;
    if (!cw) hy += (hi - lo) * tr.idy;
  }
}

// Contact frame and normal gap of a foot at world position p (see the definition above).
WBC_DEV void terrain_contact(const TerrainRec& tr, const double* heights, V3 p, double (&d)[3][3], double& phi) {
  double h, hx, hy;
  terrain_height(tr, heights, p.x, p.y, h, hx, hy);
  const double in = 1.0 / sqrt(hx * hx + hy * hy + 1.0);
  const V3 n = mk(-hx * in, -hy * in, in);
  const V3 e = mk(1.0 - n.x * n.x, -n.x * n.y, -n.x * n.z);
  const V3 t1 = (1.0 / sqrt(dot(e, e))) * e, t2 = cross(n, t1);
  d[0][0] = t1.x; d[0][1] = t1.y; d[0][2] = t1.z;
  d[1][0] = t2.x; d[1][1] = t2.y; d[1][2] = t2.z;
  d[2][0] = n.x; d[2][1] = n.y; d[2][2] = n.z;
  phi = (p.z - h) * n.z;
}

// PERTURB = false: the unperturbed step (md = the handle's model, a.mu). PERTURB = true: md is the robot's variant and `pt`
// adds its friction, its push and the freeze of a bad variant index; nothing else differs. TERRAIN = true (with PERTURB): the
// contacts are against the robot's terrain of `ta`, with the per-foot frames and gaps in `ts`; a bad terrain index freezes.
template <bool PERTURB = false, bool TERRAIN = false>
WBC_DEV void plant_step_instance(WarpSmem& s, PlantSmem& ps, const wbc_model& md, const PlantArgs& a, long long inst, int lane,
                                 const Perturb& pt = Perturb{}, TerrainSmem* ts = nullptr, const TerrainArgs& ta = TerrainArgs{}) {
  static_assert(!TERRAIN || PERTURB, "the terrain step is a perturbed step");
  constexpr int FREEZE = TERRAIN ? (PLANT_FREEZE | WBC_ST_BADVARIANT | WBC_ST_BADTERRAIN)
                                 : PERTURB ? (PLANT_FREEZE | WBC_ST_BADVARIANT) : PLANT_FREEZE;
  int status = a.ctrl_status ? a.ctrl_status[inst] : 0;
  if (PERTURB && pt.bad_variant) status |= WBC_ST_BADVARIANT;
  int terrain = 0;
  if constexpr (TERRAIN) {
    terrain = plant_terrain(ta, inst);
    if (terrain < 0) status |= WBC_ST_BADTERRAIN;
  }
  for (int i = lane; i < WBC_NQ; i += 32) s.q[i] = a.q[inst * WBC_NQ + i];
  for (int i = lane; i < WBC_NV; i += 32) s.v[i] = a.v[inst * WBC_NV + i];
  if (lane < 12) ps.tauk[lane] = a.tau[inst * WBC_NU + md.act_index[lane]];
  __syncwarp();
  dynamics_phase<DYN_STEP>(s, md, lane, status, nullptr);
  if constexpr (TERRAIN) {
    // ---- lane k < 4: the frame and gap of foot k on its terrain (a bad index is frozen: flat ground will do)
    if (lane < 4) {
      const TerrainRec tr = (ta.set && terrain >= 0) ? ta.set[terrain] : TerrainRec{};
      const V3 pf = mk(s.q[4] + s.rho[lane][0], s.q[5] + s.rho[lane][1], s.q[6] + s.rho[lane][2]);
      terrain_contact(tr, ta.heights, pf, ts->d[lane], ts->phi[lane]);
    }
    __syncwarp();
    // ---- lane r < 12: the coefficients of contact row r = 3 k + i, d' J_k = [-d' skew(rho) | d' | d' L_k] with d = d[k][i]
    if (lane < 12) {
      const int k = lane / 3, i = lane % 3;
      const V3 rh = ld3(s.rho[k]), d = ld3(ts->d[k][i]);
      double* cf = ts->cf[lane];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        cf[c] = d.x * -skew_ent(rh, 0, c) + d.y * -skew_ent(rh, 1, c) + d.z * -skew_ent(rh, 2, c);
        cf[3 + c] = comp(d, c);
        cf[6 + c] = d.x * s.L[k][0][c] + d.y * s.L[k][1][c] + d.z * s.L[k][2][c];
      }
    }
  }
  // ---- M^-1 through the block-arrow structure
  if (lane < 4) {
    const double* d = s.Mleg[lane];
    const double aa = d[0], b = d[1], c = d[2], e = d[3], f = d[4], g = d[5];     // [[a b c],[b e f],[c f g]]
    const double c00 = e * g - f * f, c01 = c * f - b * g, c02 = b * f - c * e;
    const double det = aa * c00 + b * c01 + c * c02, id = 1.0 / det;
    ps.Dinv[lane][0] = c00 * id; ps.Dinv[lane][1] = c01 * id; ps.Dinv[lane][2] = c02 * id;
    ps.Dinv[lane][3] = (aa * g - c * c) * id; ps.Dinv[lane][4] = (b * c - aa * f) * id; ps.Dinv[lane][5] = (aa * e - b * b) * id;
  }
  __syncwarp();
  for (int e = lane; e < 36; e += 32) {
    const int i = e / 6, j = e % 6;
    double acc = s.Mb[j][i];
    for (int k = 0; k < 4; ++k)
      for (int x = 0; x < 3; ++x)
        for (int y = 0; y < 3; ++y) acc = fma(-s.Mb[6 + 3 * k + x][i] * sym3get(ps.Dinv[k], x, y), s.Mb[6 + 3 * k + y][j], acc);
    ps.Sb[i][j] = acc;
  }
  __syncwarp();
  for (int j = 0; j < 6; ++j) {                     // Cholesky of Sb (lower), lanes = rows
    const double dj = ps.Sb[j][j];
    if (!(dj > 1e-300)) status |= WBC_ST_NOTPD;
    const double inv = 1.0 / sqrt(dj > 1e-300 ? dj : 1.0);
    __syncwarp();
    if (lane < 6 && lane >= j) ps.Sb[lane][j] *= inv;
    __syncwarp();
    if (lane < 6 && lane > j)
      for (int k = j + 1; k <= lane; ++k) ps.Sb[lane][k] = fma(-ps.Sb[lane][j], ps.Sb[k][j], ps.Sb[lane][k]);
    __syncwarp();
  }
  // ---- column c = lane < 13 of X = M^-1 [J_c' | B tau - h]
  if (lane < 13) {
    double rb[6], rl[4][3];
    if (TERRAIN && lane < 12) {                     // (d' J_k)' = the row's coefficients
      const int k = lane / 3;
      const double* cf = ts->cf[lane];
#pragma unroll
      for (int c = 0; c < 6; ++c) rb[c] = cf[c];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int x = 0; x < 3; ++x) rl[kk][x] = (kk == k) ? cf[6 + x] : 0.0;
    } else if (lane < 12) {
      const int k = lane / 3, i = lane % 3;
      const V3 rh = ld3(s.rho[k]);
      // J_k = [-skew(rho) | 1 | L_k]  ->  J_k' e_i = [skew(rho) e_i ; e_i ; L_k[i][:]]
#pragma unroll
      for (int c = 0; c < 3; ++c) { rb[c] = -skew_ent(rh, i, c); rb[3 + c] = (c == i) ? 1.0 : 0.0; }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int x = 0; x < 3; ++x) rl[kk][x] = (kk == k) ? s.L[k][i][x] : 0.0;
    } else {
#pragma unroll
      for (int c = 0; c < 6; ++c) rb[c] = -s.hb[c];
      if (PERTURB && pt.push) {                     // generalized force J_p' F of the push: [(R0 r) x F ; F], none on the joints
        const V3 F = ld3(pt.push), r = ld3(pt.push + 3);
        const V3 rw = r.x * ld3(&s.task[7]) + r.y * ld3(&s.task[10]) + r.z * ld3(&s.task[13]);
        const V3 m = cross(rw, F);
        rb[0] += m.x; rb[1] += m.y; rb[2] += m.z;
        rb[3] += F.x; rb[4] += F.y; rb[5] += F.z;
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int x = 0; x < 3; ++x) rl[kk][x] = ps.tauk[3 * kk + x] - s.hj[3 * kk + x];
    }
    double tl[4][3];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
      for (int x = 0; x < 3; ++x)
        tl[kk][x] = sym3get(ps.Dinv[kk], x, 0) * rl[kk][0] + sym3get(ps.Dinv[kk], x, 1) * rl[kk][1] + sym3get(ps.Dinv[kk], x, 2) * rl[kk][2];
    double xb[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      double acc = rb[i];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int x = 0; x < 3; ++x) acc = fma(-s.Mb[6 + 3 * kk + x][i], tl[kk][x], acc);
      xb[i] = acc;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) {                   // L y = cb
      double acc = xb[i];
#pragma unroll
      for (int k = 0; k < 6; ++k) if (k < i) acc = fma(-ps.Sb[i][k], xb[k], acc);
      xb[i] = acc / ps.Sb[i][i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {                  // L' x = y
      double acc = xb[i];
#pragma unroll
      for (int k = 0; k < 6; ++k) if (k > i) acc = fma(-ps.Sb[k][i], xb[k], acc);
      xb[i] = acc / ps.Sb[i][i];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) ps.X[i][lane] = xb[i];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      double c3[3];
#pragma unroll
      for (int x = 0; x < 3; ++x) {
        double acc = rl[kk][x];
#pragma unroll
        for (int i = 0; i < 6; ++i) acc = fma(-s.Mb[6 + 3 * kk + x][i], xb[i], acc);
        c3[x] = acc;
      }
#pragma unroll
      for (int x = 0; x < 3; ++x)
        ps.X[6 + 3 * kk + x][lane] = sym3get(ps.Dinv[kk], x, 0) * c3[0] + sym3get(ps.Dinv[kk], x, 1) * c3[1] + sym3get(ps.Dinv[kk], x, 2) * c3[2];
    }
  }
  __syncwarp();
  // ---- contact rows: lane r < 12 owns row r = 3 k + i of J_c: A[r][:] = J_r X[:, :12], u_free = J_r (v + dt X[:, 12])
  const int rk = lane < 12 ? lane / 3 : 0, ri = lane < 12 ? lane % 3 : 0;
  double u = 0.0, ainv = 0.0, bias = 0.0;
  if (TERRAIN && lane < 12) {                       // the same chains with the row's coefficients
    const double* cf = ts->cf[lane];
    auto jrow = [&](int c) {
      double val = cf[3] * ps.X[3][c];
      val = fma(cf[4], ps.X[4][c], val);
      val = fma(cf[5], ps.X[5][c], val);
#pragma unroll
      for (int x = 0; x < 3; ++x) val = fma(cf[x], ps.X[x][c], val);
#pragma unroll
      for (int x = 0; x < 3; ++x) val = fma(cf[6 + x], ps.X[6 + 3 * rk + x][c], val);
      return val;
    };
    for (int c = 0; c < 12; ++c) ps.A[lane][c] = jrow(c);
    const double uf = fma(cf[5], s.vf[rk][2], fma(cf[4], s.vf[rk][1], cf[3] * s.vf[rk][0]));   // d' (foot velocity)
    u = fma(a.dt, jrow(12), uf);
    ainv = 1.0 / ps.A[lane][lane];
    if (ri == 2) {
      const double phi = ts->phi[rk];               // gap along the terrain normal
      bias = (phi > 0.0 ? phi : a.erp * phi) / a.dt;
    }
  } else if (lane < 12) {
    const V3 rh = ld3(s.rho[rk]);
    auto jrow = [&](int c) {
      double val = ps.X[3 + ri][c];
#pragma unroll
      for (int x = 0; x < 3; ++x) val = fma(-skew_ent(rh, ri, x), ps.X[x][c], val);
#pragma unroll
      for (int x = 0; x < 3; ++x) val = fma(s.L[rk][ri][x], ps.X[6 + 3 * rk + x][c], val);
      return val;
    };
    for (int c = 0; c < 12; ++c) ps.A[lane][c] = jrow(c);
    u = fma(a.dt, jrow(12), s.vf[rk][ri]);
    ainv = 1.0 / ps.A[lane][lane];
    if (ri == 2) {
      const double phi = s.q[6] + s.rho[rk][2];      // foot height over the ground plane z = 0
      bias = (phi > 0.0 ? phi : a.erp * phi) / a.dt;
    }
  }
  __syncwarp();
  // ---- projected Gauss-Seidel from p = 0: feet in order, normal row first, then the two tangential rows
  double p = 0.0;
  for (int it = 0; it < a.iters; ++it) {
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
      double pn;
      {
        const int r = 3 * k + 2;
        const double pnew = fmax(0.0, p - (u + bias) * ainv);
        const double dl = shfl(pnew - p, r);
        pn = shfl(pnew, r);
        if (lane == r) p = pnew;
        if (lane < 12) u = fma(ps.A[lane][r], dl, u);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int r = 3 * k + i;
        const double lim = (PERTURB ? pt.mu : a.mu) * pn;
        const double pnew = fmin(fmax(p - u * ainv, -lim), lim);
        const double dl = shfl(pnew - p, r);
        if (lane == r) p = pnew;
        if (lane < 12) u = fma(ps.A[lane][r], dl, u);
      }
    }
  }
  if (lane < 12) ps.p[lane] = p;
  __syncwarp();
  // ---- v+ = v + dt X[:, 12] + X[:, :12] p (rows in internal joint order), then q+ = q + dt N(q) v+
  double vn = 0.0;
  int vi = 0;
  if (lane < 18) {
    vi = lane < 6 ? lane : md.v_index[lane - 6];
    double acc = fma(a.dt, ps.X[lane][12], s.v[vi]);
#pragma unroll
    for (int c = 0; c < 12; ++c) acc = fma(ps.X[lane][c], ps.p[c], acc);
    vn = acc;
  }
  const bool finite = __all_sync(WBC_FULL, lane >= 18 || fabs(vn) < 1e6);
  if (!finite) status |= WBC_ST_DIVERGED;
  if (lane == 0 && a.status_or) a.status_or[inst] |= status;
  if (a.metrics) {
    if (lane == 0 && a.err_max) { const double e = a.metrics[inst * WBC_NMETRIC + 1]; if (e > a.err_max[inst]) a.err_max[inst] = e; }
    if (a.metrics_log && lane < WBC_NMETRIC)
      a.metrics_log[((long long)(*a.step_counter) * a.n + inst) * WBC_NMETRIC + lane] = a.metrics[inst * WBC_NMETRIC + lane];
  }
  if constexpr (TERRAIN) {                          // world axes: f_k = R_k p_k / dt
    if (a.f_contact && lane < 12) {
      const double(&d)[3][3] = ts->d[rk];
      const double pw = d[0][ri] * ps.p[3 * rk] + d[1][ri] * ps.p[3 * rk + 1] + d[2][ri] * ps.p[3 * rk + 2];
      a.f_contact[inst * 12 + lane] = (status & FREEZE) ? 0.0 : pw / a.dt;
    }
  } else {
    if (a.f_contact && lane < 12) a.f_contact[inst * 12 + lane] = (status & FREEZE) ? 0.0 : p / a.dt;
  }
  if (lane == 0 && a.t) a.t[inst] += a.dt;
  if (status & FREEZE) return;
  const double wx = shfl(vn, 0), wy = shfl(vn, 1), wz = shfl(vn, 2);
  if (lane < 18) a.v[inst * WBC_NV + vi] = vn;
  if (lane == 0) {
    const double qw = s.q[0], qx = s.q[1], qy = s.q[2], qz = s.q[3];
    const double nw = qw + 0.5 * a.dt * (-wx * qx - wy * qy - wz * qz);
    const double nx = qx + 0.5 * a.dt * (wx * qw + wy * qz - wz * qy);
    const double ny = qy + 0.5 * a.dt * (wy * qw + wz * qx - wx * qz);
    const double nz = qz + 0.5 * a.dt * (wz * qw + wx * qy - wy * qx);
    const double inv = 1.0 / sqrt(nw * nw + nx * nx + ny * ny + nz * nz);
    double* qo = a.q + inst * WBC_NQ;
    qo[0] = nw * inv; qo[1] = nx * inv; qo[2] = ny * inv; qo[3] = nz * inv;
  }
  if (lane >= 3 && lane < 18) a.q[inst * WBC_NQ + 1 + vi] = fma(a.dt, vn, s.q[1 + vi]);   // base position (q 4..6) and joints
  __syncwarp();
}

}  // namespace wbcplant
