"""TEST INFRASTRUCTURE ONLY: a torch float64 restatement of the problem's F (S10 and G7; wind models 0, 1 and 3, the
wind cube's trilinear interpolation included), so that second derivatives of the Jacobian can be formed with
torch.func.  Used by tests/test_lagrangian_hessian.py; the product package never imports it.

What G is a derivative of.  The reference's G (oracle/fg_oracle.c, compute_g) is the Jacobian of F with three
exceptions, which the restatement keeps so that `jacobian` reproduces G exactly:
  * G7's objective row is the gradient of 1/2 kT sum T^2 + kp ts dt / dist, where F[0] uses kv (sic, fg_kernels.cu
    traj_epilogue);
  * G7's boundary row 11 (dist - dmax) has the gradient of dist alone: the node-0 derivative of dmax is left out;
  * the wind and its gradient enter G as constants: under wind models 1 and 3 the defect rows have no entries for the
    wind's own dependence on the node position (F1 has no z entry, for instance).
F_tilde(y; W) below is F with G7's rows 0 and 11 replaced as stated and the wind quantities W taken as arguments, so
G(x) = d/dy F_tilde(y; W(x)) at y = x.  The Hessian-of-the-Lagrangian product the library computes is the
derivative of G's entries as functions of x (wind included):
    w = D_x[ G(x)^T lambda ] d,
which is the Hessian of lambda^T F_tilde times d under wind model 0, and not symmetric under models 1 and 3."""
import math

import numpy as np
import torch
from torch.func import jacfwd, jvp, vjp, vmap

PX, PF = 11, 8
G_ACC, RHO = 9.81, 1.2682


class Problem:
    """from a golden fixture (tests/golden/*.npz); wind_model overrides the fixture's (0, 1; 3 needs its cube), ts its
    number of windows"""

    def __init__(self, g, wind_model=None, ts=None):
        self.mission = str(g["mission"])
        self.ts = int(g["ts"]) if ts is None else int(ts)
        ac, gn, goal = g["ac"], g["gn"], g["goal_ned"]
        self.mm, self.SS, self.ee, self.AR, self.Cd0 = (float(ac[i]) for i in (0, 2, 3, 4, 5))
        self.kT, self.kp, self.kv, self.kdt = float(gn[0]), float(gn[1]), float(gn[2]), float(gn[4])
        self.xg, self.yg, self.rg = float(goal[0]), float(goal[1]), float(goal[3])
        self.chi_d = math.atan2(self.yg - 0.0, self.xg - 0.0) if self.mission == "G7" else 0.0
        self.wind = int(g["wind_model"]) if wind_model is None else int(wind_model)
        self.nb = 12 if self.mission == "G7" else 11
        self.n = 1 + PX * (self.ts + 1)
        self.neF = 1 + PF * self.ts + self.nb
        if self.wind == 3:
            t = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64))
            self.gx, self.gy, self.gz, self.gv = t(g["grid_x"]), t(g["grid_y"]), t(g["grid_z"]), t(g["grid_v"])
            self.datum = [float(v) for v in g["grid_datum"]]
            self.spacing = [float(v) for v in g["grid_spacing"]]

    # ---- wind: (Wx, dWx/dx, dWx/dy, dWx/dz) in NED at nodes N[..., 11] (src/problem.cpp:475-695) ----
    def wind_at(self, N):
        z = N[..., 2]
        zero = torch.zeros_like(z)
        if self.wind == 0:
            return zero, zero, zero, zero
        if self.wind == 1:
            Vref, href = 2.4, 10.0
            return -Vref * (-z) / href, zero, zero, zero - (-Vref / href)
        return self._cube(N[..., 0], N[..., 1], z)

    def _cube(self, xn, yn, zn):
        xs, ys, zs = yn + self.datum[0], xn + self.datum[1], -zn + self.datum[2]
        dx, dy, dz = self.spacing
        ne, nn, nu = self.gv.shape

        def search(v, grid, lim, sp, cap):  # first index with v - grid < spacing, among the first `lim`; values only
            hit = (v.detach()[..., None] - grid[:lim]) < sp
            i = torch.where(hit.any(-1), hit.to(torch.int64).argmax(-1), torch.full_like(v, lim, dtype=torch.int64))
            return torch.clamp(i, max=cap)
        xi = search(xs, self.gx, nn, dx, ne - 2)  # (sic) bounded by the second dimension, as the reference
        yi = search(ys, self.gy, ne, dy, nn - 2)
        zi = search(zs, self.gz, nu, dz, nu - 2)
        V = self.gv
        vc = [V[xi, yi, zi], V[xi + 1, yi, zi], V[xi, yi + 1, zi], V[xi + 1, yi + 1, zi],
              V[xi, yi, zi + 1], V[xi + 1, yi, zi + 1], V[xi, yi + 1, zi + 1], V[xi + 1, yi + 1, zi + 1]]
        xrel, yrel, zrel = xs - self.gx[xi], ys - self.gy[yi], zs - self.gz[zi]
        zeta, eta, mu = xrel / dx, yrel / dy, zrel / dz
        N = [(1 - zeta) * (1 - eta) * (1 - mu), zeta * (1 - eta) * (1 - mu), (1 - zeta) * eta * (1 - mu),
             zeta * eta * (1 - mu), (1 - zeta) * (1 - eta) * mu, zeta * (1 - eta) * mu, (1 - zeta) * eta * mu,
             zeta * eta * mu]
        NX = [-((eta - 1.0) * (mu - 1.0)) / dx, ((eta - 1.0) * (mu - 1.0)) / dx, (yrel * (mu - 1.0)) / (dx * dy),
              -(yrel * (mu - 1.0)) / (dx * dy), (zrel * (eta - 1.0)) / (dx * dz), -(zrel * (eta - 1.0)) / (dx * dz),
              -(yrel * zrel) / (dx * dy * dz), (yrel * zrel) / (dx * dy * dz)]
        NY = [-((zeta - 1.0) * (mu - 1.0)) / dy, (xrel * (mu - 1.0)) / (dx * dy), ((zeta - 1.0) * (mu - 1.0)) / dy,
              -(xrel * (mu - 1.0)) / (dx * dy), (zrel * (zeta - 1.0)) / (dy * dz), -(xrel * zrel) / (dx * dy * dz),
              -(zrel * (zeta - 1.0)) / (dy * dz), (xrel * zrel) / (dx * dy * dz)]
        NZ = [-((zeta - 1.0) * (eta - 1.0)) / dz, (xrel * (eta - 1.0)) / (dx * dz), (yrel * (zeta - 1.0)) / (dy * dz),
              -(xrel * yrel) / (dx * dy * dz), ((zeta - 1.0) * (eta - 1.0)) / dz, -(xrel * (eta - 1.0)) / (dx * dz),
              -(yrel * (zeta - 1.0)) / (dy * dz), (xrel * yrel) / (dx * dy * dz)]
        v = dvx = dvy = dvz = 0.0
        for i in range(8):
            v, dvx, dvy, dvz = v + N[i] * vc[i], dvx + NX[i] * vc[i], dvy + NY[i] * vc[i], dvz + NZ[i] * vc[i]
        return v, dvy, dvx, -dvz  # NED <- ENU: Wx = v, dWx/dx = dv/dy, dWx/dy = dv/dx, dWx/dz = -dv/dz

    # ---- the 8 defects of windows (s0, s1 [..., 11]) with wind W at s0, src/problem.cpp:929-1021 ----
    def defects(self, dt, s0, s1, W):
        Wx, Wxx, Wxy, Wxz = W
        Va, gam, chi, phi, CL = s0[..., 3], s0[..., 4], s0[..., 5], s0[..., 6], s0[..., 7]
        dphi, dCL, T = s0[..., 8], s0[..., 9], s0[..., 10]
        cc, sc, cg, sg, cp, sp = torch.cos(chi), torch.sin(chi), torch.cos(gam), torch.sin(gam), torch.cos(phi), torch.sin(phi)
        vx, vy, vz = Wx + Va * cc * cg, 0.0 + Va * cg * sc, 0.0 - Va * sg
        ax, ay, az = Wxx * cc * cg, Wxy * cc * cg, Wxz * cc * cg
        bx, by, bz = Wxx * cc * sg, Wxy * cc * sg, Wxz * cc * sg
        cx, cy, cz = -(Wxx * sc), -(Wxy * sc), -(Wxz * sc)
        mm, rho, SS = self.mm, RHO, self.SS
        dx3 = (T / mm - vy * ay - vz * az - vx * ax - G_ACC * sg
               - (rho * SS * Va * Va * (self.Cd0 + CL * CL / (self.AR * math.pi * self.ee))) / (2.0 * mm))
        dx4 = (vx * bx + vy * by + vz * bz - G_ACC * cg + (CL * rho * SS * Va * Va * cp) / (2 * mm)) / Va
        dx5 = -(vz * cz + cx * vx + vy * cy - (CL * rho * SS * Va * Va * sp) / (2.0 * mm)) / (Va * cg)
        rates = [vx, vy, vz, dx3, dx4, dx5, dphi, dCL]
        return torch.stack([s1[..., s] - rates[s] * dt - s0[..., s] for s in range(PF)], -1)

    def _nodes(self, x):
        return x[1:].reshape(self.ts + 1, PX)

    def _ends(self, x):
        """G7 objective and boundary rows of node 0 / node ts"""
        N = self._nodes(x)
        xf, x0, yf, y0 = N[-1, 0], N[0, 0], N[-1, 1], N[0, 1]
        return xf, x0, yf, y0, torch.sqrt((xf - x0) * (xf - x0) + (yf - y0) * (yf - y0))

    def F(self, x):
        """F as the reference computes it (oracle/fg_oracle.c), in F order"""
        return self._F(x, self.wind_at(self._nodes(x)[:-1]), tilde=False)

    def F_tilde(self, y, W):
        """F with G7's rows 0 and 11 as G differentiates them, the wind quantities W given (module docstring)"""
        return self._F(y, W, tilde=True)

    def _F(self, x, W, tilde):
        N, dt, ts = self._nodes(x), x[0], self.ts
        f = self.defects(dt, N[:-1], N[1:], W).reshape(-1)
        T2 = (N[:, 10] * N[:, 10]).sum()
        if self.mission == "S10":
            r = torch.sqrt((N[:, 0] - self.xg) * (N[:, 0] - self.xg) + (N[:, 1] - self.yg) * (N[:, 1] - self.yg))
            f0 = 0.5 * self.kT * T2 + 0.5 * self.kp * ((r - self.rg) * (r - self.rg)).sum() + self.kdt * dt
            bnd = N[-1] - N[0] - torch.tensor([0.0] * 5 + [2.0 * math.pi] + [0.0] * 5, dtype=x.dtype)
        else:
            xf, x0, yf, y0, dist = self._ends(x)
            f0 = self.kT * 0.5 * T2 + (self.kp if tilde else self.kv) * ts * dt / dist
            dmax = torch.sqrt((self.xg - x0) * (self.xg - x0) + (self.yg - y0) * (self.yg - y0))
            if tilde:
                dmax = dmax.detach()
            bnd = torch.cat([torch.stack([xf - x0 - dist * math.cos(self.chi_d), yf - y0 - dist * math.sin(self.chi_d)]),
                             N[-1, 2:] - N[0, 2:], (dist - dmax)[None]])
        return torch.cat([f0[None], f, bnd])

    # ---- derived quantities ----
    def jacobian(self, x):
        """dense J = G(x) [neF, n] (the Jacobian of F_tilde with the wind held at W(x))"""
        x = torch.as_tensor(x, dtype=torch.float64)
        W = self.wind_at(self._nodes(x)[:-1])
        return jacfwd(lambda y: self.F_tilde(y, W))(x)

    def jt_lambda(self, x, lam):
        """G(x)^T lambda"""
        W = self.wind_at(self._nodes(x)[:-1])
        return vjp(lambda y: self.F_tilde(y, W), x)[1](lam)[0]

    def lag_hess_vec(self, x, lam, d):
        """w = D_x[G(x)^T lambda] d"""
        x, lam, d = (torch.as_tensor(a, dtype=torch.float64) for a in (x, lam, d))
        return jvp(lambda xx: self.jt_lambda(xx, lam), (x,), (d,))[1]

    def term_scale(self, x, lam, d):
        """sum_i sum_l |lambda_i dG_ij/dx_l d_l| for every column j: from per-window derivatives of each window's
        Jacobian block (functions of dt, node k and node k+1), plus the objective and boundary rows"""
        x, lam, d = (torch.as_tensor(a, dtype=torch.float64) for a in (x, lam, d))
        ts, N, Nd = self.ts, self._nodes(x), self._nodes(d)
        u = torch.cat([x[0].expand(ts, 1), N[:-1], N[1:]], 1)        # [ts, 23]: dt, node k, node k+1
        du = torch.cat([d[0].expand(ts, 1), Nd[:-1], Nd[1:]], 1)

        # the windows are independent, so one tangent that is e_j in every window gives column j of every window's
        # block at once: 23 tangents for the blocks, 23 x 23 for their derivatives (wind included)
        basis = torch.eye(23, dtype=torch.float64)[:, None, :].expand(23, ts, 23)

        def blocks(v):  # [ts, 23] -> G's blocks [ts, 8, 23], the wind held at its value at v
            Wv = self.wind_at(v[:, 1:12])
            f = lambda vv: self.defects(vv[:, 0], vv[:, 1:12], vv[:, 12:23], Wv)
            return vmap(lambda t: jvp(f, (v,), (t,))[1])(basis).permute(1, 2, 0)
        Tw = vmap(lambda t: jvp(blocks, (u,), (t,))[1])(basis).permute(1, 2, 3, 0)   # [ts, 8, 23, 23]
        lw = lam[1:1 + PF * ts].reshape(ts, PF)
        terms = (lw[:, :, None, None] * Tw * du[:, None, None, :]).abs().sum((1, 3))   # [ts, 23]
        out = torch.zeros(self.n, dtype=torch.float64)
        out[0] += terms[:, 0].sum()
        idx = 1 + PX * torch.arange(ts)[:, None] + torch.arange(PX)[None, :]
        out.index_add_(0, idx.reshape(-1), terms[:, 1:12].reshape(-1))
        out.index_add_(0, (idx + PX).reshape(-1), terms[:, 12:23].reshape(-1))
        # objective and boundary rows: F[0] is a sum of per-node functions of (x, y, T) (plus, for G7, a function of
        # dt and the end nodes' (x, y)); S10's boundary rows are linear, G7's rows 0, 1 and 11 functions of the ends
        def node_cost(v):
            c = 0.5 * self.kT * v[2] * v[2]
            if self.mission == "S10":
                r = torch.sqrt((v[0] - self.xg) * (v[0] - self.xg) + (v[1] - self.yg) * (v[1] - self.yg))
                c = c + 0.5 * self.kp * (r - self.rg) * (r - self.rg)
            return c
        sel = torch.tensor([0, 1, 10])
        Hn = vmap(jacfwd(jacfwd(node_cost)))(N[:, sel])               # [ts+1, 3, 3]
        tn = (lam[0] * Hn * Nd[:, sel][:, None, :]).abs().sum(2)     # [ts+1, 3]
        out.index_add_(0, (1 + PX * torch.arange(ts + 1)[:, None] + sel[None, :]).reshape(-1), tn.reshape(-1))
        if self.mission == "G7":
            def ends(e):  # e = dt, x0, y0, xf, yf -> the dist term of row 0, boundary rows 0, 1, 11
                dist = torch.sqrt((e[3] - e[1]) * (e[3] - e[1]) + (e[4] - e[2]) * (e[4] - e[2]))
                return torch.stack([self.kp * ts * e[0] / dist, e[3] - e[1] - dist * math.cos(self.chi_d),
                                    e[4] - e[2] - dist * math.sin(self.chi_d), dist])
            ce = torch.tensor([0, 1, 2, 1 + PX * ts, 2 + PX * ts])
            le = lam[torch.tensor([0, self.neF - 12, self.neF - 11, self.neF - 1])]
            He = jacfwd(jacfwd(ends))(x[ce])                          # [4, 5, 5]
            out.index_add_(0, ce, (le[:, None, None] * He * d[ce][None, None, :]).abs().sum((0, 2)))
        return out
