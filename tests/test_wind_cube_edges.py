"""Wind model 3 where trilinear interpolation goes wrong: nodes exactly on a cell plane and one ulp either side of it,
nodes outside the cube, non-square and minimal cubes, a cube whose `spacing` is not its grid step, and a cube replaced
between launches.

The cubes and states are built here from exactly representable values (integer grid coordinates, datum and spacing),
so that `yn + datum[0]` lands exactly on a plane.  References:
  * the CPU port (oracle/fg_oracle.c), bit for bit the reference, wherever its cell search and the cell's corners stay
    inside its arrays (port_reads_inside);
  * the torch float64 restatement (oracle/lagrangian_torch.py) everywhere: it implements the clamp the library
    documents for nodes outside the cube (the nearest cell) and the reference's swapped search bounds (the x search
    runs over the cube's second dimension, the y search over its first).
Without a GPU the restatement is checked against the port on every port-safe state used here; on the GPU the kernels
are checked against both: F, G, the summary, J d, J^T lambda and w, through kernel A with 1 and 3 trajectories per
CTA, kernel L (option "kernel" = 2, and ts = 257), the F-only and summary instances and the matrix-free products."""
import numpy as np
import pytest
import torch

import tol_b200 as T
from conftest import ATOL, RTOL, assert_parity, load_golden

import lagrangian_torch as LT

# name -> (shape ne x nn x nu, grid origin, grid step, spacing given to the kernels, datum).  Every grid coordinate is
# within a factor of 2 of its axis' datum, so node coordinate = plane -+ one ulp - datum is exact (Sterbenz) and the
# kernels' `yn + datum[0]` gives back the plane's neighbour exactly
CUBES = {
    "13x7x3": ((13, 7, 3), (100.0, 200.0, 20.0), (10.0, 10.0, 10.0), (10.0, 10.0, 10.0), (150.0, 230.0, 25.0)),
    "5x17x2": ((5, 17, 2), (-48.0, 64.0, 96.0), (8.0, 4.0, 16.0), (8.0, 4.0, 16.0), (-24.0, 100.0, 100.0)),
    "2x2x2": ((2, 2, 2), (64.0, 32.0, 16.0), (64.0, 32.0, 16.0), (64.0, 32.0, 16.0), (96.0, 48.0, 24.0)),
    "spacing!=step": ((6, 6, 4), (1000.0, 2000.0, 40.0), (50.0, 50.0, 25.0), (40.0, 60.0, 25.0), (1100.0, 2100.0, 80.0)),
}
_BASE = {"S10": "S10_tempest_ts100_wind3", "G7": "G7_skywalker_ts45_wind3"}


def cube(name, seed=0):
    shape, org, step, spacing, datum = CUBES[name]
    axes = [o + s * np.arange(k, dtype=np.float64) for o, s, k in zip(org, step, shape)]
    v = np.random.default_rng(seed).uniform(-4.0, 4.0, shape)
    return dict(grid_x=axes[0], grid_y=axes[1], grid_z=axes[2], grid_v=v, grid_datum=np.array(datum),
                grid_spacing=np.array(spacing))


def _mids(a):
    return [0.5 * (a[0] + a[1]), 0.5 * (a[-2] + a[-1])]


def plane_points(c):
    """(xs, ys, zs) in cube coordinates: every axis' first, second, middle and last plane exactly, and one ulp below
    and above each, the other two coordinates at cell midpoints"""
    axes = [c["grid_x"], c["grid_y"], c["grid_z"]]
    pts = []
    for a in range(3):
        planes = sorted({0, 1, len(axes[a]) // 2, len(axes[a]) - 1})
        others = [_mids(axes[b]) for b in range(3) if b != a]
        for p in planes:
            v = axes[a][p]
            for t in (v, np.nextafter(v, -np.inf), np.nextafter(v, np.inf)):
                for k in range(2):
                    q = [others[0][k], others[1][1 - k]]
                    q.insert(a, t)
                    pts.append(q)
    return np.array(pts)


def outside_points(c):
    """beyond the last plane and before the first on each of the six faces (half a step and three steps out), and
    at two opposite corners"""
    axes = [c["grid_x"], c["grid_y"], c["grid_z"]]
    pts = []
    for a in range(3):
        step = axes[a][1] - axes[a][0]
        others = [_mids(axes[b])[0] for b in range(3) if b != a]
        for t in (axes[a][-1] + 0.5 * step, axes[a][-1] + 3 * step, axes[a][0] - 0.5 * step, axes[a][0] - 3 * step):
            q = list(others)
            q.insert(a, t)
            pts.append(q)
    pts.append([ax[-1] + 2 * (ax[1] - ax[0]) for ax in axes])
    pts.append([ax[0] - 2 * (ax[1] - ax[0]) for ax in axes])
    return np.array(pts)


def states(mission, c, pts, B, ts=None, seed=0):
    """B trajectories of ts windows (default: one per point) whose window nodes 0..ts-1 sit on the points (rolled by b
    in trajectory b, tiled when ts exceeds the number of points); node ts keeps the initial guess' position"""
    g = load_golden(_BASE[mission])
    ts = ts or len(pts)
    lm = g["lm"]
    cfg = T.make_config(mission, ts, g["ac"], g["gn"], g["goal_ned"],
                        limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]])
    X = T.synth.batch(T.initial_guess(cfg), 6000 + seed, 0, B)
    d = c["grid_datum"]
    for b in range(B):
        P = np.roll(np.resize(pts, (ts, 3)), b, axis=0)
        N = X[b, 1:].reshape(ts + 1, 11)
        N[:ts, 1], N[:ts, 0], N[:ts, 2] = P[:, 0] - d[0], P[:, 1] - d[1], d[2] - P[:, 2]
        # the cube coordinates the kernels form are the points exactly
        assert (N[:ts, 1] + d[0] == P[:, 0]).all() and (N[:ts, 0] + d[1] == P[:, 1]).all()
        assert (-N[:ts, 2] + d[2] == P[:, 2]).all()
    return g, X


def _port_cell(v, grid, bound, sp):
    """the port's cell search: the first i < bound with v - grid[i] < sp, else bound; None if it reads past grid"""
    for i in range(bound):
        if i >= grid.size:
            return None
        if v - grid[i] < sp:
            return i
    return bound


def port_reads_inside(c, X, ts):
    """True if the port's cell search and corner reads stay inside its arrays for every window node of every row: the
    reference's loops (x over the second dimension, y over the first) and no clamp"""
    ne, nn, nu = c["grid_v"].shape
    sx, sy, sz = c["grid_spacing"]
    d = c["grid_datum"]
    for x in X:
        for xn, yn, zn in x[1:].reshape(ts + 1, 11)[:ts, :3]:
            xi = _port_cell(yn + d[0], c["grid_x"], nn, sx)
            yi = _port_cell(xn + d[1], c["grid_y"], ne, sy)
            zi = _port_cell(-zn + d[2], c["grid_z"], nu, sz)
            if xi is None or yi is None or zi is None or xi > ne - 2 or yi > nn - 2 or zi > nu - 2:
                return False
    return True


class Ref:
    """the restatement's F, G (at the pattern), J d, J^T lambda, w and their term scales, and the port's F and G where
    its reads stay inside the cube"""

    def __init__(self, mission, g, c, X, D, Lam):
        import portclient as P
        ts = (X.shape[1] - 1) // 11 - 1
        gd = dict(g)
        gd.update(c)
        gd["wind_model"] = 3
        o = LT.Problem(gd, ts=ts)
        p = P.PortProblem(mission, ts, g["ac"], g["gn"], g["goal_ned"], 3)
        p.set_wind_grid(c["grid_x"], c["grid_y"], c["grid_z"], c["grid_v"], c["grid_datum"], c["grid_spacing"])
        self.iG, self.jG = p.pattern()
        self.n, self.neF, self.neG, self.nb = p.n, p.neF, p.neG, p.nb
        B = X.shape[0]
        self.F, self.G = np.empty((B, p.neF)), np.empty((B, p.neG))
        self.Y, self.Ya, self.Z, self.Za = np.empty((B, p.neF)), np.empty((B, p.neF)), np.empty((B, p.n)), np.empty((B, p.n))
        self.W, self.Ws = np.empty((B, p.n)), np.empty((B, p.n))
        for b in range(B):
            xt = torch.from_numpy(X[b])
            self.F[b] = o.F(xt).numpy()
            J = o.jacobian(xt).numpy()
            self.G[b] = J[self.iG, self.jG]
            self.Y[b], self.Ya[b] = J @ D[b], np.abs(J) @ np.abs(D[b])
            self.Z[b], self.Za[b] = J.T @ Lam[b], np.abs(J).T @ np.abs(Lam[b])
            self.W[b], self.Ws[b] = o.lag_hess_vec(X[b], Lam[b], D[b]).numpy(), o.term_scale(X[b], Lam[b], D[b]).numpy()
        self.port = None
        if port_reads_inside(c, X, ts):
            Fp, Gp = np.empty((B, p.neF)), np.empty((B, p.neG))
            p.eval_many(X, Fp, Gp)
            if mission == "S10":  # the boundary-row dt entries the reference leaves undefined: 0, as everywhere here
                Gp[:, p.ub_mask()] = 0.0
            self.port = (Fp, Gp)


def _one_node(c, q):
    """a one-window state whose node 0 sits on the point q"""
    d = c["grid_datum"]
    x = np.zeros(1 + 11 * 2)
    x[1 + 1], x[1 + 0], x[1 + 2] = q[0] - d[0], q[1] - d[1], d[2] - q[2]
    return x[None]


def points(c, kind):
    """"planes": the plane points the port can evaluate; "clamped": the outside points and the plane points where the
    port would read outside its arrays (the last planes, and overruns of a swapped search bound), defined by the clamp"""
    pl = plane_points(c)
    safe = np.array([port_reads_inside(c, _one_node(c, q), 1) for q in pl])
    if kind == "planes":
        return pl[safe]
    return np.concatenate([outside_points(c), pl[~safe]])


def _inputs(mission, cname, kind, B=7, ts=None):
    c = cube(cname)
    pts = points(c, kind)
    g, X = states(mission, c, pts, B, ts)
    rng = np.random.default_rng(len(pts))
    n = X.shape[1]
    neF = 1 + 8 * ((n - 1) // 11 - 1) + (12 if mission == "G7" else 11)
    return g, c, X, rng.uniform(-1, 1, (B, n)), rng.uniform(-1, 1, (B, neF))


CASES = [(m, cn, k) for m in ("S10", "G7") for cn in CUBES for k in ("planes", "clamped")]


def _case_id(case):
    return "-".join(case)


# ---- no GPU needed ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_the_restatement_is_the_port_where_the_port_reads_inside_the_cube(case, oracle_built):
    """every plane state is one the port evaluates, and there the restatement's F is within 1e-14 + 1e-12*|ref| of the
    port's and its G within that bar at every pattern position; the clamped points include ones the port cannot
    evaluate"""
    mission, cname, kind = case
    c = cube(cname)
    pts = points(c, kind)
    safe = np.array([port_reads_inside(c, _one_node(c, q), 1) for q in pts])
    if kind == "clamped":
        assert not safe.all()
        return
    assert safe.all() and len(pts) >= 18
    R = _ref(case)[-1]
    assert R.port is not None
    assert_parity(R.F, R.port[0], "restatement F")
    assert_parity(R.G, R.port[1], "restatement G")


# ---- GPU -------------------------------------------------------------------------------------------------------------

def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _nan(B, m):
    return torch.full((B, m), float("nan"), dtype=torch.float64, device="cuda")


def _within(got, ref, scale, what):
    assert np.isfinite(got).all(), what + ": non-finite values"
    e = np.abs(got - ref) - (ATOL + RTOL * scale)
    assert e.max() <= 0, (what, np.unravel_index(e.argmax(), e.shape), e.max())


def _evaluator(mission, g, c, ts, options):
    ev = T.Evaluator(mission, ts, g["ac"], g["gn"], g["goal_ned"], 1)
    ev.set_wind_grid(c["grid_x"], c["grid_y"], c["grid_z"], c["grid_v"], c["grid_datum"], c["grid_spacing"])
    for k, v in options.items():
        ev.set_option(k, v)
    return ev


def _check_fg(ev, R, Xd, what):
    B = Xd.shape[0]
    F, G = _nan(B, R.neF + 2), _nan(B, R.neG + 2)
    ev.eval_batch_device(Xd, F, G)
    F, G = F.cpu().numpy(), G.cpu().numpy()
    assert np.isnan(F[:, R.neF:]).all() and np.isnan(G[:, R.neG:]).all(), what + ": padding"
    F, G = F[:, :R.neF], G[:, :R.neG]
    assert_parity(F, R.F, what + " F (restatement)")
    assert_parity(G, R.G, what + " G (restatement)")
    if R.port is not None:
        assert_parity(F, R.port[0], what + " F (port)")
        assert_parity(G, R.port[1], what + " G (port)")
    return F


def _check_all_paths(mission, g, c, X, D, Lam, R, ts, what, options):
    B = X.shape[0]
    Xd, Dd, Ld = _dev(X), _dev(D), _dev(Lam)
    ev = _evaluator(mission, g, c, ts, options)
    F = _check_fg(ev, R, Xd, what)
    # F-only (kernel A's F-only instances unless kernel L is forced) and the summary with and without G
    F1, G1 = _nan(B, R.neF), _nan(B, R.neG)
    ev.eval_batch_device(Xd, F1, G1, needF=True, needG=False)
    assert np.array_equal(F1.cpu().numpy(), F) and torch.isnan(G1).all(), what + " F-only"
    for needG in (False, True):
        S = _nan(B, 4)
        flags = T.evaluator.DEVICE_PTRS | T.evaluator.NEED_F | (T.evaluator.NEED_G if needG else 0)
        F2, G2 = _nan(B, R.neF), _nan(B, R.neG)
        ev._follow_torch(Xd)
        T.lib.check(ev.L.tolcuda_eval_batch_summary(ev.h, B, Xd.data_ptr(), Xd.stride(0), F2.data_ptr(), F2.stride(0),
                                                    G2.data_ptr(), G2.stride(0), S.data_ptr(), S.stride(0), flags))
        assert np.array_equal(F2.cpu().numpy(), F), what + " summary F"
        S = S.cpu().numpy()
        d = R.F[:, 1:1 + 8 * ts]
        bnd = np.abs(R.F[:, -R.nb:])
        if mission == "G7":
            bnd[:, -1] = np.maximum(R.F[:, -1], 0.0)
        assert_parity(S[:, 0], R.F[:, 0], what + " summary objective")
        assert_parity(S[:, 1], np.abs(d).max(1), what + " summary max |defect|")
        assert_parity(S[:, 2], bnd.max(1), what + " summary max boundary violation")
        assert (np.abs(S[:, 3] - (d * d).sum(1)) <= 1e-12 * (d * d).sum(1)).all(), what + " summary sum of squares"
    # matrix-free products
    Y, Z, W, Zw = _nan(B, R.neF + 2), _nan(B, R.n + 2), _nan(B, R.n + 2), _nan(B, R.n + 2)
    ev.jac_vec(Xd, Dd, Y)
    ev.jac_tvec(Xd, Ld, Z)
    ev.lag_hess_vec(Xd, Ld, Dd, W, Zw)
    Y, Z, W = Y.cpu().numpy(), Z.cpu().numpy(), W.cpu().numpy()
    assert np.isnan(Y[:, R.neF:]).all() and np.isnan(Z[:, R.n:]).all() and np.isnan(W[:, R.n:]).all(), what + ": padding"
    _within(Y[:, :R.neF], R.Y, R.Ya, what + " J d")
    _within(Z[:, :R.n], R.Z, R.Za, what + " J^T lambda")
    _within(W[:, :R.n], R.W, R.Ws, what + " w")
    assert np.array_equal(Zw[:, :R.n].cpu().numpy(), Z[:, :R.n]), what + " z of lag_hess_vec"
    ev.close()


_REFS = {}


def _ref(case, B=7, ts=None):
    key = case + (B, ts)
    if key not in _REFS:
        mission, cname, kind = case
        g, c, X, D, Lam = _inputs(mission, cname, kind, B, ts)
        _REFS[key] = (g, c, X, D, Lam, Ref(mission, g, c, X, D, Lam))
    return _REFS[key]


PATHS = {"A-per1": {"kernel": 0, "per": 1}, "A-per3": {"kernel": 0, "per": 3, "tail_x4": 0}, "L": {"kernel": 2}}


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_edges_against_the_references(case, path):
    """7 trajectories whose window nodes sit on the case's points: every output of every instance the path reaches"""
    g, c, X, D, Lam, R = _ref(case)
    ts = (X.shape[1] - 1) // 11 - 1
    _check_all_paths(case[0], g, c, X, D, Lam, R, ts, "%s %s" % (_case_id(case), path), PATHS[path])


@pytest.mark.gpu
@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_edges_through_kernel_l_at_257_windows(mission):
    """ts = 257 (kernel L by the dispatcher's own choice): plane and outside points tiled over the trajectory"""
    c = cube("5x17x2")
    pts = np.concatenate([plane_points(c), outside_points(c)])
    g, X = states(mission, c, pts, 3, ts=257)
    rng = np.random.default_rng(257)
    D, Lam = rng.uniform(-1, 1, X.shape), rng.uniform(-1, 1, (3, 1 + 8 * 257 + (12 if mission == "G7" else 11)))
    R = Ref(mission, g, c, X, D, Lam)
    _check_all_paths(mission, g, c, X, D, Lam, R, 257, "%s ts=257" % mission, {})


@pytest.mark.gpu
def test_replacing_the_cube_between_launches():
    """launches enqueued without a synchronisation on cube A, tolcuda_set_wind_grid with a cube of another shape,
    launches again: the first results are cube A's, the second cube B's"""
    mission = "S10"
    ca, cb = cube("13x7x3", seed=1), cube("5x17x2", seed=2)
    pts = np.concatenate([plane_points(ca)[:20], outside_points(ca)[:10]])
    g, X = states(mission, ca, pts, 5)
    ts = len(pts)
    zD, zL = np.zeros(X.shape), np.zeros((5, 1 + 8 * ts + 11))
    Ra, Rb = Ref(mission, g, ca, X, zD, zL), Ref(mission, g, cb, X, zD, zL)
    assert not np.array_equal(Ra.F, Rb.F)
    ev = _evaluator(mission, g, ca, ts, {})
    Xd = _dev(X)
    out = []
    for _ in range(2):
        F, G = _nan(5, Ra.neF), _nan(5, Ra.neG)
        ev.eval_batch_device(Xd, F, G, sync=False)
        out.append((F, G))
    ev.set_wind_grid(cb["grid_x"], cb["grid_y"], cb["grid_z"], cb["grid_v"], cb["grid_datum"], cb["grid_spacing"])
    F, G = _nan(5, Ra.neF), _nan(5, Ra.neG)
    ev.eval_batch_device(Xd, F, G, sync=False)
    ev.synchronize()
    for Fa, Ga in out:
        assert_parity(Fa.cpu().numpy(), Ra.F, "cube A F")
        assert_parity(Ga.cpu().numpy(), Ra.G, "cube A G")
    assert_parity(F.cpu().numpy(), Rb.F, "cube B F")
    assert_parity(G.cpu().numpy(), Rb.G, "cube B G")
    ev.close()
