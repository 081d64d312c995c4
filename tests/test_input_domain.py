"""States across the whole bound box, and non-finite inputs, through every kernel path.

The other parity tests feed perturbations of x0 (synth.perturb), which keep gamma, z, phidot and CLdot within 0.01 of 0
and |chi| below 7.  Here:

  * box_states draws trajectories from the bounds SNOPT searches (tolcuda_problem_bounds): bounded coordinates uniform
    within their bounds or exactly on a face, unbounded ones at explicit magnitudes (|x|, |y| up to 1e4 and 1e6, z in
    [-5e3, 0], chi from whole turns up to the node-0 bound 1.745e18, where sincos takes its large-argument path), node
    0's T capped at Tmax.  Without a GPU: the states lie in the box, reach every face and every chi regime, and do not
    depend on sharding; the torch restatement (oracle/lagrangian_torch.py) is pinned to the port on them.
  * On the GPU, S10 and G7 at ts 1, 33, 100, 200 and 257 under wind models 0, 1 and 3 (positions strictly inside the
    fixture cube), through kernel A (per 1 and 3) and kernel L: F+G, F only, the summary, compact rows, the goal
    table, J d, J^T lambda and w, against the port (F with the one-ulp-of-state allowance on defect rows, G with
    1e-14 + 1e-12*|ref|), products formed from the port's G (per entry, against the sum of |terms|) and the
    restatement.
  * Non-finite inputs (singular states at node 0, an interior node and node ts; NaN in every component of those nodes
    and in dt; +-inf in Va, chi and T) interleaved with good rows: every good row keeps its bits (per 1..4, kernel L);
    the kernel is finite and within the bar where the port is finite and non-finite where the port is, but for the
    entries of _exceptions (terms of zero wind gradients the kernels leave out); the summary is what numpy's
    NaN-propagating reductions give on the kernel's own F.
  * NaN in one coordinate of d or lambda reaches only the product entries the pattern connects to it."""
import functools

import numpy as np
import pytest
import torch

import tol_b200 as T
from conftest import ATOL, RTOL, load_golden
from test_instance_matrix import _BASE, _op_reference

PX, PF = 11, 8
XN, YN, ZN, VA, GAM, CHI, PHI, CL, DPHI, DCL, TT = range(PX)
COMP = ("x", "y", "z", "Va", "gamma", "chi", "phi", "CL", "phidot", "CLdot", "T")
NEED_F, NEED_G, COMPACT_G, DEV = (T.evaluator.NEED_F, T.evaluator.NEED_G, T.evaluator.COMPACT_G,
                                  T.evaluator.DEVICE_PTRS)

# ---- the box generator ----------------------------------------------------------------------------------------------

SEED_BOX = 20290000
UNBOUNDED = 1e19                          # |bound| >= this: no bound (SNOPT's infinity is 1e20)
POS, POS_FAR, Z_LOW = 1e4, 1e6, -5e3      # magnitudes of the unbounded coordinates
FACES = ("inside", "lower", "upper", "mixed")
CHI_REGIMES = ("turns", "1e6", "2^31", "1e15", "bound")


def box_kind(b):
    """(face, chi regime, far) of trajectory b: rows 0..19 hold every face with every chi regime"""
    return FACES[b % 4], CHI_REGIMES[b % 5], b % 3 == 2


def cube_ranges(g):
    """open (lo, hi) of node x, y, z strictly inside the wind cube of fixture g (the port reads past the cube outside)"""
    d = g["grid_datum"]
    return ((g["grid_y"][0] - d[1], g["grid_y"][-1] - d[1]), (g["grid_x"][0] - d[0], g["grid_x"][-1] - d[0]),
            (d[2] - g["grid_z"][-1], d[2] - g["grid_z"][0]))


def box_ranges(cfg, cube=None, far=False):
    """per entry of x: the range drawn from and whether its lower / upper end is a face of the box"""
    xl, xu, _, _ = T.bounds(cfg)
    ts = cfg.ts
    lo, up = xl.copy(), xu.copy()
    Nl, Nu = lo[1:].reshape(ts + 1, PX), up[1:].reshape(ts + 1, PX)
    Nu[0, TT] = Nu[1, TT]  # node 0's T has no upper bound: capped at Tmax
    has_lo, has_up = lo > -UNBOUNDED, up < UNBOUNDED
    R = POS_FAR if far else POS
    for c, a, b in ((XN, -R, R), (YN, -R, R), (ZN, Z_LOW, 0.0)):
        Nl[:, c] = np.where(Nl[:, c] > -UNBOUNDED, Nl[:, c], a)
        Nu[:, c] = np.where(Nu[:, c] < UNBOUNDED, Nu[:, c], b)
    if cube is not None:
        Hl, Hu = has_lo[1:].reshape(ts + 1, PX), has_up[1:].reshape(ts + 1, PX)
        for c, (a, b) in zip((XN, YN, ZN), cube_ranges(cube)):
            m = 1e-6 * (b - a)
            a, b = a + m, b - m
            free = Nl[1:, c] != Nu[1:, c]  # node 0's position is fixed at the origin
            Hl[1:, c] &= ~free | (Nl[1:, c] > a)
            Hu[1:, c] &= ~free | (Nu[1:, c] < b)
            Nl[1:, c], Nu[1:, c] = np.maximum(Nl[1:, c], a), np.minimum(Nu[1:, c], b)
    return xl, xu, lo, up, has_lo, has_up


def _chi(rng, regime, b, ts, bound):
    s = rng.choice([-1.0, 1.0], ts + 1)
    if regime == "turns":  # whole turns, half of them exactly
        k = rng.integers(0, 101, ts + 1)
        chi = s * 2.0 * np.pi * k + np.where(rng.uniform(0, 1, ts + 1) < 0.5, 0.0, rng.uniform(-np.pi, np.pi, ts + 1))
    elif regime == "1e6":
        chi = s * 1e6 * rng.uniform(0.5, 1.5, ts + 1)
    elif regime == "2^31":
        chi = s * (2.0 ** 31 + rng.uniform(-64, 64, ts + 1))
    elif regime == "1e15":
        chi = s * 1e15 * rng.uniform(0.5, 1.5, ts + 1)
    else:  # node 0 on its bound, + and - in turn; the other nodes up to it
        chi = s * bound * rng.uniform(0.5, 1.0, ts + 1)
        chi[0] = bound if (b // 5) % 2 == 0 else -bound
    return chi


def box_states(cfg, b0, b1, cube=None, seed=SEED_BOX):
    """trajectories b0..b1-1 of the box batch [b1-b0, n]; row b from numpy.random.Generator(PCG64(seed + b)) alone, so
    any sharding gives the same rows.  cube: the fixture whose wind cube must strictly contain every node"""
    ts = cfg.ts
    out = np.empty((b1 - b0, 1 + PX * (ts + 1)))
    for b in range(b0, b1):
        face, regime, far = box_kind(b)
        _, xu, lo, up, has_lo, has_up = box_ranges(cfg, cube, far and cube is None)
        rng = np.random.Generator(np.random.PCG64(seed + b))
        n = lo.size
        x = lo + (up - lo) * rng.uniform(0.0, 1.0, n)
        side = {"inside": np.full(n, 2), "lower": np.zeros(n, int), "upper": np.ones(n, int),
                "mixed": rng.integers(0, 3, n)}[face]
        x = np.where((side == 0) & has_lo, lo, x)
        x = np.where((side == 1) & has_up, up, x)
        x[1 + CHI::PX] = _chi(rng, regime, b, ts, xu[1 + CHI])
        out[b - b0] = x
    return out


def _config(mission, ts):
    g = load_golden(_BASE[mission])
    lm = g["lm"]
    return g, T.make_config(mission, ts, g["ac"], g["gn"], g["goal_ned"],
                            limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]])


def _port(g, mission, ts, wind, goal=None):
    import portclient as P
    p = P.PortProblem(mission, ts, g["ac"], g["gn"], g["goal_ned"] if goal is None else goal, 1 if wind == 3 else wind)
    if wind == 3:
        p.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
    return p


def _port_rows(p, X):
    F, G = np.empty((X.shape[0], p.neF)), np.empty((X.shape[0], p.neG))
    with np.errstate(all="ignore"):
        for b in range(X.shape[0]):
            F[b], G[b] = p.eval(X[b])
    if p.mission == "S10":
        G[:, p.ub_mask()] = 0.0  # left undefined by the reference, 0 in the kernels
    return F, G


def _f_tol(X, Fr, ts):
    """per-entry bar of F: 1e-14 + 1e-12*|ref|, plus one ulp of the larger of its two states on the defect rows (the
    documented cancellation allowance, test_gpu_parity.py::_assert_parity_F_with_cancellation_bound)"""
    tol = ATOL + RTOL * np.abs(Fr)
    N = np.nan_to_num(X[:, 1:].reshape(X.shape[0], ts + 1, PX), nan=0.0, posinf=0.0, neginf=0.0)
    scale = np.maximum(np.abs(N[:, :-1, :PF]), np.abs(N[:, 1:, :PF])).reshape(X.shape[0], -1)
    tol[:, 1:1 + PF * ts] += np.spacing(scale)
    return tol


def _misses(got, ref, tol, rows, what):
    """entries of finite ref that are non-finite in got or outside tol, reported with their trajectory"""
    with np.errstate(invalid="ignore"):
        bad = ~np.isfinite(got) | (np.abs(got - ref) > tol)
    out = []
    for b, i in zip(*np.nonzero(bad)):
        out.append("%s row %d (%s) entry %d: got %r ref %r tol %.3g" % (what, b, rows[b], i, got[b, i], ref[b, i],
                                                                       tol[b, i]))
    return out


# ---- no GPU needed ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mission", ["S10", "G7"])
@pytest.mark.parametrize("ts", [1, 33])
@pytest.mark.parametrize("cube", [False, True], ids=["free", "cube"])
def test_box_states_cover_the_box(mission, ts, cube):
    """every state lies in the bounds (and strictly inside the cube where asked), every face of every bounded entry
    occurs, and every chi regime occurs: whole turns (some exact), ~1e6, ~2^31, ~1e15 and node 0 on +-1.745e18"""
    g, cfg = _config(mission, ts)
    B = 40
    X = box_states(cfg, 0, B, g if cube else None)
    xl, xu, lo, up, has_lo, has_up = box_ranges(cfg, g if cube else None)
    assert np.isfinite(X).all() and (X >= xl).all() and (X <= xu).all()
    free = lo != up
    for face, has in ((lo, has_lo & free), (up, has_up & free)):
        hit = (X == face).any(axis=0)
        assert hit[has].all(), ("faces never reached at entries", np.nonzero(has & ~hit)[0][:10])
    N = X[:, 1:].reshape(B, ts + 1, PX)
    if cube:
        for c, (a, b) in zip((XN, YN, ZN), cube_ranges(g)):
            assert (N[..., c] > a).all() and (N[..., c] < b).all()
    else:
        assert np.abs(N[..., :2]).max() > POS and np.abs(N[..., :2]).max() <= POS_FAR
        assert N[..., ZN].min() >= Z_LOW and N[..., ZN].max() == 0.0
    assert (N[:, 0, TT] <= N[:, 1, TT].max()).all() and (N[:, 0, TT] == up[1 + TT]).any()
    chi, bound = np.abs(N[..., CHI]), xu[1 + CHI]
    assert bound == 1.7453292519943296e18 or bound == 1e20 * np.pi / 180.0
    assert set(N[:, 0, CHI][N[:, 0, CHI] ** 2 == bound ** 2]) == {bound, -bound}
    turns = chi[chi <= 2 * np.pi * 100 + np.pi]
    assert turns.size and (turns[turns > 0] == 2 * np.pi * np.round(turns[turns > 0] / (2 * np.pi))).any()
    for a, b in ((5e5, 1.5e6), (2.0 ** 31 - 64, 2.0 ** 31 + 64), (5e14, 1.5e15), (bound / 2, bound)):
        assert ((chi >= a) & (chi <= b)).any(), (a, b)


def test_box_states_do_not_depend_on_sharding():
    g, cfg = _config("G7", 33)
    for cube in (None, g):
        X = box_states(cfg, 0, 23, cube)
        assert np.array_equal(np.concatenate([box_states(cfg, 0, 5, cube), box_states(cfg, 5, 17, cube),
                                              box_states(cfg, 17, 23, cube)]), X)
        assert np.array_equal(box_states(cfg, 7, 8, cube)[0], X[7])


@pytest.mark.parametrize("mission", ["S10", "G7"])
@pytest.mark.parametrize("wind", [0, 1, 3])
@pytest.mark.parametrize("ts", [1, 33])
def test_restatement_is_pinned_to_the_port_on_box_states(mission, wind, ts, oracle_built):
    """the torch restatement (the reference w is checked against) on box states: F within the bar of the port (with
    the defect rows' one-ulp-of-state allowance), the Jacobian of F_tilde within 1e-14 + 1e-12*|ref| of the port's
    G at every pattern position and exactly 0 off the pattern"""
    import lagrangian_torch as LT
    g, cfg = _config(mission, ts)
    p, o = _port(g, mission, ts, wind), LT.Problem(g, wind_model=wind, ts=ts)
    iG, jG = p.pattern()
    X = box_states(cfg, 0, 20, g if wind == 3 else None)
    Fr, Gr = _port_rows(p, X)
    rows = [box_kind(b) for b in range(X.shape[0])]
    F, J = np.empty_like(Fr), np.empty((X.shape[0], p.neF, p.n))
    for b, x in enumerate(X):
        xt = torch.from_numpy(x)
        F[b], J[b] = o.F(xt).numpy(), o.jacobian(xt).numpy()
    miss = _misses(F, Fr, _f_tol(X, Fr, ts), rows, "F")
    miss += _misses(J[:, iG, jG], Gr, ATOL + RTOL * np.abs(Gr), rows, "G")
    assert not miss, "%d misses: %s" % (len(miss), miss[:10])
    J[:, iG, jG] = 0.0
    assert not J.any()


# ---- GPU: the paths ------------------------------------------------------------------------------------------------

PAD = 3


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _nan(B, m):
    return torch.full((B, m), float("nan"), dtype=torch.float64, device="cuda")


class _Ctx:
    """one (mission, ts, wind): the context, the port and the pattern"""

    def __init__(self, mission, ts, wind):
        self.g, self.cfg = _config(mission, ts)
        self.mission, self.ts, self.wind = mission, ts, wind
        g = self.g
        self.ev = T.Evaluator(mission, ts, g["ac"], g["gn"], g["goal_ned"], 1 if wind == 3 else wind)
        if wind == 3:
            self.ev.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
        self.port = _port(g, mission, ts, wind)
        p = self.port
        self.n, self.neF, self.neG, self.nb = p.n, p.neF, p.neG, p.nb
        self.iG, self.jG = p.pattern()
        self._lt = None

    def restatement(self):
        import lagrangian_torch as LT
        if self._lt is None:
            self._lt = LT.Problem(self.g, wind_model=self.wind, ts=self.ts)
        return self._lt

    def configs(self):
        """(name, kernel, per): kernel A one trajectory per CTA and runs of 3, kernel L; kernel L alone above 256"""
        if self.ts > 256:
            return [("L", 0, 0)]
        return [("A per1", 0, 1), ("A per3", 0, 3), ("L", 2, 0)]

    def run(self, X, D, Lam, kernel, per, goals=None):
        """every path on X: F+G, F only, summary (with F+G, with F only, alone), compact rows, the goal table
        (F+G+summary), J d, J^T lambda, w with z.  Padding columns must stay NaN."""
        ev, B, n, neF, neG = self.ev, X.shape[0], self.n, self.neF, self.neG
        ev.set_option("kernel", kernel)
        ev.set_option("per", per)
        ev.set_option("tail_x4", 0)
        L, Xd = ev.L, _dev(X)
        ev._follow_torch(Xd)
        ptr = lambda t: None if t is None else t.data_ptr()
        ld = lambda t: 0 if t is None else t.stride(0)
        out = {}

        def launch(tag, flags, glen=neG, summary=False, goal_table=False):
            F = _nan(B, neF + PAD) if flags & NEED_F else None
            G = _nan(B, glen + PAD) if flags & NEED_G else None
            S = _nan(B, 4 + PAD) if summary else None
            if goal_table:
                T.lib.check(L.tolcuda_eval_batch_goals(ev.h, 0, B, Xd.data_ptr(), Xd.stride(0), ptr(F), ld(F), ptr(G),
                                                       ld(G), ptr(S), ld(S), flags | DEV))
            else:
                T.lib.check(L.tolcuda_eval_batch_summary(ev.h, B, Xd.data_ptr(), Xd.stride(0), ptr(F), ld(F), ptr(G),
                                                         ld(G), ptr(S), ld(S), flags | DEV))
            for name, t, m in (("F", F, neF), ("G", G, glen), ("S", S, 4)):
                if t is not None:
                    a = t.cpu().numpy()
                    assert np.isnan(a[:, m:]).all(), "%s: padding of %s written" % (tag, name)
                    out[tag + "." + name] = a[:, :m]

        launch("fg", NEED_F | NEED_G)
        launch("f", NEED_F)
        launch("fgs", NEED_F | NEED_G, summary=True)
        launch("fs", NEED_F, summary=True)
        launch("s", 0, summary=True)
        launch("c", NEED_F | NEED_G | COMPACT_G, glen=ev.compact_len)
        out["c.G"] = T.evaluator.expand_compact_g(self.mission, self.ts, np.ascontiguousarray(out["c.G"]))
        if goals is not None:
            ev.set_goals(goals)
            launch("goal", NEED_F | NEED_G, summary=True, goal_table=True)
            launch("goalf", NEED_F, summary=True, goal_table=True)
        Dd, Ld = _dev(D), _dev(Lam)
        Y, Z, W, Wz = _nan(B, neF + PAD), _nan(B, n + PAD), _nan(B, n + PAD), _nan(B, n + PAD)
        ev.jac_vec(Xd, Dd, Y)
        ev.jac_tvec(Xd, Ld, Z)
        ev.lag_hess_vec(Xd, Ld, Dd, W, Wz)
        for name, t, m in (("Y", Y, neF), ("Z", Z, n), ("W", W, n), ("Wz", Wz, n)):
            a = t.cpu().numpy()
            assert np.isnan(a[:, m:]).all(), "padding of %s written" % name
            out[name] = a[:, :m]
        return out


@functools.lru_cache(maxsize=None)
def _ctx(mission, ts, wind):
    return _Ctx(mission, ts, wind)


def _summary_of(F, nb, mission, ts):
    """[objective, max |defect|, max boundary violation, sum of defect^2] of F rows with numpy's NaN-propagating
    reductions"""
    d = F[:, 1:1 + PF * ts]
    bnd = np.abs(F[:, -nb:])
    if mission == "G7":
        bnd[:, -1] = np.maximum(F[:, -1], 0.0)
    return F[:, 0], np.abs(d).max(axis=1), bnd.max(axis=1), (d * d).sum(axis=1)


def _summary_misses(S, F, c, what, rows):
    """S against _summary_of(F): the objective and both maxima value for value with NaN where numpy has NaN, the sum
    of squares within 1e-12 relative (the kernel sums in another order) and non-finite where numpy's is"""
    obj, dmax, bmax, ssq = _summary_of(F, c.nb, c.mission, c.ts)
    out = []
    for k, ref in ((0, obj), (1, dmax), (2, bmax)):
        for b in np.nonzero(~((S[:, k] == ref) | (np.isnan(S[:, k]) & np.isnan(ref))))[0]:
            out.append("%s summary[%d] row %d (%s): got %r, numpy on the kernel's F %r" % (what, k, b, rows[b], S[b, k],
                                                                                         ref[b]))
    fin = np.isfinite(ssq)
    with np.errstate(invalid="ignore"):
        ok = np.where(fin, np.abs(S[:, 3] - ssq) <= 1e-12 * np.abs(ssq),
                      (np.isnan(ssq) & np.isnan(S[:, 3])) | (S[:, 3] == ssq))
    for b in np.nonzero(~ok)[0]:
        out.append("%s summary[3] row %d (%s): got %r, numpy %r" % (what, b, rows[b], S[b, 3], ssq[b]))
    return out


def _op_refs(c, Gr, D, Lam):
    return _op_reference(c.iG, c.jG, Gr, D, Lam, c.neF, c.n)


def _hvp_refs(c, X, Lam, D):
    o = c.restatement()
    W = np.stack([o.lag_hess_vec(x, lam, d).numpy() for x, lam, d in zip(X, Lam, D)])
    S = np.stack([o.term_scale(x, lam, d).numpy() for x, lam, d in zip(X, Lam, D)])
    return W, S


BOX_TS = (1, 33, 100, 200, 257)
BOX_B = 20


@pytest.mark.gpu
@pytest.mark.parametrize("wind", [0, 1, 3])
@pytest.mark.parametrize("ts", BOX_TS)
@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_box_states_through_every_path(mission, ts, wind):
    """20 box states (every face with every chi regime) through every path and launch configuration: F, G, compact
    rows and the goal table against the port, the summary against numpy on the kernel's F, J d and J^T lambda against
    the port's G, w against the restatement and z bit for bit J^T lambda"""
    c = _ctx(mission, ts, wind)
    X = box_states(c.cfg, 0, BOX_B, c.g if wind == 3 else None)
    rows = ["%s, chi %s%s" % (k[0], k[1], ", far" if k[2] and wind != 3 else "") for k in map(box_kind, range(BOX_B))]
    rng = np.random.default_rng(ts * 10 + wind)
    D, Lam = rng.uniform(-1, 1, (BOX_B, c.n)), rng.uniform(-1, 1, (BOX_B, c.neF))
    goals = T.synth.goals(mission, 0, BOX_B)
    Fr, Gr = _port_rows(c.port, X)
    Fq, Gq = np.empty_like(Fr), np.empty_like(Gr)  # row b with goal b
    for b in range(BOX_B):
        Fq[b:b + 1], Gq[b:b + 1] = _port_rows(_port(c.g, mission, ts, wind, goals[b]), X[b:b + 1])
    assert np.isfinite(Fr).all() and np.isfinite(Gr).all() and np.isfinite(Fq).all() and np.isfinite(Gq).all()
    Yr, Ya, Zr, Za = _op_refs(c, Gr, D, Lam)
    Wr, Ws = _hvp_refs(c, X, Lam, D)
    ftol, gtol = _f_tol(X, Fr, ts), ATOL + RTOL * np.abs(Gr)
    ftolq, gtolq = _f_tol(X, Fq, ts), ATOL + RTOL * np.abs(Gq)
    miss = []
    for name, kernel, per in c.configs():
        o = c.run(X, D, Lam, kernel, per, goals)
        for tag in ("fg", "f", "fgs", "fs", "c"):
            miss += _misses(o[tag + ".F"], Fr, ftol, rows, name + " " + tag + " F")
        for tag in ("fg", "fgs", "c"):
            miss += _misses(o[tag + ".G"], Gr, gtol, rows, name + " " + tag + " G")
        miss += _misses(o["goal.F"], Fq, ftolq, rows, name + " goal F")
        miss += _misses(o["goalf.F"], Fq, ftolq, rows, name + " goal F-only F")
        miss += _misses(o["goal.G"], Gq, gtolq, rows, name + " goal G")
        for tag, ftag in (("fgs", "fgs"), ("fs", "fs"), ("s", "f"), ("goal", "goal"), ("goalf", "goalf")):
            miss += _summary_misses(o[tag + ".S"], o[ftag + ".F"], c, name + " " + tag, rows)
        miss += _misses(o["Y"], Yr, ATOL + RTOL * Ya, rows, name + " J d")
        miss += _misses(o["Z"], Zr, ATOL + RTOL * Za, rows, name + " J^T lambda")
        miss += _misses(o["W"], Wr, ATOL + RTOL * Ws, rows, name + " w")
        assert np.array_equal(o["Wz"], o["Z"]), name + ": z of lag_hess_vec differs from jac_tvec's"
    assert not miss, "%d misses:\n%s" % (len(miss), "\n".join(miss[:40]))


# ---- GPU: non-finite inputs ------------------------------------------------------------------------------------------

def _bad_rows(c):
    """(label, kind, node, component) of the bad rows: kind 'nan' / 'inf' / 'singular'; component None for dt.  Under
    wind model 3 no position is made non-finite (the port does not clamp its cube indices)"""
    ts, mid = c.ts, c.ts // 2 + (c.ts > 1)
    nodes = sorted({0, mid, ts})
    out = [("NaN dt", "nan", None, None, np.nan)]
    for k in nodes:
        for comp in range(PX):
            if c.wind == 3 and comp in (XN, YN, ZN):
                continue
            out.append(("NaN %s[%d]" % (COMP[comp], k), "nan", k, comp, np.nan))
        for comp in (VA, CHI, TT):
            for v in (np.inf, -np.inf):
                out.append(("%sinf %s[%d]" % ("+" if v > 0 else "-", COMP[comp], k), "inf", k, comp, v))
        out.append(("Va = 0 at %d" % k, "singular", k, VA, 0.0))
        out.append(("gamma = pi/2 at %d" % k, "singular", k, GAM, np.pi / 2))
        out.append(("gamma = -pi/2 at %d" % k, "singular", k, GAM, -np.pi / 2))
        out.append(("node %d on the goal" % k, "singular", k, "goal", None))
    if c.mission == "G7":
        out.append(("G7 dist = 0", "singular", ts, "dist", None))
    return out


def _make_bad(x, c, node, comp, v):
    x = x.copy()
    if node is None:
        x[0] = v
        return x
    N = x[1:].reshape(c.ts + 1, PX)
    if comp == "goal":
        N[node, XN], N[node, YN] = c.g["goal_ned"][0], c.g["goal_ned"][1]
    elif comp == "dist":
        N[c.ts, XN], N[c.ts, YN] = N[0, XN], N[0, YN]
    else:
        N[node, comp] = v
    return x


def _exceptions(c, node, comp, Fb, Gb):
    """flat indices into F and into G of the entries where the port is non-finite on the bad row although it does not
    depend on the bad value in finite arithmetic.  Under wind models 0 and 1 the kernels leave out the terms multiplied
    by wind-gradient components that are identically zero (DESIGN.md section 3: all of them under model 0, dWx/dx and
    dWx/dy under model 1); the reference multiplies those zeros by the NaN or inf and gets NaN.  On the B200 this shows
    as, for instance, F rows 3 and 4 of window k non-finite in the port and finite in the kernel for a NaN chi_k, and
    the chi columns of rows 3-5 (finite-state values 0, -0, -1) for a NaN dt.  The table is explicit in its scope --
    wind models 0 and 1, defect rows 3, 4 and 5 of the windows whose state holds the bad value (every window for dt)
    -- and per entry the port's own structure: at a probe state six finite values of the bad coordinate give the port
    the same bits there.  The probe state is a perturbation of x0 (no chi of 1e18 to absorb other terms) with gamma =
    0.3 and dt = 1e6, so that the rates dominate the defect rows and their constant +-1 entries: a term that depends
    on the bad value only up to rounding (Va cancels from Wxz sin(gamma) cos(chi) Va / (Va cos(gamma)) in row 5's
    chi entry under wind model 1, which the kernels evaluate with Va) changes bits there instead of vanishing in the
    sum.  The kernel must hold its finite-state value (the good row's) on every such entry."""
    none = (np.zeros(0, int), np.zeros(0, int))
    if c.wind not in (0, 1) or isinstance(comp, str) or node == c.ts:
        return none
    j = 0 if node is None else 1 + PX * node + comp
    windows = range(c.ts) if node is None else [node]
    rows = np.zeros(c.neF, bool)
    for k in windows:
        rows[1 + PF * k + 3:1 + PF * k + 6] = True
    x = T.synth.perturb(T.initial_guess(c.cfg), 4321)
    x[0], x[1 + GAM::PX] = 1e6, 0.3
    X = np.tile(x, (7, 1))
    X[1:, j] = x[j] * (1.0 + 0.25 * np.arange(1, 7)) + 0.125 * np.arange(1, 7)
    Fp, Gp = _port_rows(c.port, X)
    same = lambda P: (P.view(np.int64) == P[:1].view(np.int64)).all(axis=0)
    fexc = rows & same(Fp) & ~np.isfinite(Fb)
    gexc = rows[c.iG] & same(Gp) & ~np.isfinite(Gb)
    return np.nonzero(fexc)[0], np.nonzero(gexc)[0]


def _non_finite_misses(got, ref, tol, exc, base, weak, what, label):
    """the contract on one bad row: finite ref -> got finite (unless weak) and within tol; non-finite ref -> got
    non-finite; entries of exc hold the base row's value bit for bit"""
    out = []
    keep = np.ones(got.shape, bool)
    for i in exc:
        keep[i] = False
        if got[i].tobytes() != base[i].tobytes():
            out.append("%s %s: exception entry %d is %r, its finite-state value %r" % (what, label, i, got[i], base[i]))
    fin = np.isfinite(ref) & keep
    with np.errstate(invalid="ignore"):
        err = np.abs(got - ref) > tol
    bad = fin & (err if weak else (err | ~np.isfinite(got)))
    bad |= ~np.isfinite(ref) & keep & np.isfinite(got)
    for i in np.nonzero(bad)[0][:6]:
        out.append("%s %s entry %d: kernel %r port %r" % (what, label, i, got[i], ref[i]))
    if bad.sum() > 6:
        out.append("%s %s: %d entries in all" % (what, label, bad.sum()))
    return out


NONFINITE_TS = (33, 257)


@pytest.mark.gpu
@pytest.mark.parametrize("wind", [0, 1, 3])
@pytest.mark.parametrize("ts", NONFINITE_TS)
@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_non_finite_inputs(mission, ts, wind):
    """bad rows interleaved with good ones, through every path and launch configuration:
      * every good row has the bits it has in a batch without the bad rows;
      * on bad rows F and G (and compact rows, F only, the goal table) keep the port's finiteness and, where it is
        finite, its bar; +-inf rows the weaker contract (non-finite in the port -> non-finite in the kernel);
        the entries of _exceptions hold their finite-state values;
      * the summary of every row is numpy's NaN-propagating reductions of the kernel's own F (both kernels; with F+G,
        with F only, alone and with the goal table)."""
    c = _ctx(mission, ts, wind)
    c.gpos = {(i, j): k for k, (i, j) in enumerate(zip(c.iG, c.jG))}
    bad = _bad_rows(c)
    nbad = len(bad)
    good = box_states(c.cfg, 0, nbad, c.g if wind == 3 else None)
    B = 2 * nbad
    X = np.empty((B, c.n))
    X[0::2] = good
    for q, (label, kind, node, comp, v) in enumerate(bad):
        X[2 * q + 1] = _make_bad(good[q], c, node, comp, v)
    rows = sum((["good %d" % q, bad[q][0]] for q in range(nbad)), [])
    rng = np.random.default_rng(ts + wind)
    D, Lam = rng.uniform(-1, 1, (B, c.n)), rng.uniform(-1, 1, (B, c.neF))
    goals = np.tile(c.g["goal_ned"], (B, 1))  # the context's own goal in every row: bit for bit the plain path
    Fr, Gr = _port_rows(c.port, X)
    ftol = _f_tol(X, Fr, ts)
    exc = [_exceptions(c, node, comp, Fr[2 * q + 1], Gr[2 * q + 1])
           for q, (label, kind, node, comp, v) in enumerate(bad)]
    configs = c.configs()
    if ts <= 256:
        configs = [("A per%d" % p, 0, p) for p in (1, 2, 3, 4)] + [("L", 2, 0)]
    miss = []
    for name, kernel, per in configs:
        o = c.run(X, D, Lam, kernel, per, goals)
        og = c.run(X[0::2], D[0::2], Lam[0::2], kernel, per, goals[0::2])
        for key in og:  # isolation: the good rows' bits do not depend on their neighbours
            if not np.array_equal(o[key][0::2].view(np.int64), og[key].view(np.int64)):
                miss.append("%s %s: a good row changed next to bad rows" % (name, key))
        for tag, ftag in (("fgs", "fgs"), ("fs", "fs"), ("s", "f"), ("goal", "goal"), ("goalf", "goalf")):
            miss += _summary_misses(o[tag + ".S"], o[ftag + ".F"], c, name + " " + tag, rows)
        same = lambda a, b: np.array_equal(a, b, equal_nan=True)
        for k1, k2 in (("f.F", "fg.F"), ("c.G", "fg.G"), ("goal.F", "fg.F"), ("goal.G", "fg.G"), ("goalf.F", "f.F"),
                       ("goal.S", "fgs.S"), ("goalf.S", "fs.S")):
            if not same(o[k1], o[k2]):
                miss.append("%s: %s differs from %s" % (name, k1, k2))
        for q, (label, kind, node, comp, v) in enumerate(bad):
            b = 2 * q + 1
            fexc, gexc = exc[q]
            weak = kind == "inf"
            miss += _non_finite_misses(o["fg.F"][b], Fr[b], ftol[b], fexc, o["fg.F"][b - 1], weak, name + " F", label)
            miss += _non_finite_misses(o["fg.G"][b], Gr[b], ATOL + RTOL * np.abs(Gr[b]), gexc, o["fg.G"][b - 1], weak,
                                       name + " G", label)
            # the products against the port's G with the exceptions at the kernel's values
            Gp = Gr[b:b + 1].copy()
            Gp[0, gexc] = o["fg.G"][b, gexc]
            with np.errstate(all="ignore"):
                Yr, Ya, Zr, Za = _op_refs(c, Gp, D[b:b + 1], Lam[b:b + 1])
            miss += _non_finite_misses(o["Y"][b], Yr[0], ATOL + RTOL * Ya[0], [], None, weak, name + " J d", label)
            miss += _non_finite_misses(o["Z"][b], Zr[0], ATOL + RTOL * Za[0], [], None, weak, name + " J^T lambda",
                                       label)
        assert np.array_equal(o["Wz"], o["Z"], equal_nan=True), name + ": z of lag_hess_vec differs from jac_tvec's"
    assert not miss, "%d misses:\n%s" % (len(miss), "\n".join(miss[:60]))


@pytest.mark.gpu
@pytest.mark.parametrize("wind", [0, 1, 3])
@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_nan_in_one_coordinate_of_d_or_lambda(mission, wind):
    """NaN in d_j reaches the rows of J d whose pattern holds column j and the columns of w next to it (its windows'
    nodes, dt, G7's end nodes); NaN in lambda_i the columns of row i in J^T lambda and w.  Every other entry keeps its
    bar and every other trajectory its bits, on kernel A and kernel L"""
    ts = 33
    c = _ctx(mission, ts, wind)
    X = box_states(c.cfg, 100, 110, c.g if wind == 3 else None)
    B = X.shape[0]
    rng = np.random.default_rng(7 + wind)
    D, Lam = rng.uniform(-1, 1, (B, c.n)), rng.uniform(-1, 1, (B, c.neF))
    Fr, Gr = _port_rows(c.port, X)
    Yr, Ya, Zr, Za = _op_refs(c, Gr, D, Lam)
    Wr, Ws = _hvp_refs(c, X, Lam, D)
    mid = 1 + PX * 17
    dcols = [0, 1 + VA, 1 + CHI, mid + ZN, mid + GAM, mid + TT, 1 + PX * ts + XN, 1 + PX * ts + CL]
    lrows = [0, 1 + PF * 5 + 3, 1 + PF * 20 + 0, c.neF - 1, c.neF - c.nb]
    Dn = D.copy()  # trajectory b < 8: NaN in d at dcols[b]; lambda's NaN goes in launches of its own below
    for b, j in enumerate(dcols):
        Dn[b, j] = np.nan
    miss = []
    for name, kernel, per in (("A", 0, 0), ("L", 2, 0)):
        base = c.run(X, D, Lam, kernel, per)
        o = c.run(X, Dn, Lam, kernel, per)
        for b, j in enumerate(dcols):
            rows_j = set(c.iG[c.jG == j])
            free_y = np.array([i not in rows_j for i in range(c.neF)])
            if j == 0:
                cols_w = np.zeros(c.n, bool)
            else:
                k = (j - 1) // PX
                near = set(range(max(0, k - 1), min(ts, k + 1) + 1))
                if mission == "G7" and k in (0, ts):
                    near |= {0, ts}
                cols_w = np.ones(c.n, bool)
                cols_w[0] = False
                for m in near:
                    cols_w[1 + PX * m:1 + PX * (m + 1)] = False
            lab = "NaN d[%d]" % j
            miss += _misses(o["Y"][b:b + 1, free_y], Yr[b:b + 1, free_y], (ATOL + RTOL * Ya)[b:b + 1, free_y], [lab],
                            name + " J d")
            Wd = c.restatement().lag_hess_vec(X[b], Lam[b], np.where(np.isnan(Dn[b]), 0.0, Dn[b])).numpy()
            miss += _misses(o["W"][b:b + 1, cols_w], Wd[None, cols_w], (ATOL + RTOL * Ws)[b:b + 1, cols_w], [lab],
                            name + " w")
        for b in range(len(dcols), B):
            for key in ("Y", "W"):
                if not np.array_equal(o[key][b], base[key][b]):
                    miss.append("%s %s: trajectory %d changed by another's NaN d" % (name, key, b))
        assert np.array_equal(o["Z"], base["Z"]), name + ": J^T lambda depends on d"
        for q, i in enumerate(lrows):
            Lq = Lam.copy()
            Lq[q, i] = np.nan
            o = c.run(X, D, Lq, kernel, per)
            free = np.ones(c.n, bool)
            free[c.jG[c.iG == i]] = False
            lab = "NaN lambda[%d]" % i
            miss += _misses(o["Z"][q:q + 1, free], Zr[q:q + 1, free], (ATOL + RTOL * Za)[q:q + 1, free], [lab],
                            name + " J^T lambda")
            miss += _misses(o["W"][q:q + 1, free], Wr[q:q + 1, free], (ATOL + RTOL * Ws)[q:q + 1, free], [lab],
                            name + " w")
            others = np.arange(B) != q
            for key in ("Z", "W", "Wz"):
                if not np.array_equal(o[key][others], base[key][others]):
                    miss.append("%s %s: another trajectory changed by NaN lambda[%d]" % (name, key, i))
            assert np.array_equal(o["Y"], base["Y"]), name + ": J d depends on lambda"
    assert not miss, "%d misses:\n%s" % (len(miss), "\n".join(miss[:40]))
