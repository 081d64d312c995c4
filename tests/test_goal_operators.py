"""Per-trajectory goals in the matrix-free products (tolcuda_jac_vec_goals, tolcuda_jac_tvec_goals,
tolcuda_lag_hess_vec_goals; Evaluator.jac_vec / jac_tvec / lag_hess_vec with row0).

Without a GPU: the three entry points refuse a null handle before touching CUDA.
On the GPU: row b of y, z, w (and the optional z) is bit for bit what the context-goal call writes on a context created
with goal row row0 + b, under every kernel shape; the rows agree with products of the CPU port's G and with the torch
restatement built with each row's goal; a goal call runs the same entry function as the context-goal call; misuse
launches nothing; replacing the table between unsynchronised launches leaves each launch with its own table."""
import os

import numpy as np
import pytest

import tol_b200 as T
from conftest import ATOL, RTOL, load_golden

EV = T.evaluator
PAD = 3


# ---- no GPU needed ---------------------------------------------------------------------------------------------------

def test_goal_products_refuse_a_null_handle_without_cuda():
    L = T.load()
    for call in (lambda: L.tolcuda_jac_vec_goals(None, 0, 1, None, 0, None, 0, None, 0, 0),
                 lambda: L.tolcuda_jac_tvec_goals(None, 0, 1, None, 0, None, 0, None, 0, 0),
                 lambda: L.tolcuda_lag_hess_vec_goals(None, 0, 1, None, 0, None, 0, None, 0, None, 0, None, 0, 0),
                 lambda: L.tolcuda_lag_hess_vec_goals(None, 0, 0, None, 0, None, 0, None, 0, None, 0, None, 0, 0)):
        assert call() == -1
        assert b"null handle" in L.tolcuda_last_error()


# ---- GPU -------------------------------------------------------------------------------------------------------------

def _fixture(mission, wind):
    if wind == 3:
        return load_golden("S10_tempest_ts100_wind3" if mission == "S10" else "G7_skywalker_ts45_wind3")
    return load_golden("S10_tempest_ts100" if mission == "S10" else "G7_skywalker_ts100")


def _context(g, mission, ts, wind, goal, options=None):
    ev = T.Evaluator(mission, ts, g["ac"], g["gn"], goal, 1 if wind == 3 else wind)
    for k, v in (options or {}).items():
        ev.set_option(k, v)
    if wind == 3:
        ev.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
    return ev


def _inputs(g, mission, ts, B, seed=0):
    """x (synthetic trajectories around the initial guess), d and lambda (uniform in [-1, 1])"""
    x0 = T.initial_guess(T.make_config(mission, ts, g["ac"], g["gn"], g["goal_ned"]))
    X = T.synth.batch(x0, (T.synth.SEED_S10 if mission == "S10" else T.synth.SEED_G7) + seed, 0, B)
    rng = np.random.default_rng(1000 * ts + seed)
    return X, rng.uniform(-1, 1, (B, X.shape[1])), rng.uniform(-1, 1, (B, 1 + 8 * ts + (11 if mission == "S10" else 12)))


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _nan(B, m):
    import torch
    return torch.full((B, m), float("nan"), dtype=torch.float64, device="cuda")


def _products(ev, Xd, Dd, Ld, row0=None, sync=True):
    """y = J d, z = J^T lambda, w = H d alone and w with z, into NaN-filled buffers PAD columns wider than the rows;
    row0 None: the context-goal calls.  Returns the torch buffers."""
    B = Xd.shape[0]
    out = {"y": _nan(B, ev.neF + PAD), "z": _nan(B, ev.n + PAD), "w": _nan(B, ev.n + PAD), "w+z": _nan(B, ev.n + PAD),
           "z of w+z": _nan(B, ev.n + PAD)}
    ev.jac_vec(Xd, Dd, out["y"], sync=sync, row0=row0)
    ev.jac_tvec(Xd, Ld, out["z"], sync=sync, row0=row0)
    ev.lag_hess_vec(Xd, Ld, Dd, out["w"], sync=sync, row0=row0)
    ev.lag_hess_vec(Xd, Ld, Dd, out["w+z"], out["z of w+z"], sync=sync, row0=row0)
    return out


def _numpy(out):
    import torch
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _check_padding(got, ev, what):
    assert np.isnan(got["y"][:, ev.neF:]).all(), what + ": y padding"
    for k in ("z", "w", "w+z", "z of w+z"):
        assert np.isnan(got[k][:, ev.n:]).all(), "%s: %s padding" % (what, k)
    assert np.array_equal(_bits(got["z of w+z"]), _bits(got["z"])), what + ": the z of lag_hess_vec_goals differs from jac_tvec_goals'"


# kernel A with runs of 1 .. 4 trajectories per CTA (tail_x4 = 0: a batch of 64 forms runs, and a goal slot is reused
# within a run from per = 3 on) and kernel L at any ts; ts = 300 is kernel L's alone
OPTIONS = [{"per": 1}, {"per": 2, "tail_x4": 0}, {"per": 3, "tail_x4": 0}, {"per": 4, "tail_x4": 0}, {"kernel": 2}]


@pytest.mark.gpu
@pytest.mark.parametrize("ts", [1, 33, 100, 200, 300])
@pytest.mark.parametrize("wind", [0, 1, 3])
@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_rows_equal_a_context_created_with_the_rows_goal(mission, wind, ts):
    """K = 8 distinct goals (G7: every quadrant of chi_d and the axes) cycle over B = 64 rows of a table that starts 5
    rows before the call's first row; row b of y, z, w and the optional z equals bit for bit the context-goal call of
    a context created with goal b % K, under the same options"""
    g = _fixture(mission, wind)
    K, B, row0 = 8, 64, 5
    goals = T.synth.goals(mission, 0, K)
    X, D, Lam = _inputs(g, mission, ts, B)
    Xd, Dd, Ld = _dev(X), _dev(D), _dev(Lam)
    ev = _context(g, mission, ts, wind, g["goal_ned"])
    ev.set_goals(np.concatenate([T.synth.goals(mission, 100, 100 + row0), goals[np.arange(B) % K]]))
    per_goal = [_context(g, mission, ts, wind, goals[k]) for k in range(K)]
    for opts in OPTIONS if ts <= 256 else [{}]:
        for e in [ev] + per_goal:
            for k, v in {"per": 0, "tail_x4": -1, "kernel": 0, **opts}.items():
                e.set_option(k, v)
        what = "%s ts=%d wind %d %s" % (mission, ts, wind, opts)
        got = _numpy(_products(ev, Xd, Dd, Ld, row0))
        _check_padding(got, ev, what)
        for k in range(K):
            rows = np.arange(k, B, K)
            want = _numpy(_products(per_goal[k], Xd[rows].contiguous(), Dd[rows].contiguous(), Ld[rows].contiguous()))
            for name in got:
                assert np.array_equal(_bits(got[name][rows]), _bits(want[name])), "%s: %s of goal %d" % (what, name, k)
    for e in [ev] + per_goal:
        e.close()


def _port_products(mission, ts, wind, g, goal, x, d, lam):
    """y = J d, z = J^T lambda and their sums of |terms| from the CPU port's G with this goal"""
    import portclient as P
    p = P.PortProblem(mission, ts, g["ac"], g["gn"], goal, 1 if wind == 3 else wind)
    if wind == 3:
        p.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
    iG, jG = p.pattern()
    _, G = p.eval(x)
    if mission == "S10":
        G[p.ub_mask()] = 0.0  # the boundary rows' dt entries the reference leaves undefined: 0 in the kernels
    y, ya, z, za = np.zeros(p.neF), np.zeros(p.neF), np.zeros(p.n), np.zeros(p.n)
    ty, tz = G * d[jG], G * lam[iG]
    np.add.at(y, iG, ty)
    np.add.at(ya, iG, np.abs(ty))
    np.add.at(z, jG, tz)
    np.add.at(za, jG, np.abs(tz))
    return y, ya, z, za


def _assert_within(got, ref, scale, what):
    assert np.isfinite(got).all(), what + ": non-finite values"
    e = np.abs(got - ref) - (ATOL + RTOL * scale)
    assert e.max() <= 0, (what, np.unravel_index(e.argmax(), e.shape), e.max())


@pytest.mark.gpu
@pytest.mark.parametrize("ts", [64, 257])
@pytest.mark.parametrize("wind", [0, 1, 3])
@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_rows_match_the_references_with_the_rows_goal(mission, wind, ts):
    """every row against products of the CPU port's G built with that row's goal (J d, J^T lambda) and against the
    torch restatement built with it (w), with 1e-14 + 1e-12 * sum of |terms|; wind model 3 states lie inside the cube"""
    import lagrangian_torch as LT
    g = load_golden("S10_tempest_ts100_wind3" if mission == "S10" else "G7_skywalker_ts45_wind3")
    lm = g["lm"]
    cfg = T.make_config(mission, ts, g["ac"], g["gn"], g["goal_ned"],
                        limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]])
    B = 6
    X = T.synth.batch(T.initial_guess(cfg), 4321 + ts, 0, B)
    if wind == 3:
        N = X[:, 1:].reshape(B, ts + 1, 11)
        dat = g["grid_datum"]
        for s, grid in ((N[..., 1] + dat[0], g["grid_x"]), (N[..., 0] + dat[1], g["grid_y"]), (-N[..., 2] + dat[2], g["grid_z"])):
            assert (s > grid[0]).all() and (s < grid[-1]).all(), "a node outside the interior of the wind cube"
    rng = np.random.default_rng(ts * 10 + wind)
    ev = _context(g, mission, ts, wind, g["goal_ned"])
    D, Lam = rng.uniform(-1, 1, (B, ev.n)), rng.uniform(-1, 1, (B, ev.neF))
    goals = T.synth.goals(mission, 0, B + 2)
    ev.set_goals(goals)
    got = _numpy(_products(ev, _dev(X), _dev(D), _dev(Lam), row0=2))
    _check_padding(got, ev, "%s ts=%d wind %d" % (mission, ts, wind))
    for b in range(B):
        what = "%s ts=%d wind %d row %d" % (mission, ts, wind, b)
        goal = goals[2 + b]
        y, ya, z, za = _port_products(mission, ts, wind, g, goal, X[b], D[b], Lam[b])
        _assert_within(got["y"][b, :ev.neF], y, ya, what + " J d")
        _assert_within(got["z"][b, :ev.n], z, za, what + " J^T lambda")
        o = LT.Problem(dict(g, goal_ned=goal), wind_model=wind, ts=ts)
        w, ws = o.lag_hess_vec(X[b], Lam[b], D[b]).numpy(), o.term_scale(X[b], Lam[b], D[b]).numpy()
        _assert_within(got["w"][b, :ev.n], w, ws, what + " w")
        _assert_within(got["w+z"][b, :ev.n], w, ws, what + " w (with z)")
    ev.close()


def _recorded_kernels(fn):
    """fn() under torch.profiler (CUDA activity): the names of the kernels it ran"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def _profile_calls(mission, ts, opts):
    """{product: (kernels of the context-goal call, kernels of the goal call, launches the goal call counted)}"""
    g = _fixture(mission, 1)
    B = 16
    X, D, Lam = _inputs(g, mission, ts, B)
    Xd, Dd, Ld = _dev(X), _dev(D), _dev(Lam)
    ev = _context(g, mission, ts, 1, g["goal_ned"], opts)
    ev.set_goals(T.synth.goals(mission, 0, B))
    Y, Z, W = _nan(B, ev.neF), _nan(B, ev.n), _nan(B, ev.n)
    calls = {"jac_vec": lambda r: ev.jac_vec(Xd, Dd, Y, row0=r), "jac_tvec": lambda r: ev.jac_tvec(Xd, Ld, Z, row0=r),
             "lag_hess_vec": lambda r: ev.lag_hess_vec(Xd, Ld, Dd, W, Z, row0=r)}
    out = {}
    for name, call in calls.items():
        ctx = _recorded_kernels(lambda: call(None))
        n0 = ev.launches
        gl = _recorded_kernels(lambda: call(0))
        out[name] = (ctx, gl, ev.launches - n0)
    ev.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("mission", ["S10", "G7"])
@pytest.mark.parametrize("ts,opts", [(100, {"per": 1}), (200, {"per": 2, "tail_x4": 0}), (64, {"kernel": 2}), (300, {})])
def test_a_goal_call_runs_the_entry_function_of_the_context_goal_call(mission, ts, opts):
    """one launch each, and the kernel a goal call runs is the kernel the context-goal call runs: no goal instances.
    The profiler runs in a child process, so that this process's later profiler sessions start from a fresh state."""
    import json
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    code = ("import json, sys; sys.path[:0] = [%r, %r]; import test_goal_operators as t; "
            "print(json.dumps(t._profile_calls(%r, %d, %r)))" % (here, os.path.dirname(here), mission, ts, opts))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    for name, (ctx, gl, launches) in json.loads(r.stdout.strip().splitlines()[-1]).items():
        assert launches == 1 and len(ctx) == 1 and gl == ctx, (name, ctx, gl, launches)


@pytest.mark.gpu
def test_goal_product_misuse_is_refused_and_launches_nothing():
    """no table, rows outside it, null pointers, short leading dimensions and host pointers: each returns its code
    and nothing launches; B = 0 launches nothing"""
    import torch
    g = load_golden("S10_tempest_ts100")
    ev = T.Evaluator.from_golden(g)
    L, h, n, neF = ev.L, ev.h, ev.n, ev.neF
    X, D, Lam = (_dev(a) for a in _inputs(g, "S10", 100, 2))
    W, Z = torch.empty(2, n, dtype=torch.float64, device="cuda"), torch.empty(2, n, dtype=torch.float64, device="cuda")
    Y = torch.empty(2, neF, dtype=torch.float64, device="cuda")
    x, l, d, w, z, y = X.data_ptr(), Lam.data_ptr(), D.data_ptr(), W.data_ptr(), Z.data_ptr(), Y.data_ptr()

    def jv(row0, B, *a):
        return L.tolcuda_jac_vec_goals(h, row0, B, *a)

    def jt(row0, B, *a):
        return L.tolcuda_jac_tvec_goals(h, row0, B, *a)

    def hv(row0, B, *a):
        return L.tolcuda_lag_hess_vec_goals(h, row0, B, *a)

    good = {jv: (x, n, d, n, y, neF, 0), jt: (x, n, l, neF, z, n, 0), hv: (x, n, l, neF, d, n, w, n, z, n, 0)}
    before = ev.launches
    for f, a in good.items():
        assert f(0, 2, *a) == -1 and b"no goal table" in L.tolcuda_last_error()
    ev.set_goals(T.synth.goals("S10", 0, 10))
    for f, a in good.items():
        for row0, B in ((-1, 2), (9, 2), (10, 1), (0, 11), (0, -1)):
            assert f(row0, B, *a) == -1 and b"outside the goal table" in L.tolcuda_last_error(), (row0, B)
        for i in range(len(a) - 1):  # each pointer NULL, each leading dimension one short
            bad = list(a)
            bad[i] = None if i % 2 == 0 else bad[i] - 1
            if f is hv and i == 8:
                continue  # z is optional
            assert f(0, 2, *bad) == -1 and b"null pointer or leading dimension" in L.tolcuda_last_error(), (f, i)
        assert f(0, 2, *a[:-1], EV.HOST_PTRS) == -2 and b"device pointers only" in L.tolcuda_last_error()
        assert f(10, 0, *[None if i % 2 == 0 else 0 for i in range(len(a) - 1)], 0) == 0  # B = 0
    assert ev.launches == before
    for f, a in good.items():
        assert f(8, 2, *a) == 0
    assert ev.launches == before + 3
    ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_set_goals_between_unsynchronised_product_launches(mission):
    """TOLCUDA_NO_SYNC products with one table, tolcuda_set_goals with another, the same products again: each launch
    equals its own synchronous launch with its own table"""
    g = _fixture(mission, 1)
    ts, B = 200, 4096
    X, D, Lam = _inputs(g, mission, ts, B)
    Xd, Dd, Ld = _dev(X), _dev(D), _dev(Lam)
    ev = _context(g, mission, ts, 1, g["goal_ned"])
    tables = [T.synth.goals(mission, 0, B), T.synth.goals(mission, 5000, 5000 + B)]
    want = []
    for t in tables:
        ev.set_goals(t)
        want.append(_numpy(_products(ev, Xd, Dd, Ld, row0=0)))
    got = []
    for t in tables:
        ev.set_goals(t)
        got.append(_products(ev, Xd, Dd, Ld, row0=0, sync=False))
    got = [_numpy(o) for o in got]
    for i in range(2):
        for name in want[i]:
            assert np.array_equal(_bits(got[i][name]), _bits(want[i][name])), (i, name)
    assert not np.array_equal(_bits(want[0]["y"]), _bits(want[1]["y"]))  # the two tables do give different products
    ev.close()


@pytest.mark.gpu
def test_full_size_batch_of_distinct_goals():
    """65,536 x S10 ts=200 (the opbench batch) with 65,536 distinct goals: a strided sample of rows of y, z, w and the
    optional z equals bit for bit the context-goal calls of contexts created with those rows' goals"""
    g = load_golden("S10_tempest_ts200")
    B, ts = 65536, 200
    ev = _context(g, "S10", ts, 1, g["goal_ned"])
    goals = T.synth.goals("S10", 0, B)
    ev.set_goals(goals)
    X = T.synth.batch(g["x"][0], T.synth.SEED_S10, 0, B)
    rng = np.random.default_rng(65536)
    Xd, Dd, Ld = _dev(X), _dev(rng.uniform(-1, 1, (B, ev.n))), _dev(rng.uniform(-1, 1, (B, ev.neF)))
    out = _products(ev, Xd, Dd, Ld, row0=0)
    rows = np.arange(0, B, 4099)
    got = _numpy({k: v[rows] for k, v in out.items()})
    del out
    _check_padding(got, ev, "full size")
    for i, b in enumerate(rows):
        eb = _context(g, "S10", ts, 1, goals[b])
        want = _numpy(_products(eb, Xd[b:b + 1], Dd[b:b + 1], Ld[b:b + 1]))
        for name in want:
            assert np.array_equal(_bits(got[name][i:i + 1]), _bits(want[name])), (b, name)
        eb.close()
    ev.close()
