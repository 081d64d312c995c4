"""Hessian-of-the-Lagrangian products (tolcuda_lag_hess_vec): w = D_x[J(x)^T lambda] d, optionally with z = J^T lambda.

Without a GPU: the torch restatement (oracle/lagrangian_torch.py) is pinned to the CPU port -- its F within the parity
bar on every fixture, its Jacobian within the bar at every pattern position and exactly 0 elsewhere -- and checked
against itself (a central difference of the port's J^T lambda, symmetry under wind model 0); the entry point refuses
a null handle before touching CUDA.
On the GPU: w against the restatement entry by entry, z bit for bit what tolcuda_jac_tvec writes, the same bits under
every launch option (w[0] aside under kernel L), symmetry and linearity, kernel L for long and odd trajectories, the
full-size batches, degenerate inputs and misuse."""
import numpy as np
import pytest
import torch

import tol_b200 as T
from conftest import GOLDEN, load_golden, port_from_golden

import lagrangian_torch as LT


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _port_jt_lambda(p, x, lam):
    """J^T lambda formed from the port's G row and the pattern (S10's undefined boundary-row dt entries as 0)"""
    _, G = p.eval(x)
    if p.mission == "S10":
        G[p.ub_mask()] = 0.0
    iG, jG = p.pattern()
    z = np.zeros(p.n)
    np.add.at(z, jG, G * lam[iG])
    return z


def _oracle(o, X, Lam, D):
    """w and its sum of |terms| for every row"""
    W = np.stack([o.lag_hess_vec(x, l, d).numpy() for x, l, d in zip(X, Lam, D)])
    S = np.stack([o.term_scale(x, l, d).numpy() for x, l, d in zip(X, Lam, D)])
    return W, S


def _assert_within(w, wr, scale, what, rel=1e-12):
    assert np.isfinite(w).all(), what
    e = np.abs(w - wr) - (1e-14 + rel * scale)
    assert e.max() <= 0, (what, np.unravel_index(e.argmax(), e.shape), e.max())


def _inputs(g, B, seed, ts=None, x0=None):
    rng = np.random.default_rng(seed)
    X = T.synth.batch(g["x"][0] if x0 is None else x0, 555, 0, B)
    n = X.shape[1]
    nb = 12 if str(g["mission"]) == "G7" else 11
    neF = 1 + 8 * ((n - 1) // 11 - 1) + nb
    return X, rng.uniform(-1, 1, (B, neF)), rng.uniform(-1, 1, (B, n))


# ---- no GPU needed ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", GOLDEN)
def test_restatement_is_pinned_to_the_port(name, oracle_built):
    """F within 1e-14 + 1e-12*|ref| of the port; the Jacobian of F_tilde within that bar of the port's G at every
    pattern position (S10's undefined boundary-row dt entries: 0) and exactly 0 off the pattern"""
    g = load_golden(name)
    p, o = port_from_golden(g), LT.Problem(g)
    iG, jG = p.pattern()
    X = np.concatenate([g["x"][:1], T.synth.batch(g["x"][0], 555, 0, 2)])
    for x in X:
        Fr, Gr = p.eval(x)
        if p.mission == "S10":
            Gr[p.ub_mask()] = 0.0
        xt = torch.from_numpy(x)
        F = o.F(xt).numpy()
        assert (np.abs(F - Fr) <= 1e-14 + 1e-12 * np.abs(Fr)).all(), name
        J = o.jacobian(xt).numpy()
        assert (np.abs(J[iG, jG] - Gr) <= 1e-14 + 1e-12 * np.abs(Gr)).all(), name
        J[iG, jG] = 0.0
        assert not J.any(), name


@pytest.mark.parametrize("name,wind", [("S10_tempesteric_ts33", None), ("G7_tempestwences_ts45_gains", None),
                                       ("S10_tempest_ts100_wind3", None), ("G7_skywalker_ts45_wind3", None),
                                       ("S10_tempesteric_ts33", 0), ("G7_tempestwences_ts45_gains", 0)])
def test_restatement_against_a_central_difference_of_the_port(name, wind, oracle_built):
    """w against (J^T lambda)(x + h d) - (J^T lambda)(x - h d) over 2h from the port's G rows, to about 1e-6 of the
    scale; under wind model 0 also e.(H d) == d.(H e)"""
    g = load_golden(name)
    wm = int(g["wind_model"]) if wind is None else wind
    p = port_from_golden(g) if wind is None else oracle_built.PortProblem(str(g["mission"]), int(g["ts"]), g["ac"],
                                                                          g["gn"], g["goal_ned"], wm)
    o = LT.Problem(g, wind_model=wm)
    X, Lam, D = _inputs(g, 2, 11)
    for x, lam, d in zip(X, Lam, D):
        w = o.lag_hess_vec(x, lam, d).numpy()
        scale = o.term_scale(x, lam, d).numpy()
        h = 1e-6
        fd = (_port_jt_lambda(p, x + h * d, lam) - _port_jt_lambda(p, x - h * d, lam)) / (2 * h)
        assert (np.abs(w - fd) <= 1e-6 * (scale + np.abs(w)).max() + 1e-6 * scale).all(), name
    if wm == 0:
        e = np.random.default_rng(2).uniform(-1, 1, X.shape[1])
        he, hd = o.lag_hess_vec(X[0], Lam[0], e).numpy(), o.lag_hess_vec(X[0], Lam[0], D[0]).numpy()
        assert abs(D[0] @ he - e @ hd) <= 1e-12 * (np.abs(D[0]) @ o.term_scale(X[0], Lam[0], e).numpy())


def test_lag_hess_vec_refuses_a_null_handle_without_cuda():
    """argument checks come before any CUDA call; there is no CPU path"""
    L = T.load()
    assert L.tolcuda_lag_hess_vec(None, 4, None, 0, None, 0, None, 0, None, 0, None, 0, 0) == -1
    assert L.tolcuda_lag_hess_vec(None, 0, None, 0, None, 0, None, 0, None, 0, None, 0, 0) == -1


# ---- GPU -------------------------------------------------------------------------------------------------------------

def _run(ev, X, Lam, D, pad=5, with_z=True):
    Xd, Ld, Dd = _dev(X), _dev(Lam), _dev(D)
    B = X.shape[0]
    W = torch.full((B, ev.n + pad), float("nan"), dtype=torch.float64, device="cuda")
    Z = torch.full((B, ev.n + pad), float("nan"), dtype=torch.float64, device="cuda") if with_z else None
    ev.lag_hess_vec(Xd, Ld, Dd, W, Z)
    return W, Z


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN)
@pytest.mark.parametrize("kernel", [0, 2])
def test_lag_hess_vec_against_the_restatement(name, kernel):
    """21 synth.batch rows with random lambda and d: |w - w_ref| <= 1e-14 + 1e-12 * sum of |terms| per entry; padding
    untouched; z bit for bit tolcuda_jac_tvec's; a repeat launch gives the same bits"""
    g = load_golden(name)
    o = LT.Problem(g)
    ev = T.Evaluator.from_golden(g, options={"kernel": kernel})
    X, Lam, D = _inputs(g, 21, 77)
    W, Z = _run(ev, X, Lam, D)
    n = ev.n
    assert torch.isnan(W[:, n:]).all() and torch.isnan(Z[:, n:]).all()
    Wr, S = _oracle(o, X, Lam, D)
    _assert_within(W[:, :n].cpu().numpy(), Wr, S, name)
    Zt = torch.full_like(Z, float("nan"))
    ev.jac_tvec(_dev(X), _dev(Lam), Zt)
    assert torch.equal(Z[:, :n], Zt[:, :n])
    W2, Z2 = _run(ev, X, Lam, D)
    assert torch.equal(W2[:, :n], W[:, :n]) and torch.equal(Z2[:, :n], Z[:, :n])
    W3, _ = _run(ev, X, Lam, D, with_z=False)
    assert torch.equal(W3[:, :n], W[:, :n])
    ev.close()


def _long_case(mission, ts):
    g = load_golden("S10_tempest_ts100" if mission == "S10" else "G7_skywalker_ts100")
    lm = g["lm"]
    cfg = T.make_config(mission, ts, g["ac"], g["gn"], g["goal_ned"],
                        limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]])
    return g, T.initial_guess(cfg)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["G7_tempestwences_ts45_gains", ("S10", 300)])
def test_every_option_gives_the_same_bits(case):
    """"per" 1-4, "kernel" 0 and 2, "lwarps" 1-8: w and z bit-identical, except w[0] and z[0] under kernel L, which
    stay within the bar of kernel A's"""
    if isinstance(case, str):
        g, x0, ts = load_golden(case), None, None
        mk = lambda opts: T.Evaluator.from_golden(g, options=opts)
    else:
        (g, x0), ts = _long_case(*case), case[1]
        mk = lambda opts: _opts(T.Evaluator(case[0], ts, g["ac"], g["gn"], g["goal_ned"]), opts)
    X, Lam, D = _inputs(g, 9, 5, x0=x0)
    o = LT.Problem(g, ts=ts)
    _, S = _oracle(o, X[:2], Lam[:2], D[:2])
    runs = []
    opts = [{"kernel": 0, "per": p} for p in (1, 2, 3, 4)] + [{"kernel": 2, "lwarps": k} for k in range(1, 9)]
    if ts is None:
        opts += [{"kernel": 2}]
    for op in opts:
        ev = mk(op)
        W, Z = _run(ev, X, Lam, D)
        runs.append((op, W[:, :ev.n].cpu().numpy(), Z[:, :ev.n].cpu().numpy()))
        ev.close()
    op0, W0, Z0 = runs[0]
    for op, W, Z in runs[1:]:
        assert np.array_equal(W[:, 1:], W0[:, 1:]) and np.array_equal(Z[:, 1:], Z0[:, 1:]), op
        if op.get("kernel") != 2:
            assert np.array_equal(W[:, 0], W0[:, 0]) and np.array_equal(Z[:, 0], Z0[:, 0]), op
        assert (np.abs(W[:2, 0] - W0[:2, 0]) <= 1e-14 + 1e-12 * S[:, 0]).all(), op


def _opts(ev, opts):
    for k, v in opts.items():
        ev.set_option(k, v)
    return ev


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["S10_tempest_ts100", "G7_skywalker_ts100", "S10_tempest_ts100_wind3",
                                  "G7_skywalker_ts45_wind3"])
def test_symmetry_and_linearity(name):
    """e.(H d) == d.(H e) under wind model 0 (the reference's G holds the wind fixed, so models 1 and 3 have no
    symmetric Hessian); linear in d and in lambda under every model, to about 1e-11 of the terms"""
    g = load_golden(name)
    o = LT.Problem(g)
    X, Lam, D = _inputs(g, 6, 9)
    E = np.random.default_rng(10).uniform(-1, 1, D.shape)
    Mu = np.random.default_rng(11).uniform(-1, 1, Lam.shape)
    ev = T.Evaluator.from_golden(g)
    n = ev.n
    hd, he = (_run(ev, X, Lam, V)[0][:, :n].cpu().numpy() for V in (D, E))
    hde = _run(ev, X, Lam, 2.0 * D - 3.0 * E)[0][:, :n].cpu().numpy()
    hmu = _run(ev, X, Mu, D)[0][:, :n].cpu().numpy()
    hlm = _run(ev, X, 0.5 * Lam + Mu, D)[0][:, :n].cpu().numpy()
    _, Sd = _oracle(o, X, Lam, D)
    _, Se = _oracle(o, X, Lam, E)
    _, Sm = _oracle(o, X, Mu, D)
    _assert_within(hde, 2.0 * hd - 3.0 * he, 2.0 * Sd + 3.0 * Se, name + " linear in d", rel=1e-11)
    _assert_within(hlm, 0.5 * hd + hmu, 0.5 * Sd + Sm, name + " linear in lambda", rel=1e-11)
    ev.close()
    ev0 = T.Evaluator.from_golden(g, wind_model=0)
    o0 = LT.Problem(g, wind_model=0)
    hd, he = (_run(ev0, X, Lam, V)[0][:, :n].cpu().numpy() for V in (D, E))
    for b in range(X.shape[0]):
        s = np.abs(E[b]) @ o0.term_scale(X[b], Lam[b], D[b]).numpy()
        assert abs(E[b] @ hd[b] - D[b] @ he[b]) <= 1e-11 * s, (name, b)
    ev0.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mission,ts", [("S10", 300), ("G7", 300), ("S10", 513), ("G7", 513)])
def test_long_and_odd_trajectories(mission, ts):
    """ts > 256 (kernel L), odd ts (records starting 8 mod 16) against the restatement"""
    g, x0 = _long_case(mission, ts)
    o = LT.Problem(g, ts=ts)
    ev = T.Evaluator(mission, ts, g["ac"], g["gn"], g["goal_ned"])
    X, Lam, D = _inputs(g, 4, 21, x0=x0)
    W, Z = _run(ev, X, Lam, D)
    assert torch.isnan(W[:, ev.n:]).all()
    Wr, S = _oracle(o, X, Lam, D)
    _assert_within(W[:, :ev.n].cpu().numpy(), Wr, S, "%s ts=%d" % (mission, ts))
    Zt = torch.empty_like(Z)
    ev.jac_tvec(_dev(X), _dev(Lam), Zt)
    assert torch.equal(Z[:, :ev.n], Zt[:, :ev.n])
    ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("G7_skywalker_ts100", 4096), ("S10_tempest_ts200", 65536)])
def test_full_size_batches(name, B):
    """BASELINE config 3 and the bench batch: w against a central difference of jac_tvec on the GPU (relative bar
    1e-6 of the terms), and a strided sample of rows against the restatement"""
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g)
    U = 64
    Xu = _dev(T.synth.batch(g["x"][0], 1234, 0, U))
    Xd = Xu[torch.arange(B, device="cuda") % U].contiguous()
    gen = torch.Generator(device="cuda").manual_seed(5)
    D = torch.rand(B, ev.n, dtype=torch.float64, device="cuda", generator=gen) * 2 - 1
    Lam = torch.rand(B, ev.neF, dtype=torch.float64, device="cuda", generator=gen) * 2 - 1
    W = torch.empty(B, ev.n, dtype=torch.float64, device="cuda")
    Z = torch.empty_like(W)
    ev.lag_hess_vec(Xd, Lam, D, W, Z)
    h = 1e-6
    Zp, Zm = torch.empty_like(W), torch.empty_like(W)
    ev.jac_tvec(Xd + h * D, Lam, Zp)
    ev.jac_tvec(Xd - h * D, Lam, Zm)
    fd = (Zp - Zm) / (2 * h)
    rows = torch.arange(0, B, B // 16, device="cuda")
    o = LT.Problem(g)
    Xs, Ls, Ds = (t[rows].cpu().numpy() for t in (Xd, Lam, D))
    Wr, S = _oracle(o, Xs, Ls, Ds)
    _assert_within(W[rows].cpu().numpy(), Wr, S, name)
    tol = 1e-6 * (W.abs().amax(1, keepdim=True) + 1.0)
    assert bool(((W - fd).abs() <= tol).all()), name
    Zt = torch.empty_like(W)
    ev.jac_tvec(Xd, Lam, Zt)
    assert torch.equal(Z, Zt)
    ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["S10_tempest_ts100", "G7_skywalker_ts100"])
def test_degenerate_inputs_are_non_finite_where_jac_tvec_is(name):
    """Va = 0, cos(gamma) = 0, a node on the loiter centre, G7 dist = 0: no component of w is finite where z is not"""
    g = load_golden(name)
    ts = int(g["ts"])
    X, Lam, D = _inputs(g, 6, 4)
    X[1, 1 + 11 * 5 + 3] = 0.0
    X[2, 1 + 11 * 9 + 4] = np.pi / 2
    X[3, 1 + 11 * 7 + 0], X[3, 1 + 11 * 7 + 1] = g["goal_ned"][0], g["goal_ned"][1]
    X[4, 1 + 11 * ts + 0], X[4, 1 + 11 * ts + 1] = X[4, 1], X[4, 2]
    ev = T.Evaluator.from_golden(g)
    W, Z = _run(ev, X, Lam, D, pad=0)
    Zt = torch.empty_like(Z)
    ev.jac_tvec(_dev(X), _dev(Lam), Zt)
    W, Zt = W.cpu().numpy(), Zt.cpu().numpy()
    assert not np.isfinite(Zt).all()
    assert not np.isfinite(W[~np.isfinite(Zt)]).any()
    assert np.isfinite(W[[0, 5]]).all()
    ev.close()


@pytest.mark.gpu
def test_misuse_is_reported_not_executed():
    """null pointers, short leading dimensions, host pointers and B = 0: each returns its code, nothing launches"""
    g = load_golden("S10_tempest_ts100")
    ev = T.Evaluator.from_golden(g)
    L, h, n, neF = ev.L, ev.h, ev.n, ev.neF
    X, Lam, D = (_dev(a) for a in _inputs(g, 2, 1))
    W = torch.empty(2, n, dtype=torch.float64, device="cuda")
    x, l, d, w = X.data_ptr(), Lam.data_ptr(), D.data_ptr(), W.data_ptr()
    before = L.tolcuda_launch_count(h)
    cases = [(None, n, l, neF, d, n, w, n, None, 0, 0, -1), (x, n, None, neF, d, n, w, n, None, 0, 0, -1),
             (x, n, l, neF, None, n, w, n, None, 0, 0, -1), (x, n, l, neF, d, n, None, n, None, 0, 0, -1),
             (x, n - 1, l, neF, d, n, w, n, None, 0, 0, -1), (x, n, l, neF - 1, d, n, w, n, None, 0, 0, -1),
             (x, n, l, neF, d, n - 1, w, n, None, 0, 0, -1), (x, n, l, neF, d, n, w, n - 1, None, 0, 0, -1),
             (x, n, l, neF, d, n, w, n, w, n - 1, 0, -1), (x, n, l, neF, d, n, w, n, None, 0, T.evaluator.HOST_PTRS, -2)]
    for a in cases:
        assert L.tolcuda_lag_hess_vec(h, 2, *a[:-1]) == a[-1], a
    assert L.tolcuda_lag_hess_vec(h, 0, None, 0, None, 0, None, 0, None, 0, None, 0, 0) == 0
    assert L.tolcuda_lag_hess_vec(h, -1, x, n, l, neF, d, n, w, n, None, 0, 0) == -1
    assert L.tolcuda_launch_count(h) == before
    assert L.tolcuda_lag_hess_vec(h, 2, x, n, l, neF, d, n, w, n, None, 0, 0) == 0
    assert L.tolcuda_launch_count(h) == before + 1
    ev.close()
