"""Every kernel instance of the built library against a reference.

fg_kernels.cu builds one entry function per combination of family (kernel A or L; plain, goal table or HVP), formulation,
wind model, launch bounds (MAXT, MINB), mode and LOOP (runs of `per` >= 2 trajectories per CTA), and the host dispatcher
(launch_any -> launch_flavour -> launch_sel -> launch_cta / launch_long) picks one per call.  ROWS below has one row per
entry function, keyed as the function's template arguments, with the inputs that make the dispatcher pick it.

Without a GPU: the table's keys are exactly the STO_ENTRY symbols of the built libtolcuda.so (an instance added without
a row fails here, by name), and the rows spread the boundary trajectory lengths over formulations and modes.
On the GPU, one case per row:
  * the launch is recorded with torch.profiler and the kernel it ran must be the row's instance;
  * F and G (compact rows expanded first) against the CPU port with the 1e-14 + 1e-12*|ref| bar, goal-table rows against
    a port built with each row's goal;
  * the summary against the same quantities formed from the port's F;
  * J d and J^T lambda against products formed from the port's G rows and the pattern (per entry 1e-14 + 1e-12 * sum of
    |terms|); w = D_x[J^T lambda] d against the torch restatement (oracle/lagrangian_torch.py) with its sum of |terms|
    as the scale, and z bit for bit what tolcuda_jac_tvec writes;
  * padding columns stay NaN; wind model 3 rows first assert that every node lies inside the fixture cube."""
import collections
import functools
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

import tol_b200 as T
from conftest import RTOL, ATOL, assert_parity, load_golden

PLAIN, SUMMARY, COMPACT, JVP, VJP, FONLY, FSUMM, HVP = range(8)
MODE_NAMES = ("plain", "summary", "compact", "jvp", "vjp", "fonly", "fsumm", "hvp")
CTA, CTA_GOALS, CTA_HVP = "fg_cta_kernel", "fg_cta_goals_kernel", "fg_cta_hvp_kernel"
LONG, LONG_GOALS, LONG_HVP = "fg_long_kernel", "fg_long_goals_kernel", "fg_long_hvp_kernel"
FORMS = {"S10": 10, "G7": 7}

# The other two entry functions of the library, and the tests that launch them
OTHER_ENTRIES = {
    "expand_kernel": "tests/test_gpu_parity.py::test_compact_rows_path_equals_full_rows, "
                     "tests/test_gpu_parity.py::test_more_rows_than_one_grid_dimension",
    "repack_kernel": "tests/test_gpu_parity.py::test_csc_repack_on_the_device, "
                     "tests/test_gpu_parity.py::test_more_rows_than_one_grid_dimension",
}

# ---- the instance table ---------------------------------------------------------------------------------------------
#
# One shape per line: (family, MODE, MAXT, MINB, LOOP); kernel L has no launch bounds or LOOP in its template (None).
# Each shape is instantiated for both formulations and wind models 0, 1 and 3 (COMBOS), which makes one row per entry.
SHAPES = [
    # kernel A, one trajectory per CTA (LOOP false) and runs of trajectories (LOOP true)
    (CTA, PLAIN, 128, 4, False), (CTA, PLAIN, 128, 4, True), (CTA, PLAIN, 256, 2, False), (CTA, PLAIN, 256, 2, True),
    (CTA, SUMMARY, 128, 4, False), (CTA, SUMMARY, 128, 4, True), (CTA, SUMMARY, 256, 2, False), (CTA, SUMMARY, 256, 2, True),
    (CTA, COMPACT, 128, 4, False), (CTA, COMPACT, 128, 4, True), (CTA, COMPACT, 256, 2, False), (CTA, COMPACT, 256, 2, True),
    (CTA, JVP, 128, 4, False), (CTA, JVP, 128, 4, True), (CTA, JVP, 256, 2, False), (CTA, JVP, 256, 2, True),
    (CTA, VJP, 128, 4, False), (CTA, VJP, 128, 4, True), (CTA, VJP, 256, 2, False), (CTA, VJP, 256, 2, True),
    (CTA, FONLY, 128, 8, False), (CTA, FONLY, 128, 8, True), (CTA, FONLY, 256, 4, False), (CTA, FONLY, 256, 4, True),
    (CTA, FSUMM, 128, 8, False), (CTA, FSUMM, 128, 8, True), (CTA, FSUMM, 256, 4, False), (CTA, FSUMM, 256, 4, True),
    # kernel A with a goal table
    (CTA_GOALS, PLAIN, 128, 4, False), (CTA_GOALS, PLAIN, 128, 4, True),
    (CTA_GOALS, PLAIN, 256, 2, False), (CTA_GOALS, PLAIN, 256, 2, True),
    (CTA_GOALS, SUMMARY, 128, 4, False), (CTA_GOALS, SUMMARY, 128, 4, True),
    (CTA_GOALS, SUMMARY, 256, 2, False), (CTA_GOALS, SUMMARY, 256, 2, True),
    (CTA_GOALS, COMPACT, 128, 4, False), (CTA_GOALS, COMPACT, 128, 4, True),
    (CTA_GOALS, COMPACT, 256, 2, False), (CTA_GOALS, COMPACT, 256, 2, True),
    (CTA_GOALS, FONLY, 128, 8, False), (CTA_GOALS, FONLY, 128, 8, True),
    (CTA_GOALS, FONLY, 256, 4, False), (CTA_GOALS, FONLY, 256, 4, True),
    (CTA_GOALS, FSUMM, 128, 8, False), (CTA_GOALS, FSUMM, 128, 8, True),
    (CTA_GOALS, FSUMM, 256, 4, False), (CTA_GOALS, FSUMM, 256, 4, True),
    # kernel A, Hessian-of-the-Lagrangian products
    (CTA_HVP, HVP, 128, 4, False), (CTA_HVP, HVP, 128, 4, True), (CTA_HVP, HVP, 256, 2, False), (CTA_HVP, HVP, 256, 2, True),
    # kernel L: ts > 256, or option "kernel" = 2 at any ts
    (LONG, PLAIN, None, None, None), (LONG, SUMMARY, None, None, None), (LONG, COMPACT, None, None, None),
    (LONG, JVP, None, None, None), (LONG, VJP, None, None, None),
    (LONG_GOALS, PLAIN, None, None, None), (LONG_GOALS, SUMMARY, None, None, None), (LONG_GOALS, COMPACT, None, None, None),
    (LONG_HVP, HVP, None, None, None),
]
COMBOS = [("S10", 0), ("S10", 1), ("S10", 3), ("G7", 0), ("G7", 1), ("G7", 3)]

# trajectory lengths at the kernels' boundaries: the MAXT switch (128 / 129), a last tile exactly full (32, 64, 128,
# 256), kernel A's largest grid (256), odd lengths whose records start 8 mod 16 in the MAXT = 256 instances (129, 255),
# and the first length kernel L alone serves (257)
TS_A128 = (31, 32, 64, 127, 128)
TS_A256 = (129, 255, 256)
TS_L = (31, 32, 64, 127, 128, 129, 255, 256)
BOUNDARY_TS = (31, 32, 64, 127, 128, 129, 255, 256, 257)

Row = collections.namedtuple("Row", "key mission ts wind mode goals kernel per B")


def _key_name(key):
    fam, form, wind, maxt, minb, mode, loop = key
    args = [form, wind] + ([] if maxt is None else [maxt, minb]) + ([] if fam.endswith("hvp_kernel") else [mode])
    args += [] if loop is None else [int(loop)]
    return "%s<%s>" % (fam, ",".join(str(a) for a in args))


def _rows():
    rows = []
    for s, (fam, mode, maxt, minb, loop) in enumerate(SHAPES):
        for c, (mission, wind) in enumerate(COMBOS):
            key = (fam, FORMS[mission], wind, maxt, minb, mode, loop)
            if maxt is None:
                # kernel L: ts = 257 (the dispatcher's own choice) for one wind model per shape in both formulations,
                # option "kernel" = 2 at a boundary length below that for the other two
                if wind == (0, 1, 3)[s % 3]:
                    ts, kernel = 257, 0
                else:
                    ts, kernel = TS_L[(s + 3 * c) % len(TS_L)], 2
            else:
                tss = TS_A128 if maxt == 128 else TS_A256
                ts, kernel = tss[(s + c) % len(tss)], 0
            # LOOP: `per` 2, 3 or 4 with B = 2 per + 1 and tail_x4 = 0, so the grid is two runs and one single CTA
            per = 2 + (s + c) % 3 if loop else 1
            B = 2 * per + 1 if loop else 3
            rows.append(Row(key, mission, ts, wind, mode, fam in (CTA_GOALS, LONG_GOALS), kernel, per, B))
    return rows


ROWS = _rows()


def _row_id(r):
    return "%s-%s-w%d-ts%d-%s%s" % (r.key[0][3:-7], r.mission, r.wind, r.ts, MODE_NAMES[r.mode],
                                    "-loop%d" % r.per if r.key[6] else "")


# ---- no GPU needed ---------------------------------------------------------------------------------------------------

def _cuobjdump():
    exe = shutil.which("cuobjdump")
    return exe or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)


_ENTRY = re.compile(r"\d(fg_[a-z_]+?_kernel|expand_kernel|repack_kernel)(?:I(\w*?)EEv|E)")


def _parse_entry(sym):
    """(family, FORM, WIND, MAXT, MINB, MODE, LOOP) of a mangled fg_* entry; the bare name for the others"""
    m = _ENTRY.search(sym)
    assert m, "unrecognised entry function " + sym
    fam, targs = m.group(1), m.group(2)
    if not fam.startswith("fg_"):
        return fam
    args = [int(v) for _, v in re.findall(r"L([ib])(-?\d+)E", targs)]
    return _key_of(fam, args)


def _key_of(fam, args):
    """the table key from a family and its template arguments in declaration order"""
    if fam in (CTA, CTA_GOALS):
        form, wind, maxt, minb, mode, loop = args
    elif fam == CTA_HVP:
        (form, wind, maxt, minb, loop), mode = args, HVP
    elif fam in (LONG, LONG_GOALS):
        (form, wind, mode), maxt, minb, loop = args, None, None, None
    elif fam == LONG_HVP:
        (form, wind), mode, maxt, minb, loop = args, HVP, None, None, None
    else:
        raise AssertionError("unknown kernel family " + fam)
    return (fam, form, wind, maxt, minb, mode, None if loop is None else bool(loop))


def test_the_table_names_every_entry_function_of_the_library():
    """the STO_ENTRY symbols of libtolcuda.so (cuobjdump -symbols) are exactly the table's keys plus OTHER_ENTRIES"""
    exe = _cuobjdump()
    if not exe or not os.path.exists(T.lib.LIB_PATH):
        pytest.skip("cuobjdump or the built library is missing")
    out = subprocess.run([exe, "-symbols", T.lib.LIB_PATH], capture_output=True, text=True, timeout=300, check=True).stdout
    syms = [ln.split()[-1] for ln in out.splitlines() if "STO_ENTRY" in ln]
    built = [_parse_entry(s) for s in syms]
    assert len(built) == len(set(built)), "two entry functions parse to one key"
    others = {k for k in built if isinstance(k, str)}
    assert others == set(OTHER_ENTRIES), others
    built = {k for k in built if not isinstance(k, str)}
    table = [r.key for r in ROWS]
    assert len(table) == len(set(table)), "the table names an instance twice"
    missing = sorted(_key_name(k) for k in built - set(table))
    extra = sorted(_key_name(k) for k in set(table) - built)
    assert not missing, "entry functions without a row in the table: %s" % missing
    assert not extra, "rows for instances the library does not build: %s" % extra


def test_the_table_spreads_the_boundary_lengths():
    """every boundary ts reaches both formulations, and the plain, summary, JVP or VJP and HVP modes at least once
    each; every row's ts is one the dispatcher sends to the row's launch bounds"""
    seen = collections.defaultdict(set)
    for r in ROWS:
        seen[r.ts].add(r.mission)
        seen[r.ts].add({PLAIN: "plain", SUMMARY: "summary", JVP: "op", VJP: "op", HVP: "hvp"}.get(r.mode))
        fam, _, _, maxt, _, mode, loop = r.key
        if maxt is None:
            assert r.kernel == 2 or r.ts > 256, r
        else:
            assert r.kernel != 2 and (r.ts <= 128) == (maxt == 128) and r.ts <= 256, r
            assert loop == (r.per > 1), r
    for ts in BOUNDARY_TS:
        assert {"S10", "G7", "plain", "summary", "op", "hvp"} <= seen[ts], (ts, seen[ts])


def test_kernel_names_parse_like_the_mangled_symbols():
    """the profiler's demangled names give the keys the mangled symbols give"""
    ns = "_ZN46_GLOBAL__N__5e0e695b_13_fg_kernels_cu_59072e7d"
    assert _parse_entry(ns + "13fg_cta_kernelILi7ELi3ELi256ELi2ELi0ELb1EEEv7FgConstiiPKdlPdlS4_liiiS4_l") == \
        _parse_name("void (anonymous namespace)::fg_cta_kernel<7, 3, 256, 2, 0, true>(FgConst, int, int, double const*)") == \
        (CTA, 7, 3, 256, 2, PLAIN, True)
    assert _parse_entry(ns + "17fg_cta_hvp_kernelILi10ELi0ELi128ELi4ELb0EEEv7FgConstiiPKdlPdlS4_lS3_lS4_l") == \
        _parse_name("void (anonymous namespace)::fg_cta_hvp_kernel<10, 0, 128, 4, false>(FgConst, int)") == \
        (CTA_HVP, 10, 0, 128, 4, HVP, False)
    assert _parse_entry(ns + "14fg_long_kernelILi7ELi3ELi2EEEv7FgConstPKdlPdlS4_liiiS4_l") == \
        _parse_name("void (anonymous namespace)::fg_long_kernel<7, 3, 2>(FgConst, double const*, long)") == \
        (LONG, 7, 3, None, None, COMPACT, None)
    assert _parse_entry(ns + "18fg_long_hvp_kernelILi10ELi1EEEv7FgConstPKdlPdlS4_lS3_lS4_l") == (LONG_HVP, 10, 1, None, None, HVP, None)


# ---- GPU -------------------------------------------------------------------------------------------------------------

_NAME = re.compile(r"(fg_[a-z_]+?_kernel)<([^<>]*)>")


def _parse_name(name):
    """the table key of a demangled kernel name (torch.profiler), None if it is not an fg_* kernel"""
    m = _NAME.search(name)
    if not m:
        return None
    args = [1 if a.strip() == "true" else 0 if a.strip() == "false" else int(re.sub(r"\D", "", a) or 0)
            for a in m.group(2).split(",")]
    return _key_of(m.group(1), args)


def _recorded_kernels(fn):
    """fn() under torch.profiler (CUDA activity): the names of the kernels it ran"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


_BASE = {"S10": "S10_tempest_ts100_wind3", "G7": "G7_skywalker_ts45_wind3"}  # parameters, goal and wind cube
BMAX = 9


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


class _Case:
    """one (mission, ts, wind): the context, BMAX states, the port's F and G rows, random d and lambda"""

    def __init__(self, mission, ts, wind):
        g = load_golden(_BASE[mission])
        self.g, self.mission, self.ts, self.wind = g, mission, ts, wind
        lm = g["lm"]
        cfg = T.make_config(mission, ts, g["ac"], g["gn"], g["goal_ned"],
                            limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]])
        self.X = T.synth.batch(T.initial_guess(cfg), 4321 + ts, 0, BMAX)
        self.ev = T.Evaluator(mission, ts, g["ac"], g["gn"], g["goal_ned"], 1 if wind == 3 else wind)
        if wind == 3:
            self.ev.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
            self._assert_inside_the_cube(self.X)
        self.goals = T.synth.goals(mission, 0, BMAX + 1)
        self.ports = [self._port(g["goal_ned"])] + [None] * (BMAX + 1)
        p = self.ports[0]
        self.n, self.neF, self.neG, self.nb = p.n, p.neF, p.neG, p.nb
        self.iG, self.jG = p.pattern()
        rng = np.random.default_rng(ts * 10 + wind)
        self.D, self.Lam = rng.uniform(-1, 1, (BMAX, self.n)), rng.uniform(-1, 1, (BMAX, self.neF))
        self._hvp = {}

    def _port(self, goal):
        import portclient as P
        g = self.g
        p = P.PortProblem(self.mission, self.ts, g["ac"], g["gn"], goal, 1 if self.wind == 3 else self.wind)
        if self.wind == 3:
            p.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
        return p

    def _assert_inside_the_cube(self, X):
        """every node of every window strictly inside the cube (where the port is the reference bit for bit)"""
        g = self.g
        N = X[:, 1:].reshape(X.shape[0], self.ts + 1, 11)
        d = g["grid_datum"]
        for s, grid in ((N[..., 1] + d[0], g["grid_x"]), (N[..., 0] + d[1], g["grid_y"]), (-N[..., 2] + d[2], g["grid_z"])):
            assert (s > grid[0]).all() and (s < grid[-1]).all(), "a node outside the interior of the wind cube"

    def port_rows(self, B, goal_rows=None):
        """the port's F and G for states 0..B-1; goal_rows: row b with goal self.goals[goal_rows[b]]; S10's boundary-row
        dt entries, which the reference leaves undefined, as 0 (what the kernels write)"""
        F, G = np.empty((B, self.neF)), np.empty((B, self.neG))
        for b in range(B):
            if goal_rows is None:
                p = self.ports[0]
            else:
                k = goal_rows[b]
                if self.ports[1 + k] is None:
                    self.ports[1 + k] = self._port(self.goals[k])
                p = self.ports[1 + k]
            F[b], G[b] = p.eval(self.X[b])
        if self.mission == "S10":
            G[:, self.ports[0].ub_mask()] = 0.0
        return F, G

    def hvp_reference(self, B):
        """w and its sum of |terms| from the torch restatement, for states 0..B-1"""
        import lagrangian_torch as LT
        o = None
        for b in range(B):
            if b not in self._hvp:
                if o is None:
                    o = LT.Problem(self.g, wind_model=self.wind, ts=self.ts)
                x, lam, d = self.X[b], self.Lam[b], self.D[b]
                self._hvp[b] = (o.lag_hess_vec(x, lam, d).numpy(), o.term_scale(x, lam, d).numpy())
        return np.stack([self._hvp[b][0] for b in range(B)]), np.stack([self._hvp[b][1] for b in range(B)])


@functools.lru_cache(maxsize=None)
def _case(mission, ts, wind):
    return _Case(mission, ts, wind)


def _nan(B, m):
    return torch.full((B, m), float("nan"), dtype=torch.float64, device="cuda")


PAD = 3


def _summary_reference(F, nb, mission, ts):
    d = F[:, 1:1 + 8 * ts]
    bnd = np.abs(F[:, -nb:])
    if mission == "G7":
        bnd[:, -1] = np.maximum(F[:, -1], 0.0)
    return F[:, 0], np.abs(d).max(axis=1), bnd.max(axis=1), (d * d).sum(axis=1)


def _check_summary(S, Fr, c, what):
    obj, dmax, bmax, ssq = _summary_reference(Fr, c.nb, c.mission, c.ts)
    for k, (v, ref) in enumerate(((obj, "objective"), (dmax, "max |defect|"), (bmax, "max boundary violation"))):
        assert_parity(S[:, k], v, "%s summary %s" % (what, ref))
    assert (np.abs(S[:, 3] - ssq) <= 1e-12 * np.abs(ssq)).all(), (what, "sum of squared defects", S[:, 3], ssq)


def _op_reference(iG, jG, Gr, D, Lam, neF, n):
    """y = J d, z = J^T lambda and the matching sums of absolute terms, from coordinate-order G rows (float64,
    numpy scatter-adds)"""
    B = Gr.shape[0]
    Y, Ya, Z, Za = np.zeros((B, neF)), np.zeros((B, neF)), np.zeros((B, n)), np.zeros((B, n))
    for b in range(B):
        ty = Gr[b] * D[b, jG]
        np.add.at(Y[b], iG, ty)
        np.add.at(Ya[b], iG, np.abs(ty))
        tz = Gr[b] * Lam[b, iG]
        np.add.at(Z[b], jG, tz)
        np.add.at(Za[b], jG, np.abs(tz))
    return Y, Ya, Z, Za


def _assert_within(got, ref, scale, what):
    assert np.isfinite(got).all(), what + ": non-finite values"
    e = np.abs(got - ref) - (ATOL + RTOL * scale)
    assert e.max() <= 0, (what, np.unravel_index(e.argmax(), e.shape), e.max())


@pytest.mark.gpu
@pytest.mark.parametrize("row", ROWS, ids=_row_id)
def test_instance_against_the_reference(row):
    c = _case(row.mission, row.ts, row.wind)
    ev, B, mode, what = c.ev, row.B, row.mode, _key_name(row.key)
    ev.set_option("kernel", row.kernel)
    ev.set_option("per", row.per)
    ev.set_option("tail_x4", 0)
    L = ev.L
    Xd = _dev(c.X[:B])
    flags = T.evaluator.DEVICE_PTRS
    need_g = mode in (PLAIN, SUMMARY, COMPACT)
    glen = c.ev.compact_len if mode == COMPACT else c.neG
    if mode in (JVP, VJP, HVP):
        Dd, Ld = _dev(c.D[:B]), _dev(c.Lam[:B])
        Y, Z, W = _nan(B, c.neF + PAD), _nan(B, c.n + PAD), _nan(B, c.n + PAD)
        launch = {JVP: lambda: ev.jac_vec(Xd, Dd, Y), VJP: lambda: ev.jac_tvec(Xd, Ld, Z),
                  HVP: lambda: ev.lag_hess_vec(Xd, Ld, Dd, W, Z)}[mode]
    else:
        F, G = _nan(B, c.neF + PAD), _nan(B, glen + PAD)
        S = _nan(B, 4 + PAD) if mode in (SUMMARY, FSUMM) else None
        flags |= T.evaluator.NEED_F | (T.evaluator.NEED_G if need_g else 0) | (T.evaluator.COMPACT_G if mode == COMPACT else 0)
        ptr = lambda t: None if t is None else t.data_ptr()
        ld = lambda t: 0 if t is None else t.stride(0)
        if row.goals:
            ev.set_goals(c.goals)
            row0 = 1
            launch = lambda: T.lib.check(L.tolcuda_eval_batch_goals(ev.h, row0, B, Xd.data_ptr(), Xd.stride(0), F.data_ptr(),
                                                                  F.stride(0), G.data_ptr(), G.stride(0), ptr(S), ld(S), flags))
        else:
            launch = lambda: T.lib.check(L.tolcuda_eval_batch_summary(ev.h, B, Xd.data_ptr(), Xd.stride(0), F.data_ptr(),
                                                                    F.stride(0), G.data_ptr(), G.stride(0), ptr(S), ld(S),
                                                                    flags))
    ev._follow_torch(Xd)
    names = _recorded_kernels(launch)
    ran = [k for k in map(_parse_name, names) if k is not None]
    assert ran == [row.key], "%s: the launch ran %s" % (what, names)

    if mode in (JVP, VJP, HVP):
        Fr, Gr = c.port_rows(B)
        Yr, Ya, Zr, Za = _op_reference(c.iG, c.jG, Gr, c.D[:B], c.Lam[:B], c.neF, c.n)
        Yg, Zg, Wg = Y.cpu().numpy(), Z.cpu().numpy(), W.cpu().numpy()
        if mode == JVP:
            assert np.isnan(Yg[:, c.neF:]).all() and np.isnan(Zg).all() and np.isnan(Wg).all(), what + ": padding"
            _assert_within(Yg[:, :c.neF], Yr, Ya, what + " J d")
            return
        assert np.isnan(Zg[:, c.n:]).all(), what + ": padding"
        _assert_within(Zg[:, :c.n], Zr, Za, what + " J^T lambda")
        if mode == HVP:
            assert np.isnan(Wg[:, c.n:]).all(), what + ": padding"
            Wr, Ws = c.hvp_reference(B)
            _assert_within(Wg[:, :c.n], Wr, Ws, what + " w")
            Zt = _nan(B, c.n + PAD)
            ev.jac_tvec(Xd, Ld, Zt)
            assert torch.equal(Z[:, :c.n], Zt[:, :c.n]), what + ": z differs from tolcuda_jac_tvec's"
        return

    goal_rows = list(range(1, B + 1)) if row.goals else None
    Fr, Gr = c.port_rows(B, goal_rows)
    Fg, Gg = F.cpu().numpy(), G.cpu().numpy()
    assert np.isnan(Fg[:, c.neF:]).all() and np.isnan(Gg[:, glen:]).all(), what + ": padding"
    assert_parity(Fg[:, :c.neF], Fr, what + " F")
    if not need_g:
        assert np.isnan(Gg).all(), what + ": G written by an F-only launch"
    elif mode == COMPACT:
        assert_parity(T.evaluator.expand_compact_g(row.mission, row.ts, np.ascontiguousarray(Gg[:, :glen])), Gr,
                      what + " G (compact rows expanded)")
    else:
        assert_parity(Gg[:, :c.neG], Gr, what + " G")
    if S is not None:
        Sg = S.cpu().numpy()
        assert np.isnan(Sg[:, 4:]).all(), what + ": padding"
        _check_summary(Sg[:, :4], Fr, c, what)
