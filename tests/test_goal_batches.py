"""Per-trajectory goals (tolcuda_set_goals / tolcuda_eval_batch_goals, tolbatch --goals).

Without a GPU: the C entry points refuse a null handle before touching CUDA, tolbatch refuses a bad goal file and
--goals with --gather-gpu before any device query, and synth.goals does not depend on the sharding.
On the GPU: every row of a launch with a goal table is bit for bit the row a context created with that row's goal
writes for the same x, under every flavour, pointer kind and option; the rows agree with the CPU port and the
reference; misuse changes nothing."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import tol_b200 as T
from conftest import ROOT, assert_parity, load_golden

EV = T.evaluator
TOLBATCH = os.path.join(ROOT, "tol_b200", "tolbatch")
POS = ["0", "0", "70", "0", "-100", "0", "100", "tempest", "S10"]


# ---- no GPU needed ---------------------------------------------------------------------------------------------------

def test_goal_calls_refuse_a_null_handle_without_cuda():
    L = T.load()
    g = np.zeros((2, 4))
    assert L.tolcuda_set_goals(None, 2, g.ctypes.data, 4) == -1
    assert b"null handle" in L.tolcuda_last_error()
    x = np.zeros(16)
    assert L.tolcuda_eval_batch_goals(None, 0, 1, x.ctypes.data, 16, x.ctypes.data, 16, x.ctypes.data, 16, None, 0,
                                      EV.NEED_F | EV.HOST_PTRS) == -1
    assert b"null handle" in L.tolcuda_last_error()


def _tolbatch(args):
    if not os.path.exists(TOLBATCH):
        pytest.skip("tolbatch is not built")
    return subprocess.run([TOLBATCH] + POS + args, capture_output=True, text=True, timeout=60)


def test_tolbatch_refuses_bad_goal_files_before_any_device_query(tmp_path):
    """exit code 2 and a message naming the goal file -- never the device query's failure, which comes later"""
    good = tmp_path / "good.txt"
    good.write_text("0 -100 0 100\n400 0 0 0\n")
    cases = [(["--goals", str(tmp_path / "missing.txt")], "cannot open goal file")]
    for name, text, msg in (("short_line", "0 -100 0\n", "want `Eg Ng Ug Rg`"),
                            ("word", "0 -100 zero 100\n", "want `Eg Ng Ug Rg`"),
                            ("extra", "0 -100 0 100 7\n", "found more"),
                            ("blank_line", "0 -100 0 100\n\n1 2 3 4\n", "want `Eg Ng Ug Rg`"),
                            ("nan", "0 nan 0 100\n", "want `Eg Ng Ug Rg`"),
                            ("empty", "", "no goals")):
        p = tmp_path / (name + ".txt")
        p.write_text(text)
        cases.append((["--goals", str(p)], msg))
    cases.append((["--goals", str(good), "--batch", "3"], "2 goals for --batch 3"))     # short file
    cases.append((["--goals", str(good), "--batch", "1"], "2 goals for --batch 1"))
    cases.append((["--goals", str(good), "--gather-gpu", "0"], "--goals cannot be combined with --gather-gpu"))
    for args, msg in cases:
        r = _tolbatch(args)
        assert r.returncode == 2 and msg in r.stderr and r.stdout == "", (args, r.stderr)
        assert "device query" not in r.stderr


@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_synth_goals_are_shard_invariant(mission):
    full = T.synth.goals(mission, 0, 1000)
    for world in (1, 3, 8):
        parts = [T.synth.goals(mission, *T.synth.shard_range(1000, r, world)) for r in range(world)]
        assert np.array_equal(np.concatenate(parts), full)
    assert len({tuple(r) for r in full}) == 1000  # all distinct
    if mission == "G7":  # every quadrant of chi_d, and each axis from both sides
        chi = np.arctan2(full[:, 1], full[:, 0])
        for lo in (-np.pi, -np.pi / 2, 0.0, np.pi / 2):
            assert ((chi > lo) & (chi < lo + np.pi / 2)).sum() > 100
        for axis in (0.0, np.pi / 2, -np.pi / 2):
            assert (np.abs(chi - axis) < 1e-8).sum() > 50
        assert (np.abs(np.abs(chi) - np.pi) < 1e-8).sum() > 50 and (chi > 0).any() and (chi < 0).any()


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


def _inputs(g, mission, ts, B):
    x0 = T.initial_guess(T.make_config(mission, ts, g["ac"], g["gn"], g["goal_ned"]))
    return T.synth.batch(x0, T.synth.SEED_S10 if mission == "S10" else T.synth.SEED_G7, 0, B)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _call(ev, X, flags, needF, needG, summary, compact, row0=None):
    """one tolcuda_eval_batch_summary (row0 None) or tolcuda_eval_batch_goals call; numpy X: host pointers, torch X:
    device pointers.  Returns F, G, S as numpy arrays (NaN where nothing was written)."""
    import torch
    B = X.shape[0]
    dev = hasattr(X, "data_ptr")
    lenG = ev.compact_len if compact else ev.neG
    shapes = [(B, ev.neF) if needF else None, (B, lenG) if needG else None, (B, 4) if summary else None]
    if dev:
        ev._follow_torch(X)
        outs = [torch.full(s, float("nan"), dtype=torch.float64, device=X.device) if s else None for s in shapes]
        p = [o.data_ptr() if o is not None else None for o in [X] + outs]
    else:
        outs = [np.full(s, np.nan) if s else None for s in shapes]
        p = [o.ctypes.data if o is not None else None for o in [X] + outs]
    ld = [o.shape[1] if o is not None else 0 for o in [X] + outs]
    flags |= (EV.NEED_F if needF else 0) | (EV.NEED_G if needG else 0) | (EV.COMPACT_G if compact else 0)
    flags |= EV.DEVICE_PTRS if dev else EV.HOST_PTRS
    args = (p[0], ld[0], p[1], ld[1], p[2], ld[2], p[3], ld[3], flags)
    if row0 is None:
        T.lib.check(ev.L.tolcuda_eval_batch_summary(ev.h, B, *args))
    else:
        T.lib.check(ev.L.tolcuda_eval_batch_goals(ev.h, int(row0), B, *args))
    if dev:
        torch.cuda.synchronize()
        outs = [o.cpu().numpy() if o is not None else None for o in outs]
    return outs


# flavour name -> (device pointers, flags, needF, needG, summary, compact rows, options)
FLAVOURS = {
    "device F+G": (True, 0, True, True, False, False, {}),
    "device COMPACT_G": (True, 0, True, True, False, True, {}),
    "device F only": (True, 0, True, False, False, False, {}),
    "device summary only": (True, 0, False, False, True, False, {}),
    "device F+G+summary": (True, 0, True, True, True, False, {}),
    # tail_x4 = 0: no single-trajectory tail, so that a batch of 64 forms runs of `per` trajectories per CTA (and a
    # goal slot is reused within a run from per = 3 on)
    "device per=1": (True, 0, True, True, False, False, {"per": 1}),
    "device per=2": (True, 0, True, True, True, False, {"per": 2, "tail_x4": 0}),
    "device per=3": (True, 0, True, False, False, False, {"per": 3, "tail_x4": 0}),
    "device per=3 F+G": (True, 0, True, True, True, False, {"per": 3, "tail_x4": 0}),
    "device per=4": (True, 0, True, True, False, False, {"per": 4, "tail_x4": 0}),
    "device kernel=2": (True, 0, True, True, True, False, {"kernel": 2}),
    "host compact": (False, 0, True, True, False, False, {}),
    "host full rows": (False, EV.FULL_G_COPY, True, True, False, False, {}),
    "host full_rows_pct=50": (False, 0, True, True, False, False, {"full_rows_pct": 50, "chunk_mb": 1}),
    "host COMPACT_G": (False, 0, True, True, False, True, {}),
    "host summary only": (False, 0, False, False, True, False, {}),
}


@pytest.mark.gpu
@pytest.mark.parametrize("mission,ts,wind", [("S10", 1, 1), ("S10", 45, 1), ("S10", 100, 1), ("S10", 200, 1),
                                             ("S10", 300, 1), ("S10", 100, 3), ("G7", 1, 1), ("G7", 45, 1),
                                             ("G7", 100, 1), ("G7", 200, 1), ("G7", 300, 1), ("G7", 45, 3)])
def test_rows_equal_a_context_created_with_the_rows_goal(mission, ts, wind):
    """K = 8 distinct goals (G7: all four quadrants of chi_d and the axes) cycle over B rows; row b of F, G and summary
    equals bit for bit row b evaluated by a context created with goal b % K, under the same flavour and options; the
    table starts 5 rows before the call's first row (row0 = 5)"""
    import torch
    g = _fixture(mission, wind)
    K, B, row0 = 8, 64, 5
    goals = T.synth.goals(mission, 0, K)
    X = _inputs(g, mission, ts, B)
    Xd = torch.from_numpy(X).cuda()
    table = np.concatenate([T.synth.goals(mission, 100, 100 + row0), goals[np.arange(B) % K]])
    for name, (dev, flags, needF, needG, summ, compact, opts) in FLAVOURS.items():
        ev = _context(g, mission, ts, wind, g["goal_ned"], opts)
        ev.set_goals(table)
        got = _call(ev, Xd if dev else X, flags, needF, needG, summ, compact, row0)
        for k in range(K):
            rows = np.arange(k, B, K)
            ek = _context(g, mission, ts, wind, goals[k], opts)
            want = _call(ek, Xd[rows] if dev else np.ascontiguousarray(X[rows]), flags, needF, needG, summ, compact)
            for a, b, what in zip(got, want, ("F", "G", "summary")):
                if b is not None:
                    assert np.array_equal(_bits(a[rows]), _bits(b)), "%s ts=%d wind %d, %s: %s of goal %d" % (
                        mission, ts, wind, name, what, k)
            ek.close()
        ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mission", ["S10", "G7"])
def test_overlapping_launches_with_alternating_buffers(mission):
    """two TOLCUDA_OVERLAP_DISJOINT launches into two result-buffer sets, different rows of the table each, as a
    stream of SNOPT iterations enqueues them: each equals its own synchronous launch"""
    import torch
    g = _fixture(mission, 1)
    ts, B = 200, 4096
    ev = _context(g, mission, ts, 1, g["goal_ned"])
    ev.set_goals(T.synth.goals(mission, 0, 2 * B))
    Xd = torch.from_numpy(_inputs(g, mission, ts, B)).cuda()
    bufs = [(torch.empty(B, ev.neF, dtype=torch.float64, device="cuda"),
             torch.empty(B, ev.neG, dtype=torch.float64, device="cuda")) for _ in range(2)]
    ev.eval_batch_goals(Xd, *bufs[0], row0=0)  # warm-up, synchronous
    for i in range(2):
        ev.eval_batch_goals(Xd, *bufs[i], row0=i * B, sync=False, overlap=2)
    ev.synchronize()
    for i in range(2):
        F, G, _ = _call(ev, Xd, 0, True, True, False, False, i * B)
        assert np.array_equal(_bits(bufs[i][0].cpu().numpy()), _bits(F))
        assert np.array_equal(_bits(bufs[i][1].cpu().numpy()), _bits(G))


@pytest.mark.gpu
@pytest.mark.parametrize("mission,ts,wind", [("S10", 100, 1), ("S10", 200, 1), ("G7", 100, 1), ("G7", 45, 3),
                                             ("S10", 100, 3)])
def test_rows_match_the_port_with_the_rows_goal(mission, ts, wind):
    """every row against the CPU port (PortProblem with that row's goal), within 1e-14 + 1e-12*|ref|; the entries the
    reference leaves uninitialised (S10) are masked"""
    import portclient as P
    g = _fixture(mission, wind)
    B = 48
    goals = T.synth.goals(mission, 0, B)
    X = _inputs(g, mission, ts, B)
    ev = _context(g, mission, ts, wind, g["goal_ned"])
    ev.set_goals(goals)
    F, G, S = ev.eval_batch_goals(X, summary=np.empty((B, 4)))
    for b in range(B):
        port = P.PortProblem(mission, ts, g["ac"], g["gn"], goals[b], 1 if wind == 3 else wind)
        if wind == 3:
            port.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
        Fr, Gr = port.eval(X[b])
        keep = np.ones(ev.neG, bool)
        keep[port.ub_mask()] = False
        assert_parity(F[b], Fr, "%s row %d F" % (mission, b))
        assert_parity(G[b][keep], Gr[keep], "%s row %d G" % (mission, b))
        assert_parity(S[b, 0], Fr[0], "%s row %d summary objective" % (mission, b))


@pytest.mark.gpu
@pytest.mark.parametrize("mission,aircraft,ts", [("S10", "tempest", 100), ("G7", "skywalker", 100)])
def test_sampled_rows_match_the_reference_with_the_rows_goal(reference, param_root, mission, aircraft, ts):
    """a sample of rows against the reference (compiled where it is built) created with that row's goal on its
    command line; the context's parameters come from the same .param files"""
    B = 16
    goals_enu = T.synth.goals(mission, 0, B)[:, [1, 0, 2, 3]] * np.array([1.0, 1.0, -1.0, 1.0])  # NED -> E, N, U, R
    ev = T.Evaluator.from_files(param_root, aircraft, mission, (0.0, 0.0, 70.0), tuple(goals_enu[0]), ts=ts)
    cfg = T.config_from_files(param_root, aircraft, mission, (0.0, 0.0, 70.0), tuple(goals_enu[0]), ts=ts)
    ev.set_goals(np.array([T.config_from_files(param_root, aircraft, mission, (0.0, 0.0, 70.0), tuple(e), ts=ts).goal[:]
                           for e in goals_enu]))
    X = T.synth.batch(T.initial_guess(cfg), 4242, 0, B)
    F, G, _ = ev.eval_batch_goals(X)
    for b in range(0, B, 3):
        ref = reference(mission, aircraft, enu=(0.0, 0.0, 70.0), goal=tuple(goals_enu[b]), ts=ts)
        Fr, Gr = ref.eval(X[b])
        keep = np.ones(ev.neG, bool)
        keep[ref.ub_mask()] = False
        assert_parity(F[b], Fr, "%s row %d F" % (mission, b))
        assert_parity(G[b][keep], Gr[keep], "%s row %d G" % (mission, b))
        ref.close()


@pytest.mark.gpu
def test_full_size_batch_of_distinct_goals():
    """65,536 x S10 ts=200 (the bench batch) with all-distinct goals: two calls are bit-identical, and a strided sample
    of rows matches the port with each row's goal"""
    import portclient as P
    import torch
    g = load_golden("S10_tempest_ts200")
    B, ts = 65536, 200
    ev = _context(g, "S10", ts, 1, g["goal_ned"])
    goals = T.synth.goals("S10", 0, B)
    ev.set_goals(goals)
    X = T.synth.batch(g["x"][0], T.synth.SEED_S10, 0, B)
    Xd = torch.from_numpy(X).cuda()
    F1 = torch.empty(B, ev.neF, dtype=torch.float64, device="cuda")
    G1 = torch.empty(B, ev.neG, dtype=torch.float64, device="cuda")
    F2, G2 = torch.empty_like(F1), torch.empty_like(G1)
    ev.eval_batch_goals(Xd, F1, G1)
    ev.eval_batch_goals(Xd, F2, G2)
    assert torch.equal(F1.view(torch.int64), F2.view(torch.int64)) and torch.equal(G1.view(torch.int64), G2.view(torch.int64))
    rows = np.arange(0, B, 1031)
    Fs, Gs = F1[rows].cpu().numpy(), G1[rows].cpu().numpy()
    for i, b in enumerate(rows):
        port = P.PortProblem("S10", ts, g["ac"], g["gn"], goals[b], 1)
        Fr, Gr = port.eval(X[b])
        keep = np.ones(ev.neG, bool)
        keep[port.ub_mask()] = False
        assert_parity(Fs[i], Fr, "row %d F" % b)
        assert_parity(Gs[i][keep], Gr[keep], "row %d G" % b)


@pytest.mark.gpu
def test_goal_misuse_is_refused_and_changes_nothing():
    import torch
    g = load_golden("S10_tempest_ts100")
    ev = T.Evaluator.from_golden(g)
    L = ev.L
    B = 8
    X = np.ascontiguousarray(g["x"][:1].repeat(B, 0))
    F, G = np.full((B, ev.neF), np.nan), np.full((B, ev.neG), np.nan)
    flags = EV.NEED_F | EV.NEED_G | EV.HOST_PTRS

    def call(row0, nb=B):
        return L.tolcuda_eval_batch_goals(ev.h, row0, nb, X.ctypes.data, ev.n, F.ctypes.data, ev.neF, G.ctypes.data,
                                          ev.neG, None, 0, flags)
    l0 = ev.launches
    assert call(0) == -1 and b"no goal table" in L.tolcuda_last_error()
    goals = T.synth.goals("S10", 0, 10)
    ev.set_goals(goals)
    for row0, nb in ((-1, B), (3, B), (10, 1), (0, 11)):
        assert call(row0, nb) == -1 and b"outside the goal table" in L.tolcuda_last_error()
    assert L.tolcuda_set_goals(ev.h, 2, goals.ctypes.data, 3) == -1  # ldg < 4
    assert L.tolcuda_set_goals(ev.h, -1, goals.ctypes.data, 4) == -1
    assert ev.launches == l0 and np.isnan(F).all() and np.isnan(G).all()
    assert call(2) == 0 and ev.launches > l0  # the table survived the refused calls
    # set_goals while NO_SYNC launches are in flight: they finish with the table they were enqueued with
    Xd = torch.from_numpy(T.synth.batch(g["x"][0], 7, 0, 4096)).cuda()
    ev.set_goals(T.synth.goals("S10", 0, 4096))
    Fa, Ga, _ = _call(ev, Xd, 0, True, True, False, False, 0)
    Fd = torch.empty(4096, ev.neF, dtype=torch.float64, device="cuda")
    Gd = torch.empty(4096, ev.neG, dtype=torch.float64, device="cuda")
    for _ in range(3):
        ev.eval_batch_goals(Xd, Fd, Gd, sync=False)
    ev.set_goals(T.synth.goals("S10", 5000, 9096))
    assert np.array_equal(_bits(Fd.cpu().numpy()), _bits(Fa)) and np.array_equal(_bits(Gd.cpu().numpy()), _bits(Ga))
    # count 0 frees the table: the next call is refused again
    ev.set_goals(np.zeros((0, 4)))
    assert call(0, 1) == -1 and b"no goal table" in L.tolcuda_last_error()
    ev.close()


@pytest.mark.gpu
def test_tolbatch_goals_rows_and_result_files(tmp_path, param_root):
    """tolbatch --goals with --perturb 0,0 on every GPU present: row b is the reference's initial guess for goal b; its
    objective, worst defect and worst boundary value equal those of an Evaluator created with that goal, and its
    snopt_results.json is byte for byte what a single-goal run with that goal on the command line writes for row 0"""
    import torch
    B = 24
    goals_enu = T.synth.goals("G7", 0, B)[:, [1, 0, 2, 3]] * np.array([1.0, 1.0, -1.0, 1.0])
    gf = tmp_path / "goals.txt"
    gf.write_text("".join("%.17g %.17g %.17g %.17g\n" % tuple(e) for e in goals_enu))
    for mission, aircraft in (("G7", "skywalker"), ("S10", "tempest")):
        pos = ["0", "0", "70", "0", "0", "0", "0", aircraft, mission]
        out = tmp_path / mission
        out.mkdir()
        for summary in (False, True):
            js = str(out / ("s.json" if summary else "r.json"))
            extra = ["--summary-only"] if summary else ["--results", str(out), "--nresults", str(B)]
            r = subprocess.run([TOLBATCH] + pos + ["--root", param_root, "--goals", str(gf), "--perturb", "0,0",
                                                   "--steps", "1", "--gpus", str(torch.cuda.device_count()), "--json", js]
                               + extra, capture_output=True, text=True, timeout=180)
            assert r.returncode == 0, r.stdout + r.stderr
        d, s = json.load(open(out / "r.json")), json.load(open(out / "s.json"))
        assert d["batch"] == B and d["nonfinite"] == 0
        for b in range(B):
            ev = T.Evaluator.from_files(param_root, aircraft, mission, (0.0, 0.0, 70.0), tuple(goals_enu[b]))
            cfg = T.config_from_files(param_root, aircraft, mission, (0.0, 0.0, 70.0), tuple(goals_enu[b]))
            F, _ = ev.eval_batch_host(T.initial_guess(cfg)[None, :].copy())
            nb = 12 if mission == "G7" else 11
            t = d["trajectories"][b]
            assert t["objective"] == F[0, 0] and t["max_abs_defect"] == np.abs(F[0, 1:ev.neF - nb]).max()
            assert t["max_abs_boundary"] == np.abs(F[0, ev.neF - nb:]).max()
            assert s["trajectories"][b]["objective"] == F[0, 0]
            ev.close()
        for b in (0, 7, B - 1):
            one = tmp_path / ("%s_one_%d" % (mission, b))
            one.mkdir()
            args = ["0", "0", "70"] + ["%.17g" % v for v in goals_enu[b]] + [aircraft, mission]
            r = subprocess.run([TOLBATCH] + args + ["--root", param_root, "--batch", "1", "--perturb", "0,0", "--steps",
                                                    "1", "--results", str(one), "--nresults", "1"],
                               capture_output=True, text=True, timeout=120)
            assert r.returncode == 0, r.stdout + r.stderr
            assert (out / ("snopt_results_%d.json" % b)).read_bytes() == (one / "snopt_results_0.json").read_bytes()
