"""GPU: parity of the sm_100a path against the reference, through the C ABI.

  * every tests/golden fixture (outputs of the unmodified reference): pattern bit-exact, F/G within
    1e-14 + 1e-12*|ref| -- via tolcuda_eval, via the exported snOptA callback DEFINEGusrfg_, and via
    tolcuda_eval_batch with device and with host pointers;
  * SURVEY.md section 8d batches (G7 ts=100, S10 ts=200) against the oracle port (itself pinned to
    the reference bit for bit in tests/test_oracle.py) on a 64-trajectory subset;
  * size-independent properties at BASELINE.json's full sizes (structural constants, determinism,
    batch-order invariance, F/G-only consistency)."""
import numpy as np
import pytest
import torch

import tol_b200 as T
from conftest import GOLDEN, assert_parity, load_golden, port_from_golden

pytestmark = pytest.mark.gpu


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("name", GOLDEN)
def test_single_trajectory_matches_reference(name):
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g)
    assert (ev.n, ev.neF, ev.neG) == (int(g["n"]), int(g["neF"]), int(g["neG"]))
    i, j = ev.pattern()
    assert np.array_equal(i, g["iGfun"]) and np.array_equal(j, g["jGvar"])  # bit-exact pattern
    for s in range(g["x"].shape[0]):
        F, G = ev.eval(g["x"][s])
        assert_parity(F, g["F"][s], "%s[%d] F" % (name, s))
        assert_parity(G, g["G"][s], "%s[%d] G" % (name, s))
    ev.close()


def test_config2_reference_x0_and_16_perturbations_through_the_callback():
    """BASELINE.json configs[1] / SURVEY.md 8d config 2: S10, tempest, ts = 100 -- the reference's own initial guess and
    16 seeded perturbations, every one through the exported snOptA callback DEFINEGusrfg_ (reference
    src/DefineFG.cpp:9-48) against the rows the unmodified reference wrote for the same states: pattern as integer
    arrays, values within 1e-14 + 1e-12*|ref|, the 11 entries the reference leaves uninitialised masked (0.0 here)"""
    g = load_golden("S10_tempest_ts100")
    assert g["x"].shape[0] == 17 and int(g["ts"]) == 100 and str(g["aircraft"]) == "tempest"
    for s in range(1, 17):  # the fixture's states ARE the section-8d perturbations of x0
        assert np.array_equal(g["x"][s], T.synth.perturb(g["x"][0], int(g["seed0"]) + s - 1))
    ev = T.Evaluator.from_golden(g)
    i, j = ev.pattern()
    assert i.dtype == np.int32 and np.array_equal(i, g["iGfun"]) and np.array_equal(j, g["jGvar"])
    mask = g["ub_mask"]
    for s in range(17):
        st, F, G = ev.usrfun(g["x"][s], 1, 1)
        assert st == 0
        assert_parity(F, g["F"][s], "config 2 state %d F" % s)
        assert_parity(G, g["G"][s], "config 2 state %d G" % s)
        assert (G[mask] == 0.0).all()
        if s % 4 == 0:  # F alone and G alone, as SNOPT asks for them during a line search
            st, F1, G1 = ev.usrfun(g["x"][s], 1, 0)
            assert st == 0 and np.array_equal(F1, F) and np.isnan(G1).all()
            st, F1, G1 = ev.usrfun(g["x"][s], 0, 1)
            assert st == 0 and np.array_equal(G1, G) and np.isnan(F1).all()
    ev.close()


@pytest.mark.parametrize("name", ["S10_tempest_ts100", "G7_skywalker_ts100", "S10_tempesteric_ts33"])
def test_snopta_callback_drop_in(name):
    """DEFINEGusrfg_ with SNOPT's argument list; needF/needG honoured; Status untouched on success"""
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g)
    x = g["x"][1]
    st, F, G = ev.usrfun(x, 1, 1)
    assert st == 0
    assert_parity(F, g["F"][1], name + " F")
    assert_parity(G, g["G"][1], name + " G")
    st, F, G = ev.usrfun(x, 1, 0)
    assert st == 0 and np.isnan(G).all()
    assert_parity(F, g["F"][1], name + " F only")
    st, F, G = ev.usrfun(x, 0, 1)
    assert st == 0 and np.isnan(F).all()
    assert_parity(G, g["G"][1], name + " G only")
    ev.close()
    # no bound context -> Status = -2 (SNOPT: terminate), outputs untouched
    L = T.load()
    L.tolcuda_bind_global(None)
    ev2 = T.Evaluator.from_golden(g)
    st, F, G = ev2.usrfun(x, 1, 1, bind=False)
    assert st == -2 and np.isnan(F).all() and np.isnan(G).all()
    ev2.close()


@pytest.mark.parametrize("name", ["S10_skywalker_ts7_gains", "G7_tempestwill_ts7_gains"])
def test_callback_dump_files_on_request(name, tmp_path):
    """tolcuda_set_dump_dir: DEFINEGusrfg_ rewrites the reference's per-call files (src/DefineFG.cpp:16-46) --
    Xoutput.txt (what matlab/@plotSNOPT/plotSNOPT.m polls) and Woutput.txt equal to the files the unmodified
    reference wrote for the same x (tests/golden/dumps), Foutput.txt / Goutput.txt the "%.14f" lines of the arrays
    the call returned, within the parity bar of the reference's; F-only calls leave Goutput.txt alone; off again
    after set_dump_dir(None) and by default"""
    import os
    from conftest import GOLDEN_DIR
    g = load_golden(name)
    s = 3 if name.startswith("S10") else 2
    ref = os.path.join(GOLDEN_DIR, "dumps", "%s_s%d" % (name, s))
    ev = T.Evaluator.from_golden(g)
    x = g["x"][s]
    st, F, G = ev.usrfun(x, 1, 1)
    assert st == 0 and not list(tmp_path.iterdir())  # off by default
    ev.set_dump_dir(tmp_path)
    st, F, G = ev.usrfun(x, 1, 1)
    assert st == 0
    for f in ("Xoutput.txt", "Woutput.txt"):
        assert (tmp_path / f).read_bytes() == open(os.path.join(ref, f), "rb").read(), f
    for f, arr, key in (("Foutput.txt", F, "F"), ("Goutput.txt", G, "G")):
        lines = (tmp_path / f).read_text().split("\n")
        assert lines[-1] == "" and lines[:-1] == ["%.14f" % v for v in arr], f
        want = np.array([float(t) for t in open(os.path.join(ref, f)).read().split()])
        if key == "G":
            want[g["ub_mask"]] = 0.0  # printed from uninitialised memory by the reference
        assert np.abs(np.array([float(t) for t in lines[:-1]]) - want).max() <= 2e-14 + 1e-12 * np.abs(want).max()
    os.remove(tmp_path / "Goutput.txt")
    st, F, G = ev.usrfun(x, 1, 0)
    assert st == 0 and (tmp_path / "Foutput.txt").exists() and not (tmp_path / "Goutput.txt").exists()
    ev.set_dump_dir(None)
    for f in ("Xoutput.txt", "Woutput.txt", "Foutput.txt"):
        os.remove(tmp_path / f)
    st, F, G = ev.usrfun(x, 1, 1)
    assert st == 0 and not list(tmp_path.iterdir())
    ev.close()


@pytest.mark.parametrize("name", GOLDEN)
@pytest.mark.parametrize("pad", ["dense", "padded", "odd"])
def test_batch_device_pointers(name, pad):
    """fixture rows as one batch; dense / 128-byte padded / odd (8-byte aligned only) leading dims"""
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g)
    B = g["x"].shape[0]
    ld = {"dense": lambda v: v, "padded": T.evaluator.padded_ld, "odd": lambda v: v + 1 + (v % 2)}[pad]
    ldx, ldF, ldG = ld(ev.n), ld(ev.neF), ld(ev.neG)
    X = torch.zeros(B, ldx, dtype=torch.float64, device="cuda")
    X[:, :ev.n] = _dev(g["x"])
    F = torch.full((B, ldF), float("nan"), dtype=torch.float64, device="cuda")
    G = torch.full((B, ldG), float("nan"), dtype=torch.float64, device="cuda")
    ev.eval_batch_device(X, F, G)
    Fh, Gh = F.cpu().numpy(), G.cpu().numpy()
    assert_parity(Fh[:, :ev.neF], g["F"], name + " batch F")
    assert_parity(Gh[:, :ev.neG], g["G"], name + " batch G")
    assert np.isnan(Fh[:, ev.neF:]).all() and np.isnan(Gh[:, ev.neG:]).all()  # padding untouched
    ev.close()


@pytest.mark.parametrize("name", ["S10_tempest_ts200", "G7_tempestwences_ts45_gains", "S10_tempest_ts1"])
def test_batch_host_pointers_chunked(name, monkeypatch):
    """host-pointer path: pageable numpy and pinned torch memory, forced through several chunks"""
    g = load_golden(name)
    p = port_from_golden(g)
    x0 = g["x"][0]
    B = 37
    X = T.synth.batch(x0, 555, 0, B)
    Fr, Gr = np.empty((B, p.neF)), np.empty((B, p.neG))
    p.eval_many(X, Fr, Gr)
    ev = T.Evaluator.from_golden(g, options={"chunk_mb": 1})
    F, G = ev.eval_batch_host(X)
    assert_parity(F, Fr, name + " host F")
    assert_parity(G, Gr, name + " host G")
    Xp = torch.from_numpy(X).pin_memory()
    Fp = torch.empty(B, T.evaluator.padded_ld(p.neF), dtype=torch.float64).pin_memory()
    Gp = torch.empty(B, T.evaluator.padded_ld(p.neG), dtype=torch.float64).pin_memory()
    ev.eval_batch_host(Xp.numpy(), Fp.numpy(), Gp.numpy())
    assert np.array_equal(Fp.numpy()[:, :p.neF], F) and np.array_equal(Gp.numpy()[:, :p.neG], G)
    ev.close()


@pytest.mark.parametrize("name", ["S10_tempest_ts200", "G7_skywalker_ts100", "S10_tempesteric_ts33", "S10_tempest_ts1",
                                  "G7_skywalker_ts2", "S10_tempest_ts100_wind3"])
@pytest.mark.parametrize("kernel", [1, 2])
def test_compact_rows_path_equals_full_rows(name, kernel, monkeypatch):
    """The host-pointer path moves G across PCIe as compact rows (x-dependent values only) and expands them
    on host threads.  Its rows must be BIT-IDENTICAL to full rows copied from the device (TOLCUDA_FULL_G_COPY),
    for aligned and 8-byte-shifted destinations, through several chunks and lanes; compact rows requested
    by the caller (TOLCUDA_COMPACT_G, host and device pointers) expand to the same rows too."""
    g = load_golden(name)
    m, ts = str(g["mission"]), int(g["ts"])
    ev = T.Evaluator.from_golden(g, options={"kernel": kernel, "chunk_mb": 1})
    B = 101
    X = T.synth.batch(g["x"][0], 4242, 0, B)
    Ff, Gf = ev.eval_batch_host(X, full_copy=True)
    Fc, Gc = ev.eval_batch_host(X)
    assert np.array_equal(Fc.view(np.int64), Ff.view(np.int64))
    assert np.array_equal(Gc.view(np.int64), Gf.view(np.int64))
    # destination rows 8 bytes off 16-byte alignment, padding untouched; G only
    buf = np.full((B, ev.neG + 3), np.nan)
    ev.set_host_threads(3)
    ev.eval_batch_host(X, None, buf[:, 1:1 + ev.neG], needF=False)
    assert np.array_equal(buf[:, 1:1 + ev.neG].view(np.int64), Gf.view(np.int64))
    assert np.isnan(buf[:, 0]).all() and np.isnan(buf[:, 1 + ev.neG:]).all()
    # mixed mode: a share of the chunks crosses PCIe as full rows, the others as compact rows -- same bits
    for pct in (1, 30, 50, 99, 100):
        ev.set_option("full_rows_pct", pct)
        Fm, Gm = ev.eval_batch_host(X)
        assert np.array_equal(Fm.view(np.int64), Ff.view(np.int64)) and np.array_equal(Gm.view(np.int64), Gf.view(np.int64)), pct
    ev.set_option("full_rows_pct", 0)
    # caller-visible compact rows
    _, Gr = ev.eval_batch_host(X, compact_rows=True)
    assert Gr.shape == (B, T.evaluator.compact_len(m, ts))
    assert np.array_equal(T.evaluator.expand_compact_g(m, ts, Gr).view(np.int64), Gf.view(np.int64))
    Xd = _dev(X)
    Fd = torch.empty(B, ev.neF, dtype=torch.float64, device="cuda")
    Gd = torch.full((B, ev.compact_len + 5), float("nan"), dtype=torch.float64, device="cuda")
    ev.eval_batch_device(Xd, Fd, Gd, compact_rows=True)
    Gdh = Gd.cpu().numpy()
    assert np.array_equal(Gdh[:, :ev.compact_len].view(np.int64), Gr.view(np.int64)) and np.isnan(Gdh[:, ev.compact_len:]).all()
    assert np.array_equal(Fd.cpu().numpy().view(np.int64), Ff.view(np.int64))
    # expansion on the device (expand_kernel.cu): aligned rows (16-byte stores) and rows shifted by 8 bytes
    for ld, off in ((T.evaluator.padded_ld(ev.neG), 0), (ev.neG + 3, 1)):
        Gx = torch.full((B * ld + 8,), float("nan"), dtype=torch.float64, device="cuda")
        Gv = Gx[off:off + B * ld].view(B, ld)
        ev.expand_compact_device(Gd, Gv)
        Gxh = Gv.cpu().numpy()
        assert np.array_equal(np.ascontiguousarray(Gxh[:, :ev.neG]).view(np.int64), Gf.view(np.int64))
        assert np.isnan(Gxh[:, ev.neG:]).all()
    ev.close()


@pytest.mark.parametrize("name,seed0", [("G7_skywalker_ts100", T.synth.SEED_G7),
                                        ("S10_tempest_ts200", T.synth.SEED_S10)])
@pytest.mark.parametrize("kernel", [1, 2])
def test_section_8d_batches_against_oracle(name, seed0, kernel, monkeypatch, oracle_built):
    """configs 3 and 4 of BASELINE.json on a 64-trajectory subset, through both kernels (CTA per
    run of trajectories / CTA per trajectory with a tile loop); the lane-copy fallback of the TMA bulk
    stores is exercised by the odd-leading-dimension cases of test_batch_device_pointers"""
    g = load_golden(name)
    p = port_from_golden(g)
    B = 64
    X = T.synth.batch(g["x"][0], seed0, 1000, 1000 + B)
    Fr, Gr = np.empty((B, p.neF)), np.empty((B, p.neG))
    p.eval_many(X, Fr, Gr)
    ev = T.Evaluator.from_golden(g, options={"kernel": kernel})
    Xd = _dev(X)
    F = torch.empty(B, p.neF, dtype=torch.float64, device="cuda")
    G = torch.empty(B, p.neG, dtype=torch.float64, device="cuda")
    ev.eval_batch_device(Xd, F, G)
    assert_parity(F.cpu().numpy(), Fr, name + " F")
    assert_parity(G.cpu().numpy(), Gr, name + " G")
    # F-only and G-only launches give the same bits as the combined one
    F2 = torch.full_like(F, float("nan"))
    G2 = torch.full_like(G, float("nan"))
    ev.eval_batch_device(Xd, F2, G2, needF=True, needG=False)
    assert torch.equal(F2, F) and torch.isnan(G2).all()
    ev.eval_batch_device(Xd, F2, G2, needF=False, needG=True)
    assert torch.equal(G2, G)
    ev.close()


def test_wind_model_none_against_oracle(oracle_built):
    """wind model 0 (reference src/problem.cpp:480-498) cannot be reached in the reference as built
    (its constructor always falls back to model 1), so it is checked against the oracle port only"""
    for name in ("S10_tempesteric_ts33", "G7_tempestwences_ts45_gains"):
        g = load_golden(name)
        p = oracle_built.PortProblem(str(g["mission"]), int(g["ts"]), g["ac"], g["gn"], g["goal_ned"], 0)
        ev = T.Evaluator.from_golden(g, wind_model=0)
        for s in range(g["x"].shape[0]):
            Fr, Gr = p.eval(g["x"][s])
            F, G = ev.eval(g["x"][s])
            assert_parity(F, Fr, name + " wind0 F")
            assert_parity(G, Gr, name + " wind0 G")
        ev.close()


@pytest.mark.parametrize("name,seed0,B", [("G7_skywalker_ts100", T.synth.SEED_G7, 4096),
                                          ("S10_tempest_ts200", T.synth.SEED_S10, 65536)])
def test_full_size_properties(name, seed0, B, oracle_built):
    """BASELINE.json configs 3 and 4 at full size.  The oracle cannot evaluate 65,536 x 200 in
    seconds, so: (a) rows replicated from 256 distinct trajectories must come back bit-identical
    wherever they sit in the batch (batch-order invariance + determinism), (b) every structural
    constant of G holds in every row, (c) the periodic-boundary rows of F are exact differences,
    (d) a strided sample of rows matches the oracle."""
    g = load_golden(name)
    p = port_from_golden(g)
    ev = T.Evaluator.from_golden(g)
    U = 256
    Xu = T.synth.batch(g["x"][0], seed0, 0, U)
    ldx, ldF, ldG = (T.evaluator.padded_ld(v) for v in (p.n, p.neF, p.neG))
    Xd = torch.zeros(B, ldx, dtype=torch.float64, device="cuda")
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(1)).cuda() % U
    Xd[:, :p.n] = _dev(Xu)[perm]
    F = torch.empty(B, ldF, dtype=torch.float64, device="cuda")
    G = torch.empty(B, ldG, dtype=torch.float64, device="cuda")
    ev.eval_batch_device(Xd, F, G)
    # (a) group rows by source trajectory: all copies identical to the first copy
    first = torch.full((U,), -1, dtype=torch.long, device="cuda")
    idx = torch.arange(B, device="cuda")
    first.scatter_reduce_(0, perm, idx, reduce="amin", include_self=False)
    assert torch.equal(F[:, :p.neF], F[first[perm], :p.neF])
    assert torch.equal(G[:, :p.neG], G[first[perm], :p.neG])
    # (b) structural constants: entries whose reference value does not depend on x
    Gr0 = np.empty((2, p.neG))
    Fr0 = np.empty((2, p.neF))
    p.eval_many(Xu[:2], Fr0, Gr0)
    ts = int(g["ts"])
    R0 = p.neG - 104 * ts - (42 if str(g["mission"]) == "G7" else 33)
    rec = np.zeros(104, bool)
    for s in range(8):
        rec[13 * s + 12] = True  # +1 on the next node's state
    rec[[1, 15, 29, 85, 99]] = True  # -1 diagonals
    zero_like = (Gr0[0, R0:R0 + 104] == 0) & (Gr0[1, R0:R0 + 104] == 0)
    const_pos = np.where(rec | zero_like)[0]
    cols = torch.from_numpy((R0 + 104 * np.arange(ts)[:, None] + const_pos[None, :]).ravel()).cuda()
    want = _dev(np.tile(Gr0[0, R0 + const_pos], ts))
    assert torch.equal(G[:, cols], want.expand(B, -1))
    # (c) periodic boundary rows are exact differences of the inputs (states 3, 4: Va, gamma)
    nb = p.nb
    for c in (3, 4):
        assert torch.equal(F[:, p.neF - nb + c], Xd[:, 1 + 11 * ts + c] - Xd[:, 1 + c])
    # (d) strided sample against the oracle
    rows = np.arange(0, B, B // 32)
    Xs = Xd[torch.from_numpy(rows).cuda(), :p.n].cpu().numpy()
    Fr, Gr = np.empty((rows.size, p.neF)), np.empty((rows.size, p.neG))
    p.eval_many(np.ascontiguousarray(Xs), Fr, Gr)
    assert_parity(F[torch.from_numpy(rows).cuda(), :p.neF].cpu().numpy(), Fr, name + " sample F")
    assert_parity(G[torch.from_numpy(rows).cuda(), :p.neG].cpu().numpy(), Gr, name + " sample G")
    ev.close()


def test_tolbatch_driver_end_to_end(tmp_path, param_root):
    """the C++ batch driver (reference CLI arguments + reference .param files -> initial guess ->
    perturbed batch -> all visible GPUs -> host gather): trajectory 0 is the reference's x0, so its
    objective must equal the reference's F[0]; every value finite; 2 runs agree bit for bit"""
    import json
    import os
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "tol_b200", "tolbatch")
    root = param_root
    assert os.path.exists(exe), "tolbatch is not built (make -C tol_b200/csrc)"
    for args, fixture in ((["0", "0", "70", "0", "-100", "0", "100", "tempest", "S10"], "S10_tempest_ts100"),
                          (["0", "0", "70", "400", "0", "0", "0", "skywalker", "G7"], "G7_skywalker_ts100")):
        g = load_golden(fixture)
        outs = []
        for run in range(2):
            js = str(tmp_path / ("r%d.json" % run))
            r = subprocess.run([exe] + args + ["--root", root, "--batch", "300", "--steps", "1", "--json", js,
                                               "--results", str(tmp_path), "--nresults", "2"],
                               capture_output=True, text=True, timeout=120)
            assert r.returncode == 0, r.stdout + r.stderr
            outs.append(json.load(open(js)))
            # trajectory 0 is the reference's x0: its snopt_results.json is the reference's own file for x0
            ref_json = os.path.join(ROOT, "tests", "golden", "results", fixture + "_s0.json")
            if os.path.exists(ref_json):
                got = json.load(open(tmp_path / "snopt_results_0.json"))
                want = json.load(open(ref_json))
                assert abs(got.pop("FinalCost") - want.pop("FinalCost")) <= 1e-12 * abs(g["F"][0, 0])
                assert got == want
        d = outs[0]
        assert (d["n"], d["neF"], d["neG"], d["nonfinite"]) == (int(g["n"]), int(g["neF"]), int(g["neG"]), 0)
        f0 = d["trajectories"][0]["objective"]
        assert abs(f0 - g["F"][0, 0]) <= 1e-14 + 1e-12 * abs(g["F"][0, 0])
        assert outs[0]["trajectories"] == outs[1]["trajectories"]
        # screening mode: only the summary the kernels reduce on the fly comes back; same objectives and defects
        js = str(tmp_path / "summary.json")
        r = subprocess.run([exe] + args + ["--root", root, "--batch", "300", "--steps", "1", "--json", js, "--summary-only"],
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stdout + r.stderr
        sm = json.load(open(js))
        assert sm["summary_only"] is True and sm["nonfinite"] == 0
        for a, b in zip(sm["trajectories"], d["trajectories"]):
            assert a["objective"] == b["objective"] and a["max_abs_defect"] == b["max_abs_defect"]
        # --host-path full / auto: the same trajectories, bit for bit (the path only decides how G crosses PCIe)
        for hp in ("full", "auto", "40"):
            js = str(tmp_path / ("hp_%s.json" % hp))
            r = subprocess.run([exe] + args + ["--root", root, "--batch", "300", "--steps", "1", "--json", js, "--host-path", hp],
                               capture_output=True, text=True, timeout=180)
            assert r.returncode == 0, r.stdout + r.stderr
            assert json.load(open(js))["trajectories"] == d["trajectories"]
            assert (hp != "auto") or "host path calibration" in r.stdout
        # the same batch gathered on ONE GPU by the shards' own kernels (tolcuda_gather_*, the C form of
        # tol_b200.dist.eval_and_gather_peer): on every GPU count present, every choice of the gathering GPU, the
        # rows in its memory are bit for bit the rows of the host gather (tolbatch compares them and says so)
        ngpu = torch.cuda.device_count()
        for G_ in sorted({1, min(2, ngpu), ngpu}):
            for D_ in sorted({0, G_ - 1}):
                r = subprocess.run([exe] + args + ["--root", root, "--batch", "301", "--steps", "2", "--gpus", str(G_),
                                                   "--gather-gpu", str(D_)], capture_output=True, text=True, timeout=180)
                assert r.returncode == 0, r.stdout + r.stderr
                assert "gather on GPU %d" % D_ in r.stdout and "rows bit-identical to the host gather: yes" in r.stdout
            assert a["max_abs_boundary"] <= b["max_abs_boundary"]


@pytest.mark.parametrize("mission,ts", [("S10", 257), ("G7", 300), ("S10", 1100), ("G7", 2049)])
def test_long_trajectories(mission, ts, oracle_built):
    """ts > 256 is routed to kernel L (one CTA per trajectory, each warp walking several tiles);
    inputs: the restated InitialCond (bit-identical to the reference's) perturbed per SURVEY.md 8d;
    checker: the oracle port"""
    g = load_golden("S10_tempest_ts100" if mission == "S10" else "G7_skywalker_ts100")
    lm = g["lm"]
    cfg = T.make_config(mission, ts, g["ac"], g["gn"], g["goal_ned"],
                        limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]])
    x0 = T.initial_guess(cfg)
    p = oracle_built.PortProblem(mission, ts, g["ac"], g["gn"], g["goal_ned"], 1)
    B = 5
    X = T.synth.batch(x0, 77, 0, B)
    Fr, Gr = np.empty((B, p.neF)), np.empty((B, p.neG))
    p.eval_many(X, Fr, Gr)
    ev = T.Evaluator(mission, ts, g["ac"], g["gn"], g["goal_ned"])
    assert (ev.n, ev.neF, ev.neG) == (p.n, p.neF, p.neG)
    F, G = ev.eval_batch_host(X)
    assert_parity(F, Fr, "%s ts=%d F" % (mission, ts))
    assert_parity(G, Gr, "%s ts=%d G" % (mission, ts))
    F1, G1 = ev.eval(X[1])
    assert np.array_equal(F1, F[1]) and np.array_equal(G1, G[1])
    # the matrix-free products through kernel L as well, against products formed from the G rows just checked
    rng = np.random.default_rng(3)
    D, Lam = rng.uniform(-1, 1, (B, ev.n)), rng.uniform(-1, 1, (B, ev.neF))
    iG, jG = ev.pattern()
    Yr, Ya, Zr, Za = _op_reference(iG, jG, G, D, Lam, ev.neF, ev.n)
    Y = torch.empty(B, ev.neF, dtype=torch.float64, device="cuda")
    Z = torch.empty(B, ev.n, dtype=torch.float64, device="cuda")
    ev.jac_vec(_dev(X), _dev(D), Y)
    ev.jac_tvec(_dev(X), _dev(Lam), Z)
    assert (np.abs(Y.cpu().numpy() - Yr) <= 1e-14 + 1e-12 * Ya).all()
    assert (np.abs(Z.cpu().numpy() - Zr) <= 1e-14 + 1e-12 * Za).all()
    ev.close()


def _assert_parity_F_with_cancellation_bound(F, Fr, x, ts, what):
    """F against Fr at the state x: every entry within 1e-14 + 1e-12*|ref|, the defect rows x_{k+1} - xdot*dt - x_k
    within that plus ONE ULP of the larger of their two states (the documented limit of the absolute floor, see
    test_defect_cancellation_at_the_exact_initial_guess)"""
    nodes = x[1:].reshape(ts + 1, 11)
    scale = np.maximum(np.abs(nodes[:-1, :8]), np.abs(nodes[1:, :8])).ravel()  # per defect: its two states
    err = np.abs(F - Fr)
    d = slice(1, 1 + 8 * ts)
    bad = err[d] > 1e-14 + 1e-12 * np.abs(Fr[d]) + np.spacing(scale)
    assert not bad.any(), "%s: defect rows %s outside 1e-14 + 1e-12*|ref| + ulp(state): err %s" % (
        what, np.where(bad)[0][:6], err[d][bad][:6])
    assert_parity(np.delete(F, np.arange(1, 1 + 8 * ts)), np.delete(Fr, np.arange(1, 1 + 8 * ts)), what + " F[0], boundary")


def test_defect_cancellation_at_the_exact_initial_guess(oracle_built):
    """Documented limit of the 1e-14 absolute floor.  At the reference's own x0 with a fine grid the
    defects x_{k+1} - xdot*dt - x_k are ~1e-3 while the positions are ~1e2: the reference's expression
    rounds the intermediate x_{k+1} - xdot*dt to an ulp of the POSITION (2.8e-14 at 128..256 m), so a
    last-bit difference in sin/cos (CUDA libdevice vs glibc) moves such an F entry by half an ulp of the
    position, 1.4e-14, which no implementation without glibc's exact sin/cos can avoid.  The bound that
    does hold -- and is asserted here -- is one ulp of the largest state of the window; every other
    entry still meets 1e-14 + 1e-12*|ref|, as do all fixtures and all perturbed batches."""
    g = load_golden("S10_tempest_ts100")
    ts = 1100
    cfg = T.make_config("S10", ts, g["ac"], g["gn"], g["goal_ned"])
    x0 = T.initial_guess(cfg)
    p = oracle_built.PortProblem("S10", ts, g["ac"], g["gn"], g["goal_ned"], 1)
    Fr, Gr = p.eval(x0)
    ev = T.Evaluator("S10", ts, g["ac"], g["gn"], g["goal_ned"])
    F, G = ev.eval(x0)
    ev.close()
    assert_parity(G, Gr, "G at x0")
    nodes = x0[1:].reshape(ts + 1, 11)
    scale = np.maximum(np.abs(nodes[:-1, :8]), np.abs(nodes[1:, :8])).ravel()  # per defect: its two states
    err = np.abs(F - Fr)
    d = slice(1, 1 + 8 * ts)
    assert (err[d] <= 1e-14 + 1e-12 * np.abs(Fr[d]) + np.spacing(scale)).all()
    assert_parity(np.delete(F, np.arange(1, 1 + 8 * ts)), np.delete(Fr, np.arange(1, 1 + 8 * ts)), "F[0], boundary")


@pytest.mark.parametrize("name", ["S10_tempest_ts100", "G7_skywalker_ts100", "G7_tempestwences_ts45_gains",
                                  "S10_tempest_ts100_wind3"])
@pytest.mark.parametrize("kernel", [1, 2])
def test_fused_trajectory_summary(name, kernel, monkeypatch):
    """tolcuda_eval_batch_summary: objective / max|defect| / max boundary violation / sum defect^2 computed
    in the kernel equal the same quantities computed on the host from the kernel's own F (max: exactly;
    sum of squares: to rounding), with and without F/G being written"""
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g, options={"kernel": kernel})
    B = 33
    X = T.synth.batch(g["x"][0], 909, 0, B)
    S, F, G = ev.summary_host(X, needF=True, needG=True)
    S2, _, _ = ev.summary_host(X)
    assert np.array_equal(S, S2)
    ts, nb = int(g["ts"]), int(g["nb"])
    d = F[:, 1:1 + 8 * ts]
    bnd = np.abs(F[:, -nb:])
    if str(g["mission"]) == "G7":
        bnd[:, -1] = np.maximum(F[:, -1], 0.0)
    assert np.array_equal(S[:, 0], F[:, 0])
    assert np.array_equal(S[:, 1], np.abs(d).max(axis=1))
    assert np.array_equal(S[:, 2], bnd.max(axis=1))
    assert np.allclose(S[:, 3], (d * d).sum(axis=1), rtol=1e-13, atol=0)
    Fr, Gr = ev.eval_batch_host(X)
    assert np.array_equal(F, Fr) and np.array_equal(G, Gr)
    ev.close()


def _read_snmock_log(path):
    b = open(path, "rb").read()
    N, NF, NG, objrow = np.frombuffer(b[:16], np.int32)
    off = 16
    iG = np.frombuffer(b[off:off + 4 * NG], np.int32)
    jG = np.frombuffer(b[off + 4 * NG:off + 8 * NG], np.int32)
    off += 8 * NG
    calls = []
    while off < len(b):
        st, nf, ng = np.frombuffer(b[off:off + 12], np.int32)
        v = np.frombuffer(b[off + 12:off + 12 + 8 * (N + NF + NG)])
        calls.append((int(st), int(nf), int(ng), v[:N], v[N:N + NF], v[N + NF:]))
        off += 12 + 8 * (N + NF + NG)
    return int(objrow), iG, jG, calls


@pytest.mark.parametrize("args,fixture", [
    (["0", "0", "70", "0", "-100", "0", "100", "tempest", "S10"], "S10_tempest_ts100"),
    (["0", "0", "70", "400", "0", "0", "0", "skywalker", "G7"], "G7_skywalker_ts100")])
def test_reference_driver_with_libtolcuda_dropped_in(args, fixture, tmp_path):
    """The drop-in itself, executed: the UNMODIFIED reference driver objects (problem::runSNOPT ->
    snoptProblemA::solve -> f_snkera -> usrfun, then writeJSON) linked once with the reference's DefineFG.o
    and once with libtolcuda's DEFINEGusrfg_ in its place (oracle/dropin_main.cpp), SNOPT being the stand-in
    oracle/snmock.cpp that drives the callback with SNOPT's argument conventions (1-based index arrays,
    Status 1 / 0 / 2, F-only and G-only calls) and steps along the objective gradient it reads from G.
    Both runs must see the same pattern and agree call by call."""
    import json
    import os
    import subprocess
    from conftest import ROOT
    ref_exe = os.path.join(ROOT, "oracle", "_ref", "tol_dropin_ref")
    cuda_exe = os.path.join(ROOT, "oracle", "_ref", "tol_dropin_cuda")
    root = os.path.join(ROOT, "oracle", "_ref", "params") + "/"
    if not (os.path.exists(ref_exe) and os.path.exists(cuda_exe) and os.path.isdir(root)):
        pytest.skip("oracle/_ref drop-in binaries are not built (make -C oracle ref, build container only)")
    g = load_golden(fixture)
    logs, docs = {}, {}
    for tag, exe in (("ref", ref_exe), ("cuda", cuda_exe)):
        wd = tmp_path / tag
        wd.mkdir()
        log = str(wd / "calls.bin")
        r = subprocess.run([exe] + args + [root], cwd=wd, env=dict(os.environ, SNMOCK_LOG=log, SNMOCK_STEPS="7"),
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        logs[tag] = _read_snmock_log(log)
        docs[tag] = json.load(open(wd / "snopt_results.json"))
    (oref, iGr, jGr, cref), (ocuda, iGc, jGc, ccuda) = logs["ref"], logs["cuda"]
    assert oref == ocuda == 1
    assert np.array_equal(iGr, g["iGfun"] + 1) and np.array_equal(jGr, g["jGvar"] + 1)  # what SNOPT is handed
    assert np.array_equal(iGc, iGr) and np.array_equal(jGc, jGr)
    assert len(cref) == len(ccuda) == 8
    mask = np.ones(int(g["neG"]), bool)
    mask[g["ub_mask"]] = False  # left uninitialised by the reference
    for k, (a, b) in enumerate(zip(cref, ccuda)):
        assert a[:3] == b[:3] and a[0] == (1 if k == 0 else (2 if k == 7 else 0))
        assert_parity(b[3], a[3], "call %d x" % k)  # the iterates: same steps taken from the same G
        assert_parity(b[4], a[4], "call %d F" % k)
        if k == 0 or a[2]:  # G was requested in this call (otherwise the buffer keeps the last requested one)
            assert_parity(b[5][mask], a[5][mask], "call %d G" % k)
    assert_parity(cref[0][4], g["F"][0], "first call = the fixture's x0")
    # the reference's own writeJSON ran after both "solves": same document up to the parity tolerance
    assert docs["cuda"]["args"] == docs["ref"]["args"] and docs["cuda"]["snopt"] == docs["ref"]["snopt"]
    assert abs(docs["cuda"]["FinalCost"] - docs["ref"]["FinalCost"]) <= 1e-14 + 1e-12 * abs(docs["ref"]["FinalCost"])
    assert_parity(np.array(docs["cuda"]["trajectory"]["x"]), np.array(docs["ref"]["trajectory"]["x"]), "x*")


@pytest.mark.parametrize("args,fixture", [
    (["0", "0", "70", "0", "-100", "0", "100", "tempest", "S10"], "S10_tempest_ts100"),
    (["0", "0", "70", "400", "0", "0", "0", "skywalker", "G7"], "G7_skywalker_ts100")])
def test_long_callback_sequence_does_not_drift(args, fixture, tmp_path, oracle_built):
    """BASELINE.json configs[4] cannot run without the SNOPT library; what CAN be bounded is drift: the same two
    drivers (the reference's own DefineFG.o / libtolcuda's DEFINEGusrfg_) under the SNOPT stand-in for 240 calls of
    mixed kind (F+G, F only, G only), every iterate fed by the previous call's G.
      * the ITERATES of the two runs stay within the parity tolerance on every call (a last-ulp difference in G that
        fed on itself would show here);
      * on every call the CUDA run's F and G are within the tolerance of the reference arithmetic AT THE CUDA RUN'S
        OWN x (the oracle port, pinned bit for bit to the reference): F and G of the two runs cannot be compared
        directly once the iterates differ in the last bit -- a defect row is a difference of two x entries of size
        100, so one ulp of x is 1.4e-14 of F.  The defect rows carry the documented cancellation allowance of one
        ulp of their states (test_defect_cancellation_at_the_exact_initial_guess);
      * the reference run's F and G are the port's at the reference run's x, bit for bit (the pin, once more)."""
    import os
    import subprocess
    from conftest import ROOT
    ref_exe = os.path.join(ROOT, "oracle", "_ref", "tol_dropin_ref")
    cuda_exe = os.path.join(ROOT, "oracle", "_ref", "tol_dropin_cuda")
    root = os.path.join(ROOT, "oracle", "_ref", "params") + "/"
    if not (os.path.exists(ref_exe) and os.path.exists(cuda_exe) and os.path.isdir(root)):
        pytest.skip("oracle/_ref drop-in binaries are not built (make -C oracle ref, build container only)")
    g = load_golden(fixture)
    port = port_from_golden(g)
    steps, logs = 239, {}
    for tag, exe in (("ref", ref_exe), ("cuda", cuda_exe)):
        wd = tmp_path / tag
        wd.mkdir()
        log = str(wd / "calls.bin")
        r = subprocess.run([exe] + args + [root], cwd=wd, env=dict(os.environ, SNMOCK_LOG=log, SNMOCK_STEPS=str(steps)),
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        logs[tag] = _read_snmock_log(log)[3]
        os.remove(log)
    cref, ccuda = logs["ref"], logs["cuda"]
    assert len(cref) == len(ccuda) == steps + 1
    mask = np.ones(int(g["neG"]), bool)
    mask[g["ub_mask"]] = False
    kinds = set()
    moved = 0.0
    for k, (a, b) in enumerate(zip(cref, ccuda)):
        assert a[:3] == b[:3]
        kinds.add(a[1:3])
        assert_parity(b[3], a[3], "call %d x" % k)
        Fp, Gp = port.eval(b[3])
        Fr, Gr = port.eval(a[3])
        if a[1]:  # the iterates sit near x0, where the defects are ~1e-2 of positions ~1e2: cancellation bound
            _assert_parity_F_with_cancellation_bound(b[4], Fp, b[3], int(g["ts"]), "call %d F" % k)
            assert np.array_equal(a[4], Fr)
        if a[2]:
            assert_parity(b[5][mask], Gp[mask], "call %d G" % k)
            assert np.array_equal(a[5][mask], Gr[mask])
        moved = max(moved, float(np.abs(a[3] - cref[0][3]).max()))
    assert kinds == {(1, 1), (1, 0), (0, 1)} and moved > 1e-3  # all three kinds of call; the iterates did move


@pytest.mark.parametrize("name", ["S10_tempest_ts100", "G7_skywalker_ts100"])
def test_degenerate_inputs_are_non_finite_where_the_reference_is(name, oracle_built):
    """Inputs outside the bounds SNOPT keeps (Va = 0, cos(gamma) = 0, a node exactly on the loiter centre):
    the reference divides by zero there.  The kernels share reciprocals (x * (1/D) with a correction step), so
    the KIND of non-finite value can differ (NaN where the reference has +-Inf), but an entry is non-finite
    exactly where the reference's is, every other entry keeps the parity tolerance, and the other
    trajectories of the batch are unaffected."""
    g = load_golden(name)
    p = port_from_golden(g)
    ts = int(g["ts"])
    B = 6
    X = T.synth.batch(g["x"][0], 31337, 0, B)
    X[1, 1 + 11 * 5 + 3] = 0.0                    # Va = 0 at node 5
    X[2, 1 + 11 * 9 + 4] = np.pi / 2              # gamma = 90 deg at node 9
    X[3, 1 + 11 * 7 + 0], X[3, 1 + 11 * 7 + 1] = g["goal_ned"][0], g["goal_ned"][1]  # node 7 on the goal
    X[4, 1 + 11 * ts + 0], X[4, 1 + 11 * ts + 1] = X[4, 1], X[4, 2]  # G7: dist = 0
    Fr, Gr = np.empty((B, p.neF)), np.empty((B, p.neG))
    with np.errstate(all="ignore"):
        p.eval_many(X, Fr, Gr)
    ev = T.Evaluator.from_golden(g)
    F, G = ev.eval_batch_host(X)
    ev.close()
    assert not np.isfinite(Fr[1]).all() or not np.isfinite(Gr[1]).all()  # the cases do hit the singularities
    for got, ref, what in ((F, Fr, "F"), (G, Gr, "G")):
        fin = np.isfinite(ref)
        assert np.array_equal(np.isfinite(got), fin), what
        assert_parity(np.where(fin, got, 0.0), np.where(fin, ref, 0.0), name + " degenerate " + what)
    assert np.isfinite(F[[0, 5]]).all() and np.isfinite(G[[0, 5]]).all()


@pytest.mark.parametrize("name", ["S10_tempest_ts200", "G7_skywalker_ts100", "S10_tempest_ts1"])
@pytest.mark.parametrize("per", [1, 2, 3, 4])
def test_runs_of_trajectories_per_cta(name, per, monkeypatch):
    """kernel A evaluates `per` consecutive trajectories per CTA (TOLCUDA_PER; default 2 for large batches, the
    straight-line single-trajectory instance for small ones): every run length, batch sizes that leave a
    partial last run, and B = 1 must give the bits of the default configuration"""
    g = load_golden(name)
    X = T.synth.batch(g["x"][0], 777, 0, 23)
    ev = T.Evaluator.from_golden(g)
    Fd, Gd = ev.eval_batch_host(X, full_copy=True)
    ev.close()
    ev = T.Evaluator.from_golden(g, options={"per": per})
    for B in (23, 22, 1):
        F, G = ev.eval_batch_host(X[:B], full_copy=True)
        assert np.array_equal(F.view(np.int64), Fd[:B].view(np.int64))
        assert np.array_equal(G.view(np.int64), Gd[:B].view(np.int64))
    ev.close()


@pytest.mark.parametrize("name", ["S10_tempest_ts200", "G7_skywalker_ts100", "S10_tempesteric_ts33", "G7_tempestwences_ts45_gains"])
def test_launch_shapes_and_overlapped_launches_give_the_same_bits(name):
    """Every launch shape (trajectories per CTA, single-trajectory tail of the grid) and both forms of programmatic
    dependent launch (TOLCUDA_OVERLAP: the next launch starts during the previous one's tail and waits before its
    first store; TOLCUDA_OVERLAP_DISJOINT: no wait, alternating result buffers) must reproduce the bits of plain,
    serialised launches -- including when consecutive overlapped launches write DIFFERENT values into the same
    buffers (the wait is what makes that legal)."""
    g = load_golden(name)
    B = 1500  # several waves of CTAs on 148 SMs, an odd run count, a ragged end
    ev = T.Evaluator.from_golden(g)
    ldx, ldF, ldG = (T.evaluator.padded_ld(v) for v in (ev.n, ev.neF, ev.neG))
    Xs = []
    for q in range(3):
        X = np.zeros((B, ldx))
        T.synth.batch(g["x"][0], 31000 + 7 * q, 0, B, out=X)
        Xs.append(_dev(X))
    ref = []
    for X in Xs:
        F = torch.full((B, ldF), float("nan"), dtype=torch.float64, device="cuda")
        G = torch.full((B, ldG), float("nan"), dtype=torch.float64, device="cuda")
        ev.eval_batch_device(X, F, G)
        ref.append((F.cpu().numpy().view(np.int64), G.cpu().numpy().view(np.int64)))
    shapes = [(1, 0), (2, 0), (2, 1), (2, 4), (2, 64), (3, 2), (4, 3)]
    for per, tail in shapes:
        ev.set_option("per", per)
        ev.set_option("tail_x4", tail)
        for nb in (B, B - 1, 3, 1):
            F = torch.full((B, ldF), float("nan"), dtype=torch.float64, device="cuda")
            G = torch.full((B, ldG), float("nan"), dtype=torch.float64, device="cuda")
            ev.eval_batch_device(Xs[0][:nb], F[:nb], G[:nb])
            assert np.array_equal(F.cpu().numpy().view(np.int64)[:nb], ref[0][0][:nb]), (per, tail, nb)
            assert np.array_equal(G.cpu().numpy().view(np.int64)[:nb], ref[0][1][:nb]), (per, tail, nb)
            assert torch.isnan(F[nb:]).all() and torch.isnan(G[nb:]).all()
    ev.set_option("per", 0)
    ev.set_option("tail_x4", -1)
    nF, nG = ev.neF, ev.neG
    # overlap = 1: twelve launches back to back into the SAME buffers, inputs cycling; the last one's values must stand
    F = torch.empty(B, ldF, dtype=torch.float64, device="cuda")
    G = torch.empty(B, ldG, dtype=torch.float64, device="cuda")
    for rep in range(3):
        for i in range(12):
            ev.eval_batch_device(Xs[i % 3], F, G, sync=False, overlap=1)
        last = 11 % 3
        ev.synchronize()
        assert np.array_equal(F.cpu().numpy().view(np.int64)[:, :nF], ref[last][0][:, :nF])
        assert np.array_equal(G.cpu().numpy().view(np.int64)[:, :nG], ref[last][1][:, :nG])
    # overlap = 2: consecutive launches write different buffers and may run concurrently
    outs = [(torch.empty(B, ldF, dtype=torch.float64, device="cuda"), torch.empty(B, ldG, dtype=torch.float64, device="cuda"))
            for _ in range(3)]
    for i in range(12):
        ev.eval_batch_device(Xs[i % 3], outs[i % 3][0], outs[i % 3][1], sync=False, overlap=2)
    ev.synchronize()
    for q in range(3):
        assert np.array_equal(outs[q][0].cpu().numpy().view(np.int64)[:, :nF], ref[q][0][:, :nF])
        assert np.array_equal(outs[q][1].cpu().numpy().view(np.int64)[:, :nG], ref[q][1][:, :nG])
    ev.close()


@pytest.mark.parametrize("name", ["S10_tempest_ts100", "G7_tempestwences_ts45_gains", "S10_tempest_ts200"])
def test_every_execution_option_gives_the_same_bits(name):
    """tolcuda_set_option (include/tolcuda.h): every option chooses between equivalent ways of running the same
    arithmetic.  The single-trajectory callback (zero-copy kernel on mapped pinned memory / staged copies, compact or
    full G row across PCIe), the host-pointer batch path with any chunk size and any share of full-row chunks: all bit
    for bit the default's F and G; the tile-loop kernel with every warp count: bit for bit in G and in every F entry
    but the objective F[0], whose sum it associates differently (equal to a few ulp)."""
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g)
    x = g["x"][1]
    F0, G0 = ev.eval(x)
    B = 61
    X = T.synth.batch(g["x"][0], 97, 0, B)
    Fb0, Gb0 = ev.eval_batch_host(X)
    for opt, values, restore in (("zero_copy", (0, 1), 1), ("compact_host", (0, 1), 1)):
        for v in values:
            ev.set_option(opt, v)
            for needF, needG in ((1, 1), (1, 0), (0, 1)):
                st, F, G = ev.usrfun(x, needF, needG)
                assert st == 0
                assert (not needF) or np.array_equal(F.view(np.int64), F0.view(np.int64)), (opt, v)
                assert (not needG) or np.array_equal(G.view(np.int64), G0.view(np.int64)), (opt, v)
            Fb, Gb = ev.eval_batch_host(X)
            assert np.array_equal(Fb.view(np.int64), Fb0.view(np.int64)) and np.array_equal(Gb.view(np.int64), Gb0.view(np.int64)), (opt, v)
        ev.set_option(opt, restore)
    ev.set_option("kernel", 2)
    for w in range(0, 9):
        ev.set_option("lwarps", w)
        Fb, Gb = ev.eval_batch_host(X, full_copy=True)
        # the tile-loop kernel adds a trajectory's cost terms per lane over its tiles first: F[0] (and nothing else)
        # may differ from the default kernel's in the last bits
        assert np.array_equal(Gb.view(np.int64), Gb0.view(np.int64)), ("lwarps", w)
        assert np.array_equal(Fb[:, 1:].view(np.int64), Fb0[:, 1:].view(np.int64)), ("lwarps", w)
        assert (np.abs(Fb[:, 0] - Fb0[:, 0]) <= 4 * np.spacing(np.abs(Fb0[:, 0]))).all(), ("lwarps", w)
    ev.set_option("lwarps", 0)
    ev.set_option("kernel", 0)
    for mb, pct in ((1, 0), (1, 37), (2, 100), (64, 50), (4096, 0)):
        ev.set_option("chunk_mb", mb)
        ev.set_option("full_rows_pct", pct)
        Fb, Gb = ev.eval_batch_host(X)
        assert np.array_equal(Fb.view(np.int64), Fb0.view(np.int64)) and np.array_equal(Gb.view(np.int64), Gb0.view(np.int64)), (mb, pct)
    ev.close()


def test_api_misuse_is_reported_not_executed():
    """error behaviour of the C ABI on a live device: bad arguments come back as TOLCUDA_E* codes with a
    message, nothing is written, and the callback turns a mismatching problem size into Status = -2"""
    import ctypes as C
    g = load_golden("S10_tempest_ts100")
    ev = T.Evaluator.from_golden(g)
    L = ev.L
    x = np.ascontiguousarray(g["x"][0])
    F = np.full(ev.neF, np.nan)
    G = np.full(ev.neG, np.nan)
    dp = C.POINTER(C.c_double)
    assert L.tolcuda_eval(ev.h, None, 1, F.ctypes.data_as(dp), 1, G.ctypes.data_as(dp)) == -1      # EINVAL
    assert L.tolcuda_eval(ev.h, x.ctypes.data_as(dp), 1, None, 0, None) == -1
    assert L.tolcuda_eval(ev.h, x.ctypes.data_as(dp), 0, None, 0, None) == 0                        # nothing asked
    # leading dimension shorter than a row, negative batch, summary with too small a stride
    flags = T.evaluator.NEED_F | T.evaluator.NEED_G | T.evaluator.HOST_PTRS
    assert L.tolcuda_eval_batch(ev.h, 1, x.ctypes.data, ev.n - 1, F.ctypes.data, ev.neF, G.ctypes.data, ev.neG, flags) == -1
    assert b"leading dimension" in L.tolcuda_last_error()
    assert L.tolcuda_eval_batch(ev.h, -1, x.ctypes.data, ev.n, F.ctypes.data, ev.neF, G.ctypes.data, ev.neG, flags) == -1
    assert L.tolcuda_eval_batch(ev.h, 0, None, 0, None, 0, None, 0, flags) == 0                     # empty batch
    S = np.zeros(4)
    assert L.tolcuda_eval_batch_summary(ev.h, 1, x.ctypes.data, ev.n, F.ctypes.data, ev.neF, G.ctypes.data, ev.neG,
                                        S.ctypes.data, 3, flags) == -1
    assert L.tolcuda_eval_batch_summary(ev.h, 1, x.ctypes.data, ev.n, F.ctypes.data, ev.neF, G.ctypes.data, ev.neG,
                                        S.ctypes.data, 4, flags | T.evaluator.COMPACT_G) == -2     # EUNSUPPORTED
    assert np.isnan(F).all() and np.isnan(G).all()
    # flag bits the library does not define are rejected, nothing runs
    l0 = ev.launches
    for bad in (0x10000, 0x20000 | flags, 0x800 | flags, 1 << 30):
        assert L.tolcuda_eval_batch(ev.h, 1, x.ctypes.data, ev.n, F.ctypes.data, ev.neF, G.ctypes.data, ev.neG, bad | flags) == -1
        assert b"unknown flag" in L.tolcuda_last_error()
    # TOLCUDA_OVERLAP is a device-pointer, no-sync option
    assert L.tolcuda_eval_batch(ev.h, 1, x.ctypes.data, ev.n, F.ctypes.data, ev.neF, G.ctypes.data, ev.neG,
                                flags | T.evaluator.OVERLAP) == -1
    assert ev.launches == l0 and np.isnan(F).all() and np.isnan(G).all()
    # options: unknown names and values out of range are refused and change nothing
    assert L.tolcuda_set_option(ev.h, b"no_such_option", 1) == -1
    assert L.tolcuda_set_option(ev.h, b"per", 5) == -1 and L.tolcuda_set_option(ev.h, b"kernel", 3) == -1
    assert L.tolcuda_set_option(None, b"per", 1) == -1
    # unsupported configurations never reach the device
    cfg = T.make_config("S10", 100, g["ac"], g["gn"], g["goal_ned"])
    h = C.c_void_p()
    for field, bad in (("formulation", 3), ("ts", 0), ("wind_model", 2)):
        c2 = T.make_config("S10", 100, g["ac"], g["gn"], g["goal_ned"])
        setattr(c2, field, bad)
        assert L.tolcuda_create(C.byref(c2), C.byref(h)) == -2 and not h.value
    assert L.tolcuda_create(C.byref(cfg), None) == -1
    # the callback with another problem's sizes: Status = -2 (SNOPT: terminate), arrays untouched
    L.tolcuda_bind_global(ev.h)
    st = C.c_int(0)
    ints = [C.c_int(v) for v in (ev.n + 11, 1, ev.neF, 1, ev.neG, 0, 0, 0)]
    L.DEFINEGusrfg_(C.byref(st), C.byref(ints[0]), x.ctypes.data_as(dp), C.byref(ints[1]), C.byref(ints[2]),
                    F.ctypes.data_as(dp), C.byref(ints[3]), C.byref(ints[4]), G.ctypes.data_as(dp), None,
                    C.byref(ints[5]), None, C.byref(ints[6]), None, C.byref(ints[7]))
    assert st.value == -2 and np.isnan(F).all() and np.isnan(G).all()
    ev.close()


def _nccl_gather_worker(rank, world, port, name, B, out_path):
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    import tol_b200.dist as D
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g, device=rank)
    b0, b1 = D.my_shard(B)
    X = torch.from_numpy(T.synth.batch(g["x"][0], 2718, b0, b1)).cuda()
    F, G = D.eval_and_gather_device(ev, X, B, dst=0)
    if rank == 0:
        np.savez(out_path, F=F.cpu().numpy(), G=G.cpu().numpy())
    dist.barrier()
    ev.close()
    dist.destroy_process_group()


def test_shards_gathered_on_one_gpu_over_nccl(tmp_path):
    """2+ GPUs: every rank evaluates its shard into COMPACT G rows, the shards are gathered on GPU 0 with one
    NCCL gather per array (a third of the bytes of full rows) and expanded there by expand_kernel.cu; the
    result must be bit-identical to one GPU evaluating the whole batch into full rows"""
    import socket
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    name, B = "S10_tempest_ts100", 37
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = str(tmp_path / "gathered.npz")
    mp.spawn(_nccl_gather_worker, args=(2, port, name, B, out), nprocs=2, join=True)
    got = np.load(out)
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g)
    F, G = ev.eval_batch_host(T.synth.batch(g["x"][0], 2718, 0, B), full_copy=True)
    ev.close()
    assert np.array_equal(got["F"].view(np.int64), F.view(np.int64))
    assert np.array_equal(got["G"].view(np.int64), G.view(np.int64))


@pytest.mark.parametrize("name", ["S10_tempest_ts200", "G7_skywalker_ts100", "S10_tempest_ts1"])
def test_csc_repack_on_the_device(name):
    """tolcuda_repack_csc_device: G rows gathered into column-compressed order on the GPU equal the same rows
    permuted on the host with tolcuda_problem_pattern_csc's permutation (bit for bit), padding untouched"""
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g)
    B = 41
    X = T.synth.batch(g["x"][0], 99, 0, B)
    Xd = _dev(X)
    Fd = torch.empty(B, ev.neF, dtype=torch.float64, device="cuda")
    Gd = torch.empty(B, T.evaluator.padded_ld(ev.neG), dtype=torch.float64, device="cuda")
    ev.eval_batch_device(Xd, Fd, Gd)
    Gc = torch.full((B, ev.neG + 5), float("nan"), dtype=torch.float64, device="cuda")
    ev.repack_csc_device(Gd, Gc)
    _, _, pm = T.problem_pattern_csc(str(g["mission"]), int(g["ts"]))
    want = Gd.cpu().numpy()[:, :ev.neG][:, pm]
    got = Gc.cpu().numpy()
    assert np.array_equal(np.ascontiguousarray(got[:, :ev.neG]).view(np.int64), np.ascontiguousarray(want).view(np.int64))
    assert np.isnan(got[:, ev.neG:]).all()
    ev.close()


def test_more_rows_than_one_grid_dimension():
    """B > 65,535 (the y-dimension limit of a grid) through the batch kernel, the device expansion and the CSC
    repack, on a small problem: rows far apart in the batch must equal their single-trajectory evaluation"""
    g = load_golden("S10_skywalker_ts7_gains")
    ev = T.Evaluator.from_golden(g)
    B, U = 70001, 11
    Xu = T.synth.batch(g["x"][0], 8, 0, U)
    Xd = _dev(Xu)[torch.arange(B, device="cuda") % U].contiguous()
    Fd = torch.empty(B, ev.neF, dtype=torch.float64, device="cuda")
    Gd = torch.empty(B, ev.neG, dtype=torch.float64, device="cuda")
    Gc = torch.empty(B, ev.compact_len, dtype=torch.float64, device="cuda")
    ev.eval_batch_device(Xd, Fd, Gd)
    ev.eval_batch_device(Xd, Fd, Gc, compact_rows=True)
    Gx = torch.empty_like(Gd)
    ev.expand_compact_device(Gc, Gx)
    assert torch.equal(Gx, Gd)
    Gs = torch.empty_like(Gd)
    ev.repack_csc_device(Gd, Gs)
    _, _, pm = T.problem_pattern_csc("S10", 7)
    assert torch.equal(Gs, Gd[:, torch.from_numpy(pm.astype(np.int64)).cuda()])
    for b in (0, 65534, 65535, 65536, 70000):
        F1, G1 = ev.eval(Xu[b % U])
        assert np.array_equal(Fd[b].cpu().numpy(), F1) and np.array_equal(Gd[b].cpu().numpy(), G1)
    ev.close()


def test_peer_buffer_rows_on_one_gpu():
    """tolcuda_device_alloc / tolcuda_ipc_export + tolcuda_eval_batch on raw addresses (the world-size-1 leg of
    the fused evaluate + gather): the rows written into the exported buffer are bit for bit those of an ordinary
    device-pointer call, and the padding between rows is untouched"""
    import tol_b200.dist as D
    g = load_golden("S10_tempest_ts100")
    ev = T.Evaluator.from_golden(g)
    B = 29
    X = _dev(T.synth.batch(g["x"][0], 4242, 0, B))
    ldF, ldG = T.evaluator.padded_ld(ev.neF), T.evaluator.padded_ld(ev.neG)
    buf = D.open_peer_buffer(ev, B, 0, staged=False)
    assert len(buf.handle) == T.evaluator.IPC_HANDLE_BYTES and any(buf.handle)
    buf.tensor(0, 1, B * (ldF + ldG)).fill_(float("nan"))
    F, G, kept = D.eval_and_gather_peer(ev, X, B, out=buf)
    assert kept is buf and F.shape == (B, ldF) and G.shape == (B, ldG)
    Fd = torch.empty(B, ev.neF, dtype=torch.float64, device="cuda")
    Gd = torch.empty(B, ev.neG, dtype=torch.float64, device="cuda")
    ev.eval_batch_device(X, Fd, Gd)
    assert torch.equal(F[:, :ev.neF], Fd) and torch.equal(G[:, :ev.neG], Gd)
    assert torch.isnan(F[:, ev.neF:]).all() and torch.isnan(G[:, ev.neG:]).all()
    del F, G
    ev.close()
    buf.close()


def _peer_gather_worker(rank, world, port, name, B, compact, out_path):
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    import tol_b200.dist as D
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g, device=rank)
    b0, b1 = D.my_shard(B)
    X = torch.from_numpy(T.synth.batch(g["x"][0], 2718, b0, b1)).cuda()
    dst = world - 1  # not rank 0: the owner is any rank
    for _ in range(2):  # a second round maps the owner's (new) buffer again
        F, G, buf = D.eval_and_gather_peer(ev, X, B, dst=dst, compact=compact, chunks=3)
    if rank == dst:
        np.savez(out_path, F=F[:, :ev.neF].cpu().numpy(), G=G[:, :ev.neG].cpu().numpy())
    dist.barrier()
    del F, G, buf
    ev.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("name,B", [("S10_tempest_ts100", 37), ("G7_skywalker_ts100", 5), ("S10_tempest_ts200", 301)])
@pytest.mark.parametrize("compact", [True, False])
def test_shards_written_into_one_gpu_over_nvlink(name, B, compact, tmp_path):
    """2+ GPUs, fused evaluate + gather: every rank's F/G kernel stores its shard's rows directly into the
    gathering GPU's buffer (CUDA IPC mapping, NVLink peer stores: coalesced F stores and the G TMA bulk copies);
    as compact rows expanded by the owner, or as full rows at their final place; the gathered rows must be
    bit-identical to one GPU evaluating the whole batch"""
    import socket
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = str(tmp_path / "gathered.npz")
    mp.spawn(_peer_gather_worker, args=(2, port, name, B, compact, out), nprocs=2, join=True)
    got = np.load(out)
    g = load_golden(name)
    ev = T.Evaluator.from_golden(g)
    F, G = ev.eval_batch_host(T.synth.batch(g["x"][0], 2718, 0, B), full_copy=True)
    ev.close()
    assert np.array_equal(got["F"].view(np.int64), F.view(np.int64))
    assert np.array_equal(got["G"].view(np.int64), G.view(np.int64))


def test_one_process_two_devices_peer_rows():
    """2+ GPUs in ONE process (tolbatch's shape): after tolcuda_enable_peer(1, 0) the context of device 1 writes
    its F/G rows into a buffer that lives on device 0; bit-identical to device 0 evaluating the same rows"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from tol_b200 import lib as _l
    g = load_golden("G7_skywalker_ts100")
    B = 23
    X = T.synth.batch(g["x"][0], 31337, 0, B)
    ev0, ev1 = T.Evaluator.from_golden(g, device=0), T.Evaluator.from_golden(g, device=1)
    ldF, ldG = T.evaluator.padded_ld(ev0.neF), T.evaluator.padded_ld(ev0.neG)
    _l.check(_l.load().tolcuda_enable_peer(1, 0))
    _l.check(_l.load().tolcuda_enable_peer(1, 0))  # idempotent
    buf = T.PeerBuffer.alloc(0, 8 * B * (ldF + ldG))
    X1 = torch.from_numpy(X).to("cuda:1")
    ev1.eval_batch_ptrs(B, X1.data_ptr(), X1.stride(0), buf.ptr, ldF, buf.ptr + 8 * B * ldF, ldG)
    F, G = buf.tensor(0, B, ldF), buf.tensor(B * ldF, B, ldG)
    Fd = torch.empty(B, ev0.neF, dtype=torch.float64, device="cuda:0")
    Gd = torch.empty(B, ev0.neG, dtype=torch.float64, device="cuda:0")
    ev0.eval_batch_device(torch.from_numpy(X).to("cuda:0"), Fd, Gd)
    assert torch.equal(F[:, :ev0.neF], Fd) and torch.equal(G[:, :ev0.neG], Gd)
    del F, G
    ev0.close(), ev1.close(), buf.close()


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


@pytest.mark.parametrize("name", ["S10_tempest_ts200", "G7_skywalker_ts100", "S10_tempest_ts1", "S10_skywalker_ts7_gains",
                                  "G7_tempestwences_ts45_gains", "S10_tempest_ts100_wind3", "G7_skywalker_ts2", "G7_skywalker_ts45_wind3"])
@pytest.mark.parametrize("kernel", [1, 2])
def test_matrix_free_jacobian_products(name, kernel, monkeypatch, oracle_built):
    """tolcuda_jac_vec / tolcuda_jac_tvec (G never written) against products formed on the CPU from the ORACLE's G
    rows and the pattern: |err| <= 1e-14 + 1e-12 * sum of |terms| per entry; padding columns untouched; and the
    adjoint identity lambda.(J d) == (J^T lambda).d"""
    if name not in GOLDEN:
        pytest.skip("fixture not present")
    g = load_golden(name)
    p = port_from_golden(g)
    ev = T.Evaluator.from_golden(g, options={"kernel": kernel})
    iG, jG = ev.pattern()
    B = 21
    rng = np.random.default_rng(77)
    X = T.synth.batch(g["x"][0], 555, 0, B)
    D = rng.uniform(-1, 1, (B, ev.n))
    Lam = rng.uniform(-1, 1, (B, ev.neF))
    Fr, Gr = np.empty((B, p.neF)), np.empty((B, p.neG))
    p.eval_many(X, Fr, Gr)
    if str(g["mission"]) == "S10":  # the reference leaves these 11 entries uninitialised; defined as 0.0 here
        Gr[:, [ev.neG - 33 + 3 * i for i in range(11)]] = 0.0
    Yr, Ya, Zr, Za = _op_reference(iG, jG, Gr, D, Lam, ev.neF, ev.n)
    Xd, Dd, Ld = _dev(X), _dev(D), _dev(Lam)
    Y = torch.full((B, ev.neF + 3), float("nan"), dtype=torch.float64, device="cuda")
    Z = torch.full((B, ev.n + 5), float("nan"), dtype=torch.float64, device="cuda")
    ev.jac_vec(Xd, Dd, Y)
    ev.jac_tvec(Xd, Ld, Z)
    Yg, Zg = Y.cpu().numpy(), Z.cpu().numpy()
    assert np.isnan(Yg[:, ev.neF:]).all() and np.isnan(Zg[:, ev.n:]).all()
    Yg, Zg = Yg[:, :ev.neF], Zg[:, :ev.n]
    assert np.isfinite(Yg).all() and np.isfinite(Zg).all()
    ey, ez = np.abs(Yg - Yr) - (1e-14 + 1e-12 * Ya), np.abs(Zg - Zr) - (1e-14 + 1e-12 * Za)
    assert ey.max() <= 0, ("J d", np.unravel_index(ey.argmax(), ey.shape), ey.max())
    assert ez.max() <= 0, ("J^T lambda", np.unravel_index(ez.argmax(), ez.shape), ez.max())
    lhs, rhs = (Lam * Yg).sum(1), (Zg * D).sum(1)
    assert np.all(np.abs(lhs - rhs) <= 1e-11 * (np.abs(Lam) * Ya).sum(1) + 1e-13)
    # the same launches again: identical bits (no atomics, fixed summation order)
    Y2, Z2 = torch.empty_like(Y), torch.empty_like(Z)
    ev.jac_vec(Xd, Dd, Y2)
    ev.jac_tvec(Xd, Ld, Z2)
    assert torch.equal(Y2[:, :ev.neF], Y[:, :ev.neF]) and torch.equal(Z2[:, :ev.n], Z[:, :ev.n])
    ev.close()


def test_matrix_free_products_against_the_gpu_rows_at_full_size():
    """BASELINE.json config 3 size (G7 ts=100, 4,096 trajectories): J d and J^T lambda against products formed
    on the GPU from the G rows the F/G kernel writes (torch scatter-adds), and the adjoint identity"""
    g = load_golden("G7_skywalker_ts100")
    ev = T.Evaluator.from_golden(g)
    B, U = 4096, 64
    Xd = _dev(T.synth.batch(g["x"][0], T.synth.SEED_G7, 0, U))[torch.arange(B, device="cuda") % U].contiguous()
    gen = torch.Generator(device="cuda").manual_seed(5)
    D = torch.rand(B, ev.n, dtype=torch.float64, device="cuda", generator=gen) * 2 - 1
    Lam = torch.rand(B, ev.neF, dtype=torch.float64, device="cuda", generator=gen) * 2 - 1
    F = torch.empty(B, ev.neF, dtype=torch.float64, device="cuda")
    G = torch.empty(B, ev.neG, dtype=torch.float64, device="cuda")
    ev.eval_batch_device(Xd, F, G)
    iG, jG = [torch.from_numpy(a.astype(np.int64)).cuda() for a in ev.pattern()]
    ty = G * D[:, jG]
    Yr = torch.zeros(B, ev.neF, dtype=torch.float64, device="cuda").index_add_(1, iG, ty)
    Ya = torch.zeros_like(Yr).index_add_(1, iG, ty.abs())
    tz = G * Lam[:, iG]
    Zr = torch.zeros(B, ev.n, dtype=torch.float64, device="cuda").index_add_(1, jG, tz)
    Za = torch.zeros_like(Zr).index_add_(1, jG, tz.abs())
    Y, Z = torch.empty_like(Yr), torch.empty_like(Zr)
    ev.jac_vec(Xd, D, Y)
    ev.jac_tvec(Xd, Lam, Z)
    assert bool(((Y - Yr).abs() <= 1e-14 + 1e-12 * Ya).all()) and bool(((Z - Zr).abs() <= 1e-14 + 1e-12 * Za).all())
    lhs, rhs = (Lam * Y).sum(1), (Z * D).sum(1)
    assert bool(((lhs - rhs).abs() <= 1e-11 * (Lam.abs() * Ya).sum(1) + 1e-13).all())
    ev.close()


def test_stream_ordered_flags():
    """tolcuda_stream_signal / tolcuda_stream_wait (cuStreamWriteValue32 / cuStreamWaitValue32): the flag is written
    after the kernels enqueued before it, and a second context's stream passes a wait on a value already reached
    (also with the counter wrapped around)"""
    g = load_golden("S10_tempest_ts1")
    ev, ev2 = T.Evaluator.from_golden(g), T.Evaluator.from_golden(g)
    flag = torch.zeros(64, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    X = _dev(T.synth.batch(g["x"][0], 1, 0, 300))
    F = torch.empty(300, ev.neF, dtype=torch.float64, device="cuda")
    G = torch.empty(300, ev.neG, dtype=torch.float64, device="cuda")
    for value in (1, 2, 0x7fffffff, 0x80000001):
        ev.eval_batch_device(X, F, G, sync=False)
        ev.stream_signal(flag.data_ptr() + 8, value)
        ev.synchronize()
        assert int(flag[2].item()) & 0xffffffff == value and not flag[:2].any() and not flag[3:].any()
        ev2.stream_wait(flag.data_ptr() + 8, value)          # already reached: must not block
        ev2.stream_wait(flag.data_ptr() + 8, value - 1)      # (int)(*flag - value) >= 0
        ev2.eval_batch_device(X, F, G)
    L = T.load()
    assert L.tolcuda_stream_signal(ev.h, flag.data_ptr() + 2, 1) == -1   # misaligned
    assert L.tolcuda_stream_wait(None, flag.data_ptr(), 1) == -1
    ev.close(), ev2.close()
