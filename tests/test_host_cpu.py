"""CPU: the host side of libtolcuda that needs no device -- the C-ABI surface, the closed-form
sparsity pattern (vs the reference's and vs the oracle's literal countG walk) and the .param reader."""
import ctypes
import json
import os
import re

import numpy as np
import pytest

import tol_b200 as T
from conftest import GOLDEN, GOLDEN_DIR, ROOT, load_golden


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "tolcuda.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(tolcuda_[a-z_0-9]+|DEFINEGusrfg_)\s*\(", hdr))
    assert {"tolcuda_create", "tolcuda_eval", "tolcuda_eval_batch", "tolcuda_pattern", "tolcuda_dims",
            "tolcuda_bind_global", "tolcuda_destroy", "DEFINEGusrfg_"} <= names
    L = ctypes.CDLL(T.LIB_PATH)
    for nm in sorted(names):
        assert hasattr(L, nm), "libtolcuda.so does not export " + nm


@pytest.mark.parametrize("name", GOLDEN)
def test_closed_form_pattern_equals_reference(name):
    g = load_golden(name)
    m, ts = str(g["mission"]), int(g["ts"])
    assert T.problem_dims(m, ts) == (int(g["n"]), int(g["neF"]), int(g["neG"]))
    i, j = T.problem_pattern(m, ts)
    assert i.dtype == np.int32 and np.array_equal(i, g["iGfun"]) and np.array_equal(j, g["jGvar"])


@pytest.mark.parametrize("mission", ["G7", "S10"])
def test_closed_form_pattern_equals_countg_walk_for_every_small_ts(oracle_built, mission):
    g = load_golden("G7_skywalker_ts2" if mission == "G7" else "S10_tempest_ts1")
    for ts in list(range(1, 41)) + [64, 65, 127, 128, 129]:
        p = oracle_built.PortProblem(mission, ts, g["ac"], g["gn"], g["goal_ned"], 1)
        assert T.problem_dims(mission, ts) == (p.n, p.neF, p.neG)
        i, j = T.problem_pattern(mission, ts)
        oi, oj = p.pattern()
        assert np.array_equal(i, oi) and np.array_equal(j, oj), ts


def test_read_params_quirks(tmp_path):
    p = tmp_path / "q.param"
    # header comment, CRLF, literal backslash-n after the number, '/' as the real delimiter, blank and
    # text-only lines skipped, exponent and sign forms, last line without newline
    p.write_bytes(b"//header 12 // not a value\r\n4\\n    \t// Mass (kg)\r\n2.42\\n\t// span\n\n"
                  b"  -0.45\\n // min CL\nnot a number\n1e20 / single slash\n.5e-1//x\n7/3\n+3.0")
    v, cnt = T.read_params(p)
    assert cnt == 7
    assert v.tolist() == [4.0, 2.42, -0.45, 1e20, 0.05, 7.0, 3.0]
    with pytest.raises(T.TolcudaError):
        T.read_params(tmp_path / "missing.param")


def test_read_params_matches_reference_files(param_root):
    """tolcuda_read_params returns, with the reference's three degree -> radian conversions, the values the reference
    read from its .param files (tests/golden/params.json): from its own files where oracle/_ref holds a copy, else from
    files rebuilt from those values in the same layout (conftest.write_param_tree) -- then this checks the reader on
    that layout (header comment, literal backslash-n, CRLF, degrees), not the reference's exact bytes"""
    ref = param_root
    P = json.load(open(os.path.join(GOLDEN_DIR, "params.json")))
    for ac, want in P["aircraft"].items():
        v, cnt = T.read_params(os.path.join(ref, "aircraft", ac + ".param"))
        assert cnt == 15
        v[8], v[11], v[12] = v[8] * np.pi / 180.0, v[11] * np.pi / 180.0, v[12] * np.pi / 180.0
        assert v.tolist() == want, ac
    for ms, d in P["problems"].items():
        v, cnt = T.read_params(os.path.join(ref, "problems", ms, "gains.param"))
        assert cnt == 5 and v.tolist() == d["gains"]
        v, cnt = T.read_params(os.path.join(ref, "problems", ms, "snopt.param"))
        assert cnt == 6 and v.tolist() == d["snopt"]
        v, cnt = T.read_params(os.path.join(ref, "problems", ms, "limits.param"))
        lm = d["limits_member_order"]  # dtmin,dtmax,xmax,ymax,zmax,xmin,ymin,zmin
        assert cnt == 8 and v.tolist() == [lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]]


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    g = load_golden("S10_tempest_ts1")
    with pytest.raises(T.TolcudaError):
        T.Evaluator.from_golden(g)


def test_gather_and_option_entry_points_refuse_bad_arguments_without_touching_a_device():
    """tolcuda_gather_* / tolcuda_set_option / the copy wrappers (include/tolcuda.h) validate before they reach CUDA:
    null handles and null pointers come back as TOLCUDA_EINVAL on a box with no GPU, closing nothing is a no-op"""
    import ctypes as C
    L = T.load()
    out = C.c_void_p()
    hd = C.create_string_buffer(64)
    assert L.tolcuda_gather_create(None, 16, 2, 0, C.byref(out), hd) == -1 and not out.value
    assert L.tolcuda_gather_create(None, 16, 2, 0, None, hd) == -1
    assert L.tolcuda_gather_attach(None, 16, 2, 1, 0, None, hd.raw, C.byref(out)) == -1 and not out.value
    assert L.tolcuda_gather_attach(None, 16, 2, 1, 0, None, None, C.byref(out)) == -1   # neither an owner nor a handle
    assert L.tolcuda_gather_send(None, None, 0, 4) == -1
    assert L.tolcuda_gather_collect(None, None, 0, 4, None, None, None, None) == -1
    assert L.tolcuda_gather_buffer(None, None, None) == -1
    assert L.tolcuda_gather_close(None) == 0
    assert L.tolcuda_set_option(None, b"per", 1) == -1
    assert L.tolcuda_copy_to_device(0, None, None, 8) == -1 and L.tolcuda_copy_to_host(0, None, None, 8) == -1


def test_synthetic_batch_is_shard_invariant():
    g = load_golden("G7_skywalker_ts2")
    x0 = g["x"][0]
    full = T.synth.batch(x0, 99, 0, 10)
    parts = [T.synth.batch(x0, 99, *T.synth.shard_range(10, r, 4)) for r in range(4)]
    assert np.array_equal(full, np.concatenate(parts))
    # fixture sample s >= 1 is perturb(x0, seed0 + s - 1)
    assert np.array_equal(g["x"][1], T.synth.perturb(x0, int(g["seed0"])))


def _cfg_from_golden(g):
    lm = g["lm"]  # member order dtmin,dtmax,xmax,ymax,zmax,xmin,ymin,zmin -> file order
    limits = [lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]]
    return T.make_config(str(g["mission"]), int(g["ts"]), g["ac"], g["gn"], g["goal_ned"],
                         limits=limits, solver_tol=g["sn"][4:6])


@pytest.mark.parametrize("name", GOLDEN)
def test_initial_guess_is_bit_identical_to_reference_initialcond(name):
    g = load_golden(name)
    x0 = T.initial_guess(_cfg_from_golden(g))
    assert np.array_equal(x0, g["x"][0]), np.abs(x0 - g["x"][0]).max()


@pytest.mark.parametrize("name", GOLDEN)
def test_bounds_are_bit_identical_to_reference_setlimits(name):
    g = load_golden(name)
    xl, xu, fl, fu = T.bounds(_cfg_from_golden(g))
    for got, key in ((xl, "xlow"), (xu, "xupp"), (fl, "Flow"), (fu, "Fupp")):
        assert np.array_equal(got, g[key]), key


# record positions (within a window's 104 G values, row-major over the 8 defect rows x 13 columns) whose
# value depends on x; derived here from the reference fixtures themselves, not from the library
def _varying_positions():
    var = np.zeros(104, bool)
    for name in GOLDEN:
        g = load_golden(name)
        if int(g["wind_model"]) != 1:
            continue
        ts = int(g["ts"])
        R0 = int(g["neG"]) - 104 * ts - (42 if str(g["mission"]) == "G7" else 33)
        rec = g["G"][:, R0:R0 + 104 * ts].reshape(-1, 104)
        var |= ~((rec == 0).all(axis=0) | (rec == 1).all(axis=0) | (rec == -1).all(axis=0))
    return var


@pytest.mark.parametrize("name", GOLDEN)
@pytest.mark.parametrize("shift", range(8))
@pytest.mark.parametrize("wide", [True, False])
def test_compact_rows_expand_to_reference_rows(name, shift, wide, monkeypatch):
    """tolcuda_expand_compact_g (the host half of the host-pointer batch path): compact rows cut out of the
    REFERENCE's G expand back to the reference's G exactly, constants included; `shift` moves the
    destination rows through all eight 8-byte phases of a cache line (every instantiation of the AVX-512
    line path, both alignments of the SSE2 path)"""
    if not wide:
        monkeypatch.setenv("TOLCUDA_NO_AVX512", "1")
    g = load_golden(name)
    m, ts, neG = str(g["mission"]), int(g["ts"]), int(g["neG"])
    nbG = 42 if m == "G7" else 33
    R0 = neG - 104 * ts - nbG
    var = _varying_positions()
    mdt_pos = [87, 101]  # d/d(dphi) of row F7, d/d(dCL) of row F8: -dt (src/problem.cpp:1171-1172, 1183-1184)
    var[mdt_pos] = False
    pos = np.where(var)[0]
    assert pos.size == 31
    Lc = T.evaluator.compact_len(m, ts)
    assert Lc == R0 + 31 * ts + nbG + 1
    G = g["G"].copy()
    G[:, g["ub_mask"]] = 0.0  # the reference leaves these uninitialised; defined as 0.0
    B = G.shape[0]
    Gc = np.full((B, Lc + 3), np.nan)
    Gc[:, :R0] = G[:, :R0]
    Gc[:, R0:R0 + 31 * ts] = G[:, R0:R0 + 104 * ts].reshape(B, ts, 104)[:, :, pos].reshape(B, -1)
    Gc[:, R0 + 31 * ts:R0 + 31 * ts + nbG] = G[:, neG - nbG:]
    Gc[:, R0 + 31 * ts + nbG] = -g["x"][:, 0]
    buf = np.full((B, neG + 8 + (-neG) % 8), np.nan)  # rows a multiple of 64 bytes: same phase in every row
    out = buf[:, shift:shift + neG]
    T.evaluator.expand_compact_g(m, ts, Gc, out, threads=3)
    assert np.array_equal(out, G)
    assert np.array_equal(out.view(np.int64), G.view(np.int64))  # bit for bit: structural zeros are +0.0
    assert np.isnan(buf[:, :shift]).all() and np.isnan(buf[:, shift + neG:]).all()


def test_compact_expand_many_rows_threads():
    """more rows than work items per thread, odd thread counts, B = 0"""
    m, ts = "S10", 7
    _, _, neG = T.problem_dims(m, ts)
    Lc = T.evaluator.compact_len(m, ts)
    rng = np.random.default_rng(3)
    Gc = rng.standard_normal((1001, Lc))
    ref = T.evaluator.expand_compact_g(m, ts, Gc, threads=1)
    for th in (2, 5, 16):
        assert np.array_equal(T.evaluator.expand_compact_g(m, ts, Gc, threads=th), ref)
    assert T.evaluator.expand_compact_g(m, ts, Gc[:0]).shape == (0, neG)
    with pytest.raises(T.TolcudaError):
        T.evaluator.expand_compact_g(m, ts, Gc[:, :Lc - 1].copy())


RESULTS = sorted(os.path.splitext(f)[0] for f in os.listdir(os.path.join(GOLDEN_DIR, "results")) if f.endswith(".json"))


def _config_from_golden(g):
    lm = g["lm"]  # member order dtmin,dtmax,xmax,ymax,zmax,xmin,ymin,zmin -> file order
    sn = g["sn"]
    return T.make_config(str(g["mission"]), int(g["ts"]), g["ac"], g["gn"], g["goal_ned"],
                         limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]], solver_tol=[sn[4], sn[5]])


@pytest.mark.parametrize("case", RESULTS)
def test_result_files_equal_the_references_byte_for_byte(case, tmp_path):
    """tolcuda_write_results_json / _txt against the files the UNMODIFIED reference wrote for the same state
    (oracle/gen_results_golden.py): jsoncpp StyledWriter layout incl. one-line short arrays, %.17g reals,
    -0, integer-valued reals, the text table's %-4.7e columns"""
    name, s = case.rsplit("_s", 1)
    g = load_golden(name)
    cfg = _config_from_golden(g)
    x, F0 = g["x"][int(s)], g["F"][int(s), 0]
    js, tx = tmp_path / "snopt_results.json", tmp_path / "snopt_output.txt"
    T.write_results_json(cfg, str(g["aircraft"]), str(g["mission"]), g["enu"], x, F0, js)
    T.write_results_txt(cfg, x, F0, tx)
    ref = os.path.join(GOLDEN_DIR, "results", case)
    assert js.read_bytes() == open(ref + ".json", "rb").read()
    assert tx.read_bytes() == open(ref + ".txt", "rb").read()
    doc = json.load(open(js))  # and it is the document msl/mission.py:204-240 reads back
    assert len(doc["trajectory"]["time"]) == int(g["ts"]) + 1 and doc["FinalCost"] == F0
    with pytest.raises(T.TolcudaError):
        T.write_results_json(cfg, "a", "S10", (0, 0, 0), x, F0, tmp_path / "no_such_dir" / "r.json")


def test_result_json_non_finite_values(tmp_path):
    """jsoncpp spells NaN as null and infinities as +-1e+9999 (src/jsoncpp.cpp:4054-4066)"""
    g = load_golden("S10_tempest_ts1")
    cfg = _config_from_golden(g)
    x = g["x"][0].copy()
    x[1], x[2] = np.inf, -np.inf
    T.write_results_json(cfg, "tempest", "S10", (0, 0, 70), x, float("nan"), tmp_path / "r.json")
    txt = (tmp_path / "r.json").read_text()
    assert '"FinalCost" : null' in txt and "[ 1e+9999," in txt and "[ -1e+9999," in txt


def test_header_is_plain_c_and_the_callback_has_the_snopta_type(tmp_path):
    """include/tolcuda.h must compile as C99 (plain pointers and sizes, no C++/CUDA/torch types) and
    DEFINEGusrfg_ must be assignable to SNOPT's user-function pointer type snFunA as reference
    include/snopt/snopt.h:60-66 declares it (restated in the test source, not included)."""
    import subprocess
    src = tmp_path / "abi.c"
    src.write_text('''
#include "tolcuda.h"
typedef void (*snFunA)(int *Status, int *n, double x[], int *needF, int *neF, double F[], int *needG, int *neG,
                       double G[], char cu[], int *lencu, int iu[], int *leniu, double ru[], int *lenru);
snFunA user_function = DEFINEGusrfg_;
int (*batch)(tolcuda_handle, int, const double *, long, double *, long, double *, long, int) = tolcuda_eval_batch;
int main(void) { return user_function == 0 || batch == 0 || sizeof(tolcuda_config) != 4 * sizeof(int) + 34 * sizeof(double); }
''')
    for cc, std in (("gcc", "-std=c99"), ("g++", "-std=c++11")):
        exe = tmp_path / ("abi_" + cc)
        subprocess.check_call([cc, std, "-Wall", "-Wextra", "-Werror", "-pedantic", "-x", "c" if cc == "gcc" else "c++",
                               "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                               "-L", os.path.dirname(T.LIB_PATH), "-ltolcuda", "-Wl,-rpath," + os.path.dirname(T.LIB_PATH)])
        assert subprocess.run([str(exe)]).returncode == 0


@pytest.mark.parametrize("name", GOLDEN)
def test_csc_pattern_is_the_column_compressed_form_of_the_reference_pattern(name):
    """tolcuda_problem_pattern_csc against scipy's COO -> CSC conversion of the REFERENCE's (iGfun, jGvar)"""
    import scipy.sparse as sp
    g = load_golden(name)
    m, ts, n, neF, neG = str(g["mission"]), int(g["ts"]), int(g["n"]), int(g["neF"]), int(g["neG"])
    cp, ri, pm = T.problem_pattern_csc(m, ts)
    A = sp.coo_matrix((np.arange(1, neG + 1, dtype=float), (g["iGfun"], g["jGvar"])), shape=(neF, n)).tocsc()
    A.sort_indices()
    assert np.array_equal(A.indptr, cp) and np.array_equal(A.indices, ri) and np.array_equal(A.data, pm + 1.0)
    # values: G in CSC order is the reference's G permuted
    Gc = g["G"][:, pm]
    B = sp.csc_matrix((Gc[0], ri, cp), shape=(neF, n))
    C = sp.coo_matrix((g["G"][0], (g["iGfun"], g["jGvar"])), shape=(neF, n))
    assert abs(B - C).max() == 0


def test_new_entry_points_reject_misuse_without_touching_a_device():
    """argument checks of the peer-buffer and matrix-free entry points come before any CUDA call; without a
    device the allocating calls report the CUDA error and hand back NULL (never a host pointer)"""
    import ctypes as C
    import torch
    L = T.load()
    vp = C.c_void_p
    assert L.tolcuda_jac_vec(None, 4, None, 0, None, 0, None, 0, 0) == -1
    assert L.tolcuda_jac_tvec(None, 4, None, 0, None, 0, None, 0, 0) == -1
    assert L.tolcuda_ipc_export(0, None, None) == -1
    assert L.tolcuda_ipc_open(0, None, None) == -1
    assert L.tolcuda_device_alloc(0, 1024, None) == -1
    assert L.tolcuda_ipc_close(0, None) == 0 and L.tolcuda_device_free(0, None) == 0
    assert L.tolcuda_enable_peer(0, 0) == 0
    if not torch.cuda.is_available():
        p = vp(12345)
        rc = L.tolcuda_device_alloc(0, 1024, C.byref(p))
        assert rc > 0 and not p.value and L.tolcuda_last_error()
        with pytest.raises(T.TolcudaError):
            T.PeerBuffer.alloc(0, 1024)


def test_callback_without_a_bound_context_terminates_snopt(capfd):
    """SURVEY.md 8b error convention: with no context bound the exported snOptA callback writes nothing into the
    caller's arrays and sets *Status = -2 (SNOPT: terminate); the reference itself never touches Status
    (src/DefineFG.cpp:9-48).  Host logic only -- no device is touched."""
    import ctypes as C
    L = T.load()
    assert L.tolcuda_bind_global(None) == 0  # unbind whatever an earlier test left
    n, neF, neG = T.problem_dims("S10", 3)
    x, F, G = np.zeros(n), np.full(neF, 7.0), np.full(neG, 7.0)
    st = C.c_int(1)  # SNOPT's first call
    ints = [C.c_int(v) for v in (n, 1, neF, 1, neG, 0, 0, 0)]
    dp = C.POINTER(C.c_double)
    L.DEFINEGusrfg_(C.byref(st), C.byref(ints[0]), x.ctypes.data_as(dp), C.byref(ints[1]), C.byref(ints[2]),
                    F.ctypes.data_as(dp), C.byref(ints[3]), C.byref(ints[4]), G.ctypes.data_as(dp), None,
                    C.byref(ints[5]), None, C.byref(ints[6]), None, C.byref(ints[7]))
    assert st.value == -2
    assert (F == 7.0).all() and (G == 7.0).all() and (x == 0.0).all()
    assert b"no context bound" in L.tolcuda_last_error()
    assert "user function failed" in capfd.readouterr().err


def test_tolbatch_fails_loudly_on_bad_arguments_and_without_a_device():
    """the batch driver (counterpart of the reference CLI, src/tol.cpp:38-53): too few positional arguments,
    an unknown option and -- on a box without a GPU -- the missing device all end with exit code 2 and a message;
    nothing is evaluated on the CPU instead"""
    import subprocess
    import torch
    exe = os.path.join(ROOT, "tol_b200", "tolbatch")
    if not os.path.exists(exe):
        pytest.skip("tolbatch is not built")
    pos = ["0", "0", "70", "0", "-100", "0", "100", "tempest", "S10"]
    r = subprocess.run([exe] + pos[:5], capture_output=True, text=True)
    assert r.returncode == 2 and "usage: tolbatch E N U Eg Ng Ug Rg aircraft mission" in r.stderr
    r = subprocess.run([exe] + pos + ["--bogus", "1"], capture_output=True, text=True)
    assert r.returncode == 2 and "unknown option --bogus" in r.stderr
    r = subprocess.run([exe] + pos + ["--perturb", "abc"], capture_output=True, text=True)
    assert r.returncode == 2 and "--perturb wants REL,ABS" in r.stderr
    # sizes that would index an empty batch, allocate a negative size or report a timing of no step
    for opt, val, msg in (("--batch", "0", "--batch must be at least 1"), ("--batch", "-5", "--batch must be at least 1"),
                          ("--steps", "0", "--steps must be at least 1"), ("--nresults", "-1", "--nresults must not be negative"),
                          ("--gpus", "-2", "--gpus must not be negative")):
        r = subprocess.run([exe] + pos + [opt, val], capture_output=True, text=True)
        assert r.returncode == 2 and msg in r.stderr and r.stdout == "", (opt, val, r.stderr)
    r = subprocess.run([exe] + pos + ["--host-path", "sideways"], capture_output=True, text=True)
    assert r.returncode == 2 and "--host-path wants compact, full, auto or a percentage" in r.stderr
    r = subprocess.run([exe] + pos + ["--gather-gpu", "0", "--summary-only"], capture_output=True, text=True)
    assert r.returncode == 2 and "--gather-gpu" in r.stderr
    if not torch.cuda.is_available():
        r = subprocess.run([exe] + pos + ["--batch", "4"], capture_output=True, text=True)
        assert r.returncode == 2 and "failed" in r.stderr and r.stdout == ""


DUMPS = sorted(os.listdir(os.path.join(GOLDEN_DIR, "dumps")))


@pytest.mark.parametrize("case", DUMPS)
def test_dump_files_equal_the_reference_callbacks_byte_for_byte(case, tmp_path):
    """tolcuda_write_dump / tolcuda_write_wind_dump (what DEFINEGusrfg_ writes after tolcuda_set_dump_dir) against
    the four files the UNMODIFIED reference callback wrote for the same state (oracle/gen_dumps_golden.py;
    src/DefineFG.cpp:16-46, src/problem.cpp:740-756): Xoutput.txt is what matlab/@plotSNOPT/plotSNOPT.m polls.
    F and G are the reference's own values here (the fixture's); the S10 lines that print uninitialised memory
    (src/problemS10.cpp:397,414) are left out of the comparison."""
    import ctypes as C
    name, s = case.rsplit("_s", 1)
    g = load_golden(name)
    s = int(s)
    L = T.load()
    dp = C.POINTER(C.c_double)
    ref = os.path.join(GOLDEN_DIR, "dumps", case)
    for fname, arr in (("Xoutput.txt", g["x"][s]), ("Foutput.txt", g["F"][s]), ("Goutput.txt", g["G"][s])):
        arr = np.ascontiguousarray(arr)
        out = tmp_path / fname
        assert L.tolcuda_write_dump(str(out).encode(), arr.ctypes.data_as(dp), arr.size) == 0
        got, want = out.read_bytes().split(b"\n"), open(os.path.join(ref, fname), "rb").read().split(b"\n")
        assert len(got) == len(want) == arr.size + 1 and got[-1] == want[-1] == b""
        skip = set(g["ub_mask"].tolist()) if fname == "Goutput.txt" else set()
        assert [v for i, v in enumerate(got) if i not in skip] == [v for i, v in enumerate(want) if i not in skip]
    x = np.ascontiguousarray(g["x"][s])
    out = tmp_path / "Woutput.txt"
    assert L.tolcuda_write_wind_dump(str(out).encode(), int(g["wind_model"]), int(g["ts"]), x.ctypes.data_as(dp)) == 0
    assert out.read_bytes() == open(os.path.join(ref, "Woutput.txt"), "rb").read()


def test_dump_writers_reject_misuse(tmp_path):
    import ctypes as C
    L = T.load()
    v = np.array([1.5, -0.0, 1e300, -2.5e-15])
    dp = C.POINTER(C.c_double)
    out = tmp_path / "v.txt"
    assert L.tolcuda_write_dump(str(out).encode(), v.ctypes.data_as(dp), v.size) == 0
    assert out.read_text().split("\n")[:2] == ["1.50000000000000", "-0.00000000000000"]
    assert out.read_text().split("\n")[2] == "%.14f" % 1e300 and out.read_text().split("\n")[3] == "-0.00000000000000"
    assert L.tolcuda_write_dump(str(out).encode(), None, 0) == 0 and out.read_bytes() == b""
    assert L.tolcuda_write_dump(None, v.ctypes.data_as(dp), 1) == -1
    assert L.tolcuda_write_dump(str(out).encode(), None, 3) == -1
    assert L.tolcuda_write_dump(str(tmp_path / "no_such_dir" / "v.txt").encode(), v.ctypes.data_as(dp), 1) == -4
    assert b"cannot open" in L.tolcuda_last_error()
    assert L.tolcuda_write_wind_dump(str(out).encode(), 3, 2, v.ctypes.data_as(dp)) == -2  # wind cube: not written
    assert L.tolcuda_write_wind_dump(str(out).encode(), 1, 0, v.ctypes.data_as(dp)) == -1
    assert L.tolcuda_set_dump_dir(None, b".") == -1


def test_read_params_fuzz_against_the_reference_parser(tmp_path, param_root, pins):
    """tolcuda_read_params against the UNMODIFIED reference's parameters::readparams (src/parameters.cpp:14-34,
    reached through its `gain` constructor :77-94) on generated gains.param files: every line style std::stod
    accepts or rejects -- signs, exponents, hex floats, inf/nan, leading blanks, trailing text, CR, a literal
    backslash-n, a single '/' as the real delimiter, out-of-range literals and denormals (skipped), comment and
    blank lines -- five accepted values per file, as the reference's size check wants.  Against the compiled
    reference where oracle/_ref is built, against its stored pins everywhere (conftest.Pins)."""
    import shutil
    import refclient as R
    rng = np.random.default_rng(20261018)
    accepted = ["{v!r}", "  \t{v!r}", "+{v!r}", "{v:.3e}", "{v:.17g}\\n   // gain", "{v!r}// c", "{v!r} / c", "{v!r}\r",
                "{v!r}abc", "{v!r} 12", "{h}", "{v:.6f}/3", "{v:E}"]
    special = ["inf", "-inf", "INFINITY", "1e308", "-1E-300", ".5", "5.", "0x1.8p3", "-0", "1e-307", "0x10", "1e+2x"]
    rejected = ["", "   ", "// header 12", "abc 3", "/4", "e5", "1e999", "-1e999", "1e-400", "4e-320", "--3", "+-2",
                ". 5", "\t// x", "x0x10"]
    tmp = tmp_path / "root"
    for d in ("aircraft", "problems"):
        shutil.copytree(os.path.join(param_root, d), tmp / d)
    gfile = tmp / "problems" / "S10" / "gains.param"
    os.chmod(gfile, 0o644)
    compared = 0
    for trial in range(60):
        lines, count = [], 0
        while count < 5:
            kind = rng.integers(0, 10)
            if kind < 5:
                v = float(rng.standard_normal() * 10.0 ** int(rng.integers(-8, 9)))
                lines.append(accepted[int(rng.integers(len(accepted)))].format(v=v, h=v.hex()))
                count += 1
            elif kind < 7:
                lines.append(special[int(rng.integers(len(special)))])
                count += 1
            else:
                lines.append(rejected[int(rng.integers(len(rejected)))])
        for _ in range(int(rng.integers(0, 3))):
            lines.append(rejected[int(rng.integers(len(rejected)))])
        text = "\n".join(lines) + ("\n" if trial % 2 else "")
        gfile.write_bytes(text.encode())
        got, cnt = T.read_params(gfile)
        # what the reference makes of the file: rejected (not five values), or these five values bit for bit
        pins.check(np.array([cnt == 5]), got if cnt == 5 else np.zeros(0), what="trial %d: %r" % (trial, text))
        if not R.available():
            compared += cnt == 5
            continue
        p = R.RefProblem.__new__(R.RefProblem)  # a problem object on the edited tree (no ts / gains rewriting)
        p._tmp = None
        p.h = R.lib().tolref_create(b"S10", b"tempest", 0.0, 0.0, 70.0, 0.0, -100.0, 0.0, 100.0, (str(tmp) + "/").encode())
        if not p.h:  # the reference counted something other than five values ("+-3", "- 2", ...): so must the library
            assert cnt != 5, (text, got)
            continue
        want = p.params()["gn"]
        p.close()
        assert cnt == 5, (text, got)
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), (text, got, want)  # bit for bit, NaN included
        compared += 1
    assert compared >= 30
    pins.done()


def test_setup_fuzz_against_the_reference(tmp_path, reference, pins):
    """tolcuda_problem_initial_guess / tolcuda_problem_bounds against the UNMODIFIED reference's InitialCond and
    setLimits (src/problemG7.cpp:19-217, src/problemS10.cpp:19-219, src/problem.cpp:198-365) on random command
    lines: both formulations, the five shipped aircraft, ts from 1 to 150, goals in every quadrant (and on the
    axes, where atan2 and the straight-line guess have their corner cases), loiter radii from 1 m to 1 km --
    bit for bit, together with the closed-form dimensions and pattern.  Against the compiled reference where
    oracle/_ref is built, against its stored pins everywhere (conftest.Pins)."""
    rng = np.random.default_rng(20261019)
    aircraft = ["skywalker", "tempest", "tempest_eric", "tempest_wences", "tempest_will"]
    goals = [(400.0, 0.0), (0.0, 400.0), (-250.0, 0.0), (0.0, -90.0), (1e-3, 1e-3)]
    for trial in range(36):
        mission = "G7" if trial % 2 else "S10"
        ts = int(rng.choice([1, 2, 3, 7, 31, 32, 33, 64, 100, 150]))
        eg, ng = goals[trial % 9] if trial % 9 < len(goals) else tuple(rng.uniform(-800, 800, 2).tolist())
        goal = (eg, ng, float(rng.uniform(-50, 120)), float(rng.choice([0.0, 1.0, 40.0, 100.0, 1000.0])))
        enu = (float(rng.uniform(-30, 30)), float(rng.uniform(-30, 30)), float(rng.uniform(0, 150)))
        ac = aircraft[trial % 5]
        p = reference(mission, ac, enu, goal, ts=ts)
        prm = p.params()
        pins.check(prm["ac"], prm["gn"], prm["lm"], prm["sn"], prm["goal"], what="parameters of trial %d" % trial)
        lm = prm["lm"]
        cfg = T.make_config(mission, ts, prm["ac"], prm["gn"], prm["goal"],
                            limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]], solver_tol=prm["sn"][4:6])
        what = (mission, ac, ts, enu, goal)
        assert T.problem_dims(mission, ts) == (p.n, p.neF, p.neG), what
        i, j = T.problem_pattern(mission, ts)
        ri, rj = p.pattern()
        assert np.array_equal(i, ri) and np.array_equal(j, rj), what
        x0, rx0 = T.initial_guess(cfg), p.x0()
        assert np.array_equal(x0.view(np.int64), rx0.view(np.int64)), (what, np.abs(x0 - rx0).max())
        for got, want, key in zip(T.bounds(cfg), p.bounds(), ("xlow", "xupp", "Flow", "Fupp")):
            assert np.array_equal(got.view(np.int64), want.view(np.int64)), (what, key)
        pins.check(np.array(T.problem_dims(mission, ts)), i, j, x0, *T.bounds(cfg), what="setup of trial %d" % trial)
        p.close()
    pins.done()


def test_result_files_fuzz_against_the_reference(tmp_path, reference, pins):
    """tolcuda_write_results_json / _txt against the UNMODIFIED reference's writeJSON / writeTXT
    (src/problem.cpp:1247-1418, jsoncpp's StyledWriter) on random states salted with the values number
    formatting trips over: +-0, integers, powers of ten, 0.1-like decimals, huge and tiny magnitudes,
    denormals.  Against the compiled reference where oracle/_ref is built, against its stored pins everywhere
    (conftest.Pins)."""
    rng = np.random.default_rng(20261022)
    salt = np.array([0.0, -0.0, 1.0, -1.0, 10.0, 100.0, 1e5, 1e15, 1e16, 1e17, 1e21, 1e22, -1e-5, 1e-4, 0.1, 0.2, 0.3,
                     1.0 / 3.0, 2.5, 123456789.0, 1e-300, 5e-324, 1.7976931348623157e308, 4.35, 0.5, 1e-7, 123.456,
                     9007199254740993.0, 1e-10, 99999.99999999999])
    aircraft = ["skywalker", "tempest", "tempest_eric", "tempest_wences", "tempest_will"]
    for trial in range(24):
        mission = "G7" if trial % 2 else "S10"
        ts = int(rng.choice([1, 2, 3, 9, 40]))
        ac = aircraft[trial % 5]
        enu = tuple(float(v) for v in rng.choice([0.0, 70.0, -3.5, 12.25], 3))
        goal = tuple(float(v) for v in rng.uniform(-300, 300, 3)) + (float(rng.choice([0.0, 100.0, 33.3])),)
        p = reference(mission, ac, enu, goal, ts=ts)
        prm = p.params()
        lm = prm["lm"]
        cfg = T.make_config(mission, ts, prm["ac"], prm["gn"], prm["goal"],
                            limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]], solver_tol=prm["sn"][4:6])
        x = p.x0() * (1 + 0.3 * rng.uniform(-1, 1, p.n))
        k = rng.uniform(0, 1, p.n) < 0.4
        x[k] = rng.choice(salt, int(k.sum())) * rng.choice([1.0, -1.0], int(k.sum()))
        F0 = float(rng.choice(salt)) if trial % 3 else float(rng.standard_normal() * 1e3)
        d = tmp_path / ("t%d" % trial)
        d.mkdir()
        p.write_json(x, F0, d / "ref.json")
        ref_txt = p.write_txt(x, F0, str(d))
        p.close()
        T.write_results_json(cfg, ac, mission, enu, x, F0, d / "ours.json")
        T.write_results_txt(cfg, x, F0, d / "ours.txt")
        assert (d / "ours.json").read_bytes() == (d / "ref.json").read_bytes(), (trial, mission, ts)
        assert (d / "ours.txt").read_bytes() == open(ref_txt, "rb").read(), (trial, mission, ts)
        pins.check(x, (d / "ours.json").read_bytes(), (d / "ours.txt").read_bytes(), what="files of trial %d" % trial)
    pins.done()


def test_config_from_files_equals_what_the_reference_holds(tmp_path, param_root):
    """tolcuda_config_from_files (the file-reading half of tolcuda_create_from_files, host only) against the
    members of the UNMODIFIED reference's problem object built from the same files and command line
    (src/parameters.cpp:42-148, src/problem.cpp:13-60): aircraft with its degree -> radian conversions, gains,
    limits, solver tolerances, ts, the ENU -> NED goal; and the errors of the reference's own checks.  The members
    are those the reference held for the command lines of tests/golden (stored there) and, where oracle/_ref is
    built, those of live reference objects on random command lines."""
    import refclient as R
    root = param_root
    P = json.load(open(os.path.join(GOLDEN_DIR, "params.json")))
    for name in GOLDEN:
        g = load_golden(name)
        mission, ts = str(g["mission"]), int(g["ts"])
        cfg = T.config_from_files(root, str(g["aircraft"]), mission, g["enu"], g["goal_enu"], ts=ts)
        assert (cfg.formulation, cfg.ts, cfg.wind_model) == ({"G7": 7, "S10": 10}[mission], ts, 1), name
        assert list(cfg.aircraft) == g["ac"].tolist(), name
        assert list(cfg.gains) == P["problems"][mission]["gains"], name  # the *_gains fixtures edited gains.param
        lm = g["lm"]
        assert list(cfg.limits) == [lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]], name
        assert list(cfg.solver_tol) == g["sn"][4:6].tolist(), name
        assert np.array_equal(np.array(list(cfg.goal)).view(np.int64), g["goal_ned"].view(np.int64)), name
        assert np.array_equal(T.initial_guess(cfg).view(np.int64), g["x"][0].view(np.int64)), name
        for got, key in zip(T.bounds(cfg), ("xlow", "xupp", "Flow", "Fupp")):
            assert np.array_equal(got, g[key]), (name, key)
    rng = np.random.default_rng(5)
    live = ["skywalker", "tempest", "tempest_eric", "tempest_wences", "tempest_will"] * 2 if R.available() else []
    for trial, ac in enumerate(live):
        mission = "G7" if trial % 2 else "S10"
        enu = tuple(float(v) for v in rng.uniform(-50, 150, 3))
        goal = tuple(float(v) for v in rng.uniform(-400, 400, 4))
        p = R.RefProblem(mission, ac, enu, goal)
        prm = p.params()
        cfg = T.config_from_files(root, ac, mission, enu, goal)
        assert (cfg.formulation, cfg.ts, cfg.wind_model) == ({"G7": 7, "S10": 10}[mission], p.ts, prm["wind_model"])
        assert list(cfg.aircraft) == prm["ac"].tolist()
        assert list(cfg.gains) == prm["gn"].tolist()
        lm = prm["lm"]  # member order dtmin,dtmax,xmax,ymax,zmax,xmin,ymin,zmin -> file order
        assert list(cfg.limits) == [lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]]
        assert list(cfg.solver_tol) == prm["sn"][4:6].tolist()
        assert np.array_equal(np.array(list(cfg.goal)).view(np.int64), prm["goal"].view(np.int64))  # -0.0 included
        # and the setup built from it is the reference's
        assert np.array_equal(T.initial_guess(cfg), p.x0())
        for got, want in zip(T.bounds(cfg), p.bounds()):
            assert np.array_equal(got, want)
        p.close()
    assert T.config_from_files(root, "tempest", "S10", ts=37).ts == 37
    with pytest.raises(T.TolcudaError, match="not recognized"):
        T.config_from_files(root, "tempest", "S11")
    with pytest.raises(T.TolcudaError, match="cannot open parameter file"):
        T.config_from_files(root, "no_such_aircraft", "S10")
    with pytest.raises(T.TolcudaError, match="cannot open parameter file"):
        T.config_from_files(str(tmp_path) + "/", "tempest", "S10")
