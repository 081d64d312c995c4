import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
GOLDEN = sorted(os.path.splitext(os.path.basename(f))[0] for f in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))

# north_star tolerance: F/G within 1e-12 relative, 1e-14 absolute of the reference
RTOL, ATOL = 1e-12, 1e-14


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def load_golden(name):
    return np.load(os.path.join(GOLDEN_DIR, name + ".npz"))


def assert_parity(got, ref, what=""):
    """|got - ref| <= ATOL + RTOL*|ref| elementwise; reports the worst offender"""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert np.isfinite(got).all(), "%s: non-finite values at %s" % (what, np.where(~np.isfinite(got))[0][:8])
    err = np.abs(got - ref)
    tol = ATOL + RTOL * np.abs(ref)
    bad = err > tol
    if bad.any():
        i = np.unravel_index(np.argmax(err / tol), err.shape)
        raise AssertionError("%s: %d entries outside 1e-14+1e-12*|ref|; worst at %s: got %r ref %r (err %.3e)"
                             % (what, bad.sum(), i, got[i], ref[i], err[i]))


def port_from_golden(g):
    import portclient as P
    wm = int(g["wind_model"])
    p = P.PortProblem(str(g["mission"]), int(g["ts"]), g["ac"], g["gn"], g["goal_ned"], 1 if wm == 3 else wm)
    if wm == 3:
        p.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
    return p


def write_param_tree(base):
    """aircraft/<name>.param and problems/<M>/{gains,limits,snopt}.param under `base`, rebuilt from the values the
    reference read from its own files (tests/golden/params.json): a header comment, then `value\\n // comment` lines,
    angles in degrees, CRLF line ends in skywalker.param.  Not the reference's files byte for byte (their comment
    texts are not stored), but the same values in the layout its reader was written for.  Returns base + '/'."""
    import json
    P = json.load(open(os.path.join(GOLDEN_DIR, "params.json")))

    def write(rel, values, eol="\n"):
        path = os.path.join(base, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "wb") as fh:
            fh.write(("//parameters" + eol + "".join("%r\\n    // p%d%s" % (float(v), i, eol)
                                                     for i, v in enumerate(values))).encode())
    for ac, v in P["aircraft"].items():
        v = list(v)
        for i in (8, 11, 12):  # stored in radians, written in degrees (reference src/parameters.cpp:56-60)
            v[i] = round(v[i] * 180.0 / np.pi, 6)
        write("aircraft/%s.param" % ac, v, "\r\n" if ac == "skywalker" else "\n")
    for ms, d in P["problems"].items():
        lm = d["limits_member_order"]  # dtmin,dtmax,xmax,ymax,zmax,xmin,ymin,zmin -> file order
        write("problems/%s/gains.param" % ms, d["gains"])
        write("problems/%s/snopt.param" % ms, d["snopt"])
        write("problems/%s/limits.param" % ms, [lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]])
    return str(base) + "/"


@pytest.fixture
def param_root(tmp_path):
    """a .param root: the reference's own files where `make -C oracle ref` copied them into oracle/_ref/params,
    otherwise write_param_tree's rebuilt ones.  Returned with a trailing '/'."""
    ref = os.path.join(ROOT, "oracle", "_ref", "params")
    if os.path.isdir(os.path.join(ref, "aircraft")):
        return ref + "/"
    return write_param_tree(tmp_path / "params")


# ---- stored pins of what the unmodified reference returned to the tests that compare with it on fresh inputs
#
# Each such test computes its inputs from fixed seeds, compares what this project computes with what the reference
# returns, and checks a digest of every compared value (Pins.check) against tests/golden/reference_pins.json, in call
# order.  Where oracle/_ref is built the live comparison runs as well; elsewhere StandInRef supplies the inputs the
# reference would (parameters, x0, bounds) from this project's own host functions, and the pins alone decide.
# TOL_RECORD_PINS=1 records the digests instead of checking them (run with oracle/_ref built, so that every recorded
# value has been compared with the reference in the same run).
PINS_PATH = os.path.join(GOLDEN_DIR, "reference_pins.json")
RECORD_PINS = os.environ.get("TOL_RECORD_PINS") == "1"
_pins_stored, _pins_recorded = None, {}


def bits(*values):
    """16 hex digits of the sha256 of the exact bits of arrays (dtype and shape included; every NaN as one
    pattern, so NaN positions count and NaN payloads do not) and of byte strings"""
    import hashlib
    h = hashlib.sha256()
    for v in values:
        if isinstance(v, bytes):
            h.update(b"bytes%d:" % len(v) + v)
            continue
        a = np.ascontiguousarray(v)
        if a.dtype.kind == "f":
            a = np.where(np.isnan(a), np.nan, a.astype(np.float64))
        h.update(("%s%s:" % (a.dtype, a.shape)).encode() + a.tobytes())
    return h.hexdigest()[:16]


class Pins:
    def __init__(self, test):
        global _pins_stored
        if _pins_stored is None:
            import json
            _pins_stored = json.load(open(PINS_PATH)) if os.path.exists(PINS_PATH) else {}
        self.test, self.k = test, 0
        self.want = _pins_stored.get(test, [])
        if RECORD_PINS:
            self.want = _pins_recorded[test] = []
        assert RECORD_PINS or self.want, "no stored pins for " + test

    def check(self, *values, what=""):
        d = bits(*values)
        if RECORD_PINS:
            self.want.append(d)
        else:
            assert self.k < len(self.want), "%s: more values than stored pins" % self.test
            assert d == self.want[self.k], "%s: value %d (%s) differs from the reference's" % (self.test, self.k, what)
        self.k += 1

    def done(self):
        assert self.k == len(self.want), "%s: %d of %d stored pins checked" % (self.test, self.k, len(self.want))


@pytest.fixture
def pins(request):
    return Pins(request.node.name)


def pytest_sessionfinish(session):
    if RECORD_PINS and _pins_recorded:
        import json
        data = json.load(open(PINS_PATH)) if os.path.exists(PINS_PATH) else {}
        data.update(_pins_recorded)
        with open(PINS_PATH, "w") as fh:
            json.dump(data, fh, indent=0, sort_keys=True)
            fh.write("\n")


class StandInRef:
    """The refclient.RefProblem interface without the reference: parameters from the .param files through
    tolcuda_config_from_files, x0 / bounds / pattern from the library's host functions, F and G from the CPU port,
    the result files from the library's writers.  A test comparing against it compares this project with itself;
    what makes it a check is Pins."""

    def __init__(self, root, mission, aircraft, enu=(0.0, 0.0, 70.0), goal=(0.0, 0.0, 0.0, 0.0), ts=None, gains=None,
                 null_io=True):
        import portclient as P
        import tol_b200 as T
        self.T, self.mission, self.aircraft, self.enu = T, mission, aircraft, tuple(enu)
        cfg = T.config_from_files(root, aircraft, mission, enu, goal, ts=ts or 0)
        if gains is not None:
            cfg.gains[:] = [float(v) for v in gains]
        self.cfg, self.ts = cfg, cfg.ts
        self.n, self.neF, self.neG = T.problem_dims(mission, self.ts)
        self.nb = 12 if mission == "G7" else 11
        self.port = P.PortProblem(mission, self.ts, list(cfg.aircraft), list(cfg.gains), list(cfg.goal), cfg.wind_model)

    def close(self):
        pass

    def params(self):
        c, f = self.cfg, list(self.cfg.limits)  # file order dtmin dtmax xmin xmax ymin ymax zmin zmax -> member order
        return dict(ac=np.array(c.aircraft[:]), gn=np.array(c.gains[:]), lm=np.array([f[0], f[1], f[3], f[5], f[7], f[2], f[4], f[6]]),
                    sn=np.array([float(self.ts), 11.0, 8.0, float(self.nb)] + list(c.solver_tol)), goal=np.array(c.goal[:]),
                    wind_model=c.wind_model)

    def x0(self):
        return self.T.initial_guess(self.cfg)

    def bounds(self):
        return self.T.bounds(self.cfg)

    def pattern(self):
        return self.T.problem_pattern(self.mission, self.ts)

    def chi_d(self):
        return self.port.p.chi_d

    def ub_mask(self):
        return self.port.ub_mask()

    def set_wind_grid(self, gx, gy, gz, uvw, datum, spacing):
        self.port.set_wind_grid(gx, gy, gz, np.ascontiguousarray(uvw[..., 1]), datum, spacing)

    def eval(self, x):
        return self.port.eval(x)

    def write_json(self, x, F0, path):
        self.T.write_results_json(self.cfg, self.aircraft, self.mission, self.enu, x, F0, path)

    def write_txt(self, x, F0, directory):
        path = os.path.join(directory, "snopt_output.txt")
        self.T.write_results_txt(self.cfg, x, F0, path)
        return path


@pytest.fixture
def reference(param_root):
    """RefProblem(...) of the compiled reference where oracle/_ref is built, StandInRef(...) otherwise"""
    import refclient as R
    if R.available():
        return R.RefProblem
    return lambda *a, **k: StandInRef(param_root, *a, **k)


@pytest.fixture(scope="session")
def oracle_built():
    """the plain-C oracle, built on demand (gcc only)"""
    import subprocess
    import portclient as P
    if not P.available():
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "port"])
    return P
