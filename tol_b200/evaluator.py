"""Thin object wrapper over the libtolcuda C ABI: one Evaluator == one `tolcuda_handle`, i.e. what a
reference `problemG7` / `problemS10` object is to the reference callback (src/tol.cpp:5-36).  Every
evaluation goes through the C entry points a C/C++ caller would use."""
import ctypes as C

import numpy as np

from . import lib as _l

G7, S10 = 7, 10
NEED_F, NEED_G = 0x1, 0x2
HOST_PTRS, DEVICE_PTRS, NO_SYNC, COMPACT_G, FULL_G_COPY = 0x10, 0x20, 0x40, 0x80, 0x100
OVERLAP, OVERLAP_DISJOINT = 0x200, 0x400
_FORM = {"G7": G7, "S10": S10, G7: G7, S10: S10}


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def problem_dims(mission, ts):
    n, neF, neG = C.c_int(), C.c_int(), C.c_int()
    _l.check(_l.load().tolcuda_problem_dims(_FORM[mission], int(ts), C.byref(n), C.byref(neF),
                                            C.byref(neG)))
    return n.value, neF.value, neG.value


def problem_pattern(mission, ts):
    _, _, neG = problem_dims(mission, ts)
    i, j = np.empty(neG, np.int32), np.empty(neG, np.int32)
    _l.check(_l.load().tolcuda_problem_pattern(_FORM[mission], int(ts), _ip(i), _ip(j)))
    return i, j


def problem_pattern_csc(mission, ts):
    """tolcuda_problem_pattern_csc: colptr[n+1], rowidx[neG], perm[neG] (CSC position -> coordinate-order position)"""
    n, _, neG = problem_dims(mission, ts)
    cp, ri, pm = np.empty(n + 1, np.int32), np.empty(neG, np.int32), np.empty(neG, np.int32)
    _l.check(_l.load().tolcuda_problem_pattern_csc(_FORM[mission], int(ts), _ip(cp), _ip(ri), _ip(pm)))
    return cp, ri, pm


def read_params(path, cap=64):
    v = np.zeros(cap)
    cnt = C.c_int()
    _l.check(_l.load().tolcuda_read_params(str(path).encode(), _dp(v), cap, C.byref(cnt)))
    return v[:min(cnt.value, cap)].copy(), cnt.value


def make_config(mission, ts, aircraft, gains, goal_ned, wind_model=1, device=0, limits=None, solver_tol=None):
    cfg = _l.Config()
    cfg.formulation, cfg.ts, cfg.wind_model, cfg.device = _FORM[mission], int(ts), int(wind_model), int(device)
    cfg.aircraft[:] = [float(v) for v in aircraft]
    cfg.gains[:] = [float(v) for v in gains]
    cfg.goal[:] = [float(v) for v in goal_ned]
    cfg.limits[:] = [float(v) for v in (limits if limits is not None else [0.0] * 8)]
    cfg.solver_tol[:] = [float(v) for v in (solver_tol if solver_tol is not None else [0.0, 0.0])]
    return cfg


def config_from_files(root, aircraft, mission, enu=(0.0, 0.0, 0.0), goal_enu=(0.0, 0.0, 0.0, 0.0), ts=0, device=0):
    """tolcuda_config_from_files: the reference's .param files and command line as a Config (host only)"""
    cfg = _l.Config()
    _l.check(_l.load().tolcuda_config_from_files(str(root).encode(), aircraft.encode(), mission.encode(),
                                                 *[float(v) for v in enu], *[float(v) for v in goal_enu],
                                                 int(ts), int(device), C.byref(cfg)))
    return cfg


def initial_guess(cfg):
    """reference InitialCond: x0[n] (host only)"""
    n, _, _ = problem_dims(cfg.formulation, cfg.ts)
    x0 = np.empty(n)
    _l.check(_l.load().tolcuda_problem_initial_guess(C.byref(cfg), _dp(x0)))
    return x0


def bounds(cfg):
    """reference setLimits: xlow, xupp, Flow, Fupp (host only)"""
    n, neF, _ = problem_dims(cfg.formulation, cfg.ts)
    xl, xu, fl, fu = np.empty(n), np.empty(n), np.empty(neF), np.empty(neF)
    _l.check(_l.load().tolcuda_problem_bounds(C.byref(cfg), _dp(xl), _dp(xu), _dp(fl), _dp(fu)))
    return xl, xu, fl, fu


def write_results_json(cfg, aircraft, mission, enu, x, final_cost, path):
    """reference problem::writeJSON (snopt_results.json), byte for byte"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    _l.check(_l.load().tolcuda_write_results_json(C.byref(cfg), aircraft.encode(), mission.encode(),
                                                  *[float(v) for v in enu], _dp(x), float(final_cost),
                                                  str(path).encode()))


def write_results_txt(cfg, x, final_cost, path):
    """reference problem::writeTXT (snopt_output.txt), byte for byte"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    _l.check(_l.load().tolcuda_write_results_txt(C.byref(cfg), _dp(x), float(final_cost), str(path).encode()))


def padded_ld(n):
    return int(_l.load().tolcuda_padded_ld(int(n)))


def compact_len(mission, ts):
    """doubles of a compact G row (tolcuda_compact_len)"""
    v = int(_l.load().tolcuda_compact_len(_FORM[mission], int(ts)))
    _l.check(min(v, 0))
    return v


def expand_compact_g(mission, ts, Gc, G=None, threads=0):
    """tolcuda_expand_compact_g: compact rows [B, >= compact_len] -> rows in coordinate order (host only)"""
    _, _, neG = problem_dims(mission, ts)
    B = Gc.shape[0]
    assert Gc.dtype == np.float64 and (B == 0 or Gc.strides[1] == 8)
    if G is None:
        G = np.empty((B, neG))
    _l.check(_l.load().tolcuda_expand_compact_g(_FORM[mission], int(ts), B, Gc.ctypes.data, Gc.strides[0] // 8,
                                                G.ctypes.data, G.strides[0] // 8, int(threads)))
    return G


IPC_HANDLE_BYTES = 64


class PeerBuffer:
    """Device memory other GPUs of the box can write (include/tolcuda.h, "result buffers that other GPUs
    write directly").  PeerBuffer.alloc on the gathering rank, .handle sent to the others, PeerBuffer.open
    there.  .ptr is the address valid on `device`; .tensor(...) views the owner's allocation as a torch tensor."""

    def __init__(self, device, ptr, nbytes, owner, handle=None):
        self.device, self.ptr, self.nbytes, self.owner, self.handle = device, ptr, nbytes, owner, handle

    @classmethod
    def alloc(cls, device, nbytes):
        L = _l.load()
        p = C.c_void_p()
        _l.check(L.tolcuda_device_alloc(int(device), int(nbytes), C.byref(p)))
        h = C.create_string_buffer(IPC_HANDLE_BYTES)
        rc = L.tolcuda_ipc_export(int(device), p, h)
        if rc:
            L.tolcuda_device_free(int(device), p)
            _l.check(rc)
        return cls(device, p.value, nbytes, True, h.raw)

    @classmethod
    def open(cls, device, handle, nbytes):
        p = C.c_void_p()
        _l.check(_l.load().tolcuda_ipc_open(int(device), handle, C.byref(p)))
        return cls(device, p.value, nbytes, False, handle)

    def close(self):
        """owner True: frees the allocation; False: unmaps the IPC mapping; None: a view of memory owned elsewhere"""
        if getattr(self, "ptr", None):
            ptr, self.ptr = self.ptr, None
            L = _l.load()
            if self.owner is not None:
                (L.tolcuda_device_free if self.owner else L.tolcuda_ipc_close)(int(self.device), C.c_void_p(ptr))

    __del__ = close

    def tensor(self, offset_doubles, rows, ld):
        """[rows, ld] float64 torch view of the allocation, starting `offset_doubles` in (the tensor keeps
        this object alive)"""
        import torch
        assert 8 * (offset_doubles + rows * ld) <= self.nbytes

        class _View:
            pass
        v = _View()
        v.keep = self
        v.__cuda_array_interface__ = {"shape": (rows, ld), "typestr": "<f8", "version": 2, "strides": None,
                                      "data": (self.ptr + 8 * offset_doubles, False)}
        return torch.as_tensor(v, device=torch.device("cuda", self.device))


class Evaluator:
    def __init__(self, mission, ts, aircraft, gains, goal_ned, wind_model=1, device=0):
        L = _l.load()
        cfg = make_config(mission, ts, aircraft, gains, goal_ned, wind_model, device)
        self.h = C.c_void_p()
        _l.check(L.tolcuda_create(C.byref(cfg), C.byref(self.h)))
        self._finish(L, device)

    @classmethod
    def from_files(cls, root, aircraft, mission, enu=(0.0, 0.0, 0.0), goal_enu=(0.0, 0.0, 0.0, 0.0),
                   ts=0, device=0):
        L = _l.load()
        self = cls.__new__(cls)
        self.h = C.c_void_p()
        _l.check(L.tolcuda_create_from_files(str(root).encode(), aircraft.encode(), mission.encode(),
                                             *[float(v) for v in enu], *[float(v) for v in goal_enu],
                                             int(ts), int(device), C.byref(self.h)))
        self._finish(L, device)
        return self

    @classmethod
    def from_golden(cls, g, device=0, wind_model=None, options=None):
        """g: an opened tests/golden/*.npz fixture; options: {name: value} for tolcuda_set_option"""
        wm = int(g["wind_model"]) if wind_model is None else wind_model
        ev = cls(str(g["mission"]), int(g["ts"]), g["ac"], g["gn"], g["goal_ned"], 1 if wm == 3 else wm, device)
        for k, v in (options or {}).items():
            ev.set_option(k, v)
        if wm == 3:
            ev.set_wind_grid(g["grid_x"], g["grid_y"], g["grid_z"], g["grid_v"], g["grid_datum"], g["grid_spacing"])
        return ev

    def _finish(self, L, device):
        self.L, self.device = L, device
        self._stream_pinned = False  # True once the caller has chosen a stream (set_stream / use_own_stream)
        n, neF, neG = C.c_int(), C.c_int(), C.c_int()
        _l.check(L.tolcuda_dims(self.h, C.byref(n), C.byref(neF), C.byref(neG)))
        self.n, self.neF, self.neG = n.value, neF.value, neG.value
        self.compact_len = int(L.tolcuda_compact_len(self.cfg_form(), self.cfg_ts()))

    def _config(self):
        cfg = _l.Config()
        _l.check(self.L.tolcuda_get_config(self.h, C.byref(cfg)))
        return cfg

    def cfg_form(self):
        return self._config().formulation

    def cfg_ts(self):
        return self._config().ts

    def set_host_threads(self, threads):
        _l.check(self.L.tolcuda_set_host_threads(self.h, int(threads)))

    def _follow_torch(self, t):
        """Calls that take torch tensors run on torch's CURRENT stream of the tensors' device unless the caller has
        chosen a stream: the context's own stream is non-blocking, so work torch has queued on the tensors (fills,
        copies, slice assignments) would otherwise not be ordered against the kernels (include/tolcuda.h,
        tolcuda_set_stream)."""
        if not self._stream_pinned:
            import torch
            _l.check(self.L.tolcuda_set_stream(self.h, C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)))

    def set_option(self, name, value):
        """tolcuda_set_option: execution-strategy options (kernel, per, tail_x4, chunk_mb, ...); results never change"""
        _l.check(self.L.tolcuda_set_option(self.h, name.encode(), int(value)))

    def close(self):
        if getattr(self, "h", None):
            self.L.tolcuda_destroy(self.h)
            self.h = None

    __del__ = close

    def set_wind_grid(self, gx, gy, gz, v, datum, spacing):
        """tolcuda_set_wind_grid: reference wind model 3 on a wind cube v[ne, nn, nu]"""
        a = [np.ascontiguousarray(t, dtype=np.float64) for t in (gx, gy, gz, v, datum, spacing)]
        assert a[3].shape == (a[0].size, a[1].size, a[2].size)
        _l.check(self.L.tolcuda_set_wind_grid(self.h, a[0].size, a[1].size, a[2].size, *[_dp(t) for t in a]))

    def pattern(self):
        i, j = np.empty(self.neG, np.int32), np.empty(self.neG, np.int32)
        _l.check(self.L.tolcuda_pattern(self.h, _ip(i), _ip(j)))
        return i, j

    def eval(self, x, needF=True, needG=True):
        """tolcuda_eval: one trajectory, host arrays"""
        x = np.ascontiguousarray(x, dtype=np.float64)
        assert x.size == self.n
        F = np.full(self.neF, np.nan)
        G = np.full(self.neG, np.nan)
        _l.check(self.L.tolcuda_eval(self.h, _dp(x), int(needF), _dp(F), int(needG), _dp(G)))
        return F, G

    def usrfun(self, x, needF=1, needG=1, bind=True):
        """call the exported snOptA callback DEFINEGusrfg_ exactly as SNOPT would"""
        if bind:
            _l.check(self.L.tolcuda_bind_global(self.h))
        x = np.ascontiguousarray(x, dtype=np.float64)
        F = np.full(self.neF, np.nan)
        G = np.full(self.neG, np.nan)
        st = C.c_int(0)
        ints = [C.c_int(v) for v in (self.n, needF, self.neF, needG, self.neG, 0, 0, 0)]
        n_, nf_, neF_, ng_, neG_, lencu, leniu, lenru = ints
        self.L.DEFINEGusrfg_(C.byref(st), C.byref(n_), _dp(x), C.byref(nf_), C.byref(neF_), _dp(F),
                             C.byref(ng_), C.byref(neG_), _dp(G), None, C.byref(lencu), None,
                             C.byref(leniu), None, C.byref(lenru))
        return st.value, F, G

    def set_dump_dir(self, directory):
        """tolcuda_set_dump_dir: the reference callback's Xoutput/Woutput/Foutput/Goutput.txt on every usrfun call
        (src/DefineFG.cpp:16-46); None switches them off"""
        _l.check(self.L.tolcuda_set_dump_dir(self.h, None if directory is None else str(directory).encode()))

    def eval_batch_host(self, X, F=None, G=None, needF=True, needG=True, full_copy=False, compact_rows=False):
        """tolcuda_eval_batch with HOST arrays (numpy, or pinned torch tensors via .numpy());
        full_copy: TOLCUDA_FULL_G_COPY; compact_rows: G receives compact rows (TOLCUDA_COMPACT_G)"""
        B = X.shape[0]
        assert X.dtype == np.float64 and X.strides[1] == 8
        if F is None:
            F = np.empty((B, self.neF))
        if G is None:
            G = np.empty((B, self.compact_len if compact_rows else self.neG))
        flags = (NEED_F if needF else 0) | (NEED_G if needG else 0) | HOST_PTRS
        flags |= (FULL_G_COPY if full_copy else 0) | (COMPACT_G if compact_rows else 0)
        _l.check(self.L.tolcuda_eval_batch(self.h, B, X.ctypes.data, X.strides[0] // 8, F.ctypes.data,
                                           F.strides[0] // 8, G.ctypes.data, G.strides[0] // 8, flags))
        return F, G

    def eval_batch_device(self, X, F, G, needF=True, needG=True, sync=True, compact_rows=False, overlap=0):
        """tolcuda_eval_batch with torch CUDA tensors [B, ld] (float64, row-contiguous).  overlap (sync=False only):
        1 = TOLCUDA_OVERLAP, 2 = TOLCUDA_OVERLAP_DISJOINT"""
        self._follow_torch(X)
        B = X.shape[0]
        flags = (NEED_F if needF else 0) | (NEED_G if needG else 0) | DEVICE_PTRS | (0 if sync else NO_SYNC)
        flags |= COMPACT_G if compact_rows else 0
        flags |= (OVERLAP if overlap == 1 else 0) | (OVERLAP_DISJOINT if overlap == 2 else 0)
        _l.check(self.L.tolcuda_eval_batch(self.h, B, X.data_ptr(), X.stride(0), F.data_ptr(), F.stride(0),
                                           G.data_ptr(), G.stride(0), flags))

    def eval_batch_ptrs(self, B, x_ptr, ldx, F_ptr, ldF, G_ptr, ldG, needF=True, needG=True, sync=True,
                        compact_rows=False):
        """tolcuda_eval_batch with raw device addresses (integers): F_ptr / G_ptr may lie in a peer GPU's memory
        (PeerBuffer), x_ptr on this context's device"""
        flags = (NEED_F if needF else 0) | (NEED_G if needG else 0) | DEVICE_PTRS | (0 if sync else NO_SYNC)
        flags |= COMPACT_G if compact_rows else 0
        _l.check(self.L.tolcuda_eval_batch(self.h, int(B), x_ptr, int(ldx), F_ptr, int(ldF), G_ptr, int(ldG), flags))

    def expand_compact_device(self, Gc, G, sync=True):
        """tolcuda_expand_compact_g_device: compact rows (torch CUDA tensor [B, >= compact_len]) -> rows in
        coordinate order (torch CUDA tensor [B, >= neG]) on the context's stream"""
        self._follow_torch(Gc)
        _l.check(self.L.tolcuda_expand_compact_g_device(self.h, Gc.shape[0], Gc.data_ptr(), Gc.stride(0), G.data_ptr(),
                                                        G.stride(0), 0 if sync else NO_SYNC))

    def repack_csc_device(self, G, Gcsc, sync=True):
        """tolcuda_repack_csc_device: rows in coordinate order -> rows in CSC order (torch CUDA tensors)"""
        self._follow_torch(G)
        _l.check(self.L.tolcuda_repack_csc_device(self.h, G.shape[0], G.data_ptr(), G.stride(0), Gcsc.data_ptr(),
                                                  Gcsc.stride(0), 0 if sync else NO_SYNC))

    def jac_vec(self, X, D, Y, sync=True):
        """tolcuda_jac_vec: Y[b] = J(X[b]) D[b] without materialising G (torch CUDA tensors [B, >= n], [B, >= n],
        [B, >= neF])"""
        self._follow_torch(X)
        _l.check(self.L.tolcuda_jac_vec(self.h, X.shape[0], X.data_ptr(), X.stride(0), D.data_ptr(), D.stride(0),
                                        Y.data_ptr(), Y.stride(0), 0 if sync else NO_SYNC))

    def jac_tvec(self, X, Lam, Z, sync=True):
        """tolcuda_jac_tvec: Z[b] = J(X[b])^T Lam[b] (torch CUDA tensors [B, >= n], [B, >= neF], [B, >= n])"""
        self._follow_torch(X)
        _l.check(self.L.tolcuda_jac_tvec(self.h, X.shape[0], X.data_ptr(), X.stride(0), Lam.data_ptr(), Lam.stride(0),
                                         Z.data_ptr(), Z.stride(0), 0 if sync else NO_SYNC))

    def lag_hess_vec(self, X, Lam, D, W, Z=None, sync=True):
        """tolcuda_lag_hess_vec: W[b] = D_x[J(X[b])^T Lam[b]] D[b], the Hessian of the Lagrangian Lam[b]^T F times D[b],
        and, if Z is given, Z[b] = J(X[b])^T Lam[b] (torch CUDA tensors [B, >= n], [B, >= neF], [B, >= n], [B, >= n],
        [B, >= n])"""
        self._follow_torch(X)
        _l.check(self.L.tolcuda_lag_hess_vec(self.h, X.shape[0], X.data_ptr(), X.stride(0), Lam.data_ptr(), Lam.stride(0),
                                             D.data_ptr(), D.stride(0), W.data_ptr(), W.stride(0),
                                             None if Z is None else Z.data_ptr(), 0 if Z is None else Z.stride(0),
                                             0 if sync else NO_SYNC))

    def summary_host(self, X, needF=False, needG=False):
        """tolcuda_eval_batch_summary with host arrays: [B, 4] = objective, max|defect|, max boundary
        violation, sum defect^2 (F and G are not produced unless asked for)"""
        B = X.shape[0]
        S = np.empty((B, 4))
        F = np.empty((B, self.neF)) if needF else None
        G = np.empty((B, self.neG)) if needG else None
        flags = (NEED_F if needF else 0) | (NEED_G if needG else 0) | HOST_PTRS
        _l.check(self.L.tolcuda_eval_batch_summary(
            self.h, B, X.ctypes.data, X.strides[0] // 8, F.ctypes.data if needF else None, self.neF,
            G.ctypes.data if needG else None, self.neG, S.ctypes.data, 4, flags))
        return S, F, G

    def set_goals(self, goals_ned):
        """tolcuda_set_goals: the context's goal table, one row (xg, yg, zg, rg in NED) per trajectory of
        eval_batch_goals; an empty array frees it"""
        g = np.ascontiguousarray(goals_ned, dtype=np.float64).reshape(-1, 4)
        _l.check(self.L.tolcuda_set_goals(self.h, g.shape[0], g.ctypes.data if g.size else None, 4))

    def eval_batch_goals(self, X, F=None, G=None, row0=0, summary=None, needF=True, needG=True, sync=True,
                         compact_rows=False, full_copy=False, overlap=0):
        """tolcuda_eval_batch_goals: row b of X with goal row row0 + b of the table (set_goals).  X, F, G, summary are
        numpy arrays (host path; F, G allocated if None and asked for) or torch CUDA tensors (device path, like
        eval_batch_device: sync / overlap apply there).  summary: [B, >= 4] or None.  Returns F, G, summary."""
        B = X.shape[0]
        dev = hasattr(X, "data_ptr")
        if dev:
            self._follow_torch(X)
            ptr, ld = (lambda a: a.data_ptr() if a is not None else None), (lambda a: a.stride(0) if a is not None else 0)
            flags = DEVICE_PTRS | (0 if sync else NO_SYNC)
            flags |= (OVERLAP if overlap == 1 else 0) | (OVERLAP_DISJOINT if overlap == 2 else 0)
        else:
            assert X.dtype == np.float64 and X.strides[1] == 8
            if F is None and needF:
                F = np.empty((B, self.neF))
            if G is None and needG:
                G = np.empty((B, self.compact_len if compact_rows else self.neG))
            ptr, ld = (lambda a: a.ctypes.data if a is not None else None), (lambda a: a.strides[0] // 8 if a is not None else 0)
            flags = HOST_PTRS | (FULL_G_COPY if full_copy else 0)
        flags |= (NEED_F if needF else 0) | (NEED_G if needG else 0) | (COMPACT_G if compact_rows else 0)
        _l.check(self.L.tolcuda_eval_batch_goals(self.h, int(row0), B, ptr(X), ld(X), ptr(F), ld(F), ptr(G), ld(G),
                                                 ptr(summary), ld(summary), flags))
        return F, G, summary

    def stream_signal(self, flag_ptr, value):
        """tolcuda_stream_signal: *flag = value after everything enqueued so far on the context's stream"""
        _l.check(self.L.tolcuda_stream_signal(self.h, C.c_void_p(flag_ptr), int(value) & 0xffffffff))

    def stream_wait(self, flag_ptr, value):
        """tolcuda_stream_wait: the context's stream waits until (int)(*flag - value) >= 0"""
        _l.check(self.L.tolcuda_stream_wait(self.h, C.c_void_p(flag_ptr), int(value) & 0xffffffff))

    def set_stream(self, cuda_stream_ptr):
        """cudaStream_t as an integer (torch: stream.cuda_stream; 0 = legacy default stream)"""
        self._stream_pinned = True
        _l.check(self.L.tolcuda_set_stream(self.h, C.c_void_p(cuda_stream_ptr)))

    def follow_torch_stream(self):
        """back to the default: tensor calls run on torch's current stream"""
        self._stream_pinned = False

    def use_own_stream(self):
        self._stream_pinned = True
        _l.check(self.L.tolcuda_use_own_stream(self.h))

    def synchronize(self):
        _l.check(self.L.tolcuda_synchronize(self.h))

    @property
    def launches(self):
        return int(self.L.tolcuda_launch_count(self.h))
