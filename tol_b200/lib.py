"""ctypes binding of libtolcuda.so (include/tolcuda.h).  The library is built in-tree by
`make -C tol_b200/csrc` (see __graft_entry__.build); a missing library is an error, never a
fallback."""
import ctypes as C
import os

LIB_PATH = os.environ.get("TOLCUDA_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libtolcuda.so")


class TolcudaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("tolcuda error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):
    """struct tolcuda_config"""
    _fields_ = [("formulation", C.c_int), ("ts", C.c_int), ("wind_model", C.c_int),
                ("device", C.c_int), ("aircraft", C.c_double * 15), ("gains", C.c_double * 5),
                ("goal", C.c_double * 4), ("limits", C.c_double * 8), ("solver_tol", C.c_double * 2)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libtolcuda.so is not built (%s): run `python -c 'import __graft_entry__ as g; "
                          "g.build()'` or `make -C tol_b200/csrc`; there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_void_p
    L.tolcuda_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.tolcuda_create_from_files.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p] + [C.c_double] * 7 + \
        [C.c_int, C.c_int, C.POINTER(vp)]
    L.tolcuda_config_from_files.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p] + [C.c_double] * 7 + \
        [C.c_int, C.c_int, C.POINTER(Config)]
    L.tolcuda_destroy.argtypes = [vp]
    L.tolcuda_set_wind_grid.argtypes = [vp, C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, dp, dp]
    L.tolcuda_dims.argtypes = [vp, ip, ip, ip]
    L.tolcuda_pattern.argtypes = [vp, ip, ip]
    L.tolcuda_problem_dims.argtypes = [C.c_int, C.c_int, ip, ip, ip]
    L.tolcuda_problem_pattern.argtypes = [C.c_int, C.c_int, ip, ip]
    L.tolcuda_problem_initial_guess.argtypes = [C.POINTER(Config), dp]
    L.tolcuda_problem_bounds.argtypes = [C.POINTER(Config), dp, dp, dp, dp]
    L.tolcuda_write_results_json.argtypes = [C.POINTER(Config), C.c_char_p, C.c_char_p, C.c_double, C.c_double,
                                             C.c_double, dp, C.c_double, C.c_char_p]
    L.tolcuda_write_results_txt.argtypes = [C.POINTER(Config), dp, C.c_double, C.c_char_p]
    L.tolcuda_get_config.argtypes = [vp, C.POINTER(Config)]
    L.tolcuda_eval.argtypes = [vp, dp, C.c_int, dp, C.c_int, dp]
    L.tolcuda_eval_batch.argtypes = [vp, C.c_int, vp, C.c_long, vp, C.c_long, vp, C.c_long, C.c_int]
    L.tolcuda_eval_batch_summary.argtypes = [vp, C.c_int, vp, C.c_long, vp, C.c_long, vp, C.c_long, vp, C.c_long, C.c_int]
    L.tolcuda_set_goals.argtypes = [vp, C.c_long, vp, C.c_long]
    L.tolcuda_eval_batch_goals.argtypes = [vp, C.c_long, C.c_int, vp, C.c_long, vp, C.c_long, vp, C.c_long, vp, C.c_long,
                                           C.c_int]
    L.tolcuda_compact_len.argtypes = [C.c_int, C.c_int]
    L.tolcuda_compact_len.restype = C.c_long
    L.tolcuda_expand_compact_g.argtypes = [C.c_int, C.c_int, C.c_long, vp, C.c_long, vp, C.c_long, C.c_int]
    L.tolcuda_set_host_threads.argtypes = [vp, C.c_int]
    L.tolcuda_set_option.argtypes = [vp, C.c_char_p, C.c_long]
    L.tolcuda_problem_pattern_csc.argtypes = [C.c_int, C.c_int, ip, ip, ip]
    L.tolcuda_repack_csc_device.argtypes = [vp, C.c_long, vp, C.c_long, vp, C.c_long, C.c_int]
    L.tolcuda_expand_compact_g_device.argtypes = [vp, C.c_long, vp, C.c_long, vp, C.c_long, C.c_int]
    L.tolcuda_jac_vec.argtypes = [vp, C.c_int, vp, C.c_long, vp, C.c_long, vp, C.c_long, C.c_int]
    L.tolcuda_jac_tvec.argtypes = [vp, C.c_int, vp, C.c_long, vp, C.c_long, vp, C.c_long, C.c_int]
    L.tolcuda_lag_hess_vec.argtypes = [vp, C.c_int, vp, C.c_long, vp, C.c_long, vp, C.c_long, vp, C.c_long, vp,
                                       C.c_long, C.c_int]
    L.tolcuda_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.tolcuda_host_free.argtypes = [vp]
    L.tolcuda_device_count.argtypes = [ip]
    L.tolcuda_device_alloc.argtypes = [C.c_int, C.c_size_t, C.POINTER(vp)]
    L.tolcuda_device_free.argtypes = [C.c_int, vp]
    L.tolcuda_ipc_export.argtypes = [C.c_int, vp, C.c_char_p]
    L.tolcuda_ipc_open.argtypes = [C.c_int, C.c_char_p, C.POINTER(vp)]
    L.tolcuda_ipc_close.argtypes = [C.c_int, vp]
    L.tolcuda_enable_peer.argtypes = [C.c_int, C.c_int]
    L.tolcuda_stream_signal.argtypes = [vp, vp, C.c_uint]
    L.tolcuda_stream_wait.argtypes = [vp, vp, C.c_uint]
    L.tolcuda_gather_create.argtypes = [vp, C.c_long, C.c_int, C.c_int, C.POINTER(vp), C.c_char_p]
    L.tolcuda_gather_attach.argtypes = [vp, C.c_long, C.c_int, C.c_int, C.c_int, vp, C.c_char_p, C.POINTER(vp)]
    L.tolcuda_gather_send.argtypes = [vp, vp, C.c_long, C.c_int]
    L.tolcuda_gather_collect.argtypes = [vp, vp, C.c_long, C.c_int, C.POINTER(vp), C.POINTER(C.c_long), C.POINTER(vp), C.POINTER(C.c_long)]
    L.tolcuda_gather_buffer.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]
    L.tolcuda_gather_close.argtypes = [vp]
    L.tolcuda_copy_to_device.argtypes = [C.c_int, vp, vp, C.c_size_t]
    L.tolcuda_copy_to_host.argtypes = [C.c_int, vp, vp, C.c_size_t]
    L.tolcuda_padded_ld.argtypes = [C.c_long]
    L.tolcuda_padded_ld.restype = C.c_long
    L.tolcuda_set_stream.argtypes = [vp, vp]
    L.tolcuda_use_own_stream.argtypes = [vp]
    L.tolcuda_synchronize.argtypes = [vp]
    L.tolcuda_launch_count.argtypes = [vp]
    L.tolcuda_launch_count.restype = C.c_long
    L.tolcuda_bind_global.argtypes = [vp]
    L.tolcuda_set_dump_dir.argtypes = [vp, C.c_char_p]
    L.tolcuda_write_dump.argtypes = [C.c_char_p, dp, C.c_long]
    L.tolcuda_write_wind_dump.argtypes = [C.c_char_p, C.c_int, C.c_int, dp]
    L.DEFINEGusrfg_.argtypes = [ip, ip, dp, ip, ip, dp, ip, ip, dp, C.c_char_p, ip, ip, ip, dp, ip]
    L.DEFINEGusrfg_.restype = None
    L.tolcuda_read_params.argtypes = [C.c_char_p, dp, C.c_int, ip]
    L.tolcuda_last_error.restype = C.c_char_p
    L.tolcuda_version.restype = C.c_char_p
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise TolcudaError(rc, load().tolcuda_last_error().decode(errors="replace"))
