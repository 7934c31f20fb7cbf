"""
ctypes binding of ``libfcdiff_b200.so`` (C-ABI declared in ``include/fcdiff_b200.h``).

There is no CPU fallback: if the library is missing or a call fails, this module
raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C fcdiff_b200/csrc``.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfcdiff_b200.so")


class FcdTheta(ctypes.Structure):
    """``fcd_theta`` (fcdiff/model.py:31-38)."""
    _fields_ = [("pi", c_double), ("eta", c_double), ("epsilon", c_double),
                ("gamma", c_double * 3), ("mu", c_double * 3), ("sigma", c_double * 3)]


_P = c_void_p        # device pointers and streams travel as plain addresses
_D3 = POINTER(c_double)

# name -> (restype, argtypes); must list every symbol of include/fcdiff_b200.h
SIGNATURES = {
    "fcd_version": (c_int, []),
    "fcd_last_error": (c_char_p, []),
    "fcd_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "fcd_workspace_bytes": (c_int64, []),
    "fcd_download": (c_int, [_P, _P, c_int64, _P]),
    "fcd_launch_count": (c_int64, []),
    "fcd_launch_count_reset": (None, []),
    "fcd_nvtx_push": (None, [c_char_p]),
    "fcd_nvtx_pop": (None, []),
    "fcd_comm_window_bytes": (c_int64, []),
    "fcd_comm_handle_bytes": (c_int32, []),
    "fcd_comm_max_world": (c_int32, []),
    "fcd_comm_max_vals": (c_int32, []),
    "fcd_comm_window_create": (c_int, [POINTER(c_void_p)]),
    "fcd_comm_window_destroy": (c_int, [_P]),
    "fcd_comm_window_export": (c_int, [_P, _P]),
    "fcd_comm_window_open": (c_int, [_P, POINTER(c_void_p)]),
    "fcd_comm_window_close": (c_int, [_P]),
    "fcd_host_result_alloc": (c_int, [POINTER(c_void_p)]),
    "fcd_host_result_free": (c_int, [_P]),
    "fcd_allreduce_small": (c_int, [_P, c_int32, POINTER(c_void_p), c_int32, c_int32, c_uint64, _P, _P]),
    "fcd_allreduce_small_keep": (c_int, [_P, c_int32, c_int32, c_int32, POINTER(c_void_p), c_int32, c_int32, c_uint64,
                                         _P, _P]),
    "fcd_wait_result": (c_int, [_P, c_int32, c_uint64, _P, c_int32]),
    "fcd_pack_patients": (c_int, [_P, _P, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P]),
    "fcd_unpack_patients": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, _P, _P, _P]),
    "fcd_c_to_nm": (c_int, [c_int64, c_int64, _P, _P, _P]),
    "fcd_healthy_stats": (c_int, [_P, c_int64, c_int32, c_int64, _P, _P, _P, _P]),
    "fcd_row_logsums": (c_int, [_P, c_int64, c_int64, c_int32, c_int64, POINTER(FcdTheta), _P, _P]),
    "fcd_estep_qF_rowsums": (c_int, [_P, _P, _P, c_int32, _P, c_int64, _D3, POINTER(FcdTheta), _P, _P, _P]),
    "fcd_elm_rowsums": (c_int, [_P, _P, c_int64, _D3, _P, _P, _P]),
    "fcd_healthy_stats_cols": (c_int, [_P, c_int64, c_int64, _P, c_int32, _P, _P, _P, _P]),
    "fcd_gather_columns": (c_int, [_P, c_int64, c_int64, c_int32, c_int64, _P, c_int32, _P, c_int64, c_int64, _P]),
    "fcd_edge_table": (c_int, [c_int64, c_int64, _P, _P]),
    "fcd_resp_cache": (c_int, [_P, c_int64, c_int32, c_int64, POINTER(FcdTheta), _P, c_int64, _P, c_int32, _P]),
    "fcd_map_labels": (c_int, [_P, c_int64, c_int32, _P, _P]),
    "fcd_peak_states_F": (c_int, [_P, c_int64, _P, _P]),
    "fcd_peak_states_R": (c_int, [_P, c_int32, c_int32, c_int64, _P, _P]),
    "fcd_estep_qF": (c_int, [_P, _P, _P, c_int32, _P, c_int64, c_int64, c_int32, c_int64, _P, _P, c_int64, c_int32, _P,
                             POINTER(FcdTheta), _P, _P, _P]),
    "fcd_estep_qR": (c_int, [_P, c_int64, c_int32, c_int32, c_int32, c_int32, _D3, c_int32, _P, _P, _P]),
    "fcd_pstar_refresh_em": (c_int, [_P, c_int64, c_int64, c_int32, c_int32, c_int64, c_int64, _P, _P, _P, _P]),
    "fcd_region_weights_em": (c_int, [_P, c_int64, c_int64, c_int32, c_int32, c_int64, c_int64, _P, _P, _P, _P,
                                      POINTER(FcdTheta), _P, _P]),
    "fcd_mstep_stats": (c_int, [_P, c_int64, _P, c_int64, _P, _P, _P]),
    "fcd_elm_obj_grad": (c_int, [_P, c_int64, c_int64, c_int32, c_int64, _P, _P, _P, _P, c_int64, c_int32, _P,
                                 POINTER(FcdTheta), c_int32, _P, _P, _P]),
    "fcd_elm_const": (c_int, [_P, c_int64, c_int32, c_int64, _P, _P, _P, _P, c_int64, c_int32, _P, _P, _P, _P]),
    "fcd_bucket_blocks": (c_int64, [c_int64]),
    "fcd_plane_sum": (c_int, [_P, c_int64, c_int32, c_int64, _P, _P, _P]),
    "fcd_code_pitch": (c_int64, [c_int32]),
    "fcd_code_plane": (c_int, [_P, c_int64, c_int64, c_int32, c_int64, _P, _P, c_int64, _P, _P, _P, _P, c_int64, _P, _P,
                               _P, _P]),
    "fcd_code_records": (c_int, [_P, c_int64, _P, _P, c_int64, _P, _P, c_int64, c_int32, c_int64, _P, _P, _P, _P, c_int64,
                                 c_int32, _P, _P, _P, _P, _P, _P, _P, c_int64, _P, c_int64, _P, _P, _P]),
    "fcd_estep_qF_coded": (c_int, [_P, _P, _P, c_int32, _P, c_int64, c_int64, c_int32, c_int64, _P, c_int32, _P,
                                   _P, c_int64, _P, _P, _P, _P, _P, POINTER(FcdTheta), _P, c_double, c_double,
                                   _P, _P, _P]),
    "fcd_elm_coded": (c_int, [_P, _P, c_int64, _P, c_int64, _P, c_int64, POINTER(FcdTheta), c_int32, _P, _P, _P]),
    "fcd_solver_state_bytes": (c_int64, []),
    "fcd_solver_published_bytes": (c_int64, []),
    "fcd_host_mapped_alloc": (c_int, [c_int64, POINTER(c_void_p)]),
    "fcd_host_mapped_free": (c_int, [_P]),
    "fcd_solver_init": (c_int, [_P, c_double, c_double, _D3, _D3, c_double, c_int32, _P]),
    "fcd_elm_coded_solve": (c_int, [_P, _P, c_int64, _P, c_int64, _P, c_int64, c_double, c_double, _P, _P,
                                    POINTER(c_void_p), c_int32, c_int32, _P, c_uint64, c_int32, _P, _P]),
    "fcd_elm_tiered_solve": (c_int, [_P, c_int64, c_int64, c_int32, c_int64, _P, _P, _P, _P, c_int64, c_int32, _P,
                                     c_double, c_double, _P, _P, POINTER(c_void_p), c_int32, c_int32, _P, c_uint64,
                                     c_int32, _P, _P]),
    "fcd_solver_init_host": (c_int, [_P, c_double, c_double, _D3, _D3, c_double, c_int32]),
    "fcd_solver_step_host": (c_int, [_P, _D3]),
    "fcd_solver_moments": (c_int64, []),
    "fcd_solver_step_host_moments": (c_int, [_P, _D3, c_int32]),
    "fcd_solver_model_host": (c_int, [_D3, c_int32, c_double, c_double, _D3, _D3]),
    "fcd_solver_wait": (c_int, [_P, c_uint64, _P, c_int32]),
    "fcd_energy_terms": (c_int, [_P, _P, _P, c_int32, _P, _P, c_int64, _P, _P, c_int32, c_int32,
                                 POINTER(FcdTheta), c_double, _P, _P, _P, _P]),
    "fcd_patient_terms_ws_bytes": (c_int64, [c_int64, c_int32]),
    "fcd_patient_terms": (c_int, [_P, c_int64, _P, c_int64, c_int32, c_int64, _P, _P, _P, _P, c_int32, POINTER(FcdTheta),
                                  _P, _P, _P]),
    "fcd_qR_change": (c_int, [_P, _P, c_int32, c_int32, _P, _P, _P]),
    "fcd_connection_ws_bytes": (c_int64, [c_int64, c_int32]),
    "fcd_connection_posteriors": (c_int, [_P, c_int64, c_int64, c_int32, c_int64, _P, _P, _P, c_int32,
                                          POINTER(FcdTheta), _P, _P, _P, _P, _P, _P]),
    "fcd_control_terms_ws_bytes": (c_int64, [c_int64, c_int32]),
    "fcd_control_terms": (c_int, [_P, c_int64, c_int32, c_int64, _P, POINTER(FcdTheta), _P, _P, c_int32, _P]),
    "fcd_maxt_ws_bytes": (c_int64, [c_int64, c_int64]),
    "fcd_maxt_counts": (c_int, [_P, c_int64, c_int64, c_int64, _P, c_int64, c_int64, _P, _P, _P, _P]),
    "fcd_state_moments": (c_int, [_P, _P, c_int32, _P, _P, c_int64, c_int64, c_int32, c_int64, _P, _P, c_int32, _P,
                                  POINTER(FcdTheta), _P, _P, _P]),
    "fcd_materialize_lps": (c_int, [_P, _P, c_int64, c_int32, c_int32, POINTER(FcdTheta), _P, _P, _P, c_int32, _P]),
    "fcd_eval_M": (c_int, [_P, c_int64, c_double, c_double, c_int32, c_int32, _P, _P]),
    "fcd_lqF_from_arrays": (c_int, [_P, _P, c_int64, c_int32, c_int32, _P, c_int32, _D3, _P, _P]),
    "fcd_region_weights_from_lM": (c_int, [_P, c_int64, c_int32, _P, _P, _P]),
    "fcd_ElM_from_arrays": (c_int, [_P, _P, _P, c_int64, c_int32, c_int32, _P, _P, _P]),
    "fcd_dE_from_arrays": (c_int, [_P, _P, _P, _P, c_int64, c_int32, c_int32, c_double, c_double, _P, _P, _P]),
    "fcd_dlM": (c_int, [_P, _P, c_int64, c_double, c_int32, _P, _P]),
    "fcd_pair_weights": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, _P, _P]),
    "fcd_dot_broadcast": (c_int, [_P, c_int64, c_int64, _P, c_int64, c_int64, _P, _P, _P]),
    "fcd_sample_R": (c_int, [c_uint64, c_uint64, c_int32, c_int32, c_double, _P, _P]),
    "fcd_sample_T": (c_int, [c_uint64, c_uint64, _P, c_int32, c_int32, c_double, c_int64, c_int64, _P, _P]),
    "fcd_sample_F": (c_int, [c_uint64, c_uint64, c_int64, c_int64, _D3, _P, _P]),
    "fcd_sample_F_tilde": (c_int, [c_uint64, c_uint64, _P, _P, c_int64, c_int64, c_int32, c_double, _P, _P]),
    "fcd_sample_B": (c_int, [c_uint64, c_uint64, _P, c_int64, c_int64, c_int32, _D3, _D3, _P, _P]),
    "fcd_sample_B_tilde": (c_int, [c_uint64, c_uint64, _P, c_int64, c_int64, c_int32, _D3, _D3, _P, _P]),
    "fcd_corr_workspace_bytes": (c_int64, [c_int32, c_int32, c_int32]),
    "fcd_corr_fisherz": (c_int, [_P, c_int32, c_int32, c_int32, _P, c_int64, c_int32, c_int32, _P, _P]),
    "fcd_corr_mark_missing": (c_int, [_P, c_int32, c_int32, c_int32, _P, c_int64, c_int32, _P]),
    "fcd_corr_clean_workspace_bytes": (c_int64, [c_int32, c_int32, c_int32, c_int32]),
    "fcd_corr_fisherz_clean": (c_int, [_P, c_int32, c_int32, c_int32, _P, _P, c_int32, _P, c_int64, c_int32, c_int32,
                                       c_int32, _P, _P, _P]),
    "fcd_corr_partial_workspace_bytes": (c_int64, [c_int32, c_int32, c_int32, c_int32]),
    "fcd_corr_partial": (c_int, [_P, c_int32, c_int32, c_int32, _P, _P, c_int32, c_double, _P, c_int64, c_int32,
                                 c_int32, c_int32, _P, _P, _P, _P, _P]),
}

class SolverState(ctypes.Structure):
    """``fcd_solver_state`` (include/fcdiff_b200.h)."""
    _fields_ = [("x", c_double * 2), ("xprev", c_double * 2), ("fprev", c_double), ("f", c_double),
                ("g", c_double * 2), ("lo", c_double * 2), ("hi", c_double * 2), ("tol", c_double),
                ("step", c_double), ("have_prev", c_int32), ("nfev", c_int32), ("nback", c_int32),
                ("done", c_int32), ("max_evals", c_int32), ("pad_", c_int32)]


_lib = None


class FcdError(RuntimeError):
    pass


def load():
    """Loads the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise FcdError(
            "fcdiff_b200: %s not found -- the CUDA library must be built first "
            "(make -C fcdiff_b200/csrc); there is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.fcd_version() < 123:
        raise FcdError("fcdiff_b200: stale libfcdiff_b200.so (version %d)" % lib.fcd_version())
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().fcd_last_error()
        raise FcdError("%s failed (%d): %s" % (what or "libfcdiff_b200 call", rc,
                                               msg.decode() if msg else "?"))


def make_theta(pi, eta, epsilon, gamma, mu, sigma):
    th = FcdTheta()
    th.pi = float(pi)
    th.eta = float(eta)
    th.epsilon = float(epsilon)
    for k in range(3):
        th.gamma[k] = float(gamma[k])
        th.mu[k] = float(mu[k])
        th.sigma[k] = float(sigma[k])
    return th


def d3(values):
    """Host array of doubles for the ``*_host`` arguments."""
    return (c_double * len(values))(*[float(v) for v in values])
