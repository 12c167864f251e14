"""ctypes binding of ``libdgsqp_b200.so`` (C ABI declared in ``include/dgsqp_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no CPU
fallback: if the shared object is missing or no CUDA device is usable the calls raise.
"""
import ctypes as C
import os
import pathlib

MAX_AGENTS = 4
MAX_TRACK_SEGS = 8

NDIAG = 8   # DGSQP_NDIAG
PHASES = ["lin_full", "adj_full", "hessian", "pd_tridiag", "pd_eig", "cholesky", "tri_inverse", "active_set", "lsqr",
          "lin_grad", "adj_grad", "merit", "other",
          # sub-phases, non-zero only in the profiling build (-DDG_FINE_PHASES, scripts/build_prof.sh)
          "pd_sym", "pd_eigval", "pd_invit", "pd_back", "gi_slack", "gi_dz", "gi_step", "gi_add", "gi_drop", "qp_x0", "qp_warm",
          "ws_d", "ws_qr", "ws_apply", "ws_mult"]

STATUS_MSG = {0: "conv_abs_tol", 1: "conv_rel_tol", 2: "max_it", 3: "diverged", 4: "qp_fail", 5: "time_limit"}


class RacingGameStruct(C.Structure):
    _fields_ = [("M", C.c_int32), ("N", C.c_int32), ("dt", C.c_double),
                ("L_f", C.c_double), ("L_r", C.c_double),
                ("c_dr", C.c_double), ("c_da", C.c_double), ("c_s", C.c_double), ("mass", C.c_double),
                ("input_weight", C.c_double * 2), ("rate_weight", C.c_double * 2), ("comp_weights", C.c_double * 2),
                ("u_ub", C.c_double * 2), ("u_lb", C.c_double * 2),
                ("rate_ub", C.c_double * 2), ("rate_lb", C.c_double * 2),
                ("half_width", C.c_double), ("obs_r", C.c_double * MAX_AGENTS),
                ("track_nseg", C.c_int32),
                ("track_seg_len", C.c_double * MAX_TRACK_SEGS), ("track_seg_curv", C.c_double * MAX_TRACK_SEGS)]


class LaneRowStruct(C.Structure):
    _fields_ = [("brk", C.c_double), ("n_lo", C.c_double * 2), ("n_hi", C.c_double * 2), ("pt", C.c_double * 2)]


class MergeGameStruct(C.Structure):
    """dgsqp_merge_game (include/dgsqp_b200.h)."""
    _fields_ = [("M", C.c_int32), ("N", C.c_int32), ("dt", C.c_double), ("mass", C.c_double),
                ("input_weight", C.c_double * 2), ("state_weight", C.c_double * 4), ("term_scale", C.c_double),
                ("goal", (C.c_double * 4) * MAX_AGENTS),
                ("u_ub", C.c_double * 2), ("u_lb", C.c_double * 2), ("v_ub", C.c_double), ("v_lb", C.c_double),
                ("obs_r", C.c_double * MAX_AGENTS), ("lane_r", C.c_double),
                ("lane", (LaneRowStruct * 2) * MAX_AGENTS)]


class ParamsStruct(C.Structure):
    _fields_ = [("reg", C.c_double), ("p_tol", C.c_double), ("d_tol", C.c_double),
                ("beta", C.c_double), ("tau", C.c_double),
                ("line_search_iters", C.c_int32), ("sqp_iters", C.c_int32), ("nonmono_ls", C.c_int32),
                ("merit_function", C.c_int32), ("conv_approx", C.c_int32),
                ("mu_vio_thresh", C.c_double), ("time_limit", C.c_double), ("qp_warm_start", C.c_int32),
                ("iter_log", C.c_int32)]


class ParamsV2Struct(C.Structure):
    """dgsqp_v2_params (include/dgsqp_b200.h) <- DGSQPV2Params (DGSQP/solvers/solver_types.py:130-174)."""
    _fields_ = [("reg", C.c_double), ("reg_decay", C.c_double), ("p_tol", C.c_double), ("d_tol", C.c_double),
                ("beta", C.c_double), ("tau", C.c_double),
                ("line_search_iters", C.c_int32), ("sqp_iters", C.c_int32),
                ("nms", C.c_int32), ("nms_frequency", C.c_int32), ("nms_memory_size", C.c_int32),
                ("merit_function", C.c_int32), ("has_merit_parameter", C.c_int32), ("merit_parameter", C.c_double),
                ("merit_decrease", C.c_double), ("merit_decrease_condition", C.c_int32), ("delta_decay", C.c_double),
                ("mu_vio_thresh", C.c_double), ("time_limit", C.c_double), ("qp_warm_start", C.c_int32),
                ("iter_log", C.c_int32)]


class Pcg64Struct(C.Structure):
    """dgsqp_pcg64 (include/dgsqp_b200.h): the state of numpy.random.PCG64."""
    _fields_ = [("state_hi", C.c_uint64), ("state_lo", C.c_uint64), ("inc_hi", C.c_uint64), ("inc_lo", C.c_uint64)]


SAMPLE_HEAD_TO_HEAD, SAMPLE_AGENTS = 0, 1

EXPORTS = ["dgsqp_create", "dgsqp_create_v2", "dgsqp_create_merge", "dgsqp_create_merge_v2", "dgsqp_destroy", "dgsqp_dims", "dgsqp_solve_batch", "dgsqp_solve_batch_up", "dgsqp_solve_batch_async",
           "dgsqp_batch_stats", "dgsqp_last_stats", "dgsqp_pid_rollout", "dgsqp_sample_racing", "dgsqp_sample_merge", "dgsqp_last_diag", "dgsqp_iter_log_capacity", "dgsqp_last_iter_data", "dgsqp_phase_count", "dgsqp_last_phase_cycles", "dgsqp_measure_fp64_peak", "dgsqp_kernel_launches", "dgsqp_configure", "dgsqp_memory_plan", "dgsqp_set_smem_limit", "dgsqp_last_error", "dgsqp_version"]

LIB_PATH = pathlib.Path(__file__).resolve().parent / "libdgsqp_b200.so"
_lib = None


class DgsqpLibraryError(RuntimeError):
    pass


def load():
    """Load the CUDA library.  Raises DgsqpLibraryError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = pathlib.Path(os.environ.get("DGSQP_B200_LIB", LIB_PATH))
    if not path.exists():
        raise DgsqpLibraryError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  dgsqp_b200 has no CPU fallback.")
    lib = C.CDLL(str(path))
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_void_p
    lib.dgsqp_create.argtypes = [C.POINTER(RacingGameStruct), C.POINTER(ParamsStruct), C.c_int, C.POINTER(vp)]
    lib.dgsqp_create.restype = C.c_int
    lib.dgsqp_create_v2.argtypes = [C.POINTER(RacingGameStruct), C.POINTER(ParamsV2Struct), C.c_int, C.POINTER(vp)]
    lib.dgsqp_create_v2.restype = C.c_int
    lib.dgsqp_create_merge.argtypes = [C.POINTER(MergeGameStruct), C.POINTER(ParamsStruct), C.c_int, C.POINTER(vp)]
    lib.dgsqp_create_merge.restype = C.c_int
    lib.dgsqp_create_merge_v2.argtypes = [C.POINTER(MergeGameStruct), C.POINTER(ParamsV2Struct), C.c_int, C.POINTER(vp)]
    lib.dgsqp_create_merge_v2.restype = C.c_int
    lib.dgsqp_destroy.argtypes = [vp]
    lib.dgsqp_destroy.restype = C.c_int
    lib.dgsqp_dims.argtypes = [vp, ip]
    lib.dgsqp_dims.restype = C.c_int
    batch_args = [vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.dgsqp_solve_batch.argtypes = batch_args + [C.c_int32, vp]
    lib.dgsqp_solve_batch.restype = C.c_int
    lib.dgsqp_solve_batch_up.argtypes = [vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int32, vp]
    lib.dgsqp_solve_batch_up.restype = C.c_int
    lib.dgsqp_solve_batch_async.argtypes = batch_args + [vp]
    lib.dgsqp_solve_batch_async.restype = C.c_int
    lib.dgsqp_pid_rollout.argtypes = [C.POINTER(RacingGameStruct), vp, C.c_int, C.c_int32, vp, vp, vp, vp, vp, vp, C.c_int32, vp]
    lib.dgsqp_pid_rollout.restype = C.c_int
    lib.dgsqp_sample_racing.argtypes = [C.POINTER(RacingGameStruct), vp, C.c_int32, C.POINTER(Pcg64Struct), C.c_int, C.c_int32,
                                        C.c_int64, vp, vp, vp, C.POINTER(C.c_int32), C.POINTER(C.c_int64), vp]
    lib.dgsqp_sample_racing.restype = C.c_int
    lib.dgsqp_sample_merge.argtypes = [C.POINTER(MergeGameStruct), C.POINTER(Pcg64Struct), C.c_int, C.c_int32, C.c_int64, vp, vp,
                                       C.POINTER(C.c_int32), C.POINTER(C.c_int64), vp]
    lib.dgsqp_sample_merge.restype = C.c_int
    lib.dgsqp_batch_stats.argtypes = [C.c_int, C.c_int32, vp, vp, vp, vp, vp, vp]
    lib.dgsqp_batch_stats.restype = C.c_int
    lib.dgsqp_last_stats.argtypes = [vp, vp]
    lib.dgsqp_last_stats.restype = C.c_int
    lib.dgsqp_last_diag.argtypes = [vp, C.c_int32, vp]
    lib.dgsqp_last_diag.restype = C.c_int
    lib.dgsqp_iter_log_capacity.argtypes = [vp]
    lib.dgsqp_iter_log_capacity.restype = C.c_int
    lib.dgsqp_last_iter_data.argtypes = [vp, C.c_int32, vp]
    lib.dgsqp_last_iter_data.restype = C.c_int
    lib.dgsqp_phase_count.argtypes = []
    lib.dgsqp_phase_count.restype = C.c_int
    lib.dgsqp_last_phase_cycles.argtypes = [vp, C.c_int32, vp]
    lib.dgsqp_last_phase_cycles.restype = C.c_int
    lib.dgsqp_measure_fp64_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
    lib.dgsqp_measure_fp64_peak.restype = C.c_int
    lib.dgsqp_kernel_launches.argtypes = []
    lib.dgsqp_kernel_launches.restype = C.c_int64
    lib.dgsqp_configure.argtypes = [vp, C.c_int32, C.c_int32]
    lib.dgsqp_configure.restype = C.c_int
    lib.dgsqp_memory_plan.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.dgsqp_memory_plan.restype = C.c_int
    lib.dgsqp_set_smem_limit.argtypes = [vp, C.c_int64]
    lib.dgsqp_set_smem_limit.restype = C.c_int
    lib.dgsqp_last_error.argtypes = []
    lib.dgsqp_last_error.restype = C.c_char_p
    lib.dgsqp_version.argtypes = []
    lib.dgsqp_version.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().dgsqp_last_error().decode()
        raise DgsqpLibraryError(f"dgsqp_b200 error {rc}: {msg}")
