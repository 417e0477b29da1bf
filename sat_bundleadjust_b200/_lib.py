"""
ctypes binding of libsba_b200.so (the C ABI declared in include/sba_b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is visible when a
compute entry point is called, an exception is raised.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SBA_LIB_PATH") or os.path.join(HERE, "libsba_b200.so")     # override: A/B runs of two builds

MODEL_IDS = {"affine": 0, "perspective": 1, "rpc": 2}
LOSS_IDS = {"linear": 0, "huber": 1, "soft_l1": 2, "cauchy": 3, "arctan": 4}

c_double_p = ctypes.POINTER(ctypes.c_double)
c_float_p = ctypes.POINTER(ctypes.c_float)
c_int64_p = ctypes.POINTER(ctypes.c_int64)


class SbaError(RuntimeError):
    pass


class ProblemDesc(ctypes.Structure):
    _fields_ = [("cam_model", ctypes.c_int32), ("n_cam", ctypes.c_int32), ("n_pts", ctypes.c_int32),
                ("n_obs", ctypes.c_int64), ("n_params", ctypes.c_int32), ("n_cam_params", ctypes.c_int32),
                ("n_cam_fix", ctypes.c_int32), ("n_pts_fix", ctypes.c_int32),
                ("cam_ind", c_int64_p), ("pts_ind", c_int64_p), ("pts2d", c_double_p), ("pts2d_w", c_double_p),
                ("cam_params", c_double_p), ("rpc_coefs", c_double_p), ("rpc_float32", ctypes.c_int32),
                ("rank", ctypes.c_int32), ("world_size", ctypes.c_int32), ("n_common", ctypes.c_int32),
                ("engine", ctypes.c_int32), ("solver", ctypes.c_int32)]


class SolveOpts(ctypes.Structure):
    _fields_ = [("loss", ctypes.c_int32), ("f_scale", ctypes.c_double), ("ftol", ctypes.c_double),
                ("xtol", ctypes.c_double), ("gtol", ctypes.c_double), ("max_nfev", ctypes.c_int32),
                ("verbose", ctypes.c_int32), ("max_iterations", ctypes.c_int32), ("timed_from", ctypes.c_int32),
                ("l2_flush_bytes", ctypes.c_int64), ("no_phase_timing", ctypes.c_int32)]


class SolveInfo(ctypes.Structure):
    _fields_ = [("status", ctypes.c_int32), ("nfev", ctypes.c_int32), ("njev", ctypes.c_int32),
                ("iterations", ctypes.c_int32), ("cost_init", ctypes.c_double), ("cost", ctypes.c_double),
                ("optimality", ctypes.c_double), ("solve_ms", ctypes.c_double), ("chol_retries", ctypes.c_int32),
                ("gpu_launches", ctypes.c_int32), ("timed_iterations", ctypes.c_int32), ("iter_ms", ctypes.c_double),
                ("phase_ms", ctypes.c_double * 8), ("explicit_subspace_passes", ctypes.c_int32),
                ("pcg_solves", ctypes.c_int32), ("pcg_iterations", ctypes.c_int32)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["phase_ms"] = dict(zip(PHASES, list(self.phase_ms)))
        return d


PHASES = ["assemble", "scale_jvp", "point_prep", "schur", "cholesky", "backsub", "subspace", "step_eval"]


ALLREDUCE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64)

# every symbol include/sba_b200.h declares
EXPORTED_SYMBOLS = [
    "sba_last_error", "sba_version", "sba_problem_create", "sba_problem_destroy", "sba_release_cached_memory", "sba_problem_set_allreduce",
    "sba_problem_num_vars", "sba_problem_engine", "sba_problem_solver", "sba_residuals", "sba_jacobian_blocks", "sba_normal_blocks", "sba_reduced_system", "sba_solve", "sba_solve_errors",
    "sba_solve_device", "sba_assemble_device", "sba_tr2d", "sba_rpc_projection", "sba_rpc_projection_ecef",
    "sba_rpc_localization", "sba_rpc_throughput", "stereo_corresp_to_lonlatalt", "sba_stereo_corresp_to_lonlatalt", "sba_cholesky_solve",
    "sba_cholesky_solve_timed", "sba_outlier_elbow", "sba_outlier_mark",
    "sba_rpcfit_weighted_lsq", "sba_comm_export", "sba_comm_import", "sba_comm_try_reuse", "sba_solve_errors_device",
    "sba_init_pts3d", "sba_linear_triangulation", "sba_rpc_projection_batch", "sba_rpc_localization_batch",
    "sba_covariance", "sba_covariance_phase_ms",
]

_lib = None


def load():
    """Load libsba_b200.so (built in-tree by __graft_entry__.build()); raises if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SbaError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp = ctypes.c_void_p
    lib.sba_last_error.restype = ctypes.c_char_p
    lib.sba_problem_create.argtypes = [ctypes.POINTER(vp), ctypes.POINTER(ProblemDesc), vp]
    lib.sba_problem_destroy.argtypes = [vp]
    lib.sba_problem_set_allreduce.argtypes = [vp, ALLREDUCE_FN, vp]
    lib.sba_comm_export.argtypes = [vp, ctypes.c_char_p]
    lib.sba_comm_import.argtypes = [vp, ctypes.c_char_p]
    lib.sba_comm_try_reuse.argtypes = [vp]
    lib.sba_solve_errors_device.argtypes = [vp, vp, ctypes.POINTER(SolveOpts), vp, vp, vp, ctypes.POINTER(SolveInfo)]
    lib.sba_problem_num_vars.argtypes = [vp]
    lib.sba_problem_num_vars.restype = ctypes.c_int64
    lib.sba_problem_engine.argtypes = [vp]
    lib.sba_problem_solver.argtypes = [vp]
    lib.sba_residuals.argtypes = [vp, c_double_p, c_double_p, ctypes.c_int32, ctypes.c_double, c_double_p]
    lib.sba_jacobian_blocks.argtypes = [vp, c_double_p, c_double_p, c_double_p]
    lib.sba_normal_blocks.argtypes = [vp, c_double_p, ctypes.c_int32, ctypes.c_double, c_double_p, c_double_p, c_double_p]
    lib.sba_reduced_system.argtypes = [vp, c_double_p, ctypes.c_int32, ctypes.c_double, ctypes.c_double, c_double_p, c_double_p]
    lib.sba_covariance.argtypes = [vp, c_double_p, ctypes.c_int32, ctypes.c_double, ctypes.c_double, c_double_p, c_double_p,
                                   c_double_p, c_double_p]
    lib.sba_covariance_phase_ms.argtypes = [vp, c_double_p]
    lib.sba_solve.argtypes = [vp, c_double_p, ctypes.POINTER(SolveOpts), c_double_p, c_double_p, ctypes.POINTER(SolveInfo)]
    lib.sba_solve_device.argtypes = [vp, vp, ctypes.POINTER(SolveOpts), vp, vp, ctypes.POINTER(SolveInfo)]
    lib.sba_assemble_device.argtypes = [vp, vp, ctypes.c_int32, ctypes.c_double, c_float_p]
    lib.sba_tr2d.argtypes = [c_double_p, c_double_p, ctypes.c_double, c_double_p]
    lib.sba_rpc_projection.argtypes = [c_double_p] * 4 + [ctypes.c_int64, c_double_p, c_double_p]
    lib.sba_rpc_projection_ecef.argtypes = [c_double_p, c_double_p, ctypes.c_int64, c_double_p]
    lib.sba_rpc_localization.argtypes = [c_double_p] * 4 + [ctypes.c_int64, ctypes.c_double, c_double_p, c_double_p]
    lib.sba_rpc_projection_batch.argtypes = [c_double_p, ctypes.c_int32, c_double_p, c_double_p, c_double_p, ctypes.c_int64, ctypes.c_int32,
                                             c_double_p, c_double_p]
    lib.sba_rpc_localization_batch.argtypes = [c_double_p, ctypes.c_int32, c_double_p, c_double_p, c_double_p, ctypes.c_int64, ctypes.c_int32,
                                               ctypes.c_double, c_double_p, c_double_p]
    lib.sba_rpc_throughput.argtypes = [ctypes.c_int32, c_double_p, ctypes.c_int32, c_double_p, c_double_p, c_double_p, c_double_p,
                                       ctypes.c_int64, ctypes.c_double, ctypes.c_int32, c_double_p, c_double_p]
    lib.sba_stereo_corresp_to_lonlatalt.argtypes = [c_double_p, c_float_p, c_float_p, c_float_p, ctypes.c_int64, vp, vp]
    lib.stereo_corresp_to_lonlatalt.argtypes = [c_double_p, c_float_p, c_float_p, c_float_p, ctypes.c_int, vp, vp]
    lib.stereo_corresp_to_lonlatalt.restype = None
    lib.sba_cholesky_solve.argtypes = [c_double_p, c_double_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]
    lib.sba_rpcfit_weighted_lsq.argtypes = [c_double_p, c_double_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_double,
                                            ctypes.c_double, ctypes.c_int32, c_double_p, ctypes.POINTER(ctypes.c_int32),
                                            c_double_p]
    lib.sba_init_pts3d.argtypes = [ctypes.c_int32, c_double_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32),
                                   c_double_p, ctypes.c_int64, ctypes.POINTER(ctypes.c_int32), ctypes.c_int32, c_float_p]
    lib.sba_linear_triangulation.argtypes = [c_double_p, c_double_p, c_double_p, c_double_p, ctypes.c_int64, c_double_p]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise SbaError("libsba_b200: %s (code %d)" % (load().sba_last_error().decode(), rc))


def dptr(a):
    return a.ctypes.data_as(c_double_p)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)
