"""
Bundle-adjustment numerical core -- drop-in mirror of the reference's bundle_adjust/ba_core.py
(lines 157-349) on top of the B200 solver.

Same names, arguments, return values and defaults as the reference:
    fun(v, p)                                   ba_core.py:157-183
    build_jacobian_sparsity(p)                  ba_core.py:186-219
    init_optimization_config(config)            ba_core.py:222-241
    run_ba_optimization(p, ls_params, verbose, plots)      ba_core.py:244-332
    compute_reprojection_error(residuals, pts2d_w)         ba_core.py:335-349
    compute_mean_reprojection_error_per_track(...)         ba_core.py:352-370
`p` is an unmodified BundleAdjustmentParameters (ours or the reference's).  What differs is how the
work is done: residuals, the analytic Jacobian, robust weighting, block assembly, the Schur complement,
the dense factorisation and the trust-region steps all run in hand-written sm_100a kernels behind
libsba_b200.so.  There is no scipy call and no CPU fallback on this path.
"""
import numpy as np

from ._lib import SbaError
from .solver import DeviceProblem, initial_vars


def flush_print(*a):
    print(*a, flush=True)


def fun(v, p):
    """
    Weighted reprojection residuals (x0', y0', x1', y1', ...) of all K observations, shape (2K,).
    Like the reference this writes the frozen cameras' parameters into `v` in place.
    """
    if p.n_cam_fix > 0:
        c = p.n_params
        v[: p.n_cam * c].reshape(p.n_cam, c)[: p.n_cam_fix] = p.cam_params[: p.n_cam_fix, :c]
    with DeviceProblem(p) as prob:
        r, _ = prob.residuals(v)
    return r


def build_jacobian_sparsity(p):
    """
    0/1 sparsity of the (2K x n) Jacobian, identical (type, indices and shape) to the reference's LIL matrix
    (ba_core.py:186-219), with the row lists produced vectorised instead of by lil_matrix fancy writes.
    The B200 solver does not consume it -- its block layout is the same index formula evaluated on the
    device -- it is provided because callers and tests of the reference expect it.  The LIL format itself
    (one Python list of Python ints per row) bounds the speed: ~1.5 s at 5e5 observations.
    """
    from scipy.sparse import lil_matrix

    c = p.n_params
    nK = 3 if p.cam_model == "affine" else 5
    common = "K" in p.cam_params_to_optimize and "COMMON_K" in p.cam_params_to_optimize
    if common:
        c -= nK
    off = nK if common else 0
    K = p.pts_ind.size
    n = off + p.n_cam * c + p.n_pts * 3
    parts = []
    if common:
        parts.append(np.broadcast_to(np.arange(off), (K, off)))
    parts.append(off + np.asarray(p.cam_ind)[:, None] * c + np.arange(c))
    parts.append(off + p.n_cam * c + np.asarray(p.pts_ind)[:, None] * 3 + np.arange(3))
    cols = np.repeat(np.hstack(parts), 2, axis=0)          # ascending inside a row: shared K, camera, point
    A = lil_matrix((2 * K, n), dtype=int)
    A.rows = np.fromiter(cols.tolist(), dtype=object, count=2 * K)
    A.data = np.fromiter(np.ones(cols.shape, dtype=int).tolist(), dtype=object, count=2 * K)
    return A


def init_optimization_config(config=None):
    """Solver knobs with the reference's defaults (ba_core.py:233-234)."""
    out = {"loss": "linear", "ftol": 1e-4, "xtol": 1e-10, "f_scale": 1.0, "max_iter": 300, "verbose": 1}
    if config is not None:
        out.update({k: config[k] for k in out if k in config})
    return out


def compute_reprojection_error(residuals, pts2d_w=None):
    """Per-observation L2 norm of the un-weighted residual pair."""
    q = residuals.reshape(-1, 2)
    if pts2d_w is not None:
        q = q / np.asarray(pts2d_w)[:, np.newaxis]
    # same values as np.linalg.norm(|r / w|.reshape(n, 2), axis=1) (ba_core.py:236-238), a third of the host time
    return np.sqrt(q[:, 0] * q[:, 0] + q[:, 1] * q[:, 1])


def compute_mean_reprojection_error_per_track(err, pts_ind, cam_ind):
    """Mean reprojection error of each track (float32, like the reference)."""
    n_pts = int(np.max(pts_ind)) + 1
    s = np.bincount(pts_ind, weights=err, minlength=n_pts)
    cnt = np.bincount(pts_ind, minlength=n_pts)
    with np.errstate(invalid="ignore", divide="ignore"):
        return (s / cnt).astype(np.float32)


def run_ba_optimization(p, ls_params=None, verbose=False, plots=True, return_info=False, cam_prior=None):
    """
    Solve the bundle adjustment problem on the GPU.

    Returns (vars_init, vars_ba, err_init, err_ba, iterations) exactly like the reference
    (`iterations` = number of residual evaluations, i.e. scipy's nfev).  `plots` is accepted for
    signature compatibility; figures are out of scope.  `return_info=True` appends the solver's info dict.
    `cam_prior` (a ba_priors.CameraPrior) adds a Gaussian prior on the camera variables to the objective; the info's
    cost_init / cost then include its term, err_init / err_ba stay the pixel errors of the observations.
    """
    cfg = init_optimization_config(ls_params)
    if verbose:
        print("\nRunning bundle adjustment...")
        for k, v in cfg.items():
            print("    {}: {}".format(k, v))
    import time
    vars_init = initial_vars(p)
    t0 = time.perf_counter()
    with DeviceProblem(p, cam_prior=cam_prior) as prob:
        t1 = time.perf_counter()
        try:
            vars_ba, err_init, err_ba, info = prob.solve_with_errors(
                vars_init, loss=cfg["loss"], f_scale=cfg["f_scale"], ftol=cfg["ftol"], xtol=cfg["xtol"],
                max_nfev=cfg["max_iter"], verbose=2 if cfg["verbose"] >= 2 else 0)
        except SbaError as exc:
            if "not finite" in str(exc):      # scipy's message and exception type (least_squares.py:945-946)
                raise ValueError("Residuals are not finite in the initial point.") from exc
            raise
        t3 = time.perf_counter()
    info["wall_s"] = {"create": t1 - t0, "fun": 0.0, "solve": t3 - t1, "destroy": time.perf_counter() - t3}
    if verbose:
        flush_print("Shape of Jacobian sparsity: {}x{}".format(2 * p.pts_ind.size, vars_init.size))
        flush_print("Optimization took {:.4f} seconds on the device ({} function evaluations)\n".format(
            info["solve_ms"] * 1e-3, info["nfev"]))
    if verbose:
        flush_print("Reprojection error before BA (mean / median): {:.2f} / {:.2f}".format(np.mean(err_init), np.median(err_init)))
        flush_print("Reprojection error after  BA (mean / median): {:.2f} / {:.2f}\n".format(np.mean(err_ba), np.median(err_ba)))
        for cam_idx in range(int(p.C.shape[0] / 2)):
            sel = p.cam_ind == cam_idx
            n_obs = np.sum(1 * ~np.isnan(p.C[2 * cam_idx, :]))
            flush_print("    - cam {:3} - {:5} obs - (mean before / mean after): {:.2f} / {:.2f}".format(
                cam_idx, n_obs, np.mean(err_init[sel]), np.mean(err_ba[sel])))
        print("\n")
    out = (vars_init, vars_ba, err_init, err_ba, info["nfev"])
    return out + (info,) if return_info else out
