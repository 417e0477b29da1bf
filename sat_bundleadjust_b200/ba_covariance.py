"""
Posterior covariance of the adjusted cameras and 3-D points, computed on the device.

    cov_cam, cov_pts, sigma2, min_pivot_ratio = compute_covariance(p, vars_ba, loss="soft_l1")

At x = vars_ba, with J the Jacobian of the weighted residuals over the free variables (rescaled for a robust loss exactly
like the solver does), H = J^T J = [[U, W], [W^T, V]] and S = U - W V^-1 W^T:

  * cov_cam = sigma2 S^-1, shape (n_cam * n_params)^2 in the params_opt camera layout; rows and columns of the frozen
    cameras (the first n_cam_fix) are 0;
  * cov_pts[t] = sigma2 (V_t^-1 + V_t^-1 W_t^T S^-1 W_t V_t^-1), shape (n_pts, 3, 3); frozen points are 0;
  * sigma2: given (> 0; a weight-1 observation then has pixel standard deviation sqrt(sigma2), like curve_fit's
    absolute_sigma=True), else estimated as 2 cost(x) / (2 K - n_free) (scipy curve_fit's convention) and returned;
  * min_pivot_ratio: the smallest L_kk^2 / U_kk of the Cholesky factor S = L L^T over the free camera slots.  S is
    rejected (SbaError) as rank deficient when a ratio is <= 1e-12: the gauge is not fixed (e.g. perspective R+T with
    nothing frozen has a 7-dimensional similarity null space).  The test catches round-off pivots; it does not certify full
    rank: in ill-conditioned satellite geometry a single free direction (the scale left by ONE frozen perspective camera)
    can pass it.  Fix the gauge with at least two frozen cameras, or with frozen points.

Not available: multi-GPU problems, the matrix-free PCG path (no dense S), COMMON_K, camera-point cross-covariance.
"""
import numpy as np

from .solver import DeviceProblem, n_common_params


def degrees_of_freedom(p):
    """2 K - n_free, n_free = (n_cam - n_cam_fix) n_params + 3 (n_pts - n_pts_fix)."""
    n_free = (int(p.n_cam) - int(p.n_cam_fix)) * int(p.n_params) + 3 * (int(p.n_pts) - int(p.n_pts_fix))
    return 2 * int(np.asarray(p.pts_ind).size) - n_free


def check_covariance_supported(p, sigma2=None):
    """The checks that need no device: COMMON_K -> NotImplementedError, no degrees of freedom to estimate sigma2 -> ValueError."""
    if n_common_params(p):
        raise NotImplementedError("posterior covariance is not available with COMMON_K (shared calibration)")
    if not (sigma2 is not None and sigma2 > 0) and degrees_of_freedom(p) <= 0:
        raise ValueError("no degrees of freedom left (2 K - n_free = %d): sigma^2 cannot be estimated" % degrees_of_freedom(p))


def compute_covariance(p, vars_ba, loss="linear", f_scale=1.0, sigma2=None):
    """(cov_cam, cov_pts (N,3,3), sigma2, min_pivot_ratio) at vars_ba; see the module docstring."""
    check_covariance_supported(p, sigma2)
    with DeviceProblem(p) as prob:
        return prob.covariance(vars_ba, loss=loss, f_scale=f_scale, sigma2=sigma2)
