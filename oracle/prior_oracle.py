"""
Checker only: the bundle-adjustment objective with a Gaussian prior on the camera variables, restated on top of
ba_oracle for scipy.

    cost(x) = 0.5 f_s^2 sum_k rho(|r_k|^2 / f_s^2) + 0.5 sum_{j free} (x_j - mu_j)^T L_j (x_j - mu_j)

is scipy's least_squares on the augmented residual [r ; C_j (x_j - mu_j)] (L_j = C_j^T C_j) with the named loss applied to
the 2K observation rows and the identity to the prior rows.  `prior` is anything with .mean (n_cam, n_params) and
.information (n_cam, n_params, n_params), e.g. sat_bundleadjust_b200.ba_priors.CameraPrior; blocks of frozen cameras are
ignored.
"""
import numpy as np

from . import ba_oracle


def prior_factors(prior, n_cam_fix):
    """C_j with C_j^T C_j = L_j (from the eigen-decomposition), zero for the frozen cameras: (n_cam, n_params, n_params)."""
    L = np.asarray(prior.information, dtype=np.float64)
    ev, V = np.linalg.eigh(0.5 * (L + L.transpose(0, 2, 1)))
    C = np.sqrt(np.clip(ev, 0.0, None))[:, :, None] * V.transpose(0, 2, 1)
    C[: int(n_cam_fix)] = 0.0
    return C


def prior_rows(x, p, prior):
    """C_j (x_j - mu_j) of every camera, (n_cam * n_params,)"""
    c = int(p.n_params)
    d = np.asarray(x[: p.n_cam * c], dtype=np.float64).reshape(p.n_cam, c) - np.asarray(prior.mean)
    return np.einsum("jrc,jc->jr", prior_factors(prior, p.n_cam_fix), d).ravel()


def augmented_residuals(x, p, prior, residuals=None):
    """[r ; C_j (x_j - mu_j)]: the observation rows of ba_oracle.residuals (or `residuals`) followed by the prior rows."""
    r = (residuals or ba_oracle.residuals)(np.array(x, dtype=np.float64), p)
    return np.concatenate([r, prior_rows(x, p, prior)])


class PriorLoss:
    """Callable scipy loss: the named loss on the first n_obs_rows entries of z = (f / f_scale)^2, the identity on the rest
    (scipy multiplies rho by f_scale^2 and divides rho'' by it, so identity rows stay un-robustified whatever f_scale)."""

    def __init__(self, loss, n_obs_rows):
        from scipy.optimize._lsq.least_squares import IMPLEMENTED_LOSSES
        self.fn = IMPLEMENTED_LOSSES[loss]
        self.m = int(n_obs_rows)

    def __call__(self, z):
        rho = np.empty((3, z.size))
        rho[0], rho[1], rho[2] = z, 1.0, 0.0
        if self.fn is not None:
            sub = np.empty((3, self.m))
            self.fn(z[: self.m], sub, cost_only=False)
            rho[:, : self.m] = sub
        return rho


def augmented_cost(x, p, prior, loss="linear", f_scale=1.0, residuals=None):
    """cost(x) above"""
    r = (residuals or ba_oracle.residuals)(np.array(x, dtype=np.float64), p)
    q = prior_rows(x, p, prior)
    return ba_oracle.robust_cost(r, loss, f_scale) + 0.5 * float(q @ q)


def augmented_gradient(x, p, prior, loss="linear", f_scale=1.0, jac=None, residuals=None):
    """
    grad cost(x) = J^T (rho' r) + L (x - mu) over the free cameras.  jac(x) -> (2K, n) Jacobian of the observation rows
    (dense or sparse); default: central differences of the residual (small problems only).
    """
    from scipy.optimize._lsq.common import compute_grad, scale_for_robust_loss_function
    from scipy.optimize._lsq.least_squares import construct_loss_function
    res = residuals or ba_oracle.residuals
    x = np.array(x, dtype=np.float64)
    f = res(x.copy(), p)
    if jac is None and residuals is not None:
        raise ValueError("augmented_gradient: give jac with a custom residual")
    if jac is None:
        J = ba_oracle.dense_jacobian_fd(x, p)
        J[:, : int(p.n_cam_fix) * int(p.n_params)] = 0.0      # frozen cameras: the residual overwrites their slots (0 / 0 above)
    else:
        J = jac(x.copy())
    if loss != "linear":
        rho = construct_loss_function(f.size, loss, f_scale)(f.copy())
        J, f = scale_for_robust_loss_function(J, f.copy(), rho)
    g = np.asarray(compute_grad(J, f)).ravel().copy()
    c = int(p.n_params)
    C = prior_factors(prior, p.n_cam_fix)
    d = x[: p.n_cam * c].reshape(p.n_cam, c) - np.asarray(prior.mean)
    g[: p.n_cam * c] += np.einsum("jrc,jr->jc", C, np.einsum("jrc,jc->jr", C, d)).ravel()
    return g


def solve_converged_with_prior(p, prior, loss="linear", f_scale=1.0, x_start=None, max_nfev=300, residuals=None):
    """
    Counterpart of ba_oracle.solve_converged for the augmented problem: scipy TRF, x_scale='jac', 3-point differences, the dense
    `exact` trust-region solver and tight tolerances; small problems only.  Returns (x, augmented cost, scipy result).
    """
    from scipy.optimize import least_squares
    x0 = p.params_opt.copy() if x_start is None else np.array(x_start, dtype=np.float64)
    n_rows = 2 * int(np.asarray(p.pts_ind).size)
    res = least_squares(augmented_residuals, x0, jac="3-point", x_scale="jac", method="trf", tr_solver="exact",
                        ftol=1e-15, xtol=1e-15, gtol=1e-15, loss=PriorLoss(loss, n_rows), f_scale=f_scale, max_nfev=max_nfev,
                        args=(p, prior, residuals))
    return res.x, augmented_cost(res.x, p, prior, loss, f_scale, residuals), res
