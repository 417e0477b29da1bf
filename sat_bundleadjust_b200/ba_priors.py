"""
Gaussian priors on the camera variables.

    prior = CameraPrior.from_sigmas(np.zeros((n_cam, n_params)), sigma)      # zero-mean, e.g. RPC bias compensation
    ba_core.run_ba_optimization(p, ls_params, cam_prior=prior)

For each camera j a mean mu_j (n_params values, in the params_opt camera layout) and a symmetric positive semi-definite
information matrix L_j (n_params x n_params).  The solver then minimises

    0.5 f_scale^2 sum_k rho(|r_k|^2 / f_scale^2) + 0.5 sum_{j free} (x_j - mu_j)^T L_j (x_j - mu_j),

which is scipy's least_squares on the augmented residual [r ; C_j (x_j - mu_j)] (L_j = C_j^T C_j) with the loss applied to
the observation rows only: the prior rows are never robustified and f_scale does not touch them.  The scaling D, the
damping, the steps and every termination test are those of the augmented problem.

  * A zero L_j means no prior on camera j; a zero row / column means no prior on that parameter.
  * Blocks of frozen cameras (j < n_cam_fix) are ignored.
  * A prior of full rank on every free camera fixes the gauge: the reduced camera system is positive definite by
    construction, and the posterior covariance of every camera is available with nothing frozen.
  * COMMON_K (shared calibration) with a prior raises NotImplementedError.
"""
import numpy as np

SYM_TOL = 1e-12       # |L - L^T| <= SYM_TOL max|L_j|, per camera
PSD_TOL = 1e-12       # eigenvalues >= -PSD_TOL * the largest


class CameraPrior:
    """mean (n_cam, n_params), information (n_cam, n_params, n_params); validated and symmetrised like the C ABI does."""

    def __init__(self, mean, information):
        mean = np.array(mean, dtype=np.float64)
        info = np.array(information, dtype=np.float64)
        if mean.ndim != 2 or info.shape != (mean.shape[0], mean.shape[1], mean.shape[1]):
            raise ValueError("CameraPrior: mean must be (n_cam, n_params) and information (n_cam, n_params, n_params), got %s and %s"
                             % (mean.shape, info.shape))
        if not np.isfinite(mean).all() or not np.isfinite(info).all():
            raise ValueError("CameraPrior: non-finite values")
        amax = np.abs(info).max(axis=(1, 2))
        asym = np.abs(info - info.transpose(0, 2, 1)).max(axis=(1, 2)) if info.size else np.zeros(0)
        bad = np.nonzero(asym > SYM_TOL * amax)[0]
        if bad.size:
            raise ValueError("CameraPrior: information block of camera %d is not symmetric" % bad[0])
        info = 0.5 * (info + info.transpose(0, 2, 1))
        ev = np.linalg.eigvalsh(info) if info.size else np.zeros((mean.shape[0], 0))
        emax = ev.max(axis=1) if ev.size else np.zeros(mean.shape[0])
        bad = np.nonzero(ev.min(axis=1) < -PSD_TOL * np.maximum(emax, 0.0))[0] if ev.size else []
        if len(bad):
            raise ValueError("CameraPrior: information block of camera %d is not positive semi-definite" % bad[0])
        self.mean = mean
        self.information = info
        self.ranks = (ev > PSD_TOL * emax[:, None]).sum(axis=1) if ev.size else np.zeros(mean.shape[0], dtype=int)

    @classmethod
    def from_sigmas(cls, mean, sigma):
        """Independent parameters: information diag(1 / sigma^2); sigma (n_cam, n_params) or (n_params,), inf = no prior."""
        mean = np.array(mean, dtype=np.float64)
        sigma = np.broadcast_to(np.asarray(sigma, dtype=np.float64), mean.shape)
        if np.isnan(sigma).any() or (sigma <= 0).any():
            raise ValueError("CameraPrior.from_sigmas: sigma must be > 0 (inf: no prior)")
        with np.errstate(divide="ignore"):
            w = np.where(np.isinf(sigma), 0.0, 1.0 / sigma ** 2)
        info = np.zeros(mean.shape + (mean.shape[1],))
        idx = np.arange(mean.shape[1])
        info[:, idx, idx] = w
        return cls(mean, info)

    def free_rank(self, n_cam_fix):
        """sum of rank(L_j) over the free cameras: the rows the prior adds to the degrees of freedom."""
        return int(self.ranks[int(n_cam_fix):].sum())

    def check_for(self, p):
        """the prior fits the problem p (shape, no COMMON_K)"""
        from .solver import n_common_params
        if n_common_params(p):
            raise NotImplementedError("camera priors are not available with COMMON_K (shared calibration)")
        if self.mean.shape != (int(p.n_cam), int(p.n_params)):
            raise ValueError("CameraPrior: mean is %s, the problem has (n_cam, n_params) = (%d, %d)"
                             % (self.mean.shape, p.n_cam, p.n_params))
