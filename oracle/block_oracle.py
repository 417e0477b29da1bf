"""
Checker only: the normal equations, the reduced camera system and the posterior covariance of a bundle adjustment, formed
from the per-observation Jacobian blocks without a dense Jacobian, so that it runs at the sizes the device engines are built
for (1e6 observations in seconds on a CPU).

Inputs are the blocks Jc (K, 2, c) and Jp (K, 2, 3) (the device's sba_jacobian_blocks, or central differences), the residuals
f (2K), cam_ind / pts_ind (observations by track, pts_ind non-decreasing), the frozen counts, the loss and f_scale, and
optionally a camera prior (mean, information).  Everything is formed per observation and per track and accumulated in
np.longdouble; the 3x3 point blocks are inverted by the adjugate in np.longdouble.  The result is rounded to float64 once.

Every output comes with a per-entry magnitude A of the same shape: the sum of the absolute values of the terms the entry is
a sum of (|U_ij| + sum_t sum_{a,b,s} |Z_as,i| |W_bs,j| + reg D^2 for S, ...).  A float64 kernel that forms the entry by any
order of summation errs by a small multiple of eps A, whatever cancellation the sum has, so tolerances read
|dev - oracle| <= tau A.

    ne = NormalEquations(Jc, Jp, f, cam_ind, pts_ind, n_cam, n_pts, n_cam_fix, n_pts_fix, loss, f_scale, prior, x_cam)
    ne.U, ne.V, ne.g, ne.cost (+ .Ua, .Va, .ga, .cost_a)     U (M, c, c), V (N, 6) upper, g (M c + 3 N)
    S, rhs, Sa, rhsa = ne.reduced_system(reg, n_common)      (M c)^2 and (M c), device layout (c slots per camera)
    cov_cam, cov_pts, kappa = ne.covariance(sigma2, points)

Conventions (those of scipy's least_squares and the solver): the robust loss rescales every residual row as
scipy.optimize._lsq.common.scale_for_robust_loss_function does; D^2 = diag(J^T J) with the prior's diagonal, zeros replaced by 1;
S = U + reg D_c^2 - sum_t W_t (V_t + reg D_t^2)^-1 W_t^T and rhs = -(g_c - sum_t W_t (V_t + reg D_t^2)^-1 g_t).  Frozen cameras
have no columns: their slots are identity rows of S with a zero right-hand side; frozen points contribute nothing.  With
COMMON_K the last n_common slots of every camera are one set of unknowns, folded onto camera 0's slots (S' = P^T S P, the
damping from the folded diagonal), the others identity rows with a zero right-hand side.
"""
import numpy as np

LD = np.longdouble
IDX6 = ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))
PAIR_CHUNK = 200000


def robust_rows(Jc, Jp, f, loss="linear", f_scale=1.0):
    """(Jc, Jp, f, rho_0) after scipy's rescale of the rows for a robust loss; rho_0 (2K) are the cost terms (2 cost = sum)."""
    K, c = Jc.shape[0], Jc.shape[2]
    f = np.array(f, dtype=np.float64)
    if loss == "linear":
        return np.array(Jc, dtype=np.float64), np.array(Jp, dtype=np.float64), f, f * f
    from scipy.optimize._lsq.common import scale_for_robust_loss_function
    from scipy.optimize._lsq.least_squares import construct_loss_function
    rho = construct_loss_function(f.size, loss, f_scale)(f.copy())
    J = np.concatenate([np.reshape(Jc, (2 * K, c)), np.reshape(Jp, (2 * K, 3))], axis=1)
    J, fs = scale_for_robust_loss_function(J, f.copy(), rho)
    return J[:, :c].reshape(K, 2, c), J[:, c:].reshape(K, 2, 3), fs, rho[0].copy()


def inv3_adjugate(V):
    """(n, 3, 3) symmetric -> inverse by the adjugate, in the dtype of V; rows with det == 0 come back 0."""
    a, b, c, d, e, f = V[:, 0, 0], V[:, 0, 1], V[:, 0, 2], V[:, 1, 1], V[:, 1, 2], V[:, 2, 2]
    A = np.empty_like(V)
    A[:, 0, 0] = d * f - e * e
    A[:, 0, 1] = A[:, 1, 0] = c * e - b * f
    A[:, 0, 2] = A[:, 2, 0] = b * e - c * d
    A[:, 1, 1] = a * f - c * c
    A[:, 1, 2] = A[:, 2, 1] = b * c - a * e
    A[:, 2, 2] = a * d - b * b
    det = a * A[:, 0, 0] + b * A[:, 0, 1] + c * A[:, 0, 2]
    ok = det != 0
    A[ok] /= det[ok, None, None]
    A[~ok] = 0
    return A


def track_pairs(starts, tracks):
    """(a, b) observation pairs a <= b inside each of the given tracks (starts: (N+1) first observation of every track)."""
    tracks = np.asarray(tracks)
    s, e = starts[tracks], starts[tracks + 1]
    a = _ranges(s, e)
    ends = np.repeat(e, e - s)
    cnt = ends - a
    A = np.repeat(a, cnt)
    first = np.cumsum(cnt) - cnt
    B = A + (np.arange(A.size) - np.repeat(first, cnt))
    return A, B


def _ranges(s, e):
    n = e - s
    first = np.cumsum(n) - n
    return np.repeat(s - first, n) + np.arange(n.sum())


class NormalEquations:
    """U, V, g, cost of J^T J, J^T f at one point, and what follows from them; see the module docstring."""

    def __init__(self, Jc, Jp, f, cam_ind, pts_ind, n_cam, n_pts, n_cam_fix=0, n_pts_fix=0, loss="linear", f_scale=1.0,
                 prior=None, x_cam=None, f_tol=0.0):
        """f_tol: a bound on |f - f_kernel|, the difference between the residual given here and the one the kernel under test
        linearises (px).  It adds gt = sum |J| f_tol (gct, gpt) next to g: a kernel's g may differ from the oracle's by that
        much before any summation error."""
        cam_ind, pts_ind = np.asarray(cam_ind, dtype=np.int64), np.asarray(pts_ind, dtype=np.int64)
        assert np.all(np.diff(pts_ind) >= 0), "observations must be ordered by track"
        M, N, c, K = int(n_cam), int(n_pts), int(np.shape(Jc)[2]), cam_ind.size
        self.M, self.N, self.c, self.K = M, N, c, K
        self.n_cam_fix, self.n_pts_fix = int(n_cam_fix), int(n_pts_fix)
        self.cam_ind, self.pts_ind = cam_ind, pts_ind
        self.starts = np.searchsorted(pts_ind, np.arange(N + 1))
        raw_c, raw_p = np.abs(Jc), np.abs(Jp)
        raw_c[cam_ind < self.n_cam_fix] = 0.0
        raw_p[pts_ind < self.n_pts_fix] = 0.0
        Jc, Jp, fs, rho0 = robust_rows(Jc, Jp, f, loss, f_scale)
        Jc[cam_ind < self.n_cam_fix] = 0.0            # frozen cameras and points have no columns
        Jp[pts_ind < self.n_pts_fix] = 0.0
        self.Jc, self.Jp, self.f = Jc.astype(LD), Jp.astype(LD), fs.reshape(K, 2).astype(LD)
        self.cost = float(LD(0.5) * np.sum(rho0.astype(LD)))
        self.cost_a = float(0.5 * np.abs(rho0).sum())
        ac, ap, af = np.abs(Jc), np.abs(Jp), np.abs(fs.reshape(K, 2))
        U, Ua = np.zeros((M, c, c), LD), np.zeros((M, c, c))
        np.add.at(U, cam_ind, np.einsum("kri,krj->kij", self.Jc, self.Jc))
        np.add.at(Ua, cam_ind, np.einsum("kri,krj->kij", ac, ac))
        V, Va = np.zeros((N, 3, 3), LD), np.zeros((N, 3, 3))
        np.add.at(V, pts_ind, np.einsum("kri,krj->kij", self.Jp, self.Jp))
        np.add.at(Va, pts_ind, np.einsum("kri,krj->kij", ap, ap))
        gc, gca = np.zeros((M, c), LD), np.zeros((M, c))
        np.add.at(gc, cam_ind, np.einsum("kri,kr->ki", self.Jc, self.f))
        np.add.at(gca, cam_ind, np.einsum("kri,kr->ki", ac, af))
        gp, gpa = np.zeros((N, 3), LD), np.zeros((N, 3))
        np.add.at(gp, pts_ind, np.einsum("kri,kr->ki", self.Jp, self.f))
        np.add.at(gpa, pts_ind, np.einsum("kri,kr->ki", ap, af))
        if prior is not None:
            L = np.array(prior.information, dtype=np.float64)
            L[: self.n_cam_fix] = 0.0                   # blocks of frozen cameras are ignored
            d = np.asarray(x_cam, dtype=np.float64).reshape(M, c) - np.asarray(prior.mean)
            Ld = np.einsum("jrc,jc->jr", L.astype(LD), d.astype(LD))
            U += L.astype(LD)
            Ua += np.abs(L)
            gc += Ld
            gca += np.einsum("jrc,jc->jr", np.abs(L), np.abs(d))
            self.cost += float(LD(0.5) * np.sum(Ld * d.astype(LD)))
            self.cost_a += float(0.5 * np.einsum("jr,jr->", np.einsum("jrc,jc->jr", np.abs(L), np.abs(d)), np.abs(d)))
        self._U, self._V, self._gc, self._gp = U, V, gc, gp
        self._Ua, self._Va, self._gca, self._gpa = Ua, Va, gca, gpa
        self.U, self.Ua = U.astype(np.float64), Ua
        self.V = np.stack([V[:, a, b] for a, b in IDX6], axis=1).astype(np.float64)
        self.Va = np.stack([Va[:, a, b] for a, b in IDX6], axis=1)
        self.g = np.concatenate([gc.ravel(), gp.ravel()]).astype(np.float64)
        self.ga = np.concatenate([gca.ravel(), gpa.ravel()])
        # per row g = J^T f rho'(f^2), and |d (f rho') / df| = |rho' + 2 rho'' f^2| <= 1 for the losses of scipy: a change of f by
        # f_tol moves a row's term by at most |J| f_tol, J unscaled
        gct, gpt = np.zeros((M, c)), np.zeros((N, 3))
        if f_tol:
            np.add.at(gct, cam_ind, np.einsum("kri->ki", raw_c) * f_tol)
            np.add.at(gpt, pts_ind, np.einsum("kri->ki", raw_p) * f_tol)
        self.gt = np.concatenate([gct.ravel(), gpt.ravel()])
        self.W = np.einsum("kri,krs->kis", self.Jc, self.Jp)          # (K, c, 3): J_c^T J_p of every observation
        self.Wa = np.einsum("kri,krs->kis", ac, ap)

    # -- reduced camera system ------------------------------------------------------------------------------------------
    def _point_inverse(self, reg):
        V = self._V.copy()
        d2 = np.einsum("nii->ni", V).copy()
        d2[d2 == 0] = 1
        V[:, [0, 1, 2], [0, 1, 2]] += LD(reg) * d2
        Vi = inv3_adjugate(V)
        live = (np.arange(self.N) >= self.n_pts_fix) & (np.diff(self.starts) > 0)
        assert np.all(np.any(Vi[live] != 0, axis=(1, 2))), "a free point with observations has a singular block"
        Vi[~live] = 0
        return Vi

    def _schur(self, Vi, tracks=None):
        """(sum_t W_t Vi_t W_t^T as (M, M, c, c), its magnitude, sum_t W_t Vi_t g_t as (M, c), its magnitude)"""
        M, c = self.M, self.c
        tr = np.arange(self.N) if tracks is None else np.asarray(tracks)
        tr = tr[(tr >= self.n_pts_fix) & (self.starts[tr + 1] > self.starts[tr])]
        obs = _ranges(self.starts[tr], self.starts[tr + 1])
        t_of = self.pts_ind
        Z = np.zeros((self.K, c, 3), LD)
        Z[obs] = np.einsum("kis,kst->kit", self.W[obs], Vi[t_of[obs]])
        Za = np.abs(Z).astype(np.float64)
        R, Ra = np.zeros((M, c), LD), np.zeros((M, c))
        np.add.at(R, self.cam_ind[obs], np.einsum("kis,ks->ki", Z[obs], self._gp[t_of[obs]]))
        np.add.at(Ra, self.cam_ind[obs], np.einsum("kis,ks->ki", Za[obs], np.abs(self._gp[t_of[obs]]).astype(np.float64)))
        A, B = track_pairs(self.starts, tr)
        off = A != B
        assert not np.any(self.cam_ind[A[off]] == self.cam_ind[B[off]]), "a track observed twice by one camera"
        T, Ta = np.zeros((M * M, c, c), LD), np.zeros((M * M, c, c))
        for i in range(0, A.size, PAIR_CHUNK):
            a, b = A[i: i + PAIR_CHUNK], B[i: i + PAIR_CHUNK]
            key = self.cam_ind[a] * M + self.cam_ind[b]
            np.add.at(T, key, np.einsum("pis,pjs->pij", Z[a], self.W[b]))
            np.add.at(Ta, key, np.einsum("pis,pjs->pij", Za[a], self.Wa[b]))
        T, Ta = T.reshape(M, M, c, c), Ta.reshape(M, M, c, c)
        # the pairs a < b are accumulated once: Z_b W_a^T of the pair (b, a) is (Z_a W_b^T)^T because V_t^-1 is symmetric.  No
        # camera sees a track twice (asserted above), so the diagonal blocks of T hold the a == b terms only
        diag = np.arange(M)
        Dg, Dga = T[diag, diag].copy(), Ta[diag, diag].copy()
        T = T + T.transpose(1, 0, 3, 2)
        Ta = Ta + Ta.transpose(1, 0, 3, 2)
        T[diag, diag], Ta[diag, diag] = Dg, Dga
        return T, Ta, R, Ra

    @staticmethod
    def _square(B):
        M, c = B.shape[0], B.shape[2]
        return B.transpose(0, 2, 1, 3).reshape(M * c, M * c)

    def reduced_system(self, reg=0.0, n_common=0, tracks=None, with_cameras=True):
        """(S, rhs, Sa, rhsa), float64, ns = M c.  tracks: only these tracks' Schur terms; with_cameras=False leaves out U, g_c,
        the damping and the identity rows (the contribution of the tracks alone, for the sensitivity checks)."""
        M, c = self.M, self.c
        ns = M * c
        T, Ta, R, Ra = self._schur(self._point_inverse(reg), tracks)
        Ublk = np.zeros((M, M, c, c), LD)
        Ublka = np.zeros((M, M, c, c))
        if with_cameras:
            Ublk[np.arange(M), np.arange(M)] = self._U
            Ublka[np.arange(M), np.arange(M)] = self._Ua
        S = self._square(Ublk) - self._square(T)
        Sa = self._square(Ublka) + self._square(Ta)
        rhs = (-self._gc + R).ravel() if with_cameras else R.ravel()
        rhsa = (self._gca + Ra).ravel() if with_cameras else Ra.ravel()
        used = np.ones(ns, dtype=bool)
        used[: self.n_cam_fix * c] = False
        d2 = np.diag(self._square(Ublk)).copy()
        if n_common:
            P = np.eye(ns, dtype=LD)
            for j in range(1, M):
                for s in range(c - n_common, c):
                    P[j * c + s, j * c + s] = 0
                    P[j * c + s, s] = 1
                    used[j * c + s] = False
            S, Sa = P.T @ S @ P, (P.T @ Sa.astype(LD) @ P).astype(np.float64)
            rhs, rhsa = P.T @ rhs, (P.T @ rhsa.astype(LD)).astype(np.float64)
            d2 = np.diag(P.T @ self._square(Ublk) @ P).copy()
        if with_cameras:
            d2[d2 == 0] = 1
            k = np.where(used)[0]
            S[k, k] += LD(reg) * d2[k]
            Sa[k, k] += reg * d2[k].astype(np.float64)
            n = np.where(~used)[0]
            S[n, :], S[:, n], Sa[n, :], Sa[:, n] = 0, 0, 0, 0
            S[n, n], rhs[n], rhsa[n] = 1, 0, 0
        return S.astype(np.float64), rhs.astype(np.float64), Sa, rhsa

    # -- covariance ------------------------------------------------------------------------------------------------------
    def covariance(self, sigma2, points=None):
        """(sigma2 S^-1 (ns, ns), sigma2 C_t for the given points (all by default) (n, 3, 3), kappa): S undamped over the free
        camera slots, inverted in float64 in the Jacobi-scaled basis; C_t = V_t^-1 + Z_t^T S^-1 Z_t, Z_t = W_t V_t^-1; frozen
        cameras and points 0.  kappa: the 2-norm condition number of S scaled by diag(U) of the free slots."""
        M, c = self.M, self.c
        ns, ncf = M * c, self.n_cam_fix * c
        S, _, _, _ = self.reduced_system(0.0)
        Sinv = np.zeros((ns, ns))
        Sf = S[ncf:, ncf:]
        if Sf.size:
            d = np.sqrt(np.diag(Sf))
            Sinv[ncf:, ncf:] = np.linalg.inv(Sf / np.outer(d, d)) / np.outer(d, d)
            u = np.sqrt(np.einsum("jkk->jk", self.U).ravel()[ncf:])
            kappa = float(np.linalg.cond(Sf / np.outer(u, u)))
        else:
            kappa = 1.0
        Sinv = 0.5 * (Sinv + Sinv.T)
        pts = np.arange(self.N) if points is None else np.asarray(points)
        Vi = self._point_inverse(0.0)
        Cp = Vi[pts].astype(np.float64).copy()
        Zf = np.einsum("kis,kst->kit", self.W, Vi[self.pts_ind]).astype(np.float64)
        slots = self.cam_ind[:, None] * c + np.arange(c)[None, :]
        live = pts[(pts >= self.n_pts_fix) & (self.starts[pts + 1] > self.starts[pts])]
        where = np.full(self.N, -1)
        where[pts] = np.arange(pts.size)
        A, B = track_pairs(self.starts, live)
        for i in range(0, A.size, PAIR_CHUNK):
            a, b = A[i: i + PAIR_CHUNK], B[i: i + PAIR_CHUNK]
            blk = Sinv[slots[a][:, :, None], slots[b][:, None, :]]          # (p, c, c)
            P = np.einsum("pis,pij,pjt->pst", Zf[a], blk, Zf[b])
            off = a != b
            np.add.at(Cp, where[self.pts_ind[a]], P)
            np.add.at(Cp, where[self.pts_ind[a[off]]], P[off].transpose(0, 2, 1))
        Cp[(pts < self.n_pts_fix)] = 0.0
        Cp = 0.5 * (Cp + Cp.transpose(0, 2, 1))
        return sigma2 * Sinv, sigma2 * Cp, kappa


def fd_blocks(x, p, residuals, rel_step=1e-6):
    """Central-difference blocks (Jc, Jp) of residuals(x, p) at any size: an observation depends on its own camera and point
    only, so moving slot s of every camera (coordinate s of every point) at once gives column s of every block."""
    x = np.asarray(x, dtype=np.float64)
    M, c, N = int(p.n_cam), int(p.n_params), int(p.n_pts)
    cam, pts = np.asarray(p.cam_ind), np.asarray(p.pts_ind)
    K = cam.size
    Jc, Jp = np.zeros((K, 2, c)), np.zeros((K, 2, 3))
    for off, n, per, J, ind in ((0, M, c, Jc, cam), (M * c, N, 3, Jp, pts)):
        for s in range(per):
            idx = off + np.arange(n) * per + s
            h = rel_step * np.maximum(1.0, np.abs(x[idx]))
            a, b = x.copy(), x.copy()
            a[idx] += h
            b[idx] -= h
            step = (a[idx] - b[idx])[ind][:, None]           # before the calls: residuals() writes the frozen cameras into its vector
            J[:, :, s] = (residuals(a, p) - residuals(b, p)).reshape(K, 2) / step
    return Jc, Jp
