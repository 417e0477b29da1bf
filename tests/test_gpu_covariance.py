"""
Posterior covariance (sba_covariance / ba_covariance.compute_covariance) against dense float64 linear algebra.

The oracle follows test_reduced_camera_system: the dense Jacobian from the device's per-observation blocks plus scipy's
robust rescale, H = J^T J over the free columns inverted in the Jacobi-scaled basis D^-1 H D^-1 (so that the oracle itself is
accurate), times sigma^2.  Elements are compared scale-free: |C_dev - C_np|_ij <= tol sqrt(C_np,ii C_np,jj), so that radians
and metres compare fairly.  GPU tests are marked `gpu`; the checks that need no device are not.
"""
import re

import numpy as np
import pytest

import util
from oracle import ba_oracle, rpc_oracle
from sat_bundleadjust_b200 import _lib, synth
from sat_bundleadjust_b200.ba_covariance import compute_covariance, degrees_of_freedom
from sat_bundleadjust_b200.solver import DeviceProblem, initial_vars
from util import cond_tol, normalised_err as _normalised_err, scaled_cond, scaled_inv

NORM_TOL = 1e-7


PIVOT_THRESHOLD = 1e-12
IDX6 = ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))


def _robust_rows(J, f, loss, f_scale):
    """scipy's rescale of the Jacobian rows for a robust loss (least_squares.py / common.py)."""
    if loss == "linear":
        return J
    from scipy.optimize._lsq.common import scale_for_robust_loss_function
    from scipy.optimize._lsq.least_squares import construct_loss_function
    rho = construct_loss_function(f.size, loss, f_scale)(f.copy())
    Js, _ = scale_for_robust_loss_function(J.copy(), f.copy(), rho)
    return Js


def oracle_residuals(x, p):
    """ba_oracle.residuals, except that RPC projections stay in float64: the covariance is a float64 model of the residuals
    (the reference's fun rounds RPC projections to float32, ba_core.py:150, which moves single residuals by one float32 ulp)."""
    if p.cam_model != "rpc":
        return ba_oracle.residuals(x.copy(), p)
    pts3d, cam_params = ba_oracle.unpack_variables(x.copy(), p)
    q = ba_oracle.adjust_pts3d(pts3d[p.pts_ind], cam_params[p.cam_ind])
    rpcs = [util.rpc_from_array(t) for t in util.load_rpc_golden()["rpc_cams"]]
    proj = np.zeros((p.pts_ind.size, 2))
    for j in np.unique(p.cam_ind).tolist():
        sel = p.cam_ind == j
        lat, lon, alt = rpc_oracle.ecef_to_latlon(q[sel, 0], q[sel, 1], q[sel, 2])
        proj[sel] = np.stack(rpcs[j].projection(lon, lat, alt), axis=1)
    return np.repeat(p.pts2d_w, 2, axis=0) * (proj - p.pts2d).ravel()


def dense_oracle(p, prob, x, loss, f_scale, sigma2=None):
    """(cov_cam, cov_pts (N,3,3), sigma2, kappa) from dense linear algebra; frozen rows / points 0; kappa = scaled_cond of the
    oracle's S over the free camera slots."""
    Jc, Jp = prob.jacobian_blocks(x)
    J = util.dense_jacobian_from_blocks(p, Jc, Jp)
    f = oracle_residuals(x, p)
    J = _robust_rows(J, f, loss, f_scale)
    c, M, N = p.n_params, p.n_cam, p.n_pts
    ns = M * c
    free = np.r_[np.arange(p.n_cam_fix * c, ns), ns + np.arange(3 * p.n_pts_fix, 3 * N)]
    Jf = J[:, free]
    H = Jf.T @ Jf
    d = np.sqrt(np.diag(H))
    Hinv = np.linalg.inv(H / np.outer(d, d)) / np.outer(d, d)
    n_free = free.size
    s2 = sigma2 if sigma2 else 2.0 * ba_oracle.robust_cost(f, loss, f_scale) / (f.size - n_free)
    C = np.zeros((ns + 3 * N, ns + 3 * N))
    C[np.ix_(free, free)] = s2 * Hinv
    cov_pts = np.array([C[ns + 3 * i: ns + 3 * i + 3, ns + 3 * i: ns + 3 * i + 3] for i in range(N)])
    nfc = ns - p.n_cam_fix * c                        # S^-1 is the camera block of H^-1
    kappa = scaled_cond(scaled_inv(Hinv[:nfc, :nfc]), np.diag(H)[:nfc]) if nfc else 1.0
    return C[:ns, :ns], cov_pts, s2, kappa


def _check_against_oracle(p, prob, x, cc, cp, s2, ratio, loss, f_scale, sigma2=None):
    cc_np, cp_np, s2_np, kappa = dense_oracle(p, prob, x, loss, f_scale, sigma2)
    if sigma2:
        assert s2 == sigma2
    else:
        # the formula to 1e-12 on the device's own residuals (float64 projections); the oracle's residuals differ from them by
        # the fun parity of ~1e-9 px (CUDA sin/cos and FMA vs numpy), which moves the cost by up to ~1e-10 relative
        if p.cam_model == "rpc":
            with DeviceProblem(p, rpc_float32=False) as p64:
                r_dev, _ = p64.residuals(x, loss, f_scale)
        else:
            r_dev, _ = prob.residuals(x, loss, f_scale)
        n_free = (p.n_cam - p.n_cam_fix) * p.n_params + 3 * (p.n_pts - p.n_pts_fix)
        s2_dev = 2.0 * ba_oracle.robust_cost(r_dev, loss, f_scale) / (r_dev.size - n_free)
        assert abs(s2 - s2_dev) <= 1e-12 * s2_dev, (s2, s2_dev)
        assert abs(s2 - s2_np) <= 1e-9 * s2_np, (s2, s2_np)
    tol = cond_tol(NORM_TOL, kappa, (p.n_cam - p.n_cam_fix) * p.n_params)
    print("normalised error vs the dense oracle: cameras %.2e, points %.2e (bound %.1e, oracle kappa %.2e, min pivot ratio %.2e)"
          % (_normalised_err(cc, cc_np), max(_normalised_err(cp[i], cp_np[i]) for i in range(p.n_pts)), tol, kappa, ratio))
    assert _normalised_err(cc, cc_np) <= tol
    assert max(_normalised_err(cp[i], cp_np[i]) for i in range(p.n_pts)) <= tol
    # frozen cameras / points exactly 0; symmetric; positive definite on the free part
    ncf = p.n_cam_fix * p.n_params
    assert not cc[:ncf].any() and not cc[:, :ncf].any()
    assert not cp[: p.n_pts_fix].any()
    assert np.array_equal(cc, cc.T) and np.array_equal(cp, cp.transpose(0, 2, 1))
    if ncf < cc.shape[0]:
        np.linalg.cholesky(cc[ncf:, ncf:])
    np.linalg.cholesky(cp[p.n_pts_fix:])
    return tol


def _rpc_params(corr, n_cam_fix, seed):
    G = util.load_rpc_golden()
    sc = synth.make_rpc_scene(G["rpc_cams"], G["rpcba/camera_centers"], n_tracks=50, p_vis=0.8, seed=seed)
    return synth.SparseParams(sc, corr, n_cam_fix=n_cam_fix)


# (name, builder) of the accepted scenes: the gauge is fixed by frozen cameras or frozen points
def _scene(name):
    if name == "persp_RT_cfix2":
        return synth.scene_to_params(synth.make_scene(n_cam=5, n_tracks=50, p_vis=0.8, seed=31), ["R", "T"], n_cam_fix=2)
    if name == "persp_RT_pfix10":
        return synth.scene_to_params(synth.make_scene(n_cam=5, n_tracks=50, p_vis=0.8, seed=32), ["R", "T"], n_pts_fix=10)
    if name == "affine_RT_cfix2":
        return synth.scene_to_params(synth.make_scene(n_cam=5, n_tracks=50, p_vis=0.8, cam_model="affine", seed=33), ["R", "T"],
                                     n_cam_fix=2)
    if name == "rpc_R_cfix1":
        return _rpc_params(["R"], 1, 34)
    if name == "persp_RT_all_frozen":
        return synth.scene_to_params(synth.make_scene(n_cam=4, n_tracks=40, p_vis=0.8, seed=35), ["R", "T"], n_cam_fix=4)
    raise KeyError(name)


SCENES = ["persp_RT_cfix2", "persp_RT_pfix10", "affine_RT_cfix2", "rpc_R_cfix1", "persp_RT_all_frozen"]


def _solved(p, prob, loss):
    x, _, _ = prob.solve(initial_vars(p), want_residuals=False, loss=loss, ftol=1e-10, xtol=1e-12, max_nfev=200)
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("loss", ["linear", "soft_l1"])
@pytest.mark.parametrize("name", SCENES)
def test_covariance_dense_oracle_both_engines(built, name, loss):
    p = _scene(name)
    out = {}
    for engine in ("pattern", "generic"):
        with DeviceProblem(p, engine=engine) as prob:
            x = _solved(p, prob, loss) if engine == "pattern" else out["pattern"][4]
            cc, cp, s2, ratio = prob.covariance(x, loss=loss)
            out[engine] = (cc, cp, s2, ratio, x, _check_against_oracle(p, prob, x, cc, cp, s2, ratio, loss, 1.0))
        print("%s %s %s: sigma2 %.6e, min pivot ratio %.3e" % (name, loss, engine, s2, ratio))
        assert ratio >= 100 * PIVOT_THRESHOLD, ratio         # two orders of margin above the threshold
    (ca, pa, sa, _, _, tol), (cb, pb, sb, _, _, _) = out["pattern"], out["generic"]
    assert abs(sa - sb) <= 1e-12 * sa
    assert _normalised_err(cb, ca) <= tol
    assert max(_normalised_err(pb[i], pa[i]) for i in range(p.n_pts)) <= tol
    if p.n_cam_fix == p.n_cam:                     # pure triangulation uncertainty: sigma2 V_t^-1
        with DeviceProblem(p) as prob:
            _, V, _ = prob.normal_blocks(out["pattern"][4], loss)
        Vm = np.zeros((p.n_pts, 3, 3))
        for k, (a, b) in enumerate(IDX6):
            Vm[:, a, b] = Vm[:, b, a] = V[:, k]
        assert not ca.any()
        assert max(_normalised_err(pa[i], sa * np.linalg.inv(Vm[i])) for i in range(p.n_pts)) <= NORM_TOL


@pytest.mark.gpu
def test_covariance_given_sigma2_is_used_as_is(built):
    p = _scene("persp_RT_cfix2")
    with DeviceProblem(p) as prob:
        x = _solved(p, prob, "linear")
        cc, cp, s2, ratio = prob.covariance(x, sigma2=0.25)
        assert s2 == 0.25
        _check_against_oracle(p, prob, x, cc, cp, s2, ratio, "linear", 1.0, sigma2=0.25)


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["pattern", "generic"])
def test_covariance_unfixed_gauge_is_rejected(built, engine):
    """Perspective R+T with nothing frozen: 7-dimensional similarity null space, S singular in exact arithmetic."""
    p = synth.scene_to_params(synth.make_scene(n_cam=5, n_tracks=50, p_vis=0.8, seed=31), ["R", "T"])
    with DeviceProblem(p, engine=engine) as prob:
        x = _solved(p, prob, "linear")
        with pytest.raises(_lib.SbaError) as ei:
            prob.covariance(x)
    msg = str(ei.value)
    m = re.search(r"camera (\d+), slot (\d+): pivot ratio L_kk\^2 / U_kk = ([-+0-9.eE]+)", msg)
    assert m, msg
    ratio = float(m.group(3))
    print("gauge not fixed (%s): rejected pivot ratio %.3e (threshold %.0e)" % (engine, ratio, PIVOT_THRESHOLD))
    assert ratio <= PIVOT_THRESHOLD / 100                 # two orders of margin below the threshold


@pytest.mark.gpu
def test_covariance_monte_carlo(built):
    """
    Meaning: over 400 seeded noise draws on fixed geometry (no outliers, 0.5 px, linear loss), the empirical variance of every
    free camera parameter and of 20 free points' coordinates is within [0.75, 1.3] x the predicted one (sigma2 = 0.25 given).
    """
    sc = synth.make_scene(n_cam=6, n_tracks=300, p_vis=0.7, seed=41, noise_px=0.0, outlier_frac=0.0)
    p = synth.scene_to_params(sc, ["R", "T"], n_cam_fix=2)
    clean = p.pts2d.copy()
    x0 = initial_vars(p)
    opts = dict(want_residuals=False, loss="linear", ftol=1e-12, xtol=1e-12, gtol=1e-12, max_nfev=100)
    with DeviceProblem(p) as prob:
        xc, _, _ = prob.solve(x0, **opts)
        cc, cp, _, _ = prob.covariance(xc, sigma2=0.25)
    c, ns = p.n_params, p.n_cam * p.n_params
    pts = np.random.default_rng(7).choice(np.arange(p.n_pts_fix, p.n_pts), 20, replace=False)
    rng = np.random.default_rng(1234)
    cams, coords = [], []
    for _ in range(400):
        p.pts2d = clean + rng.normal(0.0, 0.5, size=clean.shape)
        with DeviceProblem(p) as prob:
            x, _, _ = prob.solve(xc, **opts)
        cams.append(x[p.n_cam_fix * c: ns])
        coords.append(x[ns:].reshape(-1, 3)[pts].ravel())
    p.pts2d = clean
    emp_c = np.var(np.array(cams), axis=0, ddof=1)
    emp_p = np.var(np.array(coords), axis=0, ddof=1)
    pred_c = np.diag(cc)[p.n_cam_fix * c:]
    pred_p = np.concatenate([np.diag(cp[i]) for i in pts])
    rc, rp = emp_c / pred_c, emp_p / pred_p
    print("empirical / predicted variance: cameras %.3f..%.3f, points %.3f..%.3f" % (rc.min(), rc.max(), rp.min(), rp.max()))
    assert rc.min() >= 0.75 and rc.max() <= 1.3
    assert rp.min() >= 0.75 and rp.max() <= 1.3


@pytest.mark.gpu
@pytest.mark.parametrize("loss", ["linear", "soft_l1"])
def test_covariance_many_cameras_long_tracks(built, loss):
    """
    Generic engine, 45 cameras R+T (two frozen), tracks seen by ~43 cameras: ns = 270 exercises the blocked multi-CTA Cholesky
    with its factor written back (ns > 127), k_cov_inverse over 9 column blocks with real tile steps in both substitutions and a
    padded last block, the point pass reading s2 S^-1 from L2 (ns > 113), and the chunked pair loop of tracks of more than 32
    observations (k_cov_long_tracks).  Same dense oracle as above.
    """
    p = synth.scene_to_params(synth.make_scene(n_cam=45, n_tracks=60, p_vis=0.95, seed=36), ["R", "T"], n_cam_fix=2)
    lengths = np.bincount(p.pts_ind)
    assert lengths.min() > 32 and p.n_cam * p.n_params == 270
    with DeviceProblem(p) as prob:
        assert prob.engine == "generic"
        x = _solved(p, prob, loss)
        cc, cp, s2, ratio = prob.covariance(x, loss=loss)
        _check_against_oracle(p, prob, x, cc, cp, s2, ratio, loss, 1.0)
    assert ratio >= 100 * PIVOT_THRESHOLD, ratio


@pytest.mark.gpu
def test_covariance_at_metric_size(built):
    """
    The 1e6-observation scene of the default bench workload (pattern engine, M = 10, c = 6), n_cam_fix = 2, soft_l1:
    Sigma_cc against numpy's inverse of the device's undamped reduced system, 2000 random tracks against the host formula
    from the Jacobian and normal blocks, and the generic engine against the pattern engine, all to max(1e-9, cond_tol).
    """
    sc = synth.make_scene(n_cam=10, n_tracks=200000, p_vis=0.5, cam_model="perspective", seed=0)
    # two frozen cameras: with one, the scale about its centre is still free (S singular in exact arithmetic)
    p = synth.scene_to_params(sc, ["R", "T"], n_cam_fix=2)
    loss, c = "soft_l1", p.n_params
    ns, ncf = p.n_cam * c, p.n_cam_fix * c
    with DeviceProblem(p) as prob:
        assert prob.engine == "pattern"
        x, _, _ = prob.solve(initial_vars(p), want_residuals=False, loss=loss)
        cc, cp, s2, ratio = prob.covariance(x, loss=loss)
        S, _ = prob.reduced_system(x, loss, 1.0, 0.0)
        Jc, Jp = prob.jacobian_blocks(x)
        Ublk, V, _ = prob.normal_blocks(x, loss)
        f, _ = prob.residuals(x)
    print("1e6 observations: sigma2 %.6e, min pivot ratio %.3e" % (s2, ratio))
    Sinv = np.zeros((ns, ns))
    Sinv[ncf:, ncf:] = scaled_inv(S[ncf:, ncf:])
    kappa = scaled_cond(S[ncf:, ncf:], np.concatenate([np.diag(Ub) for Ub in Ublk])[ncf:])
    tol = cond_tol(1e-9, kappa, ns - ncf)
    print("normalised error vs numpy: cameras %.2e (bound %.1e, numpy kappa %.2e)" % (_normalised_err(cc, s2 * Sinv), tol, kappa))
    assert _normalised_err(cc, s2 * Sinv) <= tol
    # host formula on 2000 random tracks
    K = p.pts_ind.size
    Jrows = _robust_rows(np.concatenate([Jc.reshape(2 * K, c), Jp.reshape(2 * K, 3)], axis=1), f, loss, 1.0)
    Jcs, Jps = Jrows[:, :c].reshape(K, 2, c), Jrows[:, c:].reshape(K, 2, 3)
    starts = np.searchsorted(p.pts_ind, np.arange(p.n_pts + 1))
    worst = 0.0
    for t in np.random.default_rng(3).choice(p.n_pts, 2000, replace=False):
        Vt = np.zeros((3, 3))
        for k, (a, b) in enumerate(IDX6):
            Vt[a, b] = Vt[b, a] = V[t, k]
        Vi = scaled_inv(Vt)
        obs = np.arange(starts[t], starts[t + 1])
        Wt = np.zeros((ns, 3))
        for a in obs:
            j = p.cam_ind[a]
            Wt[j * c:(j + 1) * c] += Jcs[a].T @ Jps[a]
        ref = s2 * (Vi + Vi @ Wt.T @ Sinv @ Wt @ Vi)
        worst = max(worst, _normalised_err(cp[t], ref))
    print("normalised error of 2000 tracks vs the host formula: %.2e" % worst)
    assert worst <= tol, worst
    with DeviceProblem(p, engine="generic") as prob:
        cg, pg, sg, _ = prob.covariance(x, loss=loss)
    assert abs(sg - s2) <= 1e-12 * s2
    dp = np.sqrt(np.einsum("nii->ni", cp))
    print("generic vs pattern engine: cameras %.2e, points %.2e" % (_normalised_err(cg, cc), (np.abs(pg - cp) / (dp[:, :, None] * dp[:, None, :])).max()))
    assert _normalised_err(cg, cc) <= tol
    assert (np.abs(pg - cp) / (dp[:, :, None] * dp[:, None, :])).max() <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["pattern", "generic"])
def test_covariance_leaves_the_handle_usable(built, engine):
    """solve, covariance, solve again from x0: bit-identical to the first solve and to a fresh handle's."""
    p = _scene("persp_RT_cfix2")
    x0 = initial_vars(p)
    kw = dict(want_residuals=True, loss="soft_l1")
    with DeviceProblem(p, engine=engine) as prob:
        x1, r1, i1 = prob.solve(x0, **kw)
        prob.covariance(x1, loss="soft_l1")
        x2, r2, i2 = prob.solve(x0, **kw)
    with DeviceProblem(p, engine=engine) as fresh:
        x3, r3, _ = fresh.solve(x0, **kw)
    assert np.array_equal(x1, x2) and np.array_equal(r1, r2) and i1["cost"] == i2["cost"] and i1["nfev"] == i2["nfev"]
    assert np.array_equal(x1, x3) and np.array_equal(r1, r3)


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["pattern", "generic"])
def test_covariance_error_leaves_the_handle_usable(built, engine):
    """A covariance call that returns SBA_E_NUMERIC (unfixed gauge) leaves the handle as usable as a successful one."""
    p = synth.scene_to_params(synth.make_scene(n_cam=5, n_tracks=50, p_vis=0.8, seed=31), ["R", "T"])
    x0 = initial_vars(p)
    kw = dict(want_residuals=True, loss="soft_l1")
    with DeviceProblem(p, engine=engine) as prob:
        x1, r1, i1 = prob.solve(x0, **kw)
        with pytest.raises(_lib.SbaError):
            prob.covariance(x1, loss="soft_l1")
        x2, r2, i2 = prob.solve(x0, **kw)
    assert np.array_equal(x1, x2) and np.array_equal(r1, r2) and i1["cost"] == i2["cost"] and i1["nfev"] == i2["nfev"]


# ---- checks that need no device -------------------------------------------------------------------------------------
def test_covariance_common_k_not_implemented():
    p = util.params_from_golden(util.load_ba_golden(), "persp_RTK_common")
    with pytest.raises(NotImplementedError):
        compute_covariance(p, p.params_opt.copy())


def test_covariance_without_degrees_of_freedom_raises():
    # 2 cameras x 10 tracks: 40 residuals, 12 + 30 free variables
    p = synth.scene_to_params(synth.make_scene(n_cam=2, n_tracks=10, p_vis=1.0, seed=5), ["R", "T"])
    assert degrees_of_freedom(p) <= 0
    with pytest.raises(ValueError):
        compute_covariance(p, p.params_opt.copy())


def test_covariance_has_no_cpu_fallback(built):
    """Without a CUDA device compute_covariance raises SbaError and never computes on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = synth.scene_to_params(synth.make_scene(n_cam=4, n_tracks=40, p_vis=0.8, seed=35), ["R", "T"], n_cam_fix=1)
    with pytest.raises(_lib.SbaError):
        compute_covariance(p, p.params_opt.copy())
