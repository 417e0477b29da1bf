"""
The normal equations (U, V, g, cost), the reduced camera system (S, rhs) and the posterior covariance of both engines against
oracle/block_oracle.py, a float64 restatement accumulated in long double from the per-observation blocks, at the layout edges
of the engines and at scale.

Tolerances are per entry: |dev - oracle| <= tau A, A the entry's sum of absolute terms (block_oracle's docstring).  The point
side of the device recomputes the Jacobian in registers (K R form), ~1e-9 relative away from sba_jacobian_blocks; that, not the
summation, is what limits V, g_p and S.  Measured maxima of |dev - oracle| / A over the scenes below (NVIDIA B200, 1000 W power
limit), both engines, both Schur kernels: U 6e-12, g_c 6.7e-14, cost 2.8e-16, V 1.3e-9, g_p 1.4e-9, S 2.1e-9, rhs 1.9e-10.  TAU
is about 10x that, within the ceilings 1e-10 (U, g, cost) and 1e-8.  For RPC, g is compared with sum |J| RPC_F_TOL on top of
tau A: the assembly linearises the derivative path's residual, 2e-9 px from sba_residuals' (oracle_f); beyond that its error
measures 0.
Each tolerance must also see the smallest change the bugs of interest make: removing one track (the last of a partial tile,
one at a warp boundary of the assignment, a random one), one observation, or rounding J to float32 moves some entry of U, g, S
or rhs by at least 10 tau A (`assert_teeth`), on every GPU scene and on a CPU scene.

The covariance uses the bound convention of test_gpu_covariance.py: normalised error <= max(1e-7, n eps kappa).
"""
import numpy as np
import pytest

import util
from oracle import ba_oracle, prior_oracle
from oracle.block_oracle import NormalEquations, fd_blocks
from sat_bundleadjust_b200 import synth
from sat_bundleadjust_b200.ba_priors import CameraPrior
from sat_bundleadjust_b200.solver import DeviceProblem, initial_vars, n_common_params

TAU = {"U": 6e-11, "g": 7e-13, "cost": 3e-15, "V": 1e-8, "gp": 1e-8, "S": 1e-8, "rhs": 2e-9}
REGS = (0.0, 0.37)
PT_MAX_NS, COV_SMEM_MAX_NS, CHUNK, SLICE = 132, 113, 1024, 1024
G = util.load_ba_golden()


def ratio(dev, ref, mag):
    """max |dev - ref| / mag; entries with mag == 0 (no terms, identity rows) must agree exactly"""
    dev, ref, mag = np.asarray(dev), np.asarray(ref), np.asarray(mag)
    z = mag == 0
    assert np.array_equal(dev[z], ref[z]), "entries without terms differ: %s" % np.abs(dev[z] - ref[z]).max()
    return float((np.abs(dev - ref)[~z] / mag[~z]).max()) if (~z).any() else 0.0


def check(tag, q, dev, ref, mag, slack=None):
    """|dev - ref| <= slack + TAU[q] mag (slack: what the oracle's inputs leave open, see RPC_F_TOL)"""
    if slack is not None:
        d = np.maximum(np.abs(np.asarray(dev) - ref) - slack, 0.0)
        dev, ref = d, np.zeros_like(d)
    r = ratio(dev, ref, mag)
    print("%-48s %-4s err/A %.2e  err/tau %.3f" % (tag, q, r, r / TAU[q]))
    assert r <= TAU[q], (tag, q, r)


# ---- scenes ---------------------------------------------------------------------------------------------------------------
def tile_tracks(L):
    return min(32 // L, 16)


def pattern_rows(M, sets, rng):
    """boolean visibility rows: `sets` = [(camera list, count), ...], rows shuffled"""
    rows = []
    for cams, n in sets:
        r = np.zeros((n, M), bool)
        r[:, list(cams)] = True
        rows.append(r)
    rows = np.concatenate(rows)
    return rows[rng.permutation(rows.shape[0])]


def pattern_scene(M, sets, frozen_sets=(), cam_model="perspective", seed=0):
    """make_scene whose tracks have exactly the given camera sets and counts; the rows of frozen_sets come first (frozen points)"""
    rng = np.random.default_rng(seed)
    free = pattern_rows(M, sets, rng)
    fro = pattern_rows(M, frozen_sets, rng) if frozen_sets else np.zeros((0, M), bool)
    vis = np.concatenate([fro, free])
    sc = synth.make_scene(n_cam=M, n_tracks=vis.shape[0], cam_model=cam_model, seed=seed, visibility=lambda r, n, m: vis)
    return sc, fro.shape[0]


def sets_every_length(M, Ls, obs_per_L, rng, must=()):
    """for every L: two camera sets (one holding the cameras `must`), track counts T k + 1 and T k - 1 (not multiples of T)"""
    out = []
    for L in Ls:
        T = tile_tracks(L)
        k = max(2, obs_per_L // (2 * L * T))
        a = sorted(set(must) | set(rng.choice([j for j in range(M) if j not in must], L - len(must), replace=False).tolist()))
        b = sorted(rng.choice(M, L, replace=False).tolist())
        out += [(a, T * k + 1), (b, T * k - 1)]
    return out


def layout_tracks(p, layout, narrow, rng):
    """caller's tracks at the edges of the pattern assignment: the last track of a partial last tile of a run, the tracks on
    both sides of a warp boundary that cuts a run (assembly and Schur assignments), one random track.  narrow = (units,
    warp_unit0) of the Schur pass."""
    t2o = layout["trk_new2old"]
    picks = {}
    for name, (units, wu) in (("assembly", (layout["units"], layout["warp_unit0"])), ("schur", narrow)):
        trk0, ntrk, L, mlo, mhi = units[:, 0], units[:, 1], units[:, 3], units[:, 4], units[:, 5]
        same_run = (trk0[:-1] + ntrk[:-1] == trk0[1:]) & (mlo[:-1] == mlo[1:]) & (mhi[:-1] == mhi[1:]) & (L[:-1] == L[1:])
        warp_start = np.zeros(units.shape[0], bool)
        warp_start[wu[(wu > 0) & (wu < units.shape[0])]] = True
        cut = np.nonzero(same_run & warp_start[1:])[0]             # unit u ends a warp's range, unit u + 1 continues the run
        if cut.size:
            u = cut[rng.integers(cut.size)]
            picks[name + " boundary, before"] = int(t2o[trk0[u] + ntrk[u] - 1])
            picks[name + " boundary, after"] = int(t2o[trk0[u + 1]])
        last = np.nonzero(np.r_[~same_run, True] & (ntrk % np.array([tile_tracks(x) for x in L]) != 0))[0]
        if last.size:
            u = last[rng.integers(last.size)]
            picks[name + " partial last tile"] = int(t2o[trk0[u] + ntrk[u] - 1])
    picks["random"] = int(rng.integers(p.n_pts_fix, p.n_pts))
    return picks


# ---- oracle inputs ------------------------------------------------------------------------------------------------------
RPC_F_TOL = 5e-9


def oracle_f(p, prob, x):
    """
    The residuals the oracle linearises: sba_residuals of the handle under test, opened with float64 RPC projections (the
    reference's fun rounds them to float32, ba_core.py:150; the assembly linearises the unrounded residual).  ba_oracle's
    residuals differ from the device's by up to ~1.5e-9 px (CUDA sin/cos and FMA against numpy), 3e-9 relative to a 0.5 px
    residual: through g = J^T f and the robust row scaling that would hide summation errors in g and U below ~6e-10 A.  The
    two are pinned to each other here at 1e-8 px.

    RPC: the assembly and sba_jacobian_blocks evaluate the projection on the derivative path (ecef_to_geodetic_d: latitude
    sine / cosine algebraically from the arguments of the arc tangents, 1 / cos through a reciprocal), sba_residuals on the
    value path (ecef_to_geodetic: the reference's atan2 / sin / cos round trips).  The two residuals differ by up to 1.9e-9 px
    (test_rpc_residual_paths_agree, host build; bound RPC_F_TOL = 5e-9 px).  A track's g_p sums two to four rows, so where
    its residuals are small that difference is 6e-8 of its A: the comparison of g allows sum |J| RPC_F_TOL on top of tau A.
    """
    f = prob.residuals(x)[0]
    if p.cam_model != "rpc":
        assert np.abs(f - ba_oracle.residuals(x.copy(), p)).max() < 1e-8
    return f


def make_ne(p, Jc, Jp, f, loss, prior=None, x=None, f_scale=1.0):
    xc = None if prior is None else x[: p.n_cam * p.n_params]
    return NormalEquations(Jc, Jp, f, p.cam_ind, p.pts_ind, p.n_cam, p.n_pts, p.n_cam_fix, p.n_pts_fix, loss, f_scale, prior, xc,
                           f_tol=RPC_F_TOL if p.cam_model == "rpc" else 0.0)


def prior_for(p, Jc, x, strength=1e-2):
    """a full-rank diagonal prior on every camera, mean at x, 1 / sigma^2 = strength x the squared column norm of J"""
    M, c = p.n_cam, p.n_params
    col = np.zeros((M, c))
    np.add.at(col, p.cam_ind, (Jc ** 2).sum(axis=1))
    sig = 1.0 / np.sqrt(strength * np.maximum(col, 1e-30))
    return CameraPrior.from_sigmas(x[: M * c].reshape(M, c).copy(), sig)


# ---- the sensitivity of the tolerances -------------------------------------------------------------------------------------
def sub_ne(p, Jc, Jp, f, loss, obs):
    """the oracle on a subset of the observations (whole tracks or one track minus an observation), same numbering"""
    obs = np.asarray(obs)
    f2 = f.reshape(-1, 2)[obs].ravel()
    return NormalEquations(Jc[obs], Jp[obs], f2, p.cam_ind[obs], p.pts_ind[obs], p.n_cam, p.n_pts, p.n_cam_fix, p.n_pts_fix, loss)


def _moves(ne, S, rhs, Sa, rhsa, dU, dg, dS, drhs, cameras_only=True):
    """max over U, g, S, rhs of |change| / (tau A); cameras_only: g_c only (a track's own g_p changes trivially)"""
    best = 0.0
    n = ne.M * ne.c if cameras_only else dg.size
    for d, a, q in ((dU, ne.Ua, "U"), (dg[:n], ne.ga[:n], "g"), (dS, Sa, "S"), (drhs, rhsa, "rhs")):
        m = a > 0
        if m.any():
            best = max(best, float((np.abs(d)[m] / (TAU[q] * a[m])).max()))
    return best


def assert_teeth(p, Jc, Jp, f, loss, tracks, seed=0):
    """Each of: removing one of `tracks` (name -> caller's track), removing one observation, rounding J to float32, moves some
    entry of U / g / S / rhs (reg 0) by >= 10 tau A."""
    ne = make_ne(p, Jc, Jp, f, loss)
    S, rhs, Sa, rhsa = ne.reduced_system(0.0)
    ncf = p.n_cam_fix * p.n_params
    starts = ne.starts

    def track_system(obs):
        s = sub_ne(p, Jc, Jp, f, loss, obs)
        Ss, rs, _, _ = s.reduced_system(0.0)
        Ss[np.arange(ncf), np.arange(ncf)] = 0.0          # identity rows of the frozen slots are there with or without the track
        return s, Ss, rs

    out = {}
    for name, t in tracks.items():
        obs = np.arange(starts[t], starts[t + 1])
        s, Ss, rs = track_system(obs)
        out["track " + name] = _moves(ne, S, rhs, Sa, rhsa, s.U, s.g, Ss, rs)
    rng = np.random.default_rng(seed)
    lens = np.diff(starts)
    t = int(rng.choice(np.nonzero((lens >= 3) & (np.arange(p.n_pts) >= p.n_pts_fix))[0]))
    obs = np.arange(starts[t], starts[t + 1])
    o = int(rng.choice(obs))
    s1, S1, r1 = track_system(obs)
    s0, S0, r0 = track_system(obs[obs != o])
    out["observation"] = _moves(ne, S, rhs, Sa, rhsa, s1.U - s0.U, s1.g - s0.g, S1 - S0, r1 - r0)
    n32 = make_ne(p, Jc.astype(np.float32).astype(np.float64), Jp.astype(np.float32).astype(np.float64), f, loss)
    out["J in float32"] = _moves(ne, S, rhs, Sa, rhsa, n32.U - ne.U, n32.g - ne.g, np.zeros_like(S), np.zeros_like(rhs),
                                   cameras_only=False)
    for k, v in out.items():
        print("teeth: %-32s moves an entry by %.3g tau A" % (k, v))
        assert v >= 10.0, (k, v)


# ---- CPU: the oracle against dense linear algebra ------------------------------------------------------------------------------
def dense_reference(p, J, f, loss, reg, prior=None, x=None):
    """U, V, g, S, rhs from the dense Jacobian (device layout), as test_reduced_camera_system and dense_oracle form them;
    frozen points' columns are dropped (their blocks are empty)"""
    from scipy.optimize._lsq.common import scale_for_robust_loss_function
    from scipy.optimize._lsq.least_squares import construct_loss_function
    M, c, N = p.n_cam, p.n_params, p.n_pts
    ns, k = M * c, n_common_params(p)
    if loss != "linear":
        rho = construct_loss_function(f.size, loss, 1.0)(f.copy())
        J, f = scale_for_robust_loss_function(J.copy(), f.copy(), rho)
    if prior is not None:
        C = prior_oracle.prior_factors(prior, p.n_cam_fix)
        Jpr = np.zeros((ns, J.shape[1]))
        for j in range(M):
            Jpr[j * c:(j + 1) * c, j * c:(j + 1) * c] = C[j]
        J = np.vstack([J, Jpr])
        f = np.concatenate([f, prior_oracle.prior_rows(x, p, prior)])
    used = np.ones(ns, bool)
    used[: p.n_cam_fix * c] = False
    if k:
        for j in range(1, M):
            J[:, c - k: c] += J[:, j * c + c - k: (j + 1) * c]
            J[:, j * c + c - k: (j + 1) * c] = 0.0
            used[j * c + c - k: (j + 1) * c] = False
    Hu, g = J.T @ J, J.T @ f
    d2 = np.diag(Hu).copy()
    d2[d2 == 0.0] = 1.0
    H = Hu + reg * np.diag(d2)
    keep = np.r_[np.nonzero(used)[0], ns + 3 * p.n_pts_fix + np.arange(3 * (N - p.n_pts_fix))]
    u = np.nonzero(used)[0]
    Hk = H[np.ix_(keep, keep)]
    nu = u.size
    X = np.linalg.solve(Hk[nu:, nu:], np.column_stack([Hk[nu:, :nu], g[keep][nu:]]))
    S = np.eye(ns)
    S[np.ix_(u, u)] = Hk[:nu, :nu] - Hk[:nu, nu:] @ X[:, :nu]
    rhs = np.zeros(ns)
    rhs[u] = -(g[u] - Hk[:nu, nu:] @ X[:, nu])
    return Hu, g, S, rhs


GOLDEN_CASES = [("persp_RT_fix", "linear", False), ("persp_RT_fix", "soft_l1", True), ("affine_RT_softl1", "soft_l1", False),
                ("persp_R", "cauchy", False), ("persp_RTK_common", "linear", False), ("affine_RTK", "soft_l1", True)]


@pytest.mark.parametrize("reg", REGS)
@pytest.mark.parametrize("name,loss,with_prior", GOLDEN_CASES)
def test_oracle_matches_dense_formulas(name, loss, with_prior, reg):
    """Golden scenes, blocks from ba_oracle.dense_jacobian_fd: the block oracle equals the dense formulas to 1e-12 (reg 0 and > 0,
    robust losses, a prior, COMMON_K, frozen cameras (persp_RT_fix: 2) and points (40))."""
    if loss == "cauchy" and reg == 0.0:
        # cauchy zeroes the Jacobian rows of outlying residuals: a point seen only through such rows has a singular block unless
        # it is damped, and there is nothing well defined to compare
        pytest.skip("undamped point blocks can be singular under cauchy")
    p = util.params_from_golden(G, name)
    x = initial_vars(p)
    M, c, k = p.n_cam, p.n_params, n_common_params(p)
    Jd = ba_oracle.dense_jacobian_fd(x.copy(), p, rel_step=1e-7)
    Jd[:, : p.n_cam_fix * c] = 0.0           # frozen cameras: the residual overwrites their slots (0 / 0 above)
    if k:                                   # caller's layout [K | cameras | points] -> c slots per camera
        ncs = c - k
        J = np.zeros((Jd.shape[0], M * c + 3 * p.n_pts))
        for j in range(M):
            J[:, j * c: j * c + ncs] = Jd[:, k + j * ncs: k + (j + 1) * ncs]
        rows = np.repeat(p.cam_ind, 2)
        for j in range(M):
            J[rows == j, j * c + ncs: (j + 1) * c] = Jd[rows == j, :k]
        J[:, M * c:] = Jd[:, k + M * ncs:]
        xd = np.zeros(M * c + 3 * p.n_pts)
    else:
        J, xd = Jd, x
    Kobs = p.pts_ind.size
    rows = np.arange(2 * Kobs).reshape(Kobs, 2)
    Jc = np.stack([J[rows[:, r][:, None], p.cam_ind[:, None] * c + np.arange(c)] for r in range(2)], axis=1)
    Jp = np.stack([J[rows[:, r][:, None], M * c + p.pts_ind[:, None] * 3 + np.arange(3)] for r in range(2)], axis=1)
    f = ba_oracle.residuals(x.copy(), p)
    prior = prior_for(p, Jc, xd) if with_prior else None
    ne = make_ne(p, Jc, Jp, f, loss, prior, xd)
    Hu, g, S, rhs = dense_reference(p, J, f, loss, reg, prior, xd)
    ns = M * c
    cost = ba_oracle.robust_cost(f, loss, 1.0) if prior is None else prior_oracle.augmented_cost(x, p, prior, loss)
    assert abs(ne.cost - cost) <= 1e-12 * cost
    if not k:
        Ud = np.array([Hu[j * c:(j + 1) * c, j * c:(j + 1) * c] for j in range(M)])
        Vd = np.array([[Hu[ns + 3 * i + a, ns + 3 * i + b] for a, b in ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))] for i in range(p.n_pts)])
        assert np.abs(ne.U - Ud).max() <= 1e-12 * np.abs(Ud).max()
        assert np.abs(ne.V - Vd).max() <= 1e-12 * np.abs(Vd).max()
        assert np.abs(ne.g - g).max() <= 1e-12 * np.abs(g).max()
    So, ro, Sa, ra = ne.reduced_system(reg, k)
    assert np.abs(So - S).max() <= 1e-12 * np.abs(S).max(), np.abs(So - S).max() / np.abs(S).max()
    assert np.abs(ro - rhs).max() <= 1e-12 * np.abs(rhs).max(), np.abs(ro - rhs).max() / np.abs(rhs).max()
    assert np.all(np.abs(So) <= Sa + (Sa == 0)) and np.all(np.abs(ro) <= ra + (ra == 0))


def test_teeth_on_a_cpu_scene(built):
    """The tolerances see one track at the edges of the pattern assignment, one observation and float32 Jacobians on a 10-view,
    5e4-observation scene (blocks from central differences, no device)."""
    sc = synth.make_scene(n_cam=10, n_tracks=10000, p_vis=0.5, seed=4)
    p = synth.SparseParams(sc, ["R", "T"], n_cam_fix=2, n_pts_fix=50)
    x = initial_vars(p)
    Jc, Jp = fd_blocks(x, p, lambda v, q: ba_oracle.residuals(v.copy(), q))
    f = ba_oracle.residuals(x.copy(), p)
    lay = util.pattern_layout(p.cam_ind, p.pts_ind, p.n_cam, p.n_pts, p.n_pts_fix)
    narrow = util.pattern_assignment(p.cam_ind, p.pts_ind, p.n_cam, p.n_pts, p.n_pts_fix, p.n_params, 2, 12)
    picks = layout_tracks(p, lay, narrow, np.random.default_rng(0))
    assert any("boundary" in k for k in picks) and any("partial" in k for k in picks)
    for loss in ("linear", "soft_l1"):
        assert_teeth(p, Jc, Jp, f, loss, picks)


# ---- GPU: both engines against the oracle ---------------------------------------------------------------------------------------
def compare_blocks(tag, p, x, engine, losses, regs, prior=None, schur=("fma", "mma"), monkeypatch=None, teeth=True,
                   normal=True, f_scale=1.0):
    """normal_blocks (U, V, g, cost) and reduced_system at each reg of the handle(s) against one oracle per loss; the pattern
    engine with each Schur kernel.  Returns the oracle inputs (Jc, Jp, f)."""
    variants = schur if engine == "pattern" else (None,)
    ne_cache = {}
    for v in variants:
        if v is not None:
            monkeypatch.setenv("SBA_PT_SCHUR", v)
        with DeviceProblem(p, engine=engine, cam_prior=prior, rpc_float32=False) as prob:
            assert prob.engine == engine
            if not ne_cache:
                Jc, Jp = prob.jacobian_blocks(x)
                f = oracle_f(p, prob, x)
                if teeth:
                    lay = util.pattern_layout(p.cam_ind, p.pts_ind, p.n_cam, p.n_pts, p.n_pts_fix)
                    rng = np.random.default_rng(1)
                    if lay is not None:
                        narrow = util.pattern_assignment(p.cam_ind, p.pts_ind, p.n_cam, p.n_pts, p.n_pts_fix, p.n_params, 2, 12)
                        picks = layout_tracks(p, lay, narrow, rng)
                        assert {"assembly boundary, before", "schur boundary, before"} <= set(picks), picks
                        assert any("partial" in k for k in picks), picks
                    else:
                        picks = {"longest": int(np.argmax(np.bincount(p.pts_ind))), "random": int(rng.integers(p.n_pts_fix, p.n_pts))}
                    assert_teeth(p, Jc, Jp, f, losses[0], picks)
                for loss in losses:
                    ne_cache[loss] = make_ne(p, Jc, Jp, f, loss, prior, x, f_scale)
            for loss in losses:
                ne = ne_cache[loss]
                t = "%s %s %s %s" % (tag, engine, v or "", loss)
                if normal and not n_common_params(p):
                    U, V, g = prob.normal_blocks(x, loss, f_scale)
                    check(t, "U", U, ne.U, ne.Ua)
                    check(t, "V", V, ne.V, ne.Va)
                    nsc = p.n_cam * p.n_params          # g_p is formed from the point side's own Jacobian, like V
                    check(t, "g", g[:nsc], ne.g[:nsc], ne.ga[:nsc], ne.gt[:nsc])
                    check(t, "gp", g[nsc:], ne.g[nsc:], ne.ga[nsc:], ne.gt[nsc:])
                    if prior is None:
                        _, cost = prob.residuals(x, loss, f_scale)
                        check(t, "cost", cost, ne.cost, ne.cost_a)
                for reg in regs:
                    S, rhs = prob.reduced_system(x, loss, f_scale, reg)
                    So, ro, Sa, ra = ne.reduced_system(reg, n_common_params(p))
                    check(t + " reg %g" % reg, "S", S, So, Sa)
                    check(t + " reg %g" % reg, "rhs", rhs, ro, ra)
    return ne_cache


def runs_of(p):
    """(L, camera mask) of every free track with observations"""
    lens = np.bincount(p.pts_ind, minlength=p.n_pts)
    mask = np.zeros(p.n_pts, dtype=np.uint64)
    np.bitwise_or.at(mask, p.pts_ind, (np.uint64(1) << p.cam_ind.astype(np.uint64)))
    return lens, mask


@pytest.mark.gpu
def test_pattern_every_tile_shape(built, monkeypatch):
    """P1: perspective R+T (c 6), 22 views (ns 132 = PT_MAX_NS), cameras 0, 1 frozen, frozen points; runs of every length 2..22
    with track counts T k +- 1, masks holding cameras 0 and 21, ~3e5 observations so that every warp of 148 x 16 holds work and
    runs are cut between warps; Schur passes 1 (L < 8), 2 (L 8) and 8 (L 22)."""
    rng = np.random.default_rng(11)
    M = 22
    sets = sets_every_length(M, range(2, 23), 14000, rng, must=(0, 21))
    sc, nfix = pattern_scene(M, sets, frozen_sets=[([0, 3, 21], 40), (list(range(4, 17)), 31)], seed=11)
    p = synth.SparseParams(sc, ["R", "T"], n_cam_fix=2, n_pts_fix=nfix)
    lens, mask = runs_of(p)
    free = np.arange(p.n_pts) >= nfix
    assert p.n_cam * p.n_params == PT_MAX_NS and 2.5e5 < p.n_obs < 4e5
    assert set(lens[free].tolist()) == set(range(2, 23))
    for L in (3, 10, 11, 16):                              # T = 10, 3, 2, 2 (T = 1 from L = 17 on)
        for m in np.unique(mask[free & (lens == L)]):
            assert int((mask[free] == m).sum()) % tile_tracks(L) != 0
    assert np.any(mask[free] & np.uint64(1)) and np.any(mask[free] & np.uint64(1 << 21))
    units, _ = util.pattern_assignment(p.cam_ind, p.pts_ind, p.n_cam, p.n_pts, p.n_pts_fix, p.n_params, 2, 12)
    passes = np.diff(units[:, 7])                          # Schur records = passes over each unit (but the last)
    for L, n in ((2, 1), (7, 1), (8, 2), (22, 8)):
        assert set(passes[units[:-1, 3] == L].tolist()) == {n}, (L, set(passes[units[:-1, 3] == L].tolist()))
    lay = util.pattern_layout(p.cam_ind, p.pts_ind, p.n_cam, p.n_pts, p.n_pts_fix)
    wu = lay["warp_unit0"]
    assert np.all(np.diff(wu) >= 1)                       # every warp of the assembly holds work
    x = initial_vars(p)
    compare_blocks("P1", p, x, "pattern", ("linear", "soft_l1"), REGS, monkeypatch=monkeypatch)


@pytest.mark.gpu
def test_pattern_cameras_above_bit_31(built, monkeypatch):
    """P2: perspective R (c 3), 44 views (ns 132): masks only above bit 31, straddling bits 31 / 32, holding camera 43; L up to 32
    (full warps, 9 DFMA passes); cauchy at reg 0.37."""
    rng = np.random.default_rng(12)
    M = 44
    sets = []
    for L in range(2, 13):
        sets.append((list(range(44 - L, 44)), 16 * tile_tracks(L) + 1))                       # bits 32..43 only, camera 43
        sets.append((sorted(rng.choice(np.arange(32, 44), L, replace=False).tolist()), 16 * tile_tracks(L) - 1))
    for L in (2, 5, 9, 16, 24, 31, 32):
        lo = min(32 - (L + 1) // 2, M - L)
        sets.append((list(range(lo, lo + L)), 40 * tile_tracks(L) + 1))                       # straddling 31 / 32
        sets.append((sorted(set([43]) | set(rng.choice(43, L - 1, replace=False).tolist())), 40 * tile_tracks(L) - 1))
    sc, _ = pattern_scene(M, sets, seed=12)
    p = synth.SparseParams(sc, ["R"], n_cam_fix=1)
    lens, mask = runs_of(p)
    hi = (mask >> np.uint64(32)).astype(np.int64)
    lo = (mask & np.uint64(0xffffffff)).astype(np.int64)
    assert p.n_cam * p.n_params == PT_MAX_NS and lens.max() == 32
    assert np.any((lo == 0) & (hi != 0)) and np.any((lo >> 31 & 1) & (hi & 1)) and np.any(hi >> 11 & 1)
    units, _ = util.pattern_assignment(p.cam_ind, p.pts_ind, p.n_cam, p.n_pts, p.n_pts_fix, p.n_params, 2, 12)
    assert set(np.diff(units[:, 7])[units[:-1, 3] == 32].tolist()) == {9}     # 9 DFMA passes over the units of L = 32
    assert np.any(units[:, 4] == 0) and np.any(units[:, 5] >> 11 & 1)         # mask_lo empty / camera 43 in the units
    x = initial_vars(p)
    compare_blocks("P2", p, x, "pattern", ("linear", "soft_l1"), REGS, monkeypatch=monkeypatch)
    compare_blocks("P2", p, x, "pattern", ("cauchy",), (0.37,), schur=("fma",), monkeypatch=monkeypatch, teeth=False)


@pytest.mark.gpu
@pytest.mark.parametrize("corr,M", [(("R", "T"), 26), (("R",), 30)])
def test_pattern_affine(built, monkeypatch, corr, M):
    """P3: affine R+T (c 5, 26 views, ns 130) and affine R (c 3)."""
    rng = np.random.default_rng(13 + M)
    sets = sets_every_length(M, range(2, min(M, 24) + 1, 2), 6000, rng, must=(0, M - 1))
    sc, nfix = pattern_scene(M, sets, frozen_sets=[([1, 2, 5], 20)], cam_model="affine", seed=13)
    p = synth.SparseParams(sc, list(corr), n_cam_fix=2, n_pts_fix=nfix)
    assert p.n_params == (5 if corr == ("R", "T") else 3) and p.n_cam * p.n_params == (130 if corr == ("R", "T") else 90)
    x = initial_vars(p)
    compare_blocks("P3 affine %s" % "".join(corr), p, x, "pattern", ("linear", "soft_l1"), REGS, monkeypatch=monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("corr", [("R",), ("R", "T")])
def test_pattern_rpc(built, monkeypatch, corr):
    """P4: RPC R and R+T on the 4 golden cameras, ~2e5 observations (g with the residual paths' difference, see oracle_f)."""
    R = util.load_rpc_golden()
    sc = synth.make_rpc_scene(R["rpc_cams"], R["rpcba/camera_centers"], n_tracks=62000, p_vis=0.8, seed=14)
    p = synth.SparseParams(sc, list(corr), n_cam_fix=1, n_pts_fix=30)
    assert p.n_obs > 1.8e5 and p.n_params == 3 * len(corr) and p.n_cam == 4
    x = initial_vars(p)
    compare_blocks("P4 rpc %s" % "".join(corr), p, x, "pattern", ("linear", "soft_l1"), REGS, monkeypatch=monkeypatch)


@pytest.mark.gpu
def test_pattern_bench_geometry_with_prior(built, monkeypatch):
    """P5: the 1m bench scene (10 views, 1e6 observations), soft_l1; without a prior at reg 0, with a full-rank prior at reg 0.37
    (the prior's lane-0 write in k_pt_reduce_assemble)."""
    sc = synth.make_scene(n_cam=10, n_tracks=200000, p_vis=0.5, seed=0)
    p = synth.SparseParams(sc, ["R", "T"])
    assert p.n_obs > 9.5e5
    x = initial_vars(p)
    compare_blocks("P5", p, x, "pattern", ("soft_l1",), (0.0,), monkeypatch=monkeypatch)
    with DeviceProblem(p) as prob:
        Jc, _ = prob.jacobian_blocks(x)
    prior = prior_for(p, Jc, x + 1e-3)
    compare_blocks("P5 prior", p, x, "pattern", ("soft_l1",), (0.37,), prior=prior, schur=("fma",), monkeypatch=monkeypatch,
                   teeth=False)


@pytest.mark.gpu
def test_generic_long_tracks_chunks_and_slices(built):
    """G1: generic engine, 66 views (the longest tracks need 65), c 6: tracks of exactly 32, 33, 64 and 65 observations, cameras
    with more than CHUNK = 1024 observations, one camera pair sharing more than SLICE = 1024 tracks, frozen cameras and points."""
    rng = np.random.default_rng(15)
    M = 66
    sets = [(sorted(rng.choice(M, L, replace=False).tolist()), 6) for L in (32, 33, 64, 65)]
    sets += [([2, 3] + sorted(rng.choice(np.arange(4, M), 2, replace=False).tolist()), 1) for _ in range(1300)]
    sets += [(sorted(rng.choice(M, int(rng.integers(2, 9)), replace=False).tolist()), 1) for _ in range(6000)]
    sc, nfix = pattern_scene(M, sets, frozen_sets=[([0, 2, 3], 30)], seed=15)
    p = synth.SparseParams(sc, ["R", "T"], n_cam_fix=2, n_pts_fix=nfix)
    lens = np.bincount(p.pts_ind)
    assert {32, 33, 64, 65} <= set(lens.tolist())
    per_cam = np.bincount(p.cam_ind, minlength=M)
    assert (per_cam + CHUNK - 1).max() // CHUNK >= 2
    both = np.zeros(p.n_pts, int)
    np.add.at(both, p.pts_ind, (p.cam_ind == 2) | (p.cam_ind == 3))
    assert (both == 2).sum() > SLICE
    x = initial_vars(p)
    compare_blocks("G1", p, x, "generic", ("linear", "soft_l1"), REGS)


@pytest.mark.gpu
@pytest.mark.parametrize("model,corr", [("perspective", ["R", "T", "K"]), ("affine", ["R", "T", "K"]),
                                        ("perspective", ["R", "T", "K", "COMMON_K"]), ("affine", ["R", "T", "K", "COMMON_K"])])
def test_generic_calibration(built, model, corr):
    """G2: generic engine, per-camera K (perspective c 11, affine c 8) and COMMON_K, >= 5e4 observations each."""
    sc = synth.make_scene(n_cam=8, n_tracks=12000, p_vis=0.7, cam_model=model, seed=16)
    p = synth.scene_to_params(sc, corr)
    assert p.pts_ind.size >= 5e4 and p.n_params == (11 if model == "perspective" else 8) and p.n_cam == 8
    x = repaired_x0(p)
    compare_blocks("G2 %s %s" % (model, "+".join(corr)), p, x, "generic", ("linear", "soft_l1"), REGS)


def repaired_x0(p):
    """initial_vars with the calibration started from the cameras' own (the reference's packing mis-initialises it)"""
    nK, c, M = (3 if p.cam_model == "affine" else 5), p.n_params, p.n_cam
    x = initial_vars(p)
    if n_common_params(p):
        x[:nK] = p.cam_params[0, -nK:]
    elif "K" in p.cam_params_to_optimize:
        x[: M * c].reshape(M, c)[:, c - nK:] = p.cam_params[:, -nK:]
    return x


# ---- GPU: covariance --------------------------------------------------------------------------------------------------------
def compare_covariance(tag, p, x, engine, loss="soft_l1", sigma2=0.25, points=None, solver=None):
    with DeviceProblem(p, engine=engine, solver=solver) as prob:
        assert prob.engine == engine and (solver is None or prob.solver == solver)
        Jc, Jp = prob.jacobian_blocks(x)
        prior = prior_for(p, Jc, x)
        prob.set_camera_prior(prior)
        f = oracle_f(p, prob, x)
        cc, cp, s2, ratio_ = prob.covariance(x, loss=loss, sigma2=sigma2)
        eng = prob.engine
    ne = make_ne(p, Jc, Jp, f, loss, prior, x)
    cc_o, cp_o, kappa = ne.covariance(sigma2, points)
    pts = np.arange(p.n_pts) if points is None else np.asarray(points)
    tol = util.cond_tol(1e-7, kappa, (p.n_cam - p.n_cam_fix) * p.n_params)
    ec = util.normalised_err(cc, cc_o)
    ep = max(util.normalised_err(cp[t], cp_o[i]) for i, t in enumerate(pts))
    print("%s (%s): covariance normalised error cameras %.2e, points %.2e, bound %.1e (kappa %.2e, min pivot ratio %.2e)"
          % (tag, eng, ec, ep, tol, kappa, ratio_))
    assert ec <= tol and ep <= tol
    assert not cp[: p.n_pts_fix].any()


@pytest.mark.gpu
@pytest.mark.parametrize("model,M", [("perspective", 10), ("perspective", 11), ("affine", 14), ("affine", 15)])
def test_covariance_calibration_smem_sides(built, model, M):
    """C1: per-camera K on both sides of the point pass's shared-memory limit (COV_SMEM_MAX: ns <= 113): c 11 at 10 / 11 views
    (ns 110 / 121), c 8 at 14 / 15 views (ns 112 / 120); the gauge fixed by a full-rank prior on every camera."""
    sc = synth.make_scene(n_cam=M, n_tracks=3000, p_vis=0.5, cam_model=model, seed=17 + M)
    p = synth.scene_to_params(sc, ["R", "T", "K"], n_pts_fix=5)
    ns = p.n_cam * p.n_params
    assert (ns <= COV_SMEM_MAX_NS) == (M in (10, 14)) and ns in (110, 121, 112, 120)
    compare_covariance("C1 %s M %d ns %d" % (model, M, ns), p, repaired_x0(p), "generic")


@pytest.mark.gpu
@pytest.mark.parametrize("model,M", [("affine", 40), ("perspective", 36)])
def test_covariance_calibration_long_tracks(built, model, M):
    """C1b: per-camera K with tracks of more than 32 observations (k_cov_long_tracks at c 8 / 11)."""
    sc = synth.make_scene(n_cam=M, n_tracks=300, p_vis=0.95, cam_model=model, seed=18)
    p = synth.scene_to_params(sc, ["R", "T", "K"], n_pts_fix=3)
    assert np.bincount(p.pts_ind).max() > 32
    assert p.n_params == (11 if model == "perspective" else 8)
    compare_covariance("C1b %s M %d" % (model, M), p, repaired_x0(p), "generic")


@pytest.mark.gpu
def test_covariance_largest_dense_size(built):
    """C2: the largest dense size, ns = 4096 (affine R+T+K, c 8, 512 views, dense solver): k_cov_inverse far above ns = 270.  Every
    camera entry and a seeded sample of 2000 points against the oracle."""
    sc = synth.make_scene_sparse(n_cam=512, n_tracks=20000, p_vis=0.012, cam_model="affine", seed=19)
    p = synth.SparseParams(sc, ["R", "T"], n_pts_fix=4)
    p.cam_params_to_optimize = ["R", "T", "K"]              # SparseParams packs R / R+T: extend it to the calibration here
    p.n_params = p.cam_params.shape[1]
    p.params_opt = np.hstack((p.cam_params.ravel(), p.pts3d.astype(np.float64).ravel()))
    assert p.n_params == 8 and p.n_cam * p.n_params == 4096 and np.bincount(p.cam_ind, minlength=512).min() > 0
    pts = np.random.default_rng(20).choice(p.n_pts, 2000, replace=False)
    compare_covariance("C2 affine M 512 ns 4096", p, initial_vars(p), "generic", points=pts, solver="dense")


def test_rpc_residual_paths_agree(built):
    """The RPC projection on the derivative path (ecef_to_geodetic_d, used by the assembly and sba_jacobian_blocks) and on the
    value path (ecef_to_geodetic, sba_residuals) agree to RPC_F_TOL / 2 (host build of csrc/sba_models.cuh; measured 1.9e-9 px
    over 400 golden ground points and a shifted, rotated camera)."""
    import ctypes
    import os
    from oracle import rpc_oracle
    from sat_bundleadjust_b200 import _lib
    lib = ctypes.CDLL(os.path.join(util.HERE, "host_harness", "libmodel_harness.so"))
    P = _lib.dptr
    R = util.load_rpc_golden()
    lla = R["lonlatalt"][:400]
    X = np.stack(rpc_oracle.latlon_to_ecef(lla[:, 1], lla[:, 0], lla[:, 2]), axis=1)
    worst = 0.0
    for tab in (R["rpc_a"][:90], R["rpc_cams"][1]):
        tab = np.ascontiguousarray(tab, dtype=np.float64)
        for v in (np.r_[0.0, 0.0, 0.0, 0.0, 0.0, 0.0, X.mean(0)], np.r_[2e-6, -1e-6, 3e-6, 0.5, -0.3, 0.2, X.mean(0)]):
            rec = np.zeros(16)
            rec[0:6] = [np.cos(v[0]), np.sin(v[0]), np.cos(v[1]), np.sin(v[1]), np.cos(v[2]), np.sin(v[2])]
            rec[6:9], rec[9:12] = v[3:6], v[6:9]
            for x in X:
                x = np.ascontiguousarray(x)
                uv, ud, Jc, Jp = np.zeros(2), np.zeros(2), np.zeros(18), np.zeros(6)
                lib.hh_project(2, P(rec), P(tab), P(x), P(uv))
                assert lib.hh_full_side(2, 6, P(rec), P(tab), P(x), P(ud), P(Jc), P(Jp)) == 0
                worst = max(worst, float(np.abs(uv - ud).max()))
    print("RPC residual, derivative path vs value path: %.2e px" % worst)
    assert worst <= RPC_F_TOL / 2
