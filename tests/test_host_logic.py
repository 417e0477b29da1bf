"""
CPU tests of the host-side mirror of the reference interface and of the C-ABI library's load/exports.
No compute call is made on the library here (there is no GPU in the build container).
"""
import ctypes
import os

import numpy as np
import pytest

import util
from oracle import ba_oracle
from oracle.ref_loader import load_reference, reference_available
from sat_bundleadjust_b200 import _lib, ba_core, ba_params, ba_rotate, cam_utils, geo_utils, synth
from sat_bundleadjust_b200.solver import DeviceProblem, initial_vars

G = util.load_ba_golden()
CASES = [str(s) for s in G["cases"]]


@pytest.mark.parametrize("name", CASES)
def test_packing_bit_exact_vs_golden(name):
    """track -> observation layout, camera vectors and params_opt equal the reference's, bit for bit."""
    p = util.params_from_golden(G, name)
    pre = name + "/"
    for k in ["pts_ind", "cam_ind", "pts2d", "params_opt", "cam_params", "pts2d_w"]:
        a, b = getattr(p, k), G[pre + "ref_" + k]
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), k
    assert np.all(np.diff(p.pts_ind) >= 0)


@pytest.mark.parametrize("name", CASES)
def test_build_jacobian_sparsity_bit_exact(name):
    p = util.params_from_golden(G, name)
    pre = name + "/"
    A = ba_core.build_jacobian_sparsity(p).tocsr()
    A.sort_indices()
    assert tuple(A.shape) == tuple(G[pre + "ref_sparsity_shape"])
    assert np.array_equal(A.indptr, G[pre + "ref_sparsity_indptr"])
    assert np.array_equal(A.indices, G[pre + "ref_sparsity_indices"])
    assert A.dtype == np.dtype(int)


@pytest.mark.skipif(not reference_available(), reason="reference tree only exists in the build container")
@pytest.mark.parametrize("name", CASES)
def test_jacobian_sparsity_is_the_reference_lil_matrix(name):
    """Same type, dtype and row / data lists as the lil_matrix the unmodified reference builds (ba_core.py:186-219)."""
    ref = load_reference()
    p = util.params_from_golden(G, name)
    A, B = ba_core.build_jacobian_sparsity(p), ref.ba_core.build_jacobian_sparsity(p)
    assert type(A) is type(B) and A.shape == B.shape and A.dtype == B.dtype
    assert all(a == b for a, b in zip(A.rows, B.rows)) and all(a == b for a, b in zip(A.data, B.data))
    A[0, A.shape[1] - 1] = 1                      # still a working LIL matrix
    assert A.nnz == B.nnz + 1


def test_get_vars_ready_for_fun_and_reconstruct():
    p = util.params_from_golden(G, "persp_RT_fix")
    v = p.params_opt.copy()
    v[:12] += 1.0
    pts, cams = p.get_vars_ready_for_fun(v)
    o_pts, o_cams = ba_oracle.unpack_variables(p.params_opt.copy() + 0.0, p)
    assert np.array_equal(cams[: p.n_cam_fix], p.cam_params[: p.n_cam_fix])      # frozen cameras restored
    assert np.array_equal(v[: p.n_cam_fix * p.n_params].reshape(p.n_cam_fix, -1), p.cam_params[: p.n_cam_fix, : p.n_params])
    assert np.array_equal(pts, o_pts)
    x0 = initial_vars(p)
    assert np.array_equal(x0, p.params_opt) or p.n_cam_fix > 0
    pts3d, cameras = p.reconstruct_vars(p.params_opt.copy(), p.pts3d.copy(), list(p.cameras))
    assert pts3d.shape == p.pts3d.shape and len(cameras) == p.n_cam
    for P0, P1 in zip(p.cameras, cameras):
        assert np.allclose(P0, P1, rtol=1e-9, atol=1e-9 * np.abs(P0).max())


def test_empty_and_ragged_inputs():
    C = np.full((4, 5), np.nan)
    cams = [np.eye(3, 4), np.eye(3, 4)]
    with pytest.raises(ValueError):      # same exception type as the reference (np.vstack of nothing)
        ba_params.BundleAdjustmentParameters(C, np.zeros((5, 3)), cams, "perspective", [], [np.zeros(3)] * 2,
                                             {"reduce": False, "verbose": False})
    # ragged tracks: lengths 1..M are all packed, order is point-major
    sc = synth.make_scene(n_cam=7, n_tracks=60, p_vis=0.4, seed=3, min_obs=1)
    p = synth.scene_to_params(sc, ["R"])
    assert p.n_obs == sc.n_obs and np.array_equal(p.pts_ind, sc.pts_ind) and np.array_equal(p.cam_ind, sc.cam_ind)


def test_camera_utils_round_trips():
    """Same checks as the reference's tests/test_functions.py:19-63, on satellite-scale matrices."""
    sc = synth.make_scene(n_cam=2, n_tracks=10, p_vis=1.0, seed=1)
    P = sc.cameras[0]
    K, R, vecT, oC = cam_utils.decompose_perspective_camera(P)
    P2 = cam_utils.compose_perspective_camera(K, R, oC)
    assert np.allclose(P, P2 / P2[2, 3])
    A = synth.affine_expansion(P, sc.pts3d_true[0])
    K, R, vecT = cam_utils.decompose_affine_camera(A)
    assert np.allclose(A, cam_utils.compose_affine_camera(K, R, vecT))
    ang = ba_rotate.euler_angles_from_R(R)
    assert np.allclose(R, ba_rotate.euler_angles_to_R(*ang))
    lat, lon, alt = geo_utils.ecef_to_latlon_custom(*geo_utils.latlon_to_ecef_custom(11.0, -72.7, 3500.0))
    assert abs(lat - 11.0) < 1e-9 and abs(lon + 72.7) < 1e-9 and abs(alt - 3500.0) < 1e-3


@pytest.mark.skipif(not reference_available(), reason="reference tree only exists in the build container")
def test_packing_against_live_reference_with_reduce():
    ref = load_reference()
    sc = synth.make_scene(n_cam=6, n_tracks=500, p_vis=0.3, cam_model="perspective", seed=2)
    d = {"correction_params": ["R", "T"], "n_cam_fix": 2, "n_pts_fix": 50, "reduce": True, "verbose": False,
         "ref_cam_weight": 3.0}
    args = (sc.correspondence_matrix(), sc.pts3d_init, list(sc.cameras_init), "perspective", [(0, 1), (1, 2), (4, 5)],
            list(sc.camera_centers), d)
    p, q = ba_params.BundleAdjustmentParameters(*args), ref.ba_params.BundleAdjustmentParameters(*args)
    for k in ["pts_ind", "cam_ind", "pts2d", "params_opt", "cam_params", "pts2d_w", "C", "pts3d", "pts_prev_indices",
              "cam_prev_indices"]:
        assert np.array_equal(getattr(p, k), getattr(q, k), equal_nan=True), k
    assert (p.n_cam_fix, p.n_pts_fix, p.n_cam_opt, p.n_pts_opt) == (q.n_cam_fix, q.n_pts_fix, q.n_cam_opt, q.n_pts_opt)
    assert p.pairs_to_triangulate == q.pairs_to_triangulate


def test_reprojection_error_and_config():
    r = np.array([3.0, 4.0, 0.0, -2.0])
    assert np.allclose(ba_core.compute_reprojection_error(r), [5.0, 2.0])
    assert np.allclose(ba_core.compute_reprojection_error(r, np.array([2.0, 1.0])), [2.5, 2.0])
    assert ba_core.init_optimization_config(None) == {"loss": "linear", "ftol": 1e-4, "xtol": 1e-10, "f_scale": 1.0,
                                                      "max_iter": 300, "verbose": 1}
    assert ba_core.init_optimization_config({"loss": "soft_l1", "bogus": 1})["loss"] == "soft_l1"
    err = np.array([1.0, 3.0, 5.0])
    assert np.allclose(ba_core.compute_mean_reprojection_error_per_track(err, np.array([0, 0, 1]), np.array([0, 1, 0])), [2.0, 5.0])


# ---------------------------------------------------------------------------------------------------
# the C-ABI library: loads, exports everything the header declares, fails loudly without a GPU
# ---------------------------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol(built):
    import re
    lib = _lib.load()
    header = open(os.path.join(os.path.dirname(util.HERE), "include", "sba_b200.h")).read()
    declared = set(re.findall(r"\b(sba_[a-z0-9_]+|stereo_corresp_to_lonlatalt)\s*\(", header))
    declared -= {"sba_allreduce_fn"}
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    for s in declared:
        assert hasattr(lib, s), s
    assert lib.sba_version() >= 100


def test_tr2d_matches_scipy(built):
    from scipy.optimize._lsq.common import solve_trust_region_2d
    lib = _lib.load()
    rng = np.random.default_rng(0)
    for t in range(3000):
        A = rng.standard_normal((2, 2))
        B = A @ A.T if t % 2 == 0 else A + A.T
        g = rng.standard_normal(2) * 10 ** rng.uniform(-3, 3)
        D = 10 ** rng.uniform(-3, 3)
        p0, newton0 = solve_trust_region_2d(B, g, D)
        p1 = np.zeros(2)
        newton1 = lib.sba_tr2d(_lib.dptr(np.ascontiguousarray(B)), _lib.dptr(g), D, _lib.dptr(p1))
        q = lambda p: 0.5 * p @ B @ p + g @ p
        assert bool(newton1) == bool(newton0)
        assert q(p1) <= q(p0) + 1e-9 * (abs(q(p0)) + 1e-12)
        assert np.linalg.norm(p1) <= D * (1 + 1e-12)


def _scipy_tr_outcome(cost, cost_new, predicted, step_h_norm, step_norm, x_norm, Delta, ftol, xtol):
    """One trial point of scipy's trf_no_bounds inner loop (trf.py:511-560): (next Delta, termination code, accepted)."""
    from scipy.optimize._lsq.common import check_termination, update_tr_radius
    if not np.isfinite(cost_new):
        return 0.25 * step_h_norm, None, False
    actual = cost - cost_new
    Delta_new, ratio = update_tr_radius(Delta, actual, predicted, step_h_norm, step_h_norm > 0.95 * Delta)
    term = check_termination(actual, cost, step_norm, x_norm, ratio, ftol, xtol)
    return (Delta if term is not None else Delta_new), term, actual > 0


def _tr_outcome_cases():
    rng = np.random.default_rng(0)
    cases = []
    for _ in range(4000):
        cost = 10 ** rng.uniform(-3, 3)
        predicted = cost * 10 ** rng.uniform(-8, 0) * rng.choice([1.0, 1.0, 1.0, -1.0, 0.0])
        ratio = rng.choice([rng.uniform(-1.0, 2.0), 0.25, 0.75, 1.0])
        actual = ratio * predicted if predicted != 0.0 else cost * rng.choice([0.0, 1e-3, -1e-3])
        Delta = 10 ** rng.uniform(-3, 3)
        step_h = Delta * rng.choice([rng.uniform(0.0, 1.0), 0.95, 1.0])
        x_norm = 10 ** rng.uniform(-2, 4)
        ftol = rng.choice([1e-4, 1e-8, 10 ** rng.uniform(-8, 0)])
        xtol = rng.choice([1e-10, 0.0, 10 ** rng.uniform(-10, -1)])
        step = xtol * (xtol + x_norm) * rng.choice([rng.uniform(0.5, 1.5), 1.0]) if rng.random() < 0.3 else step_h * x_norm
        cases.append((cost, cost - actual, predicted, step_h, step, x_norm, Delta, ftol, xtol))
    # the edges of every branch, each against a few radii, step lengths and tolerances
    edges = [(10.0, 10.0, 0.0),              # predicted = 0, actual = 0: ratio 1
             (10.0, 9.0, 0.0), (10.0, 11.0, 0.0),   # predicted = 0, actual != 0: ratio 0
             (10.0, 9.0, -1.0), (10.0, 11.0, -1.0),  # predicted < 0
             (10.0, 9.0, 4.0), (10.0, 7.0, 4.0),    # ratio exactly 0.25 and 0.75
             (1.0, 0.75, 0.5), (1.0, 0.75, 0.3),    # dF exactly ftol F (ftol = 0.25 below), ratio 0.5 and 0.83
             (10.0, np.inf, 1.0), (10.0, np.nan, 1.0), (10.0, -np.inf, 1.0)]
    for cost, cost_new, predicted in edges:
        for Delta in (1.0, 3.0):
            for step_h in (0.5 * Delta, 0.95 * Delta, Delta):
                for ftol, xtol, x_norm, step in ((0.25, 0.0, 1.0, 0.0), (1e-8, 0.0, 5.0, 1e-3), (1e-8, 0.5, 1.5, 1.0),
                                                 (1e-8, 0.5, 1.5, 0.999), (0.25, 0.5, 1.5, 0.5)):
                    cases.append((cost, cost_new, predicted, step_h, step, x_norm, Delta, ftol, xtol))
    return cases


def test_trf_update_matches_scipy(built):
    """The trust-region update of one trial point (csrc/sba_tr2d.h tr_outcome, run by the solver after every trial
    point) equals scipy's update_tr_radius + check_termination as trf_no_bounds composes them, bit for bit."""
    lib = _harness()
    f = lib.hh_tr_outcome
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_double] * 9 + [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)]
    seen = set()
    for c in _tr_outcome_cases():
        D, acc = ctypes.c_double(), ctypes.c_int()
        term = f(*c, ctypes.byref(D), ctypes.byref(acc))
        D0, term0, acc0 = _scipy_tr_outcome(*c)
        assert (term if term >= 0 else None) == term0, c
        assert D.value == D0, (c, D.value, D0)
        assert bool(acc.value) == bool(acc0), c
        seen.add((term, bool(acc.value), D.value < c[6], D.value > c[6]))
    # every outcome is exercised: each termination code, accepted and rejected steps, shrinking and growing radii
    assert {t for t, _, _, _ in seen} == {-1, 2, 3, 4}
    assert {(a, s, g) for t, a, s, g in seen if t < 0} >= {(True, True, False), (True, False, True), (True, False, False),
                                                           (False, True, False)}


def test_no_cpu_fallback(built):
    """Without a CUDA device the product path must raise, not compute on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = util.params_from_golden(G, "persp_R")
    with pytest.raises(_lib.SbaError):
        DeviceProblem(p)
    with pytest.raises(_lib.SbaError):
        ba_core.fun(p.params_opt.copy(), p)
    with pytest.raises(_lib.SbaError):
        ba_core.run_ba_optimization(p, None, False, False)


def test_unsupported_configurations_raise():
    """COMMON_K with frozen cameras: the reference packs n_cam_opt cameras but unpacks n_cam (ba_params.py:170 vs :244)."""
    from sat_bundleadjust_b200.solver import check_supported, n_common_params
    p = util.params_from_golden(G, "persp_RTK_common")
    assert n_common_params(p) == 5
    check_supported(p)
    p.n_cam_fix = 1
    with pytest.raises(NotImplementedError):
        check_supported(p)


def test_common_K_device_layout_round_trip():
    """[K | cam[:c'] ... | points] <-> n_params slots per camera with K in camera 0's slots (include/sba_b200.h n_common)."""
    from sat_bundleadjust_b200.solver import DeviceProblem as DP
    d = DP.__new__(DP)
    d.n_common, d.n_params, d.n_cam = 5, 11, 4
    n_pts = 7
    d.n_vars_device = d.n_cam * d.n_params + 3 * n_pts
    v = np.arange(5 + 4 * 6 + 3 * n_pts, dtype=np.float64) + 1.0
    x = d._to_device_layout(v)
    cams = x[:44].reshape(4, 11)
    assert np.array_equal(cams[0, 6:], v[:5]) and np.all(cams[1:, 6:] == 0.0)
    assert np.array_equal(cams[:, :6].ravel(), v[5:29]) and np.array_equal(x[44:], v[29:])
    assert np.array_equal(d._from_device_layout(x), v)
    d.handle = None


# ---------------------------------------------------------------------------------------------------
# the model math of csrc/sba_models.cuh compiled for the host (tests/host_harness)
# ---------------------------------------------------------------------------------------------------
def _harness():
    lib = ctypes.CDLL(os.path.join(util.HERE, "host_harness", "libmodel_harness.so"))
    return lib


def _camrec(model, v):
    r = np.zeros(16)
    r[0:6] = [np.cos(v[0]), np.sin(v[0]), np.cos(v[1]), np.sin(v[1]), np.cos(v[2]), np.sin(v[2])]
    if model == 1:
        r[6:9], r[9:14] = v[3:6], v[6:11]
    elif model == 0:
        r[6:8], r[9:12] = v[3:5], v[5:8]
    else:
        r[6:9], r[9:12] = v[3:6], v[6:9]
    return r


@pytest.mark.parametrize("model,name,nc", [(1, "perspective", 6), (1, "perspective", 11), (0, "affine", 5), (0, "affine", 8)])
def test_analytic_jacobian_matches_finite_differences(built, model, name, nc):
    lib = _harness()
    P = _lib.dptr
    sc = synth.make_scene(n_cam=3, n_tracks=30, p_vis=0.9, cam_model=name, seed=5)
    p = synth.scene_to_params(sc, ["R"])
    rpc = np.zeros(90)

    def proj(v, X):
        uv = np.zeros(2)
        lib.hh_project(model, P(_camrec(model, v)), P(rpc), P(np.ascontiguousarray(X)), P(uv))
        return uv

    proj_o = getattr(ba_oracle, "project_" + name)(p.pts3d.astype(np.float64), p.cam_params, p.pts_ind, p.cam_ind)
    for k in range(0, p.n_obs, 5):
        v, X = p.cam_params[p.cam_ind[k]].copy(), p.pts3d[p.pts_ind[k]].astype(np.float64)
        uv, Jc, Jp = np.zeros(2), np.zeros(2 * nc), np.zeros(6)
        assert lib.hh_project_jac(model, nc, P(_camrec(model, v)), P(rpc), P(X), P(uv), P(Jc), P(Jp)) == 0
        assert np.array_equal(uv, proj_o[k])          # same operation order as the oracle, no FMA on the host
        Jc, Jp = Jc.reshape(2, nc), Jp.reshape(2, 3)
        for s in range(nc):
            nT = 3 if model == 1 else 2
            h = 1e-7 if s < 3 else (1.0 if s < 3 + nT else 1e-3 * max(1.0, abs(v[s])))
            a, b = v.copy(), v.copy()
            a[s] += h
            b[s] -= h
            fd = (proj(a, X) - proj(b, X)) / (a[s] - b[s])
            assert np.allclose(fd, Jc[:, s], rtol=2e-6, atol=2e-6 * np.abs(fd).max() + 1e-12), (s, fd, Jc[:, s])
        for s in range(3):
            a, b = X.copy(), X.copy()
            a[s] += 0.01
            b[s] -= 0.01
            fd = (proj(v, a) - proj(v, b)) / (a[s] - b[s])
            assert np.allclose(fd, Jp[:, s], rtol=2e-6, atol=2e-6 * np.abs(fd).max())


def test_rpc_jacobian_matches_finite_differences(built):
    lib = _harness()
    P = _lib.dptr
    R = util.load_rpc_golden()
    tab = np.ascontiguousarray(R["rpc_a"][:90])
    rpc = util.rpc_from_array(R["rpc_a"])
    from oracle import rpc_oracle
    lla = R["lonlatalt"][:40]
    X = np.stack(rpc_oracle.latlon_to_ecef(lla[:, 1], lla[:, 0], lla[:, 2]), axis=1)
    v = np.array([2e-6, -1e-6, 3e-6, 0.5, -0.3, 0.2, 1.8e6, -6.1e6, 1.4e6])

    def proj(vv, x):
        uv = np.zeros(2)
        lib.hh_project(2, P(_camrec(2, vv)), P(tab), P(np.ascontiguousarray(x)), P(uv))
        return uv

    ref = rpc.project_ecef(ba_oracle.adjust_pts3d(X, np.tile(v, (X.shape[0], 1))))
    mine = np.array([proj(v, x) for x in X])
    assert np.abs(mine - ref).max() < 1e-7
    for x in X[::4]:
        uv, Jc, Jp = np.zeros(2), np.zeros(12), np.zeros(6)
        assert lib.hh_project_jac(2, 6, P(_camrec(2, v)), P(tab), P(x), P(uv), P(Jc), P(Jp)) == 0
        Jc, Jp = Jc.reshape(2, 6), Jp.reshape(2, 3)
        for s in range(6):
            h = 1e-7 if s < 3 else 0.1
            a, b = v.copy(), v.copy()
            a[s] += h
            b[s] -= h
            fd = (proj(a, x) - proj(b, x)) / (a[s] - b[s])
            assert np.allclose(fd, Jc[:, s], rtol=1e-5, atol=1e-6 * np.abs(fd).max())
        for s in range(3):
            a, b = x.copy(), x.copy()
            a[s] += 0.1
            b[s] -= 0.1
            fd = (proj(v, a) - proj(v, b)) / (a[s] - b[s])
            assert np.allclose(fd, Jp[:, s], rtol=1e-5, atol=1e-6 * np.abs(fd).max())


@pytest.mark.parametrize("loss", ["linear", "huber", "soft_l1", "cauchy", "arctan"])
def test_robust_rescale_matches_scipy(built, loss):
    from scipy.optimize._lsq.common import scale_for_robust_loss_function
    from scipy.optimize._lsq.least_squares import construct_loss_function
    lib = _harness()
    lib.hh_loss_rescale.restype = ctypes.c_double
    lib.hh_loss_rescale.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.POINTER(ctypes.c_double),
                                    ctypes.POINTER(ctypes.c_double)]
    f = np.array([-30.0, -2.0, -0.5, 0.0, 0.3, 1.0, 1.5, 4.0, 100.0])
    fs = 1.7
    if loss == "linear":
        exp_scale, exp_f, exp_cost = np.ones_like(f), f.copy(), 0.5 * f ** 2
    else:
        lf = construct_loss_function(f.size, loss, fs)
        rho = lf(f.copy())
        exp_cost = 0.5 * rho[0].copy()
        J = np.ones((f.size, 1))
        ff = f.copy()
        J, ff = scale_for_robust_loss_function(J, ff, rho)
        exp_scale, exp_f = J[:, 0], ff
    for i, fi in enumerate(f):
        fo, co = ctypes.c_double(), ctypes.c_double()
        s = lib.hh_loss_rescale(_lib.LOSS_IDS[loss], fs, fi, ctypes.byref(fo), ctypes.byref(co))
        assert np.isclose(s, exp_scale[i], rtol=1e-10, atol=0)
        assert np.isclose(fo.value, exp_f[i], rtol=1e-10, atol=1e-300)
        assert np.isclose(co.value, exp_cost[i], rtol=1e-10, atol=1e-300)


# ---------------------------------------------------------------------------------------------------
# host index construction of a device problem (csrc/sba_index.h), compiled into the host harness
# ---------------------------------------------------------------------------------------------------
def _host_index(cam_ind, pts_ind, M, N, chunk=1024, threads=8):
    lib = _harness()
    ip, lp = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_longlong)
    cam_ind, pts_ind = np.ascontiguousarray(cam_ind, dtype=np.int64), np.ascontiguousarray(pts_ind, dtype=np.int64)
    K = cam_ind.size
    sizes = np.zeros(2, dtype=np.int32)
    null = ctypes.cast(None, ip)
    args = [cam_ind.ctypes.data_as(lp), pts_ind.ctypes.data_as(lp), ctypes.c_longlong(K), M, N, chunk, threads,
            sizes.ctypes.data_as(ip)]
    rc = lib.hh_host_index(*args, *([null] * 10))
    if rc:
        return rc, None
    out = {"cam": np.zeros(K, np.int32), "pts": np.zeros(K, np.int32), "track_ptr": np.zeros(N + 1, np.int32),
           "cam_cnt": np.zeros(M + 1, np.int32), "cm_obs": np.zeros(K, np.int32), "ch_cam": np.zeros(sizes[0], np.int32),
           "ch_beg": np.zeros(sizes[0], np.int32), "ch_end": np.zeros(sizes[0], np.int32),
           "first_chunk": np.zeros(M + 1, np.int32), "tile_obs": np.zeros(sizes[1], np.int32)}
    rc = lib.hh_host_index(*args, *[out[k].ctypes.data_as(ip) for k in
                                    ("cam", "pts", "track_ptr", "cam_cnt", "cm_obs", "ch_cam", "ch_beg", "ch_end", "first_chunk", "tile_obs")])
    return rc, out


@pytest.mark.parametrize("M,N,p_vis,threads", [(10, 100000, 0.5, 8), (10, 100000, 0.5, 1), (40, 3000, 0.9, 8), (3, 50, 0.5, 8),
                                                 (7, 200000, 0.3, 5)])
def test_host_index_tables(built, M, N, p_vis, threads):
    """track offsets, camera-major permutation, chunks and warp tiles against their numpy definitions (threaded build)."""
    rng = np.random.default_rng(M * 1000 + N)
    seen = rng.random((N, M)) < p_vis
    seen[rng.random(N) < 0.05] = False                     # some tracks without any observation
    pts_ind, cam_ind = np.nonzero(seen)                    # the reference's order: by track, cameras ascending
    K = pts_ind.size
    rc, h = _host_index(cam_ind, pts_ind, M, N, chunk=1024, threads=threads)
    assert rc == 0
    assert np.array_equal(h["cam"], cam_ind) and np.array_equal(h["pts"], pts_ind)
    assert np.array_equal(h["track_ptr"], np.searchsorted(pts_ind, np.arange(N + 1), side="left"))
    assert np.array_equal(h["cam_cnt"], np.concatenate([[0], np.cumsum(np.bincount(cam_ind, minlength=M))]))
    assert np.array_equal(h["cm_obs"], np.argsort(cam_ind, kind="stable"))
    # chunks: consecutive ranges of <= 1024 observations, never across cameras, covering [0, K)
    assert h["ch_beg"][0] == 0 and h["ch_end"][-1] == K and np.array_equal(h["ch_beg"][1:], h["ch_end"][:-1])
    assert np.all(h["ch_end"] - h["ch_beg"] <= 1024) and np.all(h["ch_end"] > h["ch_beg"])
    for c in range(h["ch_cam"].size):
        assert h["cam_cnt"][h["ch_cam"][c]] <= h["ch_beg"][c] and h["ch_end"][c] <= h["cam_cnt"][h["ch_cam"][c] + 1]
    assert np.array_equal(h["first_chunk"], np.searchsorted(h["ch_cam"], np.arange(M + 1), side="left"))
    # warp tiles: whole tracks, <= 32 observations unless the tile is a single longer track, covering [0, K)
    t = h["tile_obs"]
    assert t[0] == 0 and t[-1] == K and np.all(np.diff(t) > 0)
    starts = set(h["track_ptr"].tolist())
    assert all(int(v) in starts for v in t)
    lens = np.diff(t)
    track_len = np.diff(h["track_ptr"])
    for a0, L in zip(t[:-1][lens > 32], lens[lens > 32]):
        i = pts_ind[a0]
        assert track_len[i] == L                          # an over-long tile is exactly one track


def test_host_index_rejects_bad_input(built):
    assert _host_index([0, 1, 5], [0, 0, 1], 3, 2)[0] == 1          # camera out of range
    assert _host_index([0, 1, 0], [0, 2, 1], 3, 3)[0] == 2          # tracks not sorted
    assert _host_index([0, 1], [0, 7], 3, 3)[0] == 1                # track out of range


_pattern_layout = util.pattern_layout


@pytest.mark.parametrize("M,N,p_vis,fix", [(10, 100000, 0.5, 0), (10, 5000, 0.5, 37), (22, 3000, 0.3, 0), (3, 50, 0.5, 5), (6, 2000, 0.9, 0)])
def test_pattern_layout(built, M, N, p_vis, fix):
    """csrc/sba_pattern.h: the internal order is a permutation that groups tracks by (frozen, camera set); units tile every
    track with observations exactly once; inside a unit all tracks see the unit's camera list; every warp of the persistent
    grid owns a contiguous, equally long tile range."""
    rng = np.random.default_rng(M * 100 + N)
    seen = rng.random((N, M)) < p_vis
    seen[rng.random(N) < 0.05] = False
    pts_ind, cam_ind = np.nonzero(seen)
    K = pts_ind.size
    n_cta, warps = 148, 16
    lay = _pattern_layout(cam_ind, pts_ind, M, N, n_pts_fix=fix, n_cta=n_cta, warps=warps)
    assert lay is not None
    t2o, o2o, tp = lay["trk_new2old"], lay["obs_new2old"], lay["track_ptr"]
    assert np.array_equal(np.sort(t2o), np.arange(N)) and np.array_equal(np.sort(o2o), np.arange(K))
    lens_old = np.bincount(pts_ind, minlength=N)
    assert np.array_equal(np.diff(tp), lens_old[t2o])
    # observations of an internal track are the caller's observations of that track, cameras ascending
    tp_old = np.searchsorted(pts_ind, np.arange(N + 1))
    first = o2o[tp[:-1][lens_old[t2o] > 0]]
    assert np.array_equal(first, tp_old[t2o][lens_old[t2o] > 0])
    assert np.all(pts_ind[o2o] == np.repeat(t2o, lens_old[t2o]))
    # frozen tracks (with observations) come first
    nf = int(np.sum(lens_old[:fix] > 0))
    assert lay["n_frozen"] == nf and set(t2o[:nf].tolist()) == set(np.nonzero(lens_old[:fix] > 0)[0].tolist())
    # units: disjoint, in track order, cover all tracks with observations, uniform camera list
    covered = np.zeros(N, bool)
    units = lay["units"]
    tiles = []
    for trk0, ntrk, obs0, L, mlo, mhi, free, rec in units.tolist():
        assert 1 <= L <= 32 and ntrk >= 1 and obs0 == tp[trk0]
        assert not covered[trk0: trk0 + ntrk].any()
        covered[trk0: trk0 + ntrk] = True
        mask = (mlo & 0xffffffff) | ((mhi & 0xffffffff) << 32)
        cams = np.array([j for j in range(64) if (mask >> j) & 1])
        assert cams.size == L
        obs = cam_ind[o2o[obs0: obs0 + ntrk * L]].reshape(ntrk, L)
        assert np.all(obs == cams[None, :])
        assert np.all((t2o[trk0: trk0 + ntrk] >= fix) == bool(free))
        T = min(32 // L, 16)
        tiles.append((ntrk + T - 1) // T)
    assert np.array_equal(covered, lens_old[t2o] > 0)
    assert np.all(np.diff(units[:, 0]) > 0)
    tiles = np.array(tiles)
    assert tiles.sum() == lay["n_tiles"]
    wu = lay["warp_unit0"]
    assert wu[0] == 0 and wu[-1] == len(units) and np.all(np.diff(wu) >= 0)
    # the warps' ranges are balanced by the cost model (clocks per tile of a track length and per unit start, csrc/sba_pattern.h): their
    # modelled costs differ by at most about two tiles and two unit starts (kind 1 = the assembly kernel's assignment, which the harness returns)
    import ctypes
    hl = ctypes.CDLL(os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness", "libmodel_harness.so"))
    tcost = np.array([hl.hh_tile_cost(int(L), 6, 3, 1) for L in units[:, 3]])
    ucost = hl.hh_unit_cost(1, 3)
    per_warp = np.array([(tiles[wu[g]: wu[g + 1]] * tcost[wu[g]: wu[g + 1]]).sum() + ucost * (wu[g + 1] - wu[g]) for g in range(n_cta * warps)])
    if tiles.sum() >= 4 * n_cta * warps:
        assert per_warp.max() - per_warp.min() <= 2 * tcost.max() + 2 * ucost, (per_warp.min(), per_warp.max())
    passes = (units[:, 3] * (units[:, 3] + 1) // 2 * 2 + 63) // 64      # Schur records: one per pass over a unit (n_params 6: 2 row chunks)
    assert np.array_equal(units[:, 7], np.concatenate([[0], np.cumsum(passes)[:-1]]))


def test_pattern_layout_rejects(built):
    # cameras not ascending inside a track / a track longer than 32 observations -> generic engine
    assert _pattern_layout([1, 0], [0, 0], 2, 1) is None
    assert _pattern_layout(np.arange(40), np.zeros(40, int), 40, 1) is None


def test_pattern_layout_tile_fill(built):
    """Tile fill = observations per lane slot: high when many tracks share a camera set (10 views), low when nearly every track has
    its own (50 views seen with probability 0.1) -- sba_problem_create then prefers the generic engine (fill < 0.5, >= 65536 obs)."""
    rng = np.random.default_rng(0)
    fills = {}
    for M, N, p_vis in ((10, 20000, 0.5), (50, 20000, 0.1)):
        vis = rng.random((N, M)) < p_vis
        vis[vis.sum(axis=1) < 2, :2] = True
        pts_ind, cam_ind = np.nonzero(vis)
        lay = _pattern_layout(cam_ind, pts_ind, M, N)
        assert lay is not None
        fills[M] = lay["fill"]
        assert abs(lay["fill"] - cam_ind.size / (32.0 * lay["n_tiles"])) < 2e-3
    assert fills[10] > 0.7 and fills[50] < 0.3, fills


def test_sparse_scene_matches_dense_packing():
    """synth.SparseParams (no dense correspondence matrix, used for the time-series scale configs) packs exactly like the class."""
    sc = synth.make_scene_sparse(n_cam=12, n_tracks=500, p_vis=0.3, seed=2)
    q = synth.scene_to_params(sc, ["R", "T"])
    r = synth.SparseParams(sc, ["R", "T"])
    for k in ("pts_ind", "cam_ind", "pts2d", "params_opt", "cam_params", "pts2d_w"):
        assert np.array_equal(getattr(q, k), getattr(r, k)), k
    assert (q.n_params, q.n_obs, q.n_cam, q.n_pts) == (r.n_params, r.n_obs, r.n_cam, r.n_pts)
    same = r.pts_ind[1:] == r.pts_ind[:-1]
    assert np.all(np.diff(r.pts_ind) >= 0) and np.all(r.cam_ind[1:][same] > r.cam_ind[:-1][same])


def test_common_k_vector_layouts():
    """COMMON_K: the caller's [K | cameras | points] vector (ba_params.py:167-171) <-> the device's n_params slots per camera."""
    from sat_bundleadjust_b200.solver import from_device_layout, to_device_layout
    rng = np.random.default_rng(0)
    for k, c, m, n_pts in ((5, 11, 4, 7), (3, 8, 3, 5), (0, 6, 4, 3)):
        v = rng.standard_normal(k + m * (c - k) + 3 * n_pts)
        x = to_device_layout(v, k, c, m)
        assert x.size == m * c + 3 * n_pts
        cams = x[: m * c].reshape(m, c)
        assert np.array_equal(cams[0, c - k:], v[:k]) and np.all(cams[1:, c - k:] == 0.0)
        assert np.array_equal(cams[:, : c - k].ravel(), v[k: k + m * (c - k)]) and np.array_equal(x[m * c:], v[k + m * (c - k):])
        assert np.array_equal(from_device_layout(x, k, c, m), v)
