"""
Generates the golden fixtures in tests/golden/ by running the UNMODIFIED reference
(/root/reference, imported through oracle/ref_loader.py; its C sources compiled in place into
oracle/_ref/disp_to_h.so) on small seeded inputs.  Run in the build container only:

    python tests/golden/make_golden.py

Fixtures (all inputs are stored next to the outputs, so the tests never need the reference):
  ba_golden.npz     per case: scene inputs, reference packing (pts_ind/cam_ind/pts2d/params_opt/cam_params),
                    reference `fun` at the initial point and at a perturbed point, the sparsity pattern,
                    the reference `run_ba_optimization` result (x, err, nfev, cost), and the reference's cost
                    function at a true local minimum (`conv_*`, oracle.ba_oracle.solve_converged)
  rpcfit_golden.npz ba_rpcfit.weighted_lsq of the reference on 12 Rt-corrected 10x10x10 samplings (targets, inputs, fitted RPC, errors)
  rpc_golden.npz    the two SkySat RPCs of the reference's tests/data/images (coefficients as arrays),
                    projections / localisations / two-view triangulations computed by the compiled reference C,
                    and the reference `fun` for cam_model='rpc' driven through oracle.rpc_oracle.RPCModel
"""
import glob
import io
import os
import sys
import contextlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import rpc_ctypes, rpc_oracle  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402
from sat_bundleadjust_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

BA_CASES = [
    # name, cam_model, correction_params, n_cam, n_tracks, p_vis, n_cam_fix, n_pts_fix, ref_w, ls_params
    ("persp_R", "perspective", ["R"], 5, 300, 0.6, 0, 0, 1.0, None),
    ("persp_RT_softl1", "perspective", ["R", "T"], 6, 400, 0.5, 0, 0, 1.0, {"loss": "soft_l1", "f_scale": 1.0, "max_iter": 300}),
    ("persp_RT_fix", "perspective", ["R", "T"], 6, 400, 0.5, 2, 40, 3.0, None),
    ("persp_RT_huber", "perspective", ["R", "T"], 5, 300, 0.6, 1, 0, 1.0, {"loss": "huber", "f_scale": 2.0}),
    ("affine_R", "affine", ["R"], 5, 300, 0.6, 0, 0, 1.0, None),
    ("affine_RT_softl1", "affine", ["R", "T"], 6, 400, 0.5, 1, 0, 1.0, {"loss": "soft_l1", "f_scale": 1.0, "max_iter": 300}),
    ("persp_RTK", "perspective", ["R", "T", "K"], 4, 200, 0.7, 0, 0, 1.0, "nosolve"),
    ("affine_RTK", "affine", ["R", "T", "K"], 4, 200, 0.7, 0, 0, 1.0, "nosolve"),
    ("persp_RTK_common", "perspective", ["R", "T", "K", "COMMON_K"], 4, 200, 0.7, 0, 0, 1.0, "nosolve"),
]


def quiet(f, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return f(*a, **k)


def make_ba_golden(ref):
    out = {"cases": np.array([c[0] for c in BA_CASES])}
    for seed, (name, model, corr, n_cam, n_tracks, p_vis, ncf, npf, refw, ls) in enumerate(BA_CASES):
        sc = synth.make_scene(n_cam=n_cam, n_tracks=n_tracks, p_vis=p_vis, cam_model=model, seed=100 + seed)
        p = synth.scene_to_params(sc, corr, n_cam_fix=ncf, n_pts_fix=npf, ref_cam_weight=refw,
                                  params_cls=ref.ba_params.BundleAdjustmentParameters)
        pre = name + "/"
        out[pre + "cam_model"] = np.array(model)
        out[pre + "correction_params"] = np.array(corr)
        out[pre + "opts"] = np.array([ncf, npf, refw], dtype=np.float64)
        out[pre + "C"] = sc.correspondence_matrix()
        out[pre + "pts3d_init"] = sc.pts3d_init
        out[pre + "cameras_init"] = np.array(sc.cameras_init)
        out[pre + "camera_centers"] = np.array(sc.camera_centers)
        for k in ["pts_ind", "cam_ind", "pts2d", "params_opt", "cam_params", "pts2d_w"]:
            out[pre + "ref_" + k] = getattr(p, k)
        x0 = p.params_opt.copy()
        out[pre + "ref_fun_x0"] = ref.ba_core.fun(x0, p)
        rng = np.random.default_rng(7)
        x1 = p.params_opt.copy()
        x1 *= 1.0 + 1e-9 * rng.standard_normal(x1.size)
        out[pre + "x1"] = x1.copy()
        out[pre + "ref_fun_x1"] = ref.ba_core.fun(x1, p)
        A = ref.ba_core.build_jacobian_sparsity(p).tocsr()
        A.sort_indices()
        out[pre + "ref_sparsity_indptr"] = A.indptr.astype(np.int64)
        out[pre + "ref_sparsity_indices"] = A.indices.astype(np.int64)
        out[pre + "ref_sparsity_shape"] = np.array(A.shape)
        if ls != "nosolve":
            cfg = dict(ls or {})
            cfg["verbose"] = 0
            v0, v1, e0, e1, nfev = quiet(ref.ba_core.run_ba_optimization, p, cfg, False, False)
            out[pre + "ls_keys"] = np.array(list(cfg.keys()))
            out[pre + "ls_vals"] = np.array([str(v) for v in cfg.values()])
            out[pre + "ref_vars_init"], out[pre + "ref_vars_ba"] = v0, v1
            out[pre + "ref_err_init"], out[pre + "ref_err_ba"] = e0, e1
            out[pre + "ref_nfev"] = np.array(nfev)
            # same problem driven to tight convergence (SURVEY.md H1); only its residual is kept, which keeps the
            # fixture under 1 MB
            cfg_t = dict(cfg, ftol=1e-14, xtol=1e-14, max_iter=400)
            _, v1t, _, _, nfev_t = quiet(ref.ba_core.run_ba_optimization, p, cfg_t, False, False)
            out[pre + "ref_tight_nfev"] = np.array(nfev_t)
            out[pre + "ref_tight_fun"] = ref.ba_core.fun(v1t.copy(), p)
            # the reference's cost function at a true local minimum (scipy TRF, dense exact solver)
            from oracle import ba_oracle
            xc, cc, rc = ba_oracle.solve_converged(p, cfg.get("loss", "linear"), cfg.get("f_scale", 1.0), x_start=v1t)
            assert np.array_equal(ba_oracle.residuals(xc.copy(), p), ref.ba_core.fun(xc.copy(), p))
            out[pre + "conv_vars"], out[pre + "conv_cost"], out[pre + "conv_status"] = xc, np.array(cc), np.array(rc.status)
            print("   converged cost %.12e status %d nfev %d" % (cc, rc.status, rc.nfev))
        print("ba case", name, "K =", p.pts_ind.size, "n =", p.params_opt.size)
    np.savez_compressed(os.path.join(HERE, "ba_golden.npz"), **out)


def rpc_arrays(r):
    return np.concatenate([[r.row_offset, r.col_offset, r.lat_offset, r.lon_offset, r.alt_offset,
                            r.row_scale, r.col_scale, r.lat_scale, r.lon_scale, r.alt_scale],
                           r.row_num, r.row_den, r.col_num, r.col_den])


def approx_center(r):
    """A point ~500 km up the viewing ray through the image centre (stands in for the camera centre)."""
    lon0, lat0 = r.localization(r.col_offset, r.row_offset, r.alt_offset)
    lon1, lat1 = r.localization(r.col_offset, r.row_offset, r.alt_offset + 1000.0)
    a = np.array(rpc_oracle.latlon_to_ecef(lat0, lon0, r.alt_offset))
    b = np.array(rpc_oracle.latlon_to_ecef(lat1, lon1, r.alt_offset + 1000.0))
    return a + 500e3 * (b - a) / np.linalg.norm(b - a)


def make_rpc_golden(ref):
    files = sorted(glob.glob(os.path.join(os.environ.get("SBA_REFERENCE_ROOT", "/root/reference"),
                                          "tests/data/images/*.rpc")))
    ra, rb = [rpc_oracle.RPCModel.from_file(f) for f in files]
    lib = rpc_ctypes.load_ref()
    assert lib is not None, "run `make -C oracle ref` first"
    rng = np.random.default_rng(5)
    n = 500
    lla = np.stack([ra.lon_offset + rng.uniform(-.04, .04, n), ra.lat_offset + rng.uniform(-.04, .04, n),
                    ra.alt_offset + rng.uniform(-800, 800, n)], axis=1)
    out = {"rpc_a": rpc_arrays(ra), "rpc_b": rpc_arrays(rb), "lonlatalt": lla}
    out["ref_proj_a"] = rpc_ctypes.ref_project(lib, ra, lla)
    out["ref_proj_b"] = rpc_ctypes.ref_project(lib, rb, lla)
    cra = np.stack([rng.uniform(0, 3200, n), rng.uniform(0, 1350, n), ra.alt_offset + rng.uniform(-800, 800, n)], axis=1)
    out["colrowalt"] = cra
    out["ref_loc_a_delta1"] = rpc_ctypes.ref_localize(lib, ra, cra, delta=1.0)
    out["ref_loc_a_delta01"] = rpc_ctypes.ref_localize(lib, ra, cra, delta=0.1)
    kp_a = out["ref_proj_a"] + rng.normal(0, 0.3, (n, 2))
    kp_b = out["ref_proj_b"] + rng.normal(0, 0.3, (n, 2))
    out["kp_a"], out["kp_b"] = kp_a, kp_b
    out["ref_tri_lonlatalt"], out["ref_tri_err"] = rpc_ctypes.triangulate(lib, ra, rb, kp_a, kp_b, delta=0.1, ref=True)

    # reference `fun` with cam_model='rpc': 4 cameras (the two real RPCs and two footprint-shifted copies)
    cams = [ra, rb]
    for src, dlon, dlat in [(ra, 0.002, -0.001), (rb, -0.0015, 0.002)]:
        c = rpc_oracle.RPCModel(src.to_dict())
        c.lon_offset += dlon
        c.lat_offset += dlat
        cams.append(c)
    out["rpc_cams"] = np.array([rpc_arrays(c) for c in cams])
    centers = [approx_center(c) for c in cams]
    npts = 250
    g = np.stack([ra.lon_offset + rng.uniform(-.01, .01, npts), ra.lat_offset + rng.uniform(-.004, .004, npts),
                  ra.alt_offset + rng.uniform(-200, 200, npts)], axis=1)
    X = np.stack(rpc_oracle.latlon_to_ecef(g[:, 1], g[:, 0], g[:, 2]), axis=1)
    C = np.full((8, npts), np.nan)
    seen = rng.random((4, npts)) < 0.7
    seen[:2] |= ~(seen.sum(axis=0) >= 2)
    for j, c in enumerate(cams):
        uv = c.project_ecef(X) + rng.normal(0, 0.5, (npts, 2))
        C[2 * j, seen[j]] = uv[seen[j], 0]
        C[2 * j + 1, seen[j]] = uv[seen[j], 1]
    pts_init = (X + rng.normal(0, 1.0, X.shape)).astype(np.float32)
    out["rpcba/C"], out["rpcba/pts3d_init"], out["rpcba/camera_centers"] = C, pts_init, np.array(centers)
    for corr in (["R"], ["R", "T"]):
        d = {"correction_params": corr, "reduce": False, "verbose": False}
        p = ref.ba_params.BundleAdjustmentParameters(C, pts_init, list(cams), "rpc", [(0, 1)], centers, d)
        tag = "rpcba/" + "".join(corr) + "/"
        x1 = p.params_opt.copy()
        x1[: p.n_cam * p.n_params] += 1e-6 * rng.standard_normal(p.n_cam * p.n_params)
        out[tag + "params_opt"], out[tag + "x1"] = p.params_opt, x1.copy()
        out[tag + "ref_fun_x0"] = ref.ba_core.fun(p.params_opt.copy(), p)
        out[tag + "ref_fun_x1"] = ref.ba_core.fun(x1, p)
        print("rpc ba case", corr, "K =", p.pts_ind.size)
    np.savez_compressed(os.path.join(HERE, "rpc_golden.npz"), **out)


def make_rpcfit_golden(ref):
    """ba_rpcfit.weighted_lsq of the UNMODIFIED reference (its `rpcm.RPCModel` is the oracle's look-alike, see
    oracle/ref_loader.py) on the Rt-corrected sampling of the two SkySat RPCs."""
    from oracle import rpcfit_oracle
    R = np.load(os.path.join(HERE, "rpc_golden.npz"))
    out = {}
    crop = {"col0": 0.0, "row0": 0.0, "width": 3199.0, "height": 1349.0}
    rts = [np.array([3e-6, -2e-6, 4e-6, 0.8, -0.5, 0.3]), np.array([-5e-6, 1e-6, 2e-6, -1.0, 0.4, 0.7]),
           np.array([0.0, 0.0, 0.0, 0.0, 0.0, 0.0])]
    k = 0
    for key in ("rpc_a", "rpc_b"):
        a = R[key]
        rpc = rpc_oracle.RPCModel()
        (rpc.row_offset, rpc.col_offset, rpc.lat_offset, rpc.lon_offset, rpc.alt_offset,
         rpc.row_scale, rpc.col_scale, rpc.lat_scale, rpc.lon_scale, rpc.alt_scale) = [float(v) for v in a[:10]]
        rpc.row_num, rpc.row_den, rpc.col_num, rpc.col_den = [list(a[10 + 20 * i: 30 + 20 * i]) for i in range(4)]
        center = approx_center(rpc)
        for rt in rts:
            for margin in (10, 160):
                Rt = np.concatenate([rt, center])
                target, locs, _ = rpcfit_oracle.rt_corrected_samples(Rt, rpc, crop, margin=margin)
                fit = ref.ba_rpcfit.weighted_lsq(target, locs)
                err = ref.ba_rpcfit.check_errors(fit, locs, target)
                pre = "case%d/" % k
                out[pre + "Rt"], out[pre + "src"], out[pre + "margin"] = Rt, np.array(key), np.array(margin)
                out[pre + "target"], out[pre + "input_locs"] = target, locs
                out[pre + "ref_rpc"] = rpc_arrays(fit)
                out[pre + "ref_err"] = err
                k += 1
    out["n_cases"] = np.array(k)
    np.savez_compressed(os.path.join(HERE, "rpcfit_golden.npz"), **out)
    print("rpcfit cases", k)


if __name__ == "__main__":
    ref = load_reference()
    if "--only-rpcfit" in sys.argv:
        make_rpcfit_golden(ref)
        sys.exit(0)
    make_ba_golden(ref)
    make_rpc_golden(ref)
    make_rpcfit_golden(ref)
    for f in ("ba_golden.npz", "rpc_golden.npz", "rpcfit_golden.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")
