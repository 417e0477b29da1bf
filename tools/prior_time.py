"""
Overhead of a camera prior on the trust-region iteration: ms per iteration without a prior against a zero-information prior
(which gives identical iterations, so the difference is the cost of the prior terms alone), on the bench's `1m` workload
(pattern engine) and on a 50-view generic-engine scene (`cfg3`), L2-cold like bench.py (timed_from, L2 flush).  The two
variants alternate over `--rounds` rounds on the same handle.  Prints one JSON object with the GPU's name and power limit
(queried, not set).

    python tools/prior_time.py [--iters 20] [--rounds 5]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from cov_time import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--workloads", default="1m,cfg3")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("prior_time.py needs a CUDA device")
    from sat_bundleadjust_b200 import synth
    from sat_bundleadjust_b200.ba_priors import CameraPrior
    from sat_bundleadjust_b200.solver import DeviceProblem, initial_vars
    res = {"gpu": gpu_info(), "iters": args.iters, "rounds": args.rounds}
    for wl in args.workloads.split(","):
        n_cam, tracks, p_vis, model, corr, _ = bench.WORKLOADS[wl]
        sc = synth.make_scene(n_cam=n_cam, n_tracks=tracks, p_vis=p_vis, cam_model=model, seed=0)
        p = synth.scene_to_params(sc, corr)
        x0 = initial_vars(p)
        zero = CameraPrior(np.zeros((p.n_cam, p.n_params)), np.zeros((p.n_cam, p.n_params, p.n_params)))
        kw = dict(want_residuals=False, ftol=0.0, xtol=0.0, gtol=0.0, max_nfev=10 ** 6, max_iterations=2 + args.iters, timed_from=2,
                  l2_flush_bytes=bench.L2_FLUSH_BYTES, no_phase_timing=1, **bench.LS)
        out = {"none": [], "zero": []}
        with DeviceProblem(p) as prob:
            engine = prob.engine
            prob.solve(x0, **kw)                                   # warm-up
            for _ in range(args.rounds):
                for name in ("none", "zero"):
                    prob.set_camera_prior(zero if name == "zero" else None)
                    x, _, info = prob.solve(x0, **kw)
                    out[name].append((info["iter_ms"] / info["timed_iterations"], x, info["cost"]))
        same = all(np.array_equal(a[1], b[1]) and a[2] == b[2] for a, b in zip(out["none"], out["zero"]))
        med = {k: float(np.median([v[0] for v in out[k]])) for k in out}
        res[wl] = {"engine": engine, "n_obs": int(p.pts_ind.size), "n_cam": int(p.n_cam),
                   "ms_per_iteration_median": med, "ms_all": {k: [round(v[0], 4) for v in out[k]] for k in out},
                   "overhead_rel": med["zero"] / med["none"] - 1.0, "iterates_identical": bool(same)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
