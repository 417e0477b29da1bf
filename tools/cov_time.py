"""
Device time of the posterior covariance (sba_covariance) at the bench's `1m` workload, against the trust-region iterations of the
same problem, in one run.  Prints one JSON object: the GPU's name and power limit (queried, not set), the covariance call's
phases (CUDA events: reduced system, factor + pivot test, inverse, point pass) and a host clock around the synchronising call,
and the device time of one trust-region iteration (L2-cold, like bench.py).

    python tools/cov_time.py [--workload 1m] [--reps 10] [--iters 8]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as exc:  # the measurement itself does not depend on it
        return {"error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="1m")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--iters", type=int, default=8)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("cov_time.py needs a CUDA device")
    from sat_bundleadjust_b200 import synth
    from sat_bundleadjust_b200.solver import DeviceProblem, initial_vars
    n_cam, tracks, p_vis, model, corr, _ = bench.WORKLOADS[args.workload]
    sc = synth.make_scene(n_cam=n_cam, n_tracks=tracks, p_vis=p_vis, cam_model=model, seed=0)
    p = synth.scene_to_params(sc, corr, n_cam_fix=2)     # two frozen cameras fix the similarity gauge (one leaves the scale free)
    ls = bench.LS
    x0 = initial_vars(p)
    res = {"gpu": gpu_info(), "workload": args.workload, "n_obs": int(p.pts_ind.size), "n_pts": int(p.n_pts), "n_cam": int(p.n_cam),
           "n_params": int(p.n_params), "n_cam_fix": 2, "loss": ls["loss"]}
    with DeviceProblem(p) as prob:
        res["engine"] = prob.engine
        x, _, info = prob.solve(x0, want_residuals=False, **ls)
        res["solve_iterations"], res["solve_ms"] = info["iterations"], info["solve_ms"]
        # trust-region iterations of the same problem: W untimed, then `iters` timed, L2 flushed between them
        it = prob.solve(x0, want_residuals=False, ftol=0.0, xtol=0.0, gtol=0.0, max_nfev=10 ** 6, max_iterations=2 + args.iters,
                        timed_from=2, l2_flush_bytes=bench.L2_FLUSH_BYTES, no_phase_timing=1, **ls)[2]
        res["iteration_ms"] = it["iter_ms"] / it["timed_iterations"]
        prob.covariance(x, **ls)                               # warm-up: first-call allocations, module loads
        phases, walls = [], []
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, _, s2, ratio = prob.covariance(x, **ls)
            walls.append((time.perf_counter() - t0) * 1e3)
            phases.append(prob.covariance_phase_ms())
    keys = list(phases[0].keys())
    med = {k: float(np.median([ph[k] for ph in phases])) for k in keys}
    res["covariance"] = {"phase_ms_median": med, "device_ms_median": float(np.median([sum(ph.values()) for ph in phases])),
                         "device_ms_all": [round(sum(ph.values()), 4) for ph in phases],
                         "host_wall_ms_median": float(np.median(walls)), "host_wall_ms_all": [round(w, 3) for w in walls],
                         "sigma2": s2, "min_pivot_ratio": ratio}
    res["covariance_over_iteration"] = res["covariance"]["device_ms_median"] / res["iteration_ms"]
    print(json.dumps(res))


if __name__ == "__main__":
    main()
