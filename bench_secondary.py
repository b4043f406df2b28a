#!/usr/bin/env python
"""Secondary measurements (SURVEY.md 8(d)): obs/s per LM iteration for global
positioning and edges/s per IRLS iteration for rotation averaging, 1 GPU.
Not the driver's bench (that is bench.py); results are copied to profiles/.

  python bench_secondary.py --what gp --workload config2
  python bench_secondary.py --what ra --frames 100000 --neighbours 50
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from glomap_b200 import estimators as E, geometry as G, synthetic as S  # noqa: E402


def bench_gp(args):
    C, P = (1000, 200_000) if args.workload == "config2" else (200, 20_000)
    sc = S.make_scene(C, P, 10.0, seed=1, pixel_sigma=0.5, chunk=25_000)
    prob = E.PositioningProblem(sc.quat, sc.pt_obs_begin, sc.obs_cam, S.bearings_from_scene(sc))
    opts = E.GlobalPositionerOptions(profile_kernels=True)
    opts.solver_options.pcg_rel_tolerance = args.pcg_tol
    gp = E.GlobalPositioner(opts)
    res = []
    for it in range(args.warmup + args.steps):
        gp.rng = np.random.default_rng(1)
        prob.centers = prob.points = prob.scales = None
        t0 = time.perf_counter()
        ok = gp.Solve(prob)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            res.append((dt, gp.summary.as_dict()))
    st = res[-1][1]
    R = G.quat_xyzw_to_rotmat(sc.quat)
    cg = G.centers_from_pose(R, sc.trans)
    s, Rr, t = G.umeyama_sim3(prob.centers, cg)
    err = float(np.linalg.norm((s * (Rr @ prob.centers.T)).T + t - cg, axis=1).max())
    n_used = st["num_observations"]
    dev_ms = np.mean([r[1]["ms_total"] for r in res])
    line = {"what": "global positioning (BATA) from random initialisation", "workload": f"{C} cams / {P} pts / {sc.N} obs, 0.5 px noise",
            "ok": bool(ok), "lm_iterations": st["iterations"], "pcg_iterations": st["pcg_iterations"],
            "device_ms_per_solve": dev_ms, "wall_ms_per_solve_e2e": 1e3 * np.mean([r[0] for r in res]),
            "obs_per_s_per_lm_iteration": n_used * st["iterations"] / (dev_ms * 1e-3),
            "linearize_kernel_avg_ms": st["ms_linearize"] / max(st["n_linearize"], 1),
            "linearize_GBps (80*N + 96*P model)": (80 * sc.N + 96 * P) / (st["ms_linearize"] / max(st["n_linearize"], 1) * 1e-3) / 1e9,
            "matvec_kernel_avg_ms": st["ms_matvec"] / max(st["n_matvec"], 1),
            "matvec_GBps (56*N + 56*P model)": (56 * sc.N + 56 * P) / (st["ms_matvec"] / max(st["n_matvec"], 1) * 1e-3) / 1e9,
            "max_centre_error_after_sim3": err, "cost": [st["initial_cost"], st["final_cost"]], "pcg_rel_tolerance": args.pcg_tol}
    print(json.dumps(line))


def bench_ra(args):
    vg = S.make_lattice_view_graph(args.frames, args.neighbours, seed=1, noise_deg=2.0, outlier_ratio=0.05)
    opts = E.RotationEstimatorOptions(pcg_rel_tolerance=args.pcg_tol)
    est = E.RotationEstimator(opts)
    t0 = time.perf_counter()
    R0 = E.initialize_from_maximum_spanning_tree(vg)
    mst_s = time.perf_counter() - t0
    res = []
    for it in range(args.warmup + args.steps):
        opts.skip_initialization = True
        t0 = time.perf_counter()
        ok, R = est.EstimateRotations(vg, R0)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            res.append((dt, est.summary.as_dict()))
    st = res[-1][1]
    # error against ground truth on a sample of pairs (all-pairs is O(n^2))
    rng = np.random.default_rng(0)
    a, b = rng.integers(0, vg.n_images, 20000), rng.integers(0, vg.n_images, 20000)
    rel = R[b] @ np.swapaxes(R[a], -1, -2)
    rel_gt = vg.R_gt[b] @ np.swapaxes(vg.R_gt[a], -1, -2)
    err = G.rotation_angle_deg(rel, rel_gt)
    dev_ms = np.mean([r[1]["ms_total"] for r in res])
    its = st["l1_iterations"] + st["irls_iterations"]
    line = {"metric": "view-graph edges/sec per rotation-averaging outer (L1 / IRLS) iteration",
            "value": vg.E * its / (dev_ms * 1e-3), "unit": "edges/s per outer iteration", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"config5: {vg.n_images} frames / {vg.E} edges lattice view graph, 2 deg noise, 5% outliers; "
                                   "one RotationEstimator solve per step (5 L1 + IRLS to convergence), MST initialisation on the host outside the step"},
            "what": "rotation averaging (L1-ADMM + IRLS), MST initialisation on the host",
            "workload": f"{vg.n_images} frames / {vg.E} edges lattice, 2 deg noise, 5% outliers", "ok": bool(ok),
            "l1_iterations": st["l1_iterations"], "admm_iterations": st["admm_iterations"], "irls_iterations": st["irls_iterations"],
            "pcg_iterations": st["pcg_iterations"], "device_ms_per_solve": dev_ms,
            "wall_ms_per_solve_e2e": 1e3 * np.mean([r[0] for r in res]), "host_mst_init_s": mst_s,
            "edges_per_s_per_outer_iteration": vg.E * its / (dev_ms * 1e-3),
            "laplacian_matvecs_per_s": st["pcg_iterations"] / (dev_ms * 1e-3),
            "median_pair_error_deg": float(np.median(err)), "p99_pair_error_deg": float(np.percentile(err, 99)),
            "pcg_rel_tolerance": args.pcg_tol, "kernel_launches": st["kernel_launches"]}
    print(json.dumps(line))
    return R


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--what", choices=["gp", "ra"], required=True)
    ap.add_argument("--workload", default="config2")
    ap.add_argument("--frames", type=int, default=100_000)
    ap.add_argument("--neighbours", type=int, default=50)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--pcg-tol", type=float, default=1e-2)
    a = ap.parse_args()
    (bench_gp if a.what == "gp" else bench_ra)(a)
