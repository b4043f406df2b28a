#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: observations/s per BA LM-iteration on the
10k-camera / 2M-point / 20M-observation synthetic global BA (config 4), points
sharded across N GPUs (one process per GPU, NCCL all-reduce inside the solver).

  python bench.py --gpus 1 --steps 3 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      (CPU arm: the oracle port on host cores)
  python bench.py ... --dump-outputs DIR    (also write the last timed step's results as DIR/<name>.npy)

One "step" = one BundleAdjuster solve (cap of --lm-iters LM iterations, natural
Ceres termination) from the same perturbed start; `value` = observations x LM
iterations / device time with the problem resident in HBM; `e2e` = the same
through the one-shot C-ABI call b200sfm_ba_solve with pinned HOST buffers
(upload, structure build, solve, download inside the timed region).

--dump-outputs writes, after the timed steps, what the last one computed: the
refined quat / trans / points / intr_params and cost = [initial, final] (float64;
under N GPUs each rank writes its own point shard as points_rank<r>.npy), or for
config5 the estimated rotations [frames, 3, 3].  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time


def _host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# The CPU legs (cpu_baseline, --impl reference) use every host core: torchrun exports OMP_NUM_THREADS=1 to its
# workers, which would silently make the OpenMP loops and the LAPACK Cholesky single-threaded.  The thread counts
# must be in the environment before numpy / libgomp initialise, hence before the imports below.
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ[_v] = str(_host_cores())

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (C, P, mean track len, chunk)
    "config5": (0, 0, 0.0, 0),                      # rotation averaging on the 100k-frame lattice: dispatched to bench_secondary
    "config4": (10_000, 2_000_000, 10.0, 50_000),   # 10k cams / 2M pts / 20M obs  (the metric's config)
    "config2": (1_000, 200_000, 10.0, 25_000),      # 1k cams / 200k pts / 2M obs
    "tiny": (200, 20_000, 8.0, 2_500),
}
CPU_SAMPLE = "config2"   # bounded sample for the CPU baseline: 1/10 of the cameras and points
DUMP_LIMIT_BYTES = 64 << 20   # --dump-outputs: the largest workload (config4) writes ~48.6 MB


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each array as out_dir/<name>.npy in float64; refuses more than DUMP_LIMIT_BYTES in all."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  Two sources, because the timed region of the default run
    is only ~150 ms: (1) NVML in-process (pynvml), polled every 5 ms by a thread between mark_begin() and stop();
    (2) `nvidia-smi -lms 50` with timestamps, launched with start() BEFORE the warm-up (the tool needs a few hundred ms
    to come up) and filtered to the same window.  The NVML samples are used when there are any, else nvidia-smi's."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.nvml_rows, self.nvml_on, self.nvml_th = [], False, None
        self.t_begin = self.t_end = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self._mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def _poll_nvml(self):
        nv = self._nv
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap))
        while self.nvml_on:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                self.nvml_rows.append((sm, [n for n, bit in names if mask & bit]))
            except Exception:
                break
            time.sleep(0.005)

    def mark_begin(self):
        """Start of the timed region."""
        import datetime
        self.t_begin = datetime.datetime.now()
        if getattr(self, "_nv", None) is not None:
            self.nvml_on = True
            self.nvml_th = threading.Thread(target=self._poll_nvml, daemon=True)
            self.nvml_th.start()

    @staticmethod
    def parse_smi(rows, t_begin, t_end):
        """(sm clocks, max clocks, reasons) of the nvidia-smi rows whose timestamp lies in [t_begin, t_end] (no window: all)."""
        import datetime
        sm, mx, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f")
                a, b = float(f[1]), float(f[2])
            except ValueError:
                continue
            if t_begin is not None and t_end is not None and not (t_begin <= ts <= t_end):
                continue
            sm.append(a); mx.append(b)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return sm, mx, reasons

    def stop(self):
        import datetime
        self.t_end = datetime.datetime.now()
        self.nvml_on = False
        if self.nvml_th is not None:
            self.nvml_th.join(timeout=1)
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.nvml_rows:
            sm = [r[0] for r in self.nvml_rows]
            reasons = sorted({n for r in self.nvml_rows for n in r[1]})
            return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": self._mx, "reasons": reasons, "samples": len(sm),
                    "source": "NVML, 5 ms polling inside the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi / NVML unavailable"], "samples": 0}
        sm, mx, reasons = self.parse_smi(self.rows, self.t_begin, self.t_end)
        src = "nvidia-smi -lms 50, rows inside the timed region"
        if not sm:   # a region shorter than one sampling period: the rows since the warm-up (same clocks, same load pattern)
            sm, mx, reasons = self.parse_smi(self.rows, None, None)
            src = "nvidia-smi -lms 50, rows since the warm-up (none fell inside the timed region)"
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": src}


def shard_range(P, chunk, rank, world):
    from glomap_b200.dist import shard_range as sr
    return sr(P, chunk, rank, world)


def _cpu_problem():
    from glomap_b200 import synthetic as S
    C, P, L, chunk = WORKLOADS[CPU_SAMPLE]
    sc = S.make_scene(C, P, L, seed=1, pixel_sigma=0.5, chunk=chunk)
    init = S.perturb_scene(sc, chunk=chunk)
    mask = np.zeros(C, np.uint8); mask[0] = 3
    return sc, init, mask


def cpu_baseline(steps: int, lm_iters: int, natural: bool = True):
    """The oracle port (C/OpenMP + LAPACK Cholesky) on a bounded sample: `steps` timed repeats of `lm_iters` LM
    iterations (median), and -- once, untimed for the metric -- the natural solve to Ceres' termination, whose LM
    iteration count and final cost are what the GPU arm's `parity` record is checked against."""
    from oracle import ba_oracle as B, ba_oracle_fast as F
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=_host_cores())
    except Exception:
        pass
    C, P, L, chunk = WORKLOADS[CPU_SAMPLE]
    sc, init, mask = _cpu_problem()
    args = (init.quat, init.trans, init.points, sc.pt_obs_begin, sc.obs_cam, sc.obs_xy, sc.cam_intr, sc.intr_model,
            sc.intr_params, B.BAOptions(), mask)
    secs, its = [], 0
    times = {}
    for _ in range(steps):
        t0 = time.perf_counter()
        _, summ = F.solve_ba_fast(*args, fixed_num_iterations=lm_iters)
        secs.append(time.perf_counter() - t0)
        its = summ.iterations
        times = summ.times
    n_used = int((np.diff(sc.pt_obs_begin)[np.diff(sc.pt_obs_begin) >= 3]).sum())
    med = float(np.median(secs))
    out = {"value": n_used * its / med, "unit": "observations/s per LM iteration", "cores": F.num_threads(),
           "kind": "port",
           "sample": f"{CPU_SAMPLE} ({C} cams / {P} pts / {sc.N} obs = 1/10 of the workload), median of {steps} repeats of "
                     f"{its} LM iteration(s), explicit Schur + dense LAPACK Cholesky (CPU restatement, not Ceres)",
           "seconds_per_repeat": secs, "phase_seconds_last_step": times, "blas_threads": _host_cores()}
    if natural:
        t0 = time.perf_counter()
        _, full = F.solve_ba_fast(*args)
        out["natural_solve"] = {"workload": CPU_SAMPLE, "seconds": time.perf_counter() - t0, "lm_iterations": full.iterations,
                                "initial_cost": full.initial_cost, "final_cost": full.final_cost,
                                "termination": full.termination, "solver": "exact (dense Cholesky of the reduced system)"}
    return out, med


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    C, P, L, chunk = WORKLOADS[args.workload]
    steps = max(1, args.steps)
    for _ in range(min(args.warmup, 1)):
        cpu_baseline(1, 1, natural=False)
    cb, sec_per_step = cpu_baseline(steps, args.cpu_lm_iters)
    line = {"impl": "reference", "metric": "observations/sec per BA LM-iteration", "value": cb["value"],
            "unit": "observations/s per LM iteration", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sec_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {C} cams / {P} pts BA; CPU arm times a bounded sample: {cb['sample']}",
                       "natural_solve": cb.get("natural_solve"), "seconds_per_repeat": cb["seconds_per_repeat"]},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": cb["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def gpu_parity(ctx, E, cb, pcg_tol):
    """The CUDA path on the CPU arm's own problem (same generator, seed and start, all LM iterations to Ceres'
    termination at the bench's PCG forcing tolerance): final cost and LM iteration count against the exact-solve
    CPU port, and the time both take to reach it."""
    import torch
    sc, init, mask = _cpu_problem()
    opts = E.BundleAdjusterOptions(optimize_intrinsics=False)
    opts.solver_options.pcg_rel_tolerance = pcg_tol
    opts.solver_options.pcg_max_iterations = 200
    prob = E.BAProblem(ctx, sc, 3, mask)
    prob.set_state(init.intr_params, init.quat, init.trans, init.points)
    prob.save_state()
    st = None
    for _ in range(3):
        prob.restore_state()
        torch.cuda.synchronize()
        st = prob.solve(opts).as_dict()
    prob.free()
    rec = {"workload": CPU_SAMPLE, "same_problem_as_cpu_arm": True,
           "gpu": {"lm_iterations": st["iterations"], "pcg_iterations": st["pcg_iterations"], "initial_cost": st["initial_cost"],
                   "final_cost": st["final_cost"], "ms": st["ms_total"], "pcg_rel_tolerance": pcg_tol}}
    ns = (cb or {}).get("natural_solve")
    if ns:
        rec["cpu"] = ns
        rec["rel_final_cost_diff"] = abs(st["final_cost"] - ns["final_cost"]) / ns["final_cost"]
        rec["lm_iteration_diff"] = st["iterations"] - ns["lm_iterations"]
        rec["time_to_cost_ratio"] = ns["seconds"] * 1e3 / st["ms_total"]
        rec["checked"] = bool(rec["rel_final_cost_diff"] <= 1e-4 and abs(rec["lm_iteration_diff"]) <= 1)
    return rec


def run_b200(args):
    import torch
    import torch.distributed as dist
    from glomap_b200 import _lib, estimators as E, synthetic as S

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    nccl_id = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        obj = [E.Context.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        nccl_id = obj[0]
    ctx = E.Context(local, rank, world, nccl_id)
    lib = ctx.lib
    stream = torch.cuda.ExternalStream(lib.b200sfm_cuda_stream(ctx.handle), device=torch.device("cuda", local))

    C, P, L, chunk = WORKLOADS[args.workload]
    a, b = shard_range(P, chunk, rank, world)
    t0 = time.time()
    sc = S.make_scene(C, P, L, seed=1, pixel_sigma=0.5, chunk=chunk, point_range=(a, b))
    init = S.perturb_scene(sc, chunk=chunk, point_offset=a)
    gen_s = time.time() - t0
    lens = np.diff(sc.pt_obs_begin)
    n_local = int(lens[lens >= 3].sum())
    tot = torch.tensor([n_local, sc.P, sc.N], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tot)
    n_global, p_global, nraw_global = (int(x) for x in tot.tolist())
    mask = E.first_frame_mask(C)

    opt_intr = bool(args.optimize_intrinsics)   # second bench line: the reference's default BA mode (bundle_adjustment.h:18)
    opts = E.BundleAdjusterOptions(optimize_intrinsics=opt_intr, profile_kernels=True, design=args.design)
    opts.solver_options.max_num_iterations = args.lm_iters
    opts.solver_options.pcg_rel_tolerance = args.pcg_tol
    opts.solver_options.pcg_max_iterations = args.pcg_max

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxr(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- resident leg: `value` ----------------------------------------------------
    prob = E.BAProblem(ctx, sc, 3, mask)
    prob.set_state(init.intr_params, init.quat, init.trans, init.points)
    prob.save_state()
    stats = []
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()            # nvidia-smi needs a few hundred ms to come up: launched before the warm-up
    for _ in range(args.warmup):
        prob.restore_state()
        prob.solve(opts)
    barrier()
    if rank == 0:
        sampler.mark_begin()       # the samples reported are those between here and stop()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        prob.restore_state()
        stats.append(prob.solve(opts).as_dict())
    e1.record(stream)
    e1.synchronize()
    barrier()
    wall = time.perf_counter() - w0
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = maxr(e0.elapsed_time(e1))
    wall = maxr(wall)
    lm_its = sum(s["iterations"] for s in stats)
    pcg_its = sum(s["pcg_iterations"] for s in stats)
    launches = sum(s["kernel_launches"] for s in stats)
    value = n_global * lm_its / (dev_ms * 1e-3)
    # kernel roofline (this rank's shard)
    peak, peak_src = peaks()
    n_mv = sum(s["n_matvec"] for s in stats); ms_mv = sum(s["ms_matvec"] for s in stats)
    n_li = sum(s["n_linearize"] for s in stats); ms_li = sum(s["ms_linearize"] for s in stats)
    if args.design == 1:
        mv_bytes = 152 * sc.N + 56 * sc.P + 96 * C
        li_bytes = 168 * sc.N + 96 * sc.P + 64 * C
        mv_name, mv_model = "ba_schur_pass<0> (implicit-Schur mat-vec, design v1)", "152*N + 56*P + 96*C per launch"
        li_model = "168*N + 96*P + 64*C per launch"
        li_name = "ba_linearize_points<false> (Jacobian + point Schur blocks, design v1)"
    elif os.environ.get("B200SFM_ELL") == "0":
        # design v2, tile kernels: pass A streams A_o rows in point order (48 B + 2 x 4 B indices), per point X 24 + CSR 4 +
        # Vinv 48 + z 32; pass B streams {A_o, X} rows in camera order (72 B + 4 B index) and gathers z once per point (32 B)
        mv_bytes = 132 * sc.N + 140 * sc.P + 160 * C
        li_bytes = 72 * sc.N + 96 * sc.P + 64 * C
        mv_name = "ba2_pcg_direction_pack + ba2_pass_a<0> + ba2_pass_b (implicit-Schur mat-vec, design v2, tile kernels)"
        mv_model, li_model = "132*N + 140*P + 160*C per mat-vec", "72*N + 96*P + 64*C per launch"
        li_name = "ba_linearize_points<true> (Jacobian + point Schur blocks, tile kernel)"
    else:
        # design v2 with the point side in the ELL-32 layout (one thread per point): pass A streams A_o (48 B) + camera index
        # (4 B) per observation and, per point, slot -> point id 4 + length 4 + X 24 + Vinv 48 + z 32; pass B as above
        mv_bytes = 128 * sc.N + 144 * sc.P + 160 * C
        # linearisation: reads xy 16 + camera index 4, writes A_o 48 per observation; per point id 4 + length 4 + X 24 + V 48 + g 24
        li_bytes = 68 * sc.N + 104 * sc.P + 64 * C
        mv_name = "ba2_pcg_direction_pack + ba3_pass_a<0> + ba2_pass_b (implicit-Schur mat-vec, design v2, ELL-32 point side)"
        mv_model, li_model = "128*N + 144*P + 160*C per mat-vec", "68*N + 104*P + 64*C per launch"
        li_name = "ba3_linearize_points (Jacobian + point Schur blocks, one thread per point)"
        if opt_intr:
            # stored-row intrinsics path: B_o = rho' J_pt^T J_k (3 x nk doubles) streamed by both passes, written once by
            # the point-order linearisation; SIMPLE_PINHOLE with the principal point fixed has nk = 1 (the focal length)
            nk = 1
            mv_bytes += 48 * nk * sc.N
            li_bytes += 24 * nk * sc.N
            mv_name = mv_name.replace("implicit-Schur mat-vec", "implicit-Schur mat-vec with stored intrinsics rows")
            mv_model, li_model = f"(128 + 48*{nk})*N + 144*P + 160*C per mat-vec", f"(68 + 24*{nk})*N + 104*P + 64*C per launch"
    roof_mv = {"kernel": mv_name, "bound": "hbm",
               "achieved": mv_bytes / (ms_mv / max(n_mv, 1) * 1e-3) / 1e9 if n_mv else None, "peak": peak, "unit": "GB/s",
               "traffic": None, "peak_source": peak_src, "launches_timed": n_mv, "avg_ms": ms_mv / max(n_mv, 1),
               "bytes_model": mv_model}
    roof_li = {"kernel": li_name, "bound": "hbm",
               "achieved": li_bytes / (ms_li / max(n_li, 1) * 1e-3) / 1e9 if n_li else None, "peak": peak, "unit": "GB/s",
               "traffic": None, "peak_source": peak_src, "launches_timed": n_li, "avg_ms": ms_li / max(n_li, 1),
               "bytes_model": li_model}
    # DRAM traffic per launch: from the committed `ncu --set full` capture of the same kernels on the same workload (1 GPU);
    # the record carries the commit it was captured at -- null when no capture of this layout is committed
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        key = "design1" if args.design == 1 else ("design2_tiles" if os.environ.get("B200SFM_ELL") == "0" else "design2_ell")
        if tr.get("workload") == args.workload and world == 1 and key in tr:
            d = tr[key]
            roof_mv["traffic"] = sum(d["dram_bytes_per_launch"][k] for k in d["matvec_kernels"])
            roof_li["traffic"] = d["dram_bytes_per_launch"][d["linearize_kernel"]]
            roof_mv["traffic_source"] = roof_li["traffic_source"] = d["source"]
            roof_mv["traffic_captured_at_commit"] = roof_li["traffic_captured_at_commit"] = d.get("commit")
    except Exception:
        pass
    roof_mv["algorithmic_bytes"], roof_li["algorithmic_bytes"] = mv_bytes, li_bytes
    for r in (roof_mv, roof_li):
        r["frac"] = r["achieved"] / peak if r["achieved"] else None
    final_cost, init_cost = stats[-1]["final_cost"], stats[-1]["initial_cost"]
    if args.dump_outputs:
        intr, quat, trans, points = prob.get_state()
        out = {"points" if world == 1 else f"points_rank{rank}": points}
        if rank == 0:   # cameras and costs are replicated on every rank
            out.update(quat=quat, trans=trans, intr_params=intr, cost=np.array([init_cost, final_cost]))
        dump_outputs(args.dump_outputs, out)
    prob.free()

    # ---- end-to-end leg: one-shot C-ABI call with pinned host buffers ----------------
    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t.numpy(), t
    keep = []
    host = S.Scene(*[None] * 9)
    for f in ("pt_obs_begin", "obs_cam", "obs_xy", "cam_intr", "intr_model"):
        arr, t = pinned(getattr(sc, f)); keep.append(t); setattr(host, f, arr)
    state0 = {}
    for f in ("quat", "trans", "points", "intr_params"):
        arr, t = pinned(getattr(init, f)); keep.append(t); setattr(host, f, arr)
        state0[f] = np.array(arr, copy=True)
    opts_e = E.BundleAdjusterOptions(optimize_intrinsics=opt_intr, design=args.design)
    opts_e.solver_options.max_num_iterations = args.lm_iters
    opts_e.solver_options.pcg_rel_tolerance = args.pcg_tol
    opts_e.solver_options.pcg_max_iterations = args.pcg_max
    ba = E.BundleAdjuster(opts_e, ctx)
    e2e_stats = []

    def e2e_step():
        # harness work (restore the initial state in the pinned host buffers) is outside the timed region;
        # the timed region is exactly the public call: H2D of every input, solve, D2H of the result
        for f in state0:
            getattr(host, f)[...] = state0[f]
        barrier()
        t0 = time.perf_counter()
        ok = ba.Solve(host, mask)
        dt = time.perf_counter() - t0
        assert ok
        return ba.summary.as_dict(), dt

    for _ in range(min(args.warmup, 3)):
        e2e_step()
    e2e_walls = []
    for _ in range(args.e2e_steps):
        st_, dt = e2e_step()
        e2e_stats.append(st_)
        e2e_walls.append(maxr(dt))
    e2e_its = sum(s["iterations"] for s in e2e_stats)
    e2e_med = float(np.median(e2e_walls))
    e2e = {"value": n_global * (e2e_its / args.e2e_steps) / e2e_med, "unit": "observations/s per LM iteration",
           "h2d_bytes_per_step": int(e2e_stats[-1]["h2d_bytes"]), "d2h_bytes_per_step": int(e2e_stats[-1]["d2h_bytes"]),
           "steps": args.e2e_steps, "ms_per_step": 1e3 * e2e_med, "ms_per_step_all": [1e3 * w for w in e2e_walls],
           "ms_device_all": [s["ms_total"] for s in e2e_stats[-args.e2e_steps:]],
           "statistic": "median over the steps (ms_device_all: CUDA-event time of the same calls, create + H2D + solve + D2H)",
           "lm_iterations_per_step": e2e_its / args.e2e_steps,
           "ms_h2d_upload": e2e_stats[-1]["ms_h2d"], "ms_d2h": e2e_stats[-1]["ms_d2h"],
           "timed": "host wall clock around b200sfm_ba_solve with pinned host buffers, max over ranks"}

    cb = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb, _ = cpu_baseline(3, args.cpu_lm_iters)
    if rank == 0 and world == 1 and not args.no_parity:
        parity = gpu_parity(ctx, E, cb, args.pcg_tol)

    if rank == 0:
        line = {
            "metric": "observations/sec per BA LM-iteration", "value": value, "unit": "observations/s per LM iteration",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {C} cameras / {p_global} points / {nraw_global} observations "
                                   f"({n_global} in tracks >= 3 views) global BA, SIMPLE_PINHOLE, "
                                   + ("focal lengths refined (optimize_intrinsics, principal point fixed), " if opt_intr else "intrinsics constant, ") +
                                   f"0.5 px noise, start = GT perturbed 0.5 deg / 1% / 1%",
                       "parallelism": f"points sharded over {world} GPU(s), cameras replicated, NCCL all-reduce per PCG mat-vec",
                       "lm_iterations_per_step": lm_its / args.steps, "pcg_iterations_per_lm_iteration": pcg_its / max(lm_its, 1),
                       "pcg_rel_tolerance": args.pcg_tol, "preconditioner": "schur-jacobi", "design": "v1 (W blocks, atomics)" if args.design == 1 else "v2 (A_o rows, two passes)",
                       "l2_policy": "inputs_exceed_L2 (per-observation rows alone are 120-144 B x N >> 126 MB; every step restores the state and re-streams them)",
                       "cost": [init_cost, final_cost], "wall_ms_per_step": 1e3 * wall / args.steps,
                       "scene_generation_s": gen_s},
            "roofline": roof_mv, "roofline_linearize": roof_li,
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        }
        if cb:
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if parity:
            line["parity"] = parity
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config4", choices=list(WORKLOADS))
    ap.add_argument("--lm-iters", type=int, default=20, help="cap on LM iterations per solve (natural termination)")
    ap.add_argument("--pcg-tol", type=float, default=0.05,
                    help="PCG forcing tolerance: 0.05 keeps the LM iteration count within +-1 of the exact-solve CPU arm "
                         "(profiles/r2_tolerance_sweep.md); looser values buy cheaper but MORE LM iterations and would inflate the metric")
    ap.add_argument("--pcg-max", type=int, default=200)
    ap.add_argument("--optimize-intrinsics", type=int, default=0,
                    help="1: refine the camera intrinsics too (the reference's default BA mode); the headline line keeps them constant")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-lm-iters", type=int, default=1, help="LM iterations of the CPU port per step / sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the config-2 GPU-vs-CPU-port parity record")
    ap.add_argument("--design", type=int, default=0, help="BA data layout: 0 auto (v2), 1 = v1 (W blocks + atomics), 2 = v2")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's results; the CPU arm (--impl reference) has none")
    if args.workload == "config5":
        # BASELINE.json config 5 (100 k-frame view graph): rotation averaging, the secondary metric of SURVEY.md 8(d)
        # (edges/s per L1 / IRLS iteration).  Single GPU; the line is printed by bench_secondary.py in the same JSON style.
        if int(os.environ.get("RANK", "0")) != 0:
            return   # one GPU: under torchrun only rank 0 measures
        import bench_secondary as B2
        R = B2.bench_ra(argparse.Namespace(frames=100_000, neighbours=100, steps=args.steps, warmup=min(args.warmup, 1),
                                           pcg_tol=1e-6))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"rotations": R})
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
