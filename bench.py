#!/usr/bin/env python3
"""Benchmark of the calibration solve (BASELINE.json metric): trust-region
iterations per second on the 4-camera x 400-frame
LENSMODEL_SPLINED_STEREOGRAPHIC_order=3_Nx=30_Ny=20_fov_x_deg=170 synthetic
calibration (BASELINE config 3).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 3] [--dump-outputs DIR]

A "step" is one complete solve of the problem from the same seed. Prints ONE JSON
line (rank 0). See DESIGN.md "Measurement" for what every field means.

  value   iterations/s with the problem resident in HBM: Problem.reset() + Problem.optimize(),
          timed on the device with CUDA events inside the library (info.ms_total)
  e2e     the same metric through the reference-facing call mrcal_b200.optimize(**inputs)
          (C-ABI mrcal_optimize) with HOST buffers: H2D of every input and D2H of every
          output inside the timed region
  --impl reference   the CPU path on this box's host cores: the reference's own compiled
          mrcal_optimize() (oracle/_ref: mrcal.c unmodified) on top of a C restatement of
          libdogleg + a simplicial sparse Cholesky (oracle/port/dogleg_port.c); libdogleg and
          CHOLMOD themselves are not in the image. Single-threaded, like the reference.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "trust-region (LM/dogleg) iterations per second, 4cam x 400frame splined calibration"
UNIT = "iterations/s"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index=0):
        self.rows = []
        self.proc = None
        self.device_index = device_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.device_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def problem_inputs(config):
    # loaded by path: importing the package would dlopen libmrcal_b200.so, which the reference arm must not touch
    import importlib.util
    spec = importlib.util.spec_from_file_location("_mrcal_b200_synthetic", os.path.join(ROOT, "mrcal_b200", "synthetic.py"))
    synthetic = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synthetic)
    kw, truth = synthetic.baseline_config(config, pixel_noise=0.3)
    return kw


def describe(config, kw):
    return dict(workload=f"BASELINE config {config}: {kw['intrinsics'].shape[0]} cameras, "
                         f"{kw['rt_ref_frame'].shape[0]} frames, {kw['observations_board'].shape[2]}x"
                         f"{kw['observations_board'].shape[1]} board, {kw['lensmodel']}",
                lensmodel=kw["lensmodel"], Ncameras=int(kw["intrinsics"].shape[0]),
                Nframes=int(kw["rt_ref_frame"].shape[0]),
                Nobservations_board=int(kw["observations_board"].shape[0]),
                pixel_noise=0.3, seed="truth perturbed (mrcal_b200/synthetic.py, default_rng(0))",
                l2="working set per iteration (Jacobian strips 146 MB x2 + per-item Gram blocks + panels) exceeds the "
                   "126 MB L2; additionally a 256 MB buffer is written between timed steps")


def cpu_reference_run(kw, iterations):
    """`iterations` trust-region iterations of the CPU path from the seed: the reference's compiled mrcal_optimize()
    (oracle/_ref) with the iteration cap of the restated libdogleg set. Returns (iterations done, seconds, split)."""
    from oracle import ref
    if not ref.available():
        return None
    kw2 = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}
    kw2["do_apply_outlier_rejection"] = False   # a bounded sample: one pass
    P = ref.Problem(kw2)
    t0 = time.perf_counter()
    r = P.optimize(iteration_cap=iterations)
    dt = time.perf_counter() - t0
    inside = r["t_callback"] + r["t_factor"] + r["t_products"]
    return r["iterations"], dt, dict(callback_s=r["t_callback"], factor_solve_s=r["t_factor"], products_s=r["t_products"],
                                     outside_callback_and_factor_frac=(dt - r["t_callback"] - r["t_factor"]) / dt,
                                     solver_total_s=r["t_total"], wall_s=dt, accounted_frac=inside / dt,
                                     evaluations=r["evaluations"], factorizations=r["factorizations"],
                                     symbolic_analyses=r["symbolic"], nnz_L=r["Lnnz"])


CPU_SAMPLE = ("first {n} trust-region iterations of the same problem from the same seed: the reference's own compiled "
              "mrcal_optimize() (oracle/_ref; mrcal.c, its callback, pack/unpack and statistics unmodified) on a C "
              "restatement of libdogleg with a simplicial sparse Cholesky (minimum-degree ordering, up-looking LL'), "
              "oracle/port/dogleg_port.c; libdogleg/CHOLMOD themselves are absent from the image. 1 thread, as the reference")


def solve_config5(world, rank, local_rank, max_iterations):
    """BASELINE config 5 (8 cameras, 1000 frames, discrete points) solved once warm + once timed at the same N:
    the second number the verdict asks for next to config 3, whose replicated factorization caps its scaling."""
    import torch
    import mrcal_b200
    kw5 = problem_inputs(5)
    if world > 1:
        from mrcal_b200 import distributed
        kw5_local, shard5 = distributed.shard_inputs(kw5, rank, world)
    else:
        kw5_local, shard5 = kw5, None
    P5 = mrcal_b200.Problem(**kw5_local)
    if shard5 is not None:
        from mrcal_b200 import distributed
        distributed.attach(P5, shard5)
    out = None
    for k in range(2):
        P5.reset()
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        st = P5.optimize(max_iterations=max_iterations)
        ms = torch.tensor([st["ms_total"]], device="cuda", dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        out = dict(value=st["Niterations"] / (float(ms.item()) * 1e-3), unit=UNIT, iterations=st["Niterations"],
                   ms_per_solve=float(ms.item()), n_reduced=st["Nreduced"], Nstate=P5.Nstate, Nmeasurements=P5.Nmeasurements,
                   rms_reproj_error__pixels=st["rms_reproj_error__pixels"],
                   phase_ms_per_iteration={k2: st[k2] / max(1, st["Niterations"]) for k2 in ("ms_evaluate", "ms_assemble", "ms_factor", "ms_solve")},
                   collectives_per_iteration=st["Ncollectives"] / max(1, st["Niterations"]),
                   workload=f"BASELINE config 5: {kw5['intrinsics'].shape[0]} cameras, {kw5['rt_ref_frame'].shape[0]} frames, "
                            f"{kw5['points'].shape[0]} discrete points ({kw5['observations_point'].shape[0]} observations), {kw5['lensmodel']}")
    P5.close()
    return out


def dump_outputs(directory, arrays):
    """Writes what the timed path returned in its last step as DIR/<name>.npy (float64), so that two builds can be
    compared output for output: the inputs come from fixed seeds and are the same from run to run. Outputs the
    workload does not have (no discrete points, say) come back empty and are not written; scalars become 1-vectors."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        if a is None:
            continue
        a = np.atleast_1d(np.asarray(a, dtype=np.float64))
        if a.size:
            np.save(os.path.join(directory, f"{name}.npy"), a)


def measure_fp64_peak():
    """cuBLAS DGEMM throughput, the denominator for the fp64-tensor roofline (not in MEASURED_PEAKS.json)."""
    import torch
    n = 8192
    a = torch.randn(n, n, device="cuda", dtype=torch.float64)
    b = torch.randn(n, n, device="cuda", dtype=torch.float64)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--config", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true", help="skip the extra BASELINE config 5 solve reported next to config 3")
    ap.add_argument("--profile", action="store_true",
                    help="run under a profiler: only the device-resident steps (no e2e leg, no CPU baseline, no DGEMM peak "
                         "measurement); the numbers printed are not bench values")
    ap.add_argument("--max-iterations", type=int, default=300,
                    help="cap on trust-region iterations per solve (300 = the reference's; smaller only for profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the solution of the last one (b_packed, x, the unpacked state and "
                         "the observation weights; with --gpus > 1 the gathered state), its rms and outlier count as "
                         "DIR/<name>.npy in float64")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    kw = problem_inputs(args.config)
    config = describe(args.config, kw)

    ###################################################################################### reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        # a step = a bounded sample of the workload: the first 4 trust-region iterations from the seed
        iters_per_step = 4
        ncores = os.cpu_count()
        for _ in range(min(args.warmup, 1)):
            cpu_reference_run(kw, 1)
        tot_it, tot_s, split = 0, 0.0, None
        for _ in range(args.steps):
            r = cpu_reference_run(kw, iters_per_step)
            if r is None:
                print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmrcal_ref.so is missing"}))
                return 0
            tot_it += r[0]; tot_s += r[1]; split = r[2]
        v = tot_it / tot_s
        sample = CPU_SAMPLE.format(n=iters_per_step) + " (per step)"
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / args.steps,
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                                           "host_cores_available": ncores, "split": split},
                          "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    ###################################################################################### our arm
    import torch
    import mrcal_b200
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        from mrcal_b200 import distributed
        kw_local, shard = distributed.shard_inputs(kw, rank, world)
        distributed.init_comm(rank, world, local_rank)
    else:
        kw_local, shard = kw, None

    P = mrcal_b200.Problem(**kw_local)
    if shard is not None:
        from mrcal_b200 import distributed
        distributed.attach(P, shard)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize()

    def one_step():
        flush.zero_()
        torch.cuda.synchronize()
        P.reset()
        return P.optimize(max_iterations=args.max_iterations)

    for _ in range(args.warmup):
        one_step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    infos = []
    for _ in range(args.steps):
        infos.append(one_step())
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # read back before anything else runs on P; sharded, the full-size solution arrays are gathered from every rank
        if shard is None:
            sol = P.download(into_inputs=False)
        else:
            from mrcal_b200 import distributed
            sol = distributed.gather_solution(P, shard)
        if rank == 0:
            dump_outputs(args.dump_outputs, dict(sol, rms_reproj_error__pixels=infos[-1]["rms_reproj_error__pixels"],
                                                 Noutliers_board=infos[-1]["Noutliers_board"]))

    ms = np.array([i["ms_total"] for i in infos])
    its = np.array([i["Niterations"] for i in infos])
    dev_ms = float(ms.sum())
    if world > 1:
        t = torch.tensor([dev_ms], device="cuda", dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        dev_ms = float(t.item())
    value = float(its.sum()) / (dev_ms * 1e-3)

    ###### e2e: the reference-facing call with host buffers, H2D + D2H inside the timed region
    e2e = None
    if args.profile:
        print(json.dumps({"profile_run": True, "iterations": int(its.sum()), "ms": dev_ms,
                          "note": "run under a profiler: not a bench value"}))
        if world > 1:
            torch.distributed.destroy_process_group()
        return 0
    if world > 1:
        # sharded: the public multi-GPU API (mrcal_b200.distributed): each step re-uploads this rank's host
        # inputs, solves, and brings the solution back (D2H + all-gather of the frame poses)
        from mrcal_b200 import distributed
        h2d = sum(v.nbytes for v in kw_local.values() if isinstance(v, np.ndarray))
        e_it, e_s, d2h = 0, 0.0, 0
        for i in range(args.warmup + args.steps):
            flush.zero_()
            barrier()
            t0 = time.perf_counter()
            P.upload()
            st = P.optimize(max_iterations=args.max_iterations)
            sol = distributed.gather_solution(P, shard)
            barrier()
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                e_s += dt
                e_it += st["Niterations"]
                d2h = sum(v.nbytes for v in sol.values() if isinstance(v, np.ndarray)) + 8 * (P.Nstate + P.Nmeasurements)
        t = torch.tensor([e_s], device="cuda", dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e = {"value": e_it / float(t.item()), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": 1e3 * float(t.item()) / args.steps,
               "call": "mrcal_b200.distributed: Problem.upload() + Problem.optimize() + gather_solution(), per-rank host numpy buffers"}
    if world == 1:
        names = ("intrinsics", "rt_cam_ref", "rt_ref_frame", "calobject_warp", "observations_board")
        pinned = {n: torch.from_numpy(kw[n].copy()).pin_memory() for n in names}
        kw_e2e = dict(kw)
        for n in names:
            kw_e2e[n] = pinned[n].numpy()
        h2d = sum(v.nbytes for v in kw_e2e.values() if isinstance(v, np.ndarray))
        e_it, e_s, d2h = 0, 0.0, 0
        for i in range(args.warmup + args.steps):
            for n in names:
                np.copyto(kw_e2e[n], kw[n])
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = mrcal_b200.optimize(**kw_e2e)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                e_s += dt
                # the C-ABI returns no iteration count: the device-resident runs of the same problem give it
                e_it += int(round(its.mean()))
                d2h = out["b_packed"].nbytes + out["x"].nbytes + sum(kw_e2e[n].nbytes for n in names)
        e2e = {"value": e_it / e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": 1e3 * e_s / args.steps,
               "call": "mrcal_b200.optimize(**optimization_inputs) -> C-ABI mrcal_optimize(), host numpy buffers"}

    config5 = None
    if args.config == 3 and not args.no_config5:
        try:
            config5 = solve_config5(world, rank, local_rank, args.max_iterations)
        except Exception as e:   # pragma: no cover
            config5 = {"error": str(e)}
    if world > 1:
        torch.distributed.barrier()
    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return 0

    ###### roofline of the dominant kernel family
    # DRAM traffic per launch of the kernels named below, from the committed ncu capture (null if absent)
    traffic = {}
    for name in ("r02_dram_traffic.json", "r01c_dram_traffic.json"):
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", name)))
            break
        except Exception:
            pass
    last = infos[-1]
    n_c = last["Nreduced"]
    roofline = None
    try:
        peak = measure_fp64_peak()
        per_fact_s = 1e-3 * sum(i["ms_factor"] for i in infos) / max(1, sum(i["Nfactorizations"] for i in infos))
        flops = n_c ** 3 / 3.0
        achieved = flops / per_fact_s / 1e12
        roofline = {"bound": "tensor", "kernel": "reduced-system Cholesky: chol_spine_kernel (persistent, DMMA; chol_dataflow.cu)",
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "traffic": traffic.get("chol_spine_kernel", traffic.get("chol_dataflow_kernel")), "traffic_unit": "bytes per launch (ncu dram read+write)",
                    "flops_per_launch": flops, "n_reduced": n_c,
                    "peak_source": "cuBLAS DGEMM 8192^3 (torch.matmul fp64) measured in this run: MEASURED_PEAKS.json has no fp64 entry"}
    except Exception as e:   # pragma: no cover
        roofline = {"error": str(e)}
    # the Jacobian fill against HBM (SURVEY.md 8d: bytes_cb = 24 Ncorners + 8 Nstate + 8 Nmeas + 12 nnz + 4 (Nmeas+1))
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        hbm = peaks["hbm_gbs"]; hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        hbm = 6650.0; hbm_src = "fallback 6.65 TB/s (of fallback)"
    ms_cb = P.time_callback(20, True)
    ncorners = kw_local["observations_board"].shape[0] * kw_local["observations_board"].shape[1] * kw_local["observations_board"].shape[2]
    bytes_cb = 24 * ncorners + 8 * P.Nstate + 8 * P.Nmeasurements + 12 * P.N_j_nonzero + 4 * (P.Nmeasurements + 1)
    fill = {"bound": "hbm", "kernel": "eval_boards_kernel (residual + Jacobian fill)", "achieved": bytes_cb / (ms_cb * 1e-3) / 1e9,
            "peak": hbm, "unit": "GB/s", "frac": bytes_cb / (ms_cb * 1e-3) / 1e9 / hbm, "bytes_per_launch": bytes_cb,
            "ms_per_launch": ms_cb, "peak_source": hbm_src, "traffic": traffic.get("eval_boards_kernel")}

    # the assembly + Schur phase (SURVEY.md 8d): flops = sum_rows nnz(nnz+1) [JtJ] + sum_groups 6 k(k+1) [Schur, k = shared unknowns the
    # group touches]; bytes = the Jacobian read once (12 B per nonzero) + the residuals. Both rooflines are given; the phase is
    # bound by whichever takes longer at peak
    assembly = None
    try:
        idx = kw_local["indices_frame_camintrinsics_camextrinsics"]
        rows_per_obs = 2 * kw_local["observations_board"].shape[1] * kw_local["observations_board"].shape[2]
        Nreg = mrcal_b200.num_measurements_regularization(**kw_local)
        nnz_board = P.N_j_nonzero - 2 * Nreg          # splined regularization rows have 2 entries each
        n_ref = int((idx[:, 2] < 0).sum()); n_ext = idx.shape[0] - n_ref
        # widths of the two row classes (camera at the reference / with extrinsics) from the total: w_ext = w_ref + 6
        w_ref = (nnz_board / rows_per_obs - 6.0 * n_ext) / idx.shape[0]
        w_ext = w_ref + 6.0
        flops_jtj = rows_per_obs * (n_ref * w_ref * (w_ref + 1.0) + n_ext * w_ext * (w_ext + 1.0)) + Nreg * 2.0 * 3.0
        Ncam = int(kw_local["intrinsics"].shape[0])
        k_frame = Ncam * (2 * 36 + 6) + 2                  # shared unknowns a frame touches: a 6x6 knot patch per camera, extrinsics, warp
        flops_schur = float(kw_local["rt_ref_frame"].shape[0]) * 6.0 * k_frame * (k_frame + 1.0)
        flops_asm = flops_jtj + flops_schur
        bytes_asm = 12.0 * P.N_j_nonzero + 8.0 * P.Nmeasurements
        per_asm_s = 1e-3 * sum(i["ms_assemble"] for i in infos) / max(1, sum(i["Niterations"] for i in infos))
        t_flops = flops_asm / (roofline["peak"] * 1e12) if roofline and "peak" in roofline else None
        t_bytes = bytes_asm / (hbm * 1e9)
        bound = "hbm" if (t_flops is None or t_bytes >= t_flops) else "tensor"
        assembly = {"bound": bound, "kernel": "normal-equation assembly + Schur elimination per iteration: item_prepare_kernel, "
                                              "groups_panels_kernel, tile_plan_kernel, schur_tiles_kernel, reg_blocks_kernel (the observations' "
                                              "Gram blocks come from fused_boards_kernel, timed with the evaluation)",
                    "ms_per_iteration": per_asm_s * 1e3, "flops_per_assembly": flops_asm, "bytes_per_assembly": bytes_asm,
                    "achieved": (bytes_asm / per_asm_s / 1e9) if bound == "hbm" else (flops_asm / per_asm_s / 1e12),
                    "peak": hbm if bound == "hbm" else roofline["peak"], "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
                    "frac": (t_bytes if bound == "hbm" else t_flops) / per_asm_s,
                    "frac_hbm": t_bytes / per_asm_s, "frac_fp64_tensor": (t_flops / per_asm_s) if t_flops else None,
                    "traffic": (sum(traffic[k] for k in ("fused_boards_kernel", "groups_panels_kernel", "schur_tiles_kernel") if k in traffic)
                                if "schur_tiles_kernel" in traffic else None),
                    "traffic_note": "ncu dram read+write per launch: fused_boards_kernel + groups_panels_kernel + schur_tiles_kernel"}
    except Exception as e:   # pragma: no cover
        assembly = {"error": str(e)}

    ###### CPU baseline on this box's host cores: a bounded sample
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(kw, 6)
        if r is not None:
            cpu = {"value": r[0] / r[1], "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": CPU_SAMPLE.format(n=6),
                   "host_cores_available": os.cpu_count(), "split": r[2], "seconds": r[1]}

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic", "config": config,
           "iterations_per_step": float(its.mean()), "rms_reproj_error__pixels": last["rms_reproj_error__pixels"],
           "gpu_launches": int(sum(i["Nkernel_launches"] for i in infos)),
           "phase_ms_per_iteration": {k: float(sum(i[k] for i in infos) / its.sum())
                                      for k in ("ms_evaluate", "ms_assemble", "ms_factor", "ms_solve")},
           "host_syncs_per_iteration": float(sum(i["Nsyncs"] for i in infos) / its.sum()),
           "collectives_per_iteration": float(sum(i["Ncollectives"] for i in infos) / its.sum()),
           "clocks": clocks, "e2e": e2e, "roofline": roofline, "roofline_assembly": assembly,
           "roofline_jacobian_fill": fill, "config5": config5, "cpu_baseline": cpu}
    print(json.dumps(out))
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
