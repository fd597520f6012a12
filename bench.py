#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native hot path of apex-camera-models.

Metric (BASELINE.json): points/sec of the fused project + analytical Jacobian + J^T J / J^T r
pass.  Workload (BASELINE.json configs[2]): 100 M synthetic f64 correspondences per GPU, Double
Sphere model, pixel residual (project(X) - uv), inputs resident in HBM as SoA.  One step = one
streaming pass over the rank's shard (one kernel) + -- when N > 1 -- the NCCL all-reduce of the
29-double normal equations.  Weak scaling: every rank holds its own 100 M points.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port)

Prints ONE JSON result line on rank 0 (stdout); the per-kernel tables (`extras`, `roofline_by_kernel`)
follow as a second JSON line on stderr, which keeps the result line short enough for tools that
keep only the end of a command's output.  Timing: CUDA events on the launching stream, barrier +
synchronize on both sides, max over ranks.  Inputs (4 GB per rank) are far larger than the 126 MB
L2, so no explicit flush is needed between iterations.

    python bench.py --dump-outputs DIR   # also writes the normal equations of the last timed pass as DIR/*.npy
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# leave the tree as build() left it: build() never imports oracle/, so without this the first bench run would write
# oracle/__pycache__/ into a writable checkout
sys.dont_write_bytecode = True

METRIC = "points/sec project+Jacobian (fused project + analytical Jacobian + J^T J/J^T r)"
UNIT = "points/s"
N_POINTS = 100_000_000          # per GPU (BASELINE.json configs[2])
BYTES_PER_POINT = 40            # 24 B xyz + 16 B uv read per point per pass (SURVEY.md 8d)
SEED = 0xACE50003
COS_MAX = float(np.cos(np.deg2rad(85.0)))
KB_SAMPLE = [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504,
             0.0034823894022493434, 0.0007150348452162257, -0.0020532361418706202, 0.00020293673591811182]
DS_START = KB_SAMPLE[:4] + [0.6, 0.1]  # KB intrinsics with a Double Sphere guess: a model-mismatch fit like the converter's


def workload_config(n_gpus):
    return {"workload": "fused linearize (project + Jacobian + JtJ/Jtr), Double Sphere, pixel residual, f64 SoA",
            "camera_model": "double_sphere", "residual": "pixel", "points_per_gpu": N_POINTS, "global_points": N_POINTS * n_gpus,
            "correspondences": "X: seeded cone 85deg; uv = KannalaBrandt(samples/kannala_brandt.yaml).project(X)",
            "l2_policy": "inputs (4 GB/GPU) larger than L2", "parallelism": f"dp{n_gpus} (points sharded, all-reduce of 29 f64 fused into the kernel over NVLink peer memory)"}


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi in the background (B200_PROFILING.md clocks line)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.samples = []
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        atexit.register(self.stop)  # also when the run ends with an exception: nvidia-smi must not outlive bench.py
        def pump():
            for line in self.proc.stdout:
                self.samples.append((time.time(), line.strip()))
        threading.Thread(target=pump, daemon=True).start()

    def stop(self):
        if self.proc and self.proc.poll() is None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
                self.proc.wait()

    def summary(self, t0, t1):
        rows = []
        for ts, line in self.samples:
            if t0 <= ts <= t1:
                f = [x.strip() for x in line.split(",")]
                if len(f) >= 9:
                    rows.append(f)
        if not rows:
            return None
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "reasons": sorted(reasons), "samples": len(rows)}


def cpu_baseline(n_sample, min_seconds, nthreads):
    """The reference's algorithm for this path on the host: per-point residual + Jacobian
    materialised, then J^T J / J^T r (oracle port; the Rust reference cannot be built here).
    Returns points/s, passes, seconds and the normal equations (H, g, cost, n_valid) of the last pass."""
    from oracle import oracle as O
    O.build()
    kb = O.make_model(O.KB, KB_SAMPLE, 512, 512)
    ds = O.make_model(O.DS, DS_START, 512, 512)
    xyz = O.synth_points3(SEED, 0, n_sample, COS_MAX, False)
    uv, _ = O.project(kb, xyz, nthreads=max(nthreads, 1))
    O.linearize(ds, O.RES_PIXEL, xyz[:100000], uv[:100000], nthreads=nthreads)  # warm
    reps, t0 = 0, time.perf_counter()
    while True:
        last = O.linearize(ds, O.RES_PIXEL, xyz, uv, nthreads=nthreads)
        reps += 1
        el = time.perf_counter() - t0
        if el >= min_seconds and reps >= 1:
            break
    return n_sample * reps / el, reps, el, last


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    n_sample = 10_000_000
    vals = []
    for _ in range(max(args.warmup, 0)):
        cpu_baseline(200_000, 0.0, 1)
    for _ in range(args.steps):
        v, _, _, last = cpu_baseline(n_sample, 0.0, 1)
        vals.append(v)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last)
    value = float(np.median(vals))
    # beside it: the same port with OpenMP over every host core -- an upper bound the single-threaded reference does not have
    ncores = os.cpu_count() or 1
    try:
        v_all, _, _, _ = cpu_baseline(n_sample, 2.0, ncores)
        all_cores = {"value": v_all, "cores": ncores, "note": "OpenMP over every host core: a generous upper bound the single-threaded reference does not have"}
    except Exception as e:  # pragma: no cover
        all_cores = {"error": str(e)}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals), "warmup": args.warmup,
            "ms_per_step": 1e3 * n_sample / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": f"{n_sample} of the 100M correspondences per step; oracle C port of the reference algorithm (dense J then J^T J), gcc -O2 -ffp-contract=off, 1 thread (the reference is single-threaded Rust; no Rust toolchain in this image)",
                             "all_cores": all_cores},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes as C
    import torch
    import apex_camera_models_b200 as acm
    from apex_camera_models_b200 import _native as N
    lib = N.lib
    rank, local_rank, world = acm.distributed.env_rank_world()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    numa_cpus = None
    if world > 1 and not args.no_numa_bind:
        numa_cpus = acm.distributed.bind_to_gpu_numa(local_rank)   # pinned e2e buffers then sit next to their GPU
    ctx = acm.Context(local_rank)
    if world > 1:
        acm.attach_communicator(ctx)          # NCCL: linear estimation, fallback all-reduce
        if not args.no_peer:
            acm.attach_peers(ctx)             # NVLink peer exchange fused into the streaming kernel

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()
        ctx.sync()

    n = args.points
    # --- inputs generated in HBM: X from the seeded generator (rank-specific range), uv = KB.project(X)
    kb = acm.KannalaBrandtModel(acm.Intrinsics(*KB_SAMPLE[:4]), acm.Resolution(512, 512), KB_SAMPLE[4:], ctx=ctx)
    ds = acm.DoubleSphereModel(acm.Intrinsics(*DS_START[:4]), acm.Resolution(512, 512), DS_START[4:], ctx=ctx)
    X = acm.Points(ctx, 3, n)
    ctx.check(lib.acm_synth_points3(ctx.handle, SEED, rank * n, COS_MAX, 0, X.handle))
    UV, st = kb.project_batch(X)
    ctx.device_free(st)
    cam = ds.camera_block()

    def step():
        ctx.check(lib.acm_linearize_async(ctx.handle, C.byref(cam), N.RESIDUAL_PIXEL, X.handle, UV.handle))

    # --- correctness of the path that is about to be timed: the sharded pass over a fixed 2 M-point slice (every rank
    # its contiguous share, sums combined by the same fused exchange) against the CPU oracle on rank 0, and every rank
    # must hold bit-identical sums
    check = None
    if not args.no_check:
        check = oracle_check(acm, N, lib, ctx, kb, cam, rank, world, dist)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    launches0 = ctx.kernel_launches()
    wall0 = time.time()
    ctx.timer_start()
    for _ in range(args.steps):
        step()
    ms = ctx.timer_stop()
    barrier()
    wall1 = time.time()
    launches = ctx.kernel_launches() - launches0
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    value = n * world / (ms_per_step * 1e-3)

    clocks = sampler.summary(wall0, wall1) if rank == 0 else None
    probe = (wall1 - wall0) < 0.4  # same decision on every rank is not guaranteed by wall clocks -> agree on it
    if dist is not None:
        t = torch.tensor([1.0 if probe else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        probe = bool(t.item() > 0)
    if probe:
        # timed region shorter than the sampling period: run the same step for ~0.6 s on every rank
        n_probe = int(max(20, min(20000, 600.0 / max(ms_per_step, 1e-3))))
        p0 = time.time()
        for _ in range(n_probe):
            step()
        barrier()
        if rank == 0:
            clocks = sampler.summary(p0, time.time()) or clocks or {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
            clocks["sampled"] = "probe loop of the same step right after the timed region (timed region < 0.4 s)"

    # --- result of the last pass (also the d2h payload of the e2e path)
    ne = N.NormalEquations()
    ctx.check(lib.acm_linearize(ctx.handle, C.byref(cam), N.RESIDUAL_PIXEL, X.handle, UV.handle, C.byref(ne)))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *unpack_normal_equations(ne))

    # --- e2e: host AoS buffers (nalgebra layout, pinned) through acm_linearize_host, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        ne_pts = min(n, args.e2e_points)
        hx = ctx.pinned_empty((ne_pts, 3), np.float64)
        hu = ctx.pinned_empty((ne_pts, 2), np.float64)
        # fill the host buffers from the device data (download is outside the timed region)
        Xs = acm.Points(ctx, 3, ne_pts); Us = acm.Points(ctx, 2, ne_pts)
        for c in range(3):
            ctx.d2d(Xs.component_ptr(c), X.component_ptr(c), 8 * ne_pts)
        for c in range(2):
            ctx.d2d(Us.component_ptr(c), UV.component_ptr(c), 8 * ne_pts)
        ctx.check(lib.acm_points_download_aos_f64(ctx.handle, Xs.handle, hx.ctypes.data_as(C.c_void_p), ne_pts))
        ctx.check(lib.acm_points_download_aos_f64(ctx.handle, Us.handle, hu.ctypes.data_as(C.c_void_p), ne_pts))
        Xs.free(); Us.free()
        ne2 = N.NormalEquations()
        def e2e_step():
            ctx.check(lib.acm_linearize_host(ctx.handle, C.byref(cam), N.RESIDUAL_PIXEL, hx.ctypes.data_as(C.c_void_p), hu.ctypes.data_as(C.c_void_p),
                                             ne_pts, C.byref(ne2)))
        e2e_step()
        barrier()
        k = max(1, min(args.steps, args.e2e_steps))
        t0 = time.perf_counter()
        for _ in range(k):
            e2e_step()
        barrier()
        el = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([el], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            el = float(t.item())
        e2e = {"value": ne_pts * world * k / el, "unit": UNIT, "h2d_bytes_per_step": ne_pts * BYTES_PER_POINT,
               "d2h_bytes_per_step": 29 * 8, "steps": k, "points_per_gpu": ne_pts,
               "api": "acm_linearize_host (pinned nalgebra-layout AoS f64 -> chunked H2D + AoS->SoA + fused pass -> normal equations)",
               "numa_bound_cpus": len(numa_cpus) if numa_cpus else None}
        ctx.pinned_free(hx); ctx.pinned_free(hu)

    extras = None
    if not args.no_extras:
        barrier()
        mine = run_extras(acm, N, lib, ctx, X, UV, n, sampler if rank == 0 else None, barrier)
        if dist is not None:
            gathered = [None] * world
            dist.all_gather_object(gathered, mine)
        else:
            gathered = [mine]
        if rank == 0:
            extras = merge_extras(gathered, n, world)

    # --- LM conversion (BASELINE config 4): KB -> Double Sphere, 10 M correspondences sharded over the ranks
    lm = None
    if not args.no_lm:
        n_lm_total = 10_000_000
        lo, hi = acm.shard_range(n_lm_total, rank, world)
        m = hi - lo
        Xl = acm.Points(ctx, 3, m); Ul = acm.Points(ctx, 2, m)
        ctx.check(lib.acm_synth_points3(ctx.handle, 0xACE50004, lo, COS_MAX, 0, Xl.handle))
        cam_kb = kb.camera_block()
        ctx.check(lib.acm_project(ctx.handle, C.byref(cam_kb), Xl.handle, Ul.handle, None))
        dsl = acm.DoubleSphereModel(acm.Intrinsics(*KB_SAMPLE[:4]), acm.Resolution(512, 512), [0.5, 0.1], ctx=ctx)
        cost = acm.DoubleSphereOptimizationCost(dsl, Xl, Ul)  # canonical (algebraic) residual, converter bounds
        barrier()
        cost.linear_estimation()  # Gram sums are combined over the ranks inside libacm
        start = dsl.params().copy()
        cost.optimize()      # warm-up solve
        dsl.set_params(start)
        barrier()
        r = cost.optimize()
        barrier()
        ms_lm, dev_lm = r.elapsed_ms, r.device_ms
        if dist is not None:
            t = torch.tensor([ms_lm, dev_lm], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_lm, dev_lm = float(t[0].item()), float(t[1].item())
        params_raw = np.asarray(r.parameters, dtype=np.float64).tobytes()
        lm_identical = True
        if dist is not None:
            allp = acm.distributed.all_gather_bytes(params_raw)
            lm_identical = all(allp[i * len(params_raw):(i + 1) * len(params_raw)] == params_raw for i in range(world))
        lm = {"workload": "KB->DoubleSphere LM, 10M correspondences (algebraic residual, converter tolerances/bounds)", "ms": ms_lm,
              "device_ms": dev_lm, "iterations": r.iterations, "passes": r.passes, "status": r.status,
              "us_per_pass": 1e3 * ms_lm / max(r.passes, 1), "device_us_per_pass": 1e3 * dev_lm / max(r.passes, 1),
              "timing": "ms = host wall of acm_lm_solve (upload of the 1 KB state, ONE kernel launch, read-back); device_ms = %globaltimer from the first pass to the last LM step inside that kernel; max over ranks",
              "params": [float(v) for v in r.parameters], "final_cost": r.final_cost, "points_per_gpu": m, "rank_identical": bool(lm_identical)}
        # --- the converter steps around the solve, sharded the same way (SURVEY 8e rows e3, e5, e6): linear estimation,
        # reprojection statistics of the converged model over the sharded correspondences, sample_points over the sharded grid
        lin_start = [float(v) for v in start]
        err = acm.compute_reprojection_error(dsl, Xl, Ul)      # statistics of the WHOLE set on every rank (sums / histogram all-reduced)
        n_req = 1_000_000
        s_uv, s_xyz = acm.sample_points(kb, n_req, device=True, shard=(rank, world))
        su = s_uv.numpy()
        kept_local = int(su.shape[0])
        xor_local = int(np.bitwise_xor.reduce(su.view(np.uint64).ravel())) if kept_local else 0   # order-independent, exact
        s_uv.free(); s_xyz.free()
        pipe_local = np.array([kept_local, xor_local & 0xFFFFFFFF, xor_local >> 32], dtype=np.float64)
        if dist is not None:
            tl = [torch.zeros(3, dtype=torch.float64, device="cuda") for _ in range(world)]
            dist.all_gather(tl, torch.tensor(pipe_local, device="cuda"))
            pipe_all = [t.cpu().numpy() for t in tl]
            te = torch.tensor([err.mean, err.median, err.max, float(err.count)], dtype=torch.float64, device="cuda")
            tmin, tmax = te.clone(), te.clone()
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            stats_identical = bool(torch.equal(tmin, tmax))
        else:
            pipe_all = [pipe_local]; stats_identical = True
        lm["pipeline"] = {"reprojection_error": {"mean": err.mean, "median": err.median, "max": err.max, "count": int(err.count), "rank_identical": stats_identical},
                          "sample_points": {"requested": n_req, "kept_per_rank": [int(p[0]) for p in pipe_all]}}
        if rank == 0 and not args.no_lm_check:
            # the same conversion through the CPU oracle (all host threads; it walks the same algorithm): parameters <= 1e-9 relative
            from oracle import oracle as O
            O.build()
            t0 = time.perf_counter()
            xyz = O.synth_points3(0xACE50004, 0, n_lm_total, COS_MAX, False)
            uvo, _ = O.project(O.make_model(O.KB, KB_SAMPLE, 512, 512), xyz, nthreads=os.cpu_count() or 1)
            om = O.make_model(O.DS, KB_SAMPLE[:4] + [0.5, 0.1], 512, 512)
            O.linear_estimation(om, xyz, uvo)
            om_lin = om.params().copy()
            b = acm.CONVERTER_BOUNDS[5]
            po, ro = O.lm_solve(om, O.RES_ALGEBRAIC, xyz, uvo, [x[0] for x in b], [x[1] for x in b], nthreads=os.cpu_count() or 1)
            rel = float(np.max(np.abs(np.asarray(r.parameters) - po) / np.abs(po)))
            lin_o = om_lin
            lin_rel = float(np.max(np.abs(np.asarray(lin_start) - lin_o) / np.maximum(np.abs(lin_o), 1e-300)))
            omf = O.make_model(O.DS, [float(v) for v in r.parameters], 512, 512)
            eo = O.reprojection_error(omf, xyz, uvo)
            stat_rel = float(max(abs(err.mean - eo.mean) / eo.mean, abs(err.median - eo.median) / eo.median, abs(err.max - eo.max) / eo.max))
            uvs, _ = O.sample_points(O.make_model(O.KB, KB_SAMPLE, 512, 512), n_req)
            xor_o = int(np.bitwise_xor.reduce(uvs.view(np.uint64).ravel()))
            xor_g = 0
            for p in pipe_all:
                xor_g ^= int(p[1]) | (int(p[2]) << 32)
            kept_g = sum(int(p[0]) for p in pipe_all)
            lm["vs_oracle"] = {"params_rel": rel, "same_trajectory": bool((r.status, r.iterations, r.passes) == (ro.status, ro.iterations, ro.passes)),
                               "linear_estimation_rel": lin_rel, "reprojection_stats_rel": stat_rel, "reprojection_count_equal": bool(int(err.count) == int(eo.count)),
                               "sample_points_kept": [kept_g, int(uvs.shape[0])], "sample_points_pixels_identical": bool(kept_g == uvs.shape[0] and xor_g == xor_o),
                               "oracle_s": time.perf_counter() - t0}
            v = lm["vs_oracle"]
            v["ok"] = bool(rel <= 1e-9 and lin_rel <= 1e-9 and stat_rel <= 1e-9 and v["reprojection_count_equal"] and v["sample_points_pixels_identical"] and stats_identical)
            del xyz, uvo
        Xl.free(); Ul.free()

    # --- undistort (BASELINE config 5): 4096x4096 KB fisheye frames (sample intrinsics x8), 32 frames per GPU resident in
    # HBM = the per-GPU share of the 256-frame batch on 8 GPUs; frames shard over the ranks, no collective
    und = None
    if not args.no_undistort:
        Wd = Hd = 4096
        kb8 = acm.KannalaBrandtModel(acm.Intrinsics(*(v * 8 for v in KB_SAMPLE[:4])), acm.Resolution(Wd, Hd), KB_SAMPLE[4:], ctx=ctx)
        cam8 = kb8.camera_block()
        F = 32
        fb = Wd * Hd * 3
        d_in = ctx.device_alloc(fb * F); d_out = ctx.device_alloc(fb * F)
        ctx.check(lib.acm_synth_bytes(ctx.handle, 0xACE50005, rank * F * fb, C.c_void_p(d_in), fb * F))
        und = {"workload": "undistort 4096x4096 RGB8 KB fisheye frames, 32 per GPU resident in HBM (256-frame batch at 8 GPUs)", "frames_per_gpu": F}
        for interp, name in ((1, "bilinear"), (0, "nearest")):
            f_und = lambda: ctx.check(lib.acm_undistort_rgb8(ctx.handle, C.byref(cam8), None, C.c_void_p(d_in), C.c_void_p(d_out), F, interp))
            for _ in range(3):
                f_und()
            barrier()
            ctx.timer_start()
            for _ in range(5):
                f_und()
            ms_u = ctx.timer_stop() / 5
            barrier()
            if dist is not None:
                t = torch.tensor([ms_u], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms_u = float(t.item())
            und[name] = {"ms": ms_u, "frames_s": F * world / ms_u * 1e3, "gb_s_per_gpu": 2 * fb * F / ms_u / 1e6, "us_per_frame": ms_u / F * 1e3}
        ctx.device_free(d_in); ctx.device_free(d_out)

    if rank == 0:
        sampler.stop()
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback, B200_PROFILING.md)"
        achieved = n * BYTES_PER_POINT / (ms_per_step * 1e-3) / 1e9  # per GPU; at N>1 the step also holds the all-reduce
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("linearize_ds_pixel_bytes_per_launch")
        except (OSError, ValueError):
            pass
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": workload_config(world), "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                             "kernel": "linearize_kernel<DOUBLE_SPHERE, PIXEL>", "algorithmic_bytes_per_launch": n * BYTES_PER_POINT,
                             "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0},
                "e2e": e2e, "lm_conversion": lm, "undistort_batch": und, "check": check,
                "last_pass": {"n_valid": int(ne.n_valid), "cost": float(ne.cost), "H00": float(ne.H[0])}}
        if world == 1 and not args.no_cpu:
            v1, reps, el, _ = cpu_baseline(args.cpu_points, 10.0, 1)
            ncores = os.cpu_count() or 1
            vall, _, _, _ = cpu_baseline(args.cpu_points, 3.0, ncores)
            line["cpu_baseline"] = {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": f"{args.cpu_points} of the 100M correspondences x {reps} passes ({el:.1f} s); oracle C port (dense J, then J^T J), 1 thread like the single-threaded reference",
                                    "all_cores": {"value": vall, "cores": ncores, "note": "OpenMP over every host core: a generous upper bound the reference does not have"}}
        detail = None
        if extras:
            detail = {"extras": extras}
            # one roofline entry per fused kernel (model / residual), same definition as the headline entry
            detail["roofline_by_kernel"] = {k: {"bound": "hbm", "achieved": v["gb_s"], "peak": peak, "unit": "GB/s", "frac": v["gb_s"] / peak,
                                                "frac_of_nominal_8TBs": v["gb_s"] / 8000.0, "ms": v["ms"]}
                                            for k, v in extras.get("linearize_100M", {}).items()}
            for k, v in extras.get("linearize_100M", {}).items():
                if v.get("sustained_ms"):
                    gb = n * 40 / v["sustained_ms"] / 1e6
                    detail["roofline_by_kernel"][k]["sustained"] = {"achieved": gb, "frac": gb / peak, "ms": v["sustained_ms"], "sm_mhz": v.get("sm_mhz"),
                                                                    "how": "the same launch back to back for ~0.4 s; `achieved` above is a 10-launch burst"}
            # the FP64-bound ones also against the FP64 issue rate at the clock sampled during a ~0.4 s loop of that kernel
            for k, ipp in FP64_INSTR_PER_POINT.items():
                v = extras.get("linearize_100M", {}).get(k)
                if v and v.get("sustained_ms") and v.get("sm_mhz"):
                    rate = ipp * n / (v["sustained_ms"] * 1e-3)
                    detail["roofline_by_kernel"][k]["fp64"] = {
                        "instr_per_point": ipp, "sustained_ms": v["sustained_ms"], "sustained_gb_s": n * 40 / v["sustained_ms"] / 1e6, "sm_mhz": v["sm_mhz"],
                        "issue_frac_at_clock": rate / (FP64_LANES_PER_CLOCK * v["sm_mhz"] * 1e6),
                        "note": "FP64 lane-instructions issued per second / (148 SMs x 64 lanes x sampled SM clock); ncu shows ~75 % as the practical ceiling (math-pipe throttle)"
                                + ("" if world == 1 else "; N > 1: the time is the slowest rank's, the clock rank 0's, so the fraction is a lower bound")}
        if check is not None and not check.get("ok", False):
            line["check_failed"] = True
        if detail:
            print(json.dumps(detail), file=sys.stderr, flush=True)
        print(json.dumps(line), flush=True)
        if check is not None and not check.get("ok", False):
            raise SystemExit("bench.py: the sharded pass disagrees with the oracle (see \"check\")")
        if lm and lm.get("vs_oracle") and not lm["vs_oracle"].get("ok", False):
            raise SystemExit("bench.py: the sharded converter pipeline disagrees with the oracle (see \"lm_conversion.vs_oracle\")")
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def unpack_normal_equations(ne):
    """acm_normal_equations -> (H (P x P), g (P), cost, n_valid)."""
    P = ne.n_params
    return np.array(ne.H[:P * P]).reshape(P, P), np.array(ne.g[:P]), ne.cost, ne.n_valid


def dump_outputs(out_dir, H, g, cost, n_valid):
    """What a caller of the timed path receives (the normal equations H, g, cost, n_valid) as float64 DIR/<name>.npy.
    The GPU arm reads them with one more acm_linearize on the same inputs after the timed steps: the pass reduces in a
    fixed order (no float atomics), so that equals the last timed pass bit for bit (repeat runs are compared bit for bit
    in tests/test_gpu_parity.py)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in {"H": H, "g": g, "cost": [cost], "n_valid": [n_valid]}.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def merge_extras(per_rank, n, world):
    """Max over ranks of every timing; throughput = points of all ranks / that time (weak scaling: n points per rank)."""
    out = {}
    for group, rows in per_rank[0].items():
        out[group] = {}
        for name, row in rows.items():
            merged = {}
            for key, val in row.items():
                if key.endswith("ms"):
                    merged[key] = max(r[group][name][key] for r in per_rank)
                elif key.startswith("_r0_"):
                    merged[key[4:]] = val   # sampled on rank 0 only
            for key, val in row.items():
                if key.endswith("_bytes_per_point"):
                    base = key[: -len("_bytes_per_point")]
                    ms = merged[(base + "_ms") if base else "ms"]
                    merged[(base + "_" if base else "") + "gpts_s"] = n * world / ms / 1e6
                    merged[(base + "_" if base else "") + "gb_s"] = n * val / ms / 1e6          # per GPU
                    merged[(base + "_" if base else "") + "gb_s_all_gpus"] = n * world * val / ms / 1e6
            out[group][name] = merged
    return out


CHECK_POINTS = 2_000_000
CHECK_SEED = 0xACE500C3


def oracle_check(acm, N, lib, ctx, kb, cam, rank, world, dist):
    import ctypes as C
    lo, hi = acm.shard_range(CHECK_POINTS, rank, world)
    Xc = acm.Points(ctx, 3, hi - lo)
    ctx.check(lib.acm_synth_points3(ctx.handle, CHECK_SEED, lo, COS_MAX, 0, Xc.handle))
    Uc, st = kb.project_batch(Xc)
    ctx.device_free(st)
    ne = N.NormalEquations()
    ctx.check(lib.acm_linearize(ctx.handle, C.byref(cam), N.RESIDUAL_PIXEL, Xc.handle, Uc.handle, C.byref(ne)))
    Xc.free(); Uc.free()
    raw = bytes(memoryview(ne))
    identical = True
    if dist is not None:
        allraw = acm.distributed.all_gather_bytes(raw)
        identical = all(allraw[i * len(raw):(i + 1) * len(raw)] == raw for i in range(world))
    out = {"points": CHECK_POINTS, "rank_identical": bool(identical), "n_valid": int(ne.n_valid), "cost": float(ne.cost)}
    if rank == 0:
        from oracle import oracle as O
        O.build()
        xyz = O.synth_points3(CHECK_SEED, 0, CHECK_POINTS, COS_MAX, False)
        uv, _ = O.project(O.make_model(O.KB, KB_SAMPLE, 512, 512), xyz, nthreads=os.cpu_count() or 1)
        Ho, go, co, no = O.linearize(O.make_model(O.DS, DS_START, 512, 512), O.RES_PIXEL, xyz, uv, nthreads=os.cpu_count() or 1)
        H, g, _, _ = unpack_normal_equations(ne)
        # entry-wise relative error against the scale of the entry's row/column (g and the off-diagonals cancel)
        dH = np.abs(H - Ho) / np.sqrt(np.outer(np.diag(Ho), np.diag(Ho)))
        dg = np.abs(g - go) / np.sqrt(np.diag(Ho) * 2.0 * co)
        rel = float(max(dH.max(), dg.max(), abs(ne.cost - co) / co))
        out.update({"vs_oracle_rel": rel, "n_valid_oracle": int(no), "ok": bool(rel <= 1e-9 and int(no) == int(ne.n_valid) and identical)})
    return out


# FP64 instructions per point in the streaming loop of the FP64-bound fused kernels (DFMA + DMUL + DADD + DSETP, counted in the
# SASS with scripts/sass_loop_stats.py; DESIGN.md 4.1).  The B200 issues 148 SMs x 64 FP64 lane-instructions per clock.
FP64_INSTR_PER_POINT = {"double_sphere/pixel": 77, "kannala_brandt/pixel": 102, "rad_tan/pixel": 99, "fov/pixel": 82}
FP64_LANES_PER_CLOCK = 148 * 64


def run_extras(acm, N, lib, ctx, X, UV, n, sampler=None, barrier=None):
    """Every other kernel of the path on this rank's 100 M points: the fused pass of every model / residual (config 3),
    project / unproject / fused round trip for all models in f64 and f32 I/O (config 2), project + Jacobians."""
    import ctypes as C
    out = {}
    def timeit(fn, reps=10):
        for _ in range(3):
            fn()
        ctx.sync(); ctx.timer_start()
        for _ in range(reps):
            fn()
        return ctx.timer_stop() / reps
    def agree_max(v):
        import torch
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    intr = KB_SAMPLE[:4]
    dist_init = {0: [], 1: [0.01, 0.001, 0.0, 0.0, 0.0], 2: KB_SAMPLE[4:], 3: [0.6], 4: [0.6, 1.0], 5: [0.6, 0.1], 6: [0.9]}
    names = {0: "pinhole", 1: "rad_tan", 2: "kannala_brandt", 3: "ucm", 4: "eucm", 5: "double_sphere", 6: "fov"}
    lin = {}
    for mid in (5, 4, 3, 2, 6, 1, 0):
        m = acm.MODEL_CLASSES[mid](acm.Intrinsics(*intr), acm.Resolution(512, 512), dist_init[mid], ctx=ctx)
        cam = m.camera_block()
        for kind, kname in ((0, "pixel"), (1, "algebraic")):
            if kind == 1 and mid not in (3, 4, 5):
                continue
            fn = lambda: ctx.check(lib.acm_linearize_async(ctx.handle, C.byref(cam), kind, X.handle, UV.handle))
            ms = timeit(fn)
            row = {"ms": ms, "_bytes_per_point": 40}
            # the same launch for ~0.4 s with the SM clock sampled next to it: the 10-launch burst above runs at whatever
            # clock the previous kernel left behind (the power cap reacts over ~100 ms), which flatters the HBM-bound
            # kernels and penalises the FP64-bound ones; the FP64 issue rate is quoted at the clock sampled here
            # every rank must issue the same number of launches (each one is an exchange): agree on the slowest rank's time
            reps = int(max(20, min(2000, 400.0 / max(agree_max(ms), 1e-3))))
            if barrier:
                barrier()
            w0 = time.time()
            ctx.sync(); ctx.timer_start()
            for _ in range(reps):
                fn()
            row["sustained_ms"] = ctx.timer_stop() / reps
            if barrier:
                barrier()
            w1 = time.time()
            ck = sampler.summary(w0, w1) if sampler else None
            if ck:
                row["_r0_sm_mhz"] = ck["sm_mhz"]
            lin[f"{names[mid]}/{kname}"] = row
    out["linearize_100M"] = lin
    pu = {}
    UV2 = acm.Points(ctx, 2, n); X2 = acm.Points(ctx, 3, n)
    st = ctx.device_alloc(n); st2 = ctx.device_alloc(n)
    for mid in range(7):
        m = acm.MODEL_CLASSES[mid](acm.Intrinsics(*intr), acm.Resolution(512, 512), dist_init[mid], ctx=ctx)
        cam = m.camera_block()
        ms = timeit(lambda: ctx.check(lib.acm_project(ctx.handle, C.byref(cam), X.handle, UV2.handle, C.c_void_p(st))))
        ctx.check(lib.acm_synth_pixels(ctx.handle, 7, 0, 512.0, 512.0, UV2.handle))
        ms2 = timeit(lambda: ctx.check(lib.acm_unproject(ctx.handle, C.byref(cam), UV2.handle, X2.handle, C.c_void_p(st))))
        ms3 = timeit(lambda: ctx.check(lib.acm_project_unproject(ctx.handle, C.byref(cam), X.handle, UV2.handle, X2.handle, C.c_void_p(st), C.c_void_p(st2))))
        pu[names[mid]] = {"project_ms": ms, "project_bytes_per_point": 41, "unproject_ms": ms2, "unproject_bytes_per_point": 41,
                          "round_trip_fused_ms": ms3, "round_trip_fused_bytes_per_point": 66}
    out["project_unproject_100M_f64"] = pu
    # project with compute_jacobian = true (2 x P parameter Jacobian, 2 x 3 point Jacobian), on a 20 M-point prefix:
    # 24 B in + 16 B uv + 1 B status + 16 P (or 48) B of Jacobian rows out per point
    nj = min(n, 20_000_000)
    Xj = acm.Points(ctx, 3, nj); Uj = acm.Points(ctx, 2, nj)
    for c in range(3):
        ctx.d2d(Xj.component_ptr(c), X.component_ptr(c), 8 * nj)
    jac = ctx.device_alloc(8 * nj * 18)
    pj = {}
    for mid in range(7):
        m = acm.MODEL_CLASSES[mid](acm.Intrinsics(*intr), acm.Resolution(512, 512), dist_init[mid], ctx=ctx)
        cam = m.camera_block()
        P = cam.n_params
        msj = timeit(lambda: ctx.check(lib.acm_project_jacobian(ctx.handle, C.byref(cam), Xj.handle, Uj.handle, C.c_void_p(jac), C.c_void_p(st))), reps=5)
        msp = timeit(lambda: ctx.check(lib.acm_project_point_jacobian(ctx.handle, C.byref(cam), Xj.handle, Uj.handle, C.c_void_p(jac), C.c_void_p(st))), reps=5)
        pj[names[mid]] = {"param_jacobian_ms": msj * n / nj, "param_jacobian_bytes_per_point": 41 + 16 * P,
                          "point_jacobian_ms": msp * n / nj, "point_jacobian_bytes_per_point": 41 + 48}
    out["project_jacobian_f64_scaled_from_20M"] = pj
    ctx.device_free(jac); Xj.free(); Uj.free()
    UV2.free(); X2.free()
    # f32 I/O (BASELINE config 2 "f64 and f32"): 21 / 21 / 34 B per point, arithmetic still f64 so the masks stay exact
    pu32 = {}
    Xf = acm.Points(ctx, 3, n, N.F32); UVf = acm.Points(ctx, 2, n, N.F32); X2f = acm.Points(ctx, 3, n, N.F32)
    ctx.check(lib.acm_synth_points3(ctx.handle, SEED, 0, COS_MAX, 0, Xf.handle))
    for mid in range(7):
        m = acm.MODEL_CLASSES[mid](acm.Intrinsics(*intr), acm.Resolution(512, 512), dist_init[mid], ctx=ctx)
        cam = m.camera_block()
        ms = timeit(lambda: ctx.check(lib.acm_project(ctx.handle, C.byref(cam), Xf.handle, UVf.handle, C.c_void_p(st))))
        ctx.check(lib.acm_synth_pixels(ctx.handle, 7, 0, 512.0, 512.0, UVf.handle))
        ms2 = timeit(lambda: ctx.check(lib.acm_unproject(ctx.handle, C.byref(cam), UVf.handle, X2f.handle, C.c_void_p(st))))
        ms3 = timeit(lambda: ctx.check(lib.acm_project_unproject(ctx.handle, C.byref(cam), Xf.handle, UVf.handle, X2f.handle, C.c_void_p(st), C.c_void_p(st2))))
        pu32[names[mid]] = {"project_ms": ms, "project_bytes_per_point": 21, "unproject_ms": ms2, "unproject_bytes_per_point": 21,
                            "round_trip_fused_ms": ms3, "round_trip_fused_bytes_per_point": 34}
    out["project_unproject_100M_f32"] = pu32
    Xf.free(); UVf.free(); X2f.free()
    ctx.device_free(st); ctx.device_free(st2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=N_POINTS, help="points per GPU")
    ap.add_argument("--e2e-points", type=int, default=N_POINTS)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-points", type=int, default=20_000_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the pre-timing comparison of the sharded pass with the CPU oracle")
    ap.add_argument("--no-lm-check", action="store_true", help="skip the oracle LM run beside the 10 M-correspondence conversion")
    ap.add_argument("--no-lm", action="store_true")
    ap.add_argument("--no-undistort", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--no-peer", action="store_true", help="N > 1: keep the NCCL all-reduce instead of the fused NVLink exchange")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the normal equations of the last timed pass as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
