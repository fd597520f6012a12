"""Throughput of acm_render_depth and the per-sweep cost of render_depth, with the card, its power limit and SM clock read in
the same run.

    python scripts/depth_bench.py [--points 100000000] [--timed 20] [--out profiles/r03_depth_bench.log]

  * render: --points resident points of acm_synth_points3 (KB through a 100-degree cone, Pinhole through a 40-degree cone)
    into 1920x1080 and into 320x240 (heavy contention: ~1300 points per pixel), and --points / 10 into 4096x4096 (a 134 MB
    key image, beyond the 126 MB L2).  A call is the key memset, the render kernel and the resolve kernel; 3 warm-up calls,
    then the median of --timed calls between CUDA events.  Reports G points/s and algorithmic GB/s: 24 B per point read
    plus 24 B per pixel (key init, key read, range + index write).
  * per sweep: render_depth on n = 10^5 numpy points into 1920x1080 (host copies included), wall time per call.
  * CPU comparison: the depth oracle (tests/depth_oracle.c, -O2, one thread) on the same points; its images are compared with
    the GPU's (byte-identical for Pinhole; pixels that differ for KB).
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=100_000_000)
    ap.add_argument("--timed", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import apex_camera_models_b200 as acm
    from apex_camera_models_b200 import _native as N
    import depth_oracle as D
    from oracle import oracle as O
    O.build()
    cams = {  # the KB sample camera and the pinhole sample camera, focal lengths scaled to the image width
        "kannala_brandt": (2, [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434,
                               0.0007150348452162257, -0.0020532361418706202, 0.00020293673591811182], 512, 100.0),
        "pinhole": (0, [461.629, 460.152, 362.68, 246.049], 752, 40.0),
    }
    lines = [f"card: {card()}", f"points: {a.points}, timed calls: {a.timed} (median), warm-up: 3"]
    ctx = acm.Context(0)
    L = N.lib
    R9, t3 = (C.c_double * 9)(*np.eye(3).ravel()), (C.c_double * 3)()

    def run(model_id, params, W0, W, H, n, cone_deg, seed):
        s = W / W0
        p = list(params)
        p[0], p[1], p[2], p[3] = p[0] * s, p[1] * s, W / 2.0 + 0.3, H / 2.0 - 0.2
        g = acm.MODEL_CLASSES[model_id](acm.Intrinsics(*p[:4]), acm.Resolution(W, H), p[4:], ctx=ctx)
        cam = g.camera_block()
        cos = float(np.cos(np.deg2rad(cone_deg)))
        X = acm.Points(ctx, 3, n)
        ctx.check(L.acm_synth_points3(ctx.handle, seed, 0, cos, 0, X.handle))
        npix = W * H
        d = ctx.device_alloc(8 * npix)
        call = lambda: ctx.check(L.acm_render_depth(ctx.handle, C.byref(cam), R9, t3, X.handle, C.c_void_p(d), C.c_void_p(d + 4 * npix)))
        for _ in range(3):
            call()
        ctx.sync()
        ms = []
        for _ in range(a.timed):
            ctx.timer_start(); call(); ms.append(ctx.timer_stop())
        med = float(np.median(ms))
        rng, idx = np.empty((H, W), np.float32), np.empty((H, W), np.uint32)
        ctx.d2h(rng, d); ctx.d2h(idx, d + 4 * npix); ctx.sync()
        ctx.device_free(d); X.free()
        pts = O.synth_points3(seed, 0, n, cos, False)
        o = O.make_model(model_id, p, W, H)
        t0 = time.perf_counter()
        er, ei = D.render_depth(o, pts)
        cpu = time.perf_counter() - t0
        del pts
        differ = int(((rng.view(np.uint32) != er.view(np.uint32)) | (idx != ei)).sum())
        nbytes = 24 * n + 24 * npix
        return (f"{W}x{H} n={n:.0e} {cone_deg:.0f}deg: {med:.3f} ms (min {min(ms):.3f}, max {max(ms):.3f}), {n / med / 1e6:.2f} G points/s, "
                f"{nbytes / med / 1e6:.0f} GB/s algorithmic; drawn pixels {int((idx != 0xFFFFFFFF).sum())}; "
                f"oracle 1 thread {cpu:.2f} s ({cpu * 1e3 / med:.0f}x); pixels differing from the oracle: {differ}")

    for name, (mid, params, W0, cone) in cams.items():
        lines.append(f"== {name}")
        for (W, H, n) in ((1920, 1080, a.points), (320, 240, a.points), (4096, 4096, a.points // 10)):
            lines.append("  " + run(mid, params, W0, W, H, n, cone, 0xDE9B00 + W))
            print(lines[-1], flush=True)
    # per sweep through the Python API (numpy in, numpy out, host form)
    lines.append("== per sweep: render_depth(numpy, n = 1e5) into 1920x1080, wall time per call (host copies included)")
    for name, (mid, params, W0, cone) in cams.items():
        s = 1920 / W0
        p = list(params); p[0], p[1], p[2], p[3] = p[0] * s, p[1] * s, 960.3, 539.8
        g = acm.MODEL_CLASSES[mid](acm.Intrinsics(*p[:4]), acm.Resolution(1920, 1080), p[4:], ctx=ctx)
        pts = O.synth_points3(0xDE9C00, 0, 100_000, float(np.cos(np.deg2rad(cone))), False)
        for _ in range(3):
            acm.render_depth(g, pts)
        w = []
        for _ in range(a.timed):
            t0 = time.perf_counter(); acm.render_depth(g, pts); w.append(time.perf_counter() - t0)
        lines.append(f"  {name}: median {np.median(w) * 1e3:.3f} ms (min {min(w) * 1e3:.3f}, max {max(w) * 1e3:.3f})")
        print(lines[-1], flush=True)
    lines.append(f"card (end): {card()}")
    ctx.close()
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
