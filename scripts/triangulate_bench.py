"""Throughput of acm_triangulate and host overhead of triangulate_points, with the card and its power limit read in the same run.

    python scripts/triangulate_bench.py [--pairs 100000000] [--timed 20] [--out profiles/r03_triangulate_bench.log]

  * throughput: KB -> Double Sphere and Pinhole -> Pinhole, midpoint (max_iterations = 0) and refined (10), on --pairs
    resident pairs (noisy projections of seeded points, 73 algorithmic bytes per pair: 32 in, 24 xyz, 16 err, 1 status);
    3 warm-up launches, then --timed launches between CUDA events.  Reports G pairs/s and algorithmic TB/s.
  * host overhead: wall time per triangulate_points call (numpy in and out) at n = 1 000, KB / RadTan and Pinhole / Pinhole.
  * CPU comparison: the oracle (tests/triangulate_oracle.c, -O2) single-threaded and with OpenMP on all cores.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

BYTES_PER_PAIR = 73


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def axis_angle(axis, deg):
    k = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0.0, -k[2], k[1]], [k[2], 0.0, -k[0]], [-k[1], k[0], 0.0]])
    a = np.deg2rad(deg)
    return np.eye(3) + np.sin(a) * K + (1.0 - np.cos(a)) * (K @ K)


R = axis_angle([0.3, -0.8, 0.5], 10.0)
T = np.array([-0.1, 0.0, 0.0])


def pairs(O, ma, mb, n, seed):
    rng = np.random.default_rng(seed)
    uv = np.column_stack([rng.uniform(0, ma.width, 2 * n), rng.uniform(0, ma.height, 2 * n)])
    ray, st = O.unproject(ma, uv, os.cpu_count())
    X = ray * rng.uniform(0.5, 5.0, 2 * n)[:, None]
    uv1, s1 = O.project(ma, X, os.cpu_count())
    uv2, s2 = O.project(mb, X @ R.T + T, os.cpu_count())
    ok = np.flatnonzero((st == 0) & (s1 == 0) & (s2 == 0))[:n]
    return uv1[ok] + rng.normal(0, 0.5, (len(ok), 2)), uv2[ok] + rng.normal(0, 0.5, (len(ok), 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=100_000_000)
    ap.add_argument("--timed", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import ctypes as C
    import json

    import apex_camera_models_b200 as acm
    from apex_camera_models_b200 import _native as N
    from oracle import oracle as O
    import triangulate_oracle as TO
    from test_gpu_remap import gpu_model, sized
    O.build()
    cams = json.load(open(os.path.join(ROOT, "tests", "golden", "cameras.json")))
    lines = [f"card: {card()}  (name, power.limit, clocks.max.sm, clocks.sm)"]
    print(lines[0], flush=True)
    ctx = acm.Context(0)
    L = N.lib
    Rc, tc = (C.c_double * 9)(*R.ravel()), (C.c_double * 3)(*T)
    for fa, fb in (("kannala_brandt", "double_sphere"), ("pinhole", "pinhole")):
        ca, cb = sized(cams, fa, 320, 240), sized(cams, fb, 288, 224)
        ga, gb = gpu_model(acm, ctx, ca), gpu_model(acm, ctx, cb)
        oa, ob = O.make_model(ca["model_id"], ca["params"], 320, 240), O.make_model(cb["model_id"], cb["params"], 288, 224)
        # a 1 M-pair block of real pairs tiled to --pairs on the device
        u1, u2 = pairs(O, oa, ob, 1_000_000, 0x7121A7EB)
        blk = len(u1)
        n = a.pairs
        p1, p2, xyz = acm.Points(ctx, 2, n), acm.Points(ctx, 2, n), acm.Points(ctx, 3, n)
        d = ctx.device_alloc(17 * n)
        tile1, tile2 = acm.Points.from_numpy(ctx, u1), acm.Points.from_numpy(ctx, u2)
        for c in range(2):
            for src, dst in ((tile1, p1), (tile2, p2)):
                done = 0
                while done < n:
                    k = min(blk, n - done)
                    ctx.d2d(dst.component_ptr(c) + 8 * done, src.component_ptr(c), 8 * k)
                    done += k
        tile1.free(); tile2.free()
        ctx.sync()
        cam_a, cam_b = ga.camera_block(), gb.camera_block()
        for it in (0, 10):
            call = lambda: ctx.check(L.acm_triangulate(ctx.handle, C.byref(cam_a), C.byref(cam_b), Rc, tc, p1.handle, p2.handle, it,
                                                       xyz.handle, C.c_void_p(d), C.c_void_p(d + 16 * n)))
            for _ in range(3):
                call()
            ctx.sync()
            times = []
            for _ in range(a.timed):
                ctx.timer_start()
                call()
                times.append(ctx.timer_stop())
            st = np.empty(min(n, 1 << 20), np.uint8)
            ctx.d2h(st, d + 16 * n); ctx.sync()
            ms = np.array(times)
            med = float(np.median(ms))
            line = (f"{fa}->{fb} max_iterations={it:2d}  n={n}  median {med:.3f} ms (min {ms.min():.3f}, max {ms.max():.3f}, {a.timed} launches)  "
                    f"{n / med / 1e6:.3f} G pairs/s  {BYTES_PER_PAIR * n / med / 1e9:.3f} TB/s algorithmic  ok {np.mean(st == 0):.4f}")
            print(line, flush=True)
            lines.append(line)
        for p in (p1, p2, xyz):
            p.free()
        ctx.device_free(d)
        # CPU oracle on the same pairs
        m = min(200_000, blk)
        for nt in (1, os.cpu_count()):
            t0 = time.perf_counter()
            TO.triangulate(oa, ob, R, T, u1[:m], u2[:m], 10, nt)
            dt = time.perf_counter() - t0
            line = f"{fa}->{fb} oracle max_iterations=10 threads={nt}: {m / dt / 1e6:.3f} M pairs/s"
            print(line, flush=True)
            lines.append(line)
    for fa, fb in (("kannala_brandt", "rad_tan"), ("pinhole", "pinhole")):
        ca, cb = sized(cams, fa, 320, 240), sized(cams, fb, 288, 224)
        ga, gb = gpu_model(acm, ctx, ca), gpu_model(acm, ctx, cb)
        oa, ob = O.make_model(ca["model_id"], ca["params"], 320, 240), O.make_model(cb["model_id"], cb["params"], 288, 224)
        u1, u2 = pairs(O, oa, ob, 1000, 0x7121A7EC)
        for _ in range(20):
            acm.triangulate_points(ga, gb, R, T, u1, u2)
        reps = 500
        t0 = time.perf_counter()
        for _ in range(reps):
            acm.triangulate_points(ga, gb, R, T, u1, u2)
        us = (time.perf_counter() - t0) / reps * 1e6
        line = f"host overhead {fa}/{fb}: {us:.1f} us per triangulate_points call at n = {len(u1)} (numpy in and out, max_iterations=10)"
        print(line, flush=True)
        lines.append(line)
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
