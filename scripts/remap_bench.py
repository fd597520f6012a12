"""Times remap plans on one GPU, frames resident in HBM, CUDA events after warm-up, both arms in one process.

1. acm_undistort_rgb8 against an undistort plan's acm_remap_rgb8 (same camera, same output bytes) on a 4096 x 4096
   Kannala-Brandt camera, at F = 1, 4, 32 frames per call, bilinear and nearest; the two arms alternate per repeat.
2. Kannala-Brandt -> Double Sphere (focal lengths x8 as the KB camera's) to a 4096^2 and a 2048^2 output.
3. Plan build time (map + pack kernels, allocation included).

Prints the card's name and power limit beside the numbers.  Frames: 4096^2 x 3 B = 50 MB each, so batches of 4 and
more exceed the 126 MB L2; F = 1 runs partly from L2, as a one-frame-per-call pipeline would."""
import argparse, ctypes as C, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apex_camera_models_b200 as acm
from apex_camera_models_b200 import _native as N

KB = [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434, 0.0007150348452162257,
      -0.0020532361418706202, 0.00020293673591811182]
# output camera: the KB camera's intrinsics with the distortion of the reference's Double Sphere sample
# (tests/golden/cameras.json "double_sphere")
DS = KB[:4] + [0.5657413673629862, -0.24425190195168348]

ap = argparse.ArgumentParser(description=__doc__)
ap.add_argument("--frames", type=int, nargs="*", default=[1, 4, 32])
ap.add_argument("--reps", type=int, default=5, help="alternating repeats per arm")
ap.add_argument("--iters", type=int, default=20, help="calls per timed window")
ap.add_argument("--json", default=None, help="also write the results here")
args = ap.parse_args()

lib = N.lib
ctx = acm.Context(0)
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    card = q.stdout.strip()
except OSError:
    card = "unknown (nvidia-smi not found)"
print(f"card: {card}")
W = H = 4096
fb = W * H * 3
kb8 = acm.KannalaBrandtModel(acm.Intrinsics(*(v * 8 for v in KB[:4])), acm.Resolution(W, H), KB[4:], ctx=ctx)
cam = kb8.camera_block()
results = {"card": card}


def timed(fn, iters):
    ctx.sync(); ctx.timer_start()
    for _ in range(iters):
        fn()
    return ctx.timer_stop() / iters


Fmax = max(args.frames)
d_in = ctx.device_alloc(fb * Fmax); d_out = ctx.device_alloc(fb * Fmax)
ctx.check(lib.acm_synth_bytes(ctx.handle, 0xACE50005, 0, C.c_void_p(d_in), fb * Fmax))
for interp in (1, 0):
    t0 = time.perf_counter()
    plan = acm.RemapPlan(kb8, None, None, interp); ctx.sync()
    build_ms = (time.perf_counter() - t0) * 1e3
    name = "bilinear" if interp else "nearest"
    print(f"undistort plan build ({name}, 4096^2): {build_ms:.1f} ms (host clock, allocation included)")
    results[f"plan_build_ms_{name}"] = build_ms
    for F in args.frames:
        und = lambda: ctx.check(lib.acm_undistort_rgb8(ctx.handle, C.byref(cam), None, C.c_void_p(d_in), C.c_void_p(d_out), F, interp))
        pln = lambda: plan.apply_device(d_in, d_out, F)
        iters = max(args.iters, 64 // F)
        for _ in range(3):
            und(); pln()
        a, b = [], []
        for _ in range(args.reps):
            a.append(timed(und, iters)); b.append(timed(pln, iters))
        ua, pb = min(a), min(b)
        print(f"{name} F={F:2d}: undistort {F / ua * 1e3:8.0f} frames/s ({ua / F * 1e3:6.1f} us/frame)   plan {F / pb * 1e3:8.0f} frames/s "
              f"({pb / F * 1e3:6.1f} us/frame)   plan/undistort {ua / pb:.3f}x   [spread undistort {max(a) / ua - 1:.1%}, plan {max(b) / pb - 1:.1%}]")
        results[f"{name}_F{F}"] = {"undistort_fps": F / ua * 1e3, "plan_fps": F / pb * 1e3, "ratio": ua / pb}
    plan.close()

for Wo in (4096, 2048):
    s = Wo / 4096 * 8
    ds = acm.DoubleSphereModel(acm.Intrinsics(DS[0] * s, DS[1] * s, DS[2] * s, DS[3] * s), acm.Resolution(Wo, Wo), DS[4:], ctx=ctx)
    for interp in (1, 0):
        name = "bilinear" if interp else "nearest"
        t0 = time.perf_counter()
        plan = acm.RemapPlan(kb8, ds, None, interp); ctx.sync()
        build_ms = (time.perf_counter() - t0) * 1e3
        for F in args.frames:
            pln = lambda: plan.apply_device(d_in, d_out, F)
            iters = max(args.iters, 64 // F)
            for _ in range(3):
                pln()
            ms = min(timed(pln, iters) for _ in range(args.reps))
            print(f"KB 4096^2 -> DS {Wo}^2 {name} F={F:2d}: {F / ms * 1e3:8.0f} frames/s ({ms / F * 1e3:6.1f} us/frame)   plan build {build_ms:.1f} ms")
            results[f"kb_ds_{Wo}_{name}_F{F}"] = {"plan_fps": F / ms * 1e3, "plan_build_ms": build_ms}
        plan.close()
ctx.device_free(d_in); ctx.device_free(d_out)
if args.json:
    with open(args.json, "w") as f:
        json.dump(results, f, indent=1)
