"""Times the build of a rotated remap map against an unrotated one on one GPU: 4096 x 4096 output, CUDA events over
repeated builds into one preallocated map, the two arms alternating per repeat, the SM clock sampled beside each window.

Pairs: Kannala-Brandt 4096^2 (focal lengths x8 of the reference's sample) -> Pinhole 4096^2 (the rectification case) and
-> Double Sphere 4096^2; the rotation is 10 degrees about a tilted axis.  Also times whole plan builds (map + pack +
allocation, host clock) and checks that the identity-rotated map equals the unrotated one bit for bit at this size.
Prints the card's name and power limit beside the numbers."""
import argparse, ctypes as C, json, os, subprocess, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apex_camera_models_b200 as acm
from apex_camera_models_b200 import _native as N

KB = [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434, 0.0007150348452162257,
      -0.0020532361418706202, 0.00020293673591811182]
DS = [0.5657413673629862, -0.24425190195168348]

ap = argparse.ArgumentParser(description=__doc__)
ap.add_argument("--reps", type=int, default=7, help="alternating repeats per arm")
ap.add_argument("--iters", type=int, default=20, help="map builds per timed window")
ap.add_argument("--json", default=None, help="also write the results here")
args = ap.parse_args()


def smi(query):
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown (nvidia-smi not found)"


lib = N.lib
ctx = acm.Context(0)
card = smi("name,power.limit")
print(f"card: {card}")
W = H = 4096
kb8 = acm.KannalaBrandtModel(acm.Intrinsics(*(v * 8 for v in KB[:4])), acm.Resolution(W, H), KB[4:], ctx=ctx)
outputs = {"pinhole": acm.PinholeModel(acm.Intrinsics(1200.0, 1200.0, 2047.5, 2047.5), acm.Resolution(W, H), ctx=ctx),
           "double_sphere": acm.DoubleSphereModel(acm.Intrinsics(*(v * 8 for v in KB[:4])), acm.Resolution(W, H), DS, ctx=ctx)}
a = np.deg2rad(10.0)
k = np.array([0.3, -0.8, 0.5]); k /= np.linalg.norm(k)
K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
ROT = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
results = {"card": card}
d_map = ctx.device_alloc(W * H * 16)
ci = kb8.camera_block()
rot = (C.c_double * 9)(*ROT.ravel())
eye = (C.c_double * 9)(*np.eye(3).ravel())


def timed(fn):
    ctx.sync(); ctx.timer_start()
    for _ in range(args.iters):
        fn()
    return ctx.timer_stop() / args.iters


for name, out in outputs.items():
    co = out.camera_block()
    plain = lambda: ctx.check(lib.acm_remap_map(ctx.handle, C.byref(ci), C.byref(co), C.c_void_p(d_map)))
    rotated = lambda: ctx.check(lib.acm_remap_map_rotated(ctx.handle, C.byref(ci), C.byref(co), rot, C.c_void_p(d_map)))
    identity = lambda: ctx.check(lib.acm_remap_map_rotated(ctx.handle, C.byref(ci), C.byref(co), eye, C.c_void_p(d_map)))
    m0 = np.empty((H, W, 2)); m1 = np.empty((H, W, 2))
    plain(); ctx.d2h(m0, d_map); identity(); ctx.d2h(m1, d_map); ctx.sync()
    same = bool(np.array_equal(m0, m1, equal_nan=True))
    for _ in range(3):
        plain(); rotated()
    ta, tb, clocks = [], [], []
    for _ in range(args.reps):
        ta.append(timed(plain)); clocks.append(smi("clocks.sm"))
        tb.append(timed(rotated)); clocks.append(smi("clocks.sm"))
    a_ms, b_ms = min(ta), min(tb)
    t0 = time.perf_counter()
    with acm.RemapPlan(kb8, out):
        ctx.sync()
    plan_plain = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    with acm.RemapPlan(kb8, out, rotation=ROT):
        ctx.sync()
    plan_rot = (time.perf_counter() - t0) * 1e3
    print(f"KB 4096^2 -> {name} 4096^2 map build: unrotated {a_ms:.3f} ms, rotated {b_ms:.3f} ms ({b_ms / a_ms - 1:+.1%})   "
          f"[spread {max(ta) / a_ms - 1:.1%} / {max(tb) / b_ms - 1:.1%}; SM clock {', '.join(sorted(set(clocks)))}]   "
          f"plan build (host clock, allocation included) {plan_plain:.1f} / {plan_rot:.1f} ms   identity == unrotated: {same}")
    results[name] = {"map_ms_unrotated": a_ms, "map_ms_rotated": b_ms, "all_ms_unrotated": ta, "all_ms_rotated": tb, "sm_clocks": clocks,
                     "plan_build_ms_unrotated": plan_plain, "plan_build_ms_rotated": plan_rot, "identity_bit_identical": same}
ctx.device_free(d_map)
if args.json:
    with open(args.json, "w") as f:
        json.dump(results, f, indent=1)
