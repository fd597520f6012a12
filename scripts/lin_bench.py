"""Times acm_linearize_async for every model on 100 M synthetic correspondences (inputs > L2).
MODELS=5,2,... selects model ids; REPS sets the launches."""
import ctypes as C, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apex_camera_models_b200 as acm
from apex_camera_models_b200 import _native as N
lib = N.lib
KB = [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434, 0.0007150348452162257, -0.0020532361418706202, 0.00020293673591811182]
n = int(os.environ.get("N", "100000000"))
reps = int(os.environ.get("REPS", "20"))
ctx = acm.Context(0)
X = acm.Points(ctx, 3, n); UV = acm.Points(ctx, 2, n)
ctx.check(lib.acm_synth_points3(ctx.handle, 0xACE50003, 0, float(np.cos(np.deg2rad(85.0))), 0, X.handle))
kb = acm.KannalaBrandtModel(acm.Intrinsics(*KB[:4]), acm.Resolution(512, 512), KB[4:], ctx=ctx)
cam = kb.camera_block()
ctx.check(lib.acm_project(ctx.handle, C.byref(cam), X.handle, UV.handle, None))
dist_init = {0: [], 1: [0.01, 0.001, 0.0, 0.0, 0.0], 2: KB[4:], 3: [0.6], 4: [0.6, 1.0], 5: [0.6, 0.1], 6: [0.9]}
names = {0: "pinhole", 1: "rad_tan", 2: "kannala_brandt", 3: "ucm", 4: "eucm", 5: "double_sphere", 6: "fov"}
models = [int(v) for v in os.environ.get("MODELS", "5,4,3,2,6,1,0").split(",")]
for mid in models:
    m = acm.MODEL_CLASSES[mid](acm.Intrinsics(*KB[:4]), acm.Resolution(512, 512), dist_init[mid], ctx=ctx)
    cam = m.camera_block()
    for kind in ((0, 1) if mid in (3, 4, 5) else (0,)):
        f = lambda: ctx.check(lib.acm_linearize_async(ctx.handle, C.byref(cam), kind, X.handle, UV.handle))
        for _ in range(3): f()
        ctx.sync(); ctx.timer_start()
        for _ in range(reps): f()
        ms = ctx.timer_stop() / reps
        print(f"{names[mid]:15s} kind={kind}: {ms:.3f} ms  {n / ms / 1e6:.1f} Gpts/s  {n * 40 / ms / 1e6:.0f} GB/s", flush=True)
