"""Times acm_undistort_rgb8 on KB fisheye frames resident in HBM (BASELINE config 5 per-GPU share: 4096x4096).

--width picks the kernel: a multiple of 16 takes the TMA kernel, another multiple of 4 the whole-image gather kernel
(e.g. 4092), any other width the generic byte kernel (e.g. 4095).  --target-scale s undistorts to the target
intrinsics (s fx, s fy, W/2, H/2); s = 0.6 zooms out far enough that part of the patches go to the gather kernel's
leftover list."""
import argparse, ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apex_camera_models_b200 as acm
from apex_camera_models_b200 import _native as N
KB = [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434, 0.0007150348452162257, -0.0020532361418706202, 0.00020293673591811182]
ap = argparse.ArgumentParser(description=__doc__)
ap.add_argument("frames", type=int, nargs="*", default=[8, 32], help="frames per call, one run per value")
ap.add_argument("--width", type=int, default=4096, help="image width (the height stays 4096)")
ap.add_argument("--target-scale", type=float, default=None, help="target focal lengths = scale x the camera's (default: the camera's intrinsics)")
args = ap.parse_args()
lib = N.lib; ctx = acm.Context(0)
W, H = args.width, 4096
kb8 = acm.KannalaBrandtModel(acm.Intrinsics(*(v * 8 for v in KB[:4])), acm.Resolution(W, H), KB[4:], ctx=ctx)
cam = kb8.camera_block(); fb = W * H * 3
target = None if args.target_scale is None else (C.c_double * 4)(KB[0] * 8 * args.target_scale, KB[1] * 8 * args.target_scale, W / 2.0, H / 2.0)
label = f"{W}x{H} KB" + ("" if args.target_scale is None else f" target x{args.target_scale:g}")
for F in args.frames:
    d_in = ctx.device_alloc(fb * F); d_out = ctx.device_alloc(fb * F)
    ctx.check(lib.acm_synth_bytes(ctx.handle, 0xACE50005, 0, C.c_void_p(d_in), fb * F))
    for interp in (1, 0):
        f = lambda: ctx.check(lib.acm_undistort_rgb8(ctx.handle, C.byref(cam), target, C.c_void_p(d_in), C.c_void_p(d_out), F, interp))
        for _ in range(3): f()
        ctx.sync(); ctx.timer_start()
        for _ in range(5): f()
        ms = ctx.timer_stop() / 5
        print(f"undistort {label} interp={interp} frames={F}: {ms:.3f} ms  {F/ms*1e3:.0f} frames/s  {2*fb*F/ms/1e6:.0f} GB/s  ({ms/F*1e3:.1f} us/frame)")
    ctx.device_free(d_in); ctx.device_free(d_out)
