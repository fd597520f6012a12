"""Times the callers either side of the LM at the converter's 10 M scale (SURVEY 8f rows f1, f2 + linear estimation)."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apex_camera_models_b200 as acm
KB = [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434, 0.0007150348452162257, -0.0020532361418706202, 0.00020293673591811182]
ctx = acm.Context(0)
kb = acm.KannalaBrandtModel(acm.Intrinsics(*KB[:4]), acm.Resolution(512, 512), KB[4:], ctx=ctx)
def timed(f, reps=5):
    f(); ctx.sync()
    t0 = time.perf_counter()
    for _ in range(reps): r = f()
    ctx.sync()
    return (time.perf_counter() - t0) / reps * 1e3, r
ms, (uv, xyz) = timed(lambda: acm.sample_points(kb, 10_000_000, device=True))
n = len(uv)
print(f"sample_points(KB, 10M): {ms:.2f} ms -> {n} kept of {3162*3162}")
for name, cls, d in [("double_sphere", acm.DoubleSphereModel, [0.5, 0.1]), ("ucm", acm.UcmModel, [0.5]), ("eucm", acm.EucmModel, [0.5, 1.0]),
                     ("kannala_brandt", acm.KannalaBrandtModel, [0.0] * 4), ("fov", acm.FovModel, [1.0]), ("rad_tan", acm.RadTanModel, [0.0] * 5)]:
    m = cls(acm.Intrinsics(*KB[:4]), acm.Resolution(512, 512), d, ctx=ctx)
    ms_e, e = timed(lambda: acm.compute_reprojection_error(m, xyz, uv), reps=3)
    ms_l, _ = timed(lambda: m.linear_estimation(xyz, uv), reps=3)
    cost = acm.OptimizationCost(m, xyz, uv)
    t0 = time.perf_counter(); r = cost.optimize(); ms_o = (time.perf_counter() - t0) * 1e3
    e2 = acm.compute_reprojection_error(m, xyz, uv)
    print(f"{name:15s} reproj_error {ms_e:.2f} ms (mean {e.mean:.4f} px) | linear_estimation {ms_l:.2f} ms | LM {ms_o:.2f} ms it={r.iterations} status={r.status} | final mean {e2.mean:.5f} px median {e2.median:.5f}")
    ms_q, q = timed(lambda: acm.compute_image_quality_metrics(kb, m, xyz), reps=3)
    print(f"{'':15s} image_quality_metrics {ms_q:.2f} ms (512x512, {n} points): PSNR {q.psnr:.2f} dB SSIM {q.ssim:.4f}")
# the same diagnostics on a 4096^2 camera (KB sample intrinsics x 8), 10 M points
big = acm.KannalaBrandtModel(acm.Intrinsics(*[8 * v for v in KB[:4]]), acm.Resolution(4096, 4096), KB[4:], ctx=ctx)
uvb, xyzb = acm.sample_points(big, 10_000_000, device=True)
dsb = acm.DoubleSphereModel(acm.Intrinsics(*[8 * v for v in KB[:4]]), acm.Resolution(4096, 4096), [0.5, 0.1], ctx=ctx)
dsb.linear_estimation(xyzb, uvb); acm.OptimizationCost(dsb, xyzb, uvb).optimize()
ms_q, q = timed(lambda: acm.compute_image_quality_metrics(big, dsb, xyzb), reps=3)
print(f"image_quality_metrics 4096x4096, {len(uvb)} points, KB -> DS: {ms_q:.2f} ms  PSNR {q.psnr:.2f} dB SSIM {q.ssim:.4f}")
rng = np.random.default_rng(1)
a = rng.integers(0, 256, (4096, 4096, 3), dtype=np.uint8); b = rng.integers(0, 256, (4096, 4096, 3), dtype=np.uint8)
from apex_camera_models_b200.image_quality import _DeviceImage, _lib
import ctypes as C
s = ctx.staging()
da, db = _DeviceImage(s, a), _DeviceImage(s, b)
out = C.c_double()
ms_p, _ = timed(lambda: ctx.check(_lib.acm_image_psnr(ctx.handle, C.c_void_p(da.ptr), C.c_void_p(db.ptr), 4096, 4096, C.byref(out))), reps=10)
ms_s, _ = timed(lambda: ctx.check(_lib.acm_image_ssim(ctx.handle, C.c_void_p(da.ptr), C.c_void_p(db.ptr), 4096, 4096, C.byref(out))), reps=10)
print(f"resident 4096^2 RGB8 pair: psnr {ms_p:.3f} ms ({2 * a.nbytes / ms_p / 1e6:.0f} GB/s), ssim {ms_s:.3f} ms ({2 * a.nbytes / ms_s / 1e6:.0f} GB/s)")
