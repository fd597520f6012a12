"""One launch of the image-quality kernels on a 4096^2 RGB8 pair (for an `ncu --set full` capture)."""
import ctypes as C, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apex_camera_models_b200 as acm
from apex_camera_models_b200.image_quality import _DeviceImage, _lib
ctx = acm.Context(0)
rng = np.random.default_rng(1)
a = rng.integers(0, 256, (4096, 4096, 3), dtype=np.uint8); b = rng.integers(0, 256, (4096, 4096, 3), dtype=np.uint8)
s = ctx.staging()
da, db = _DeviceImage(s, a), _DeviceImage(s, b)
out = C.c_double()
for _ in range(2):
    ctx.check(_lib.acm_image_psnr(ctx.handle, C.c_void_p(da.ptr), C.c_void_p(db.ptr), 4096, 4096, C.byref(out)))
    ctx.check(_lib.acm_image_ssim(ctx.handle, C.c_void_p(da.ptr), C.c_void_p(db.ptr), 4096, 4096, C.byref(out)))
KB = [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434, 0.0007150348452162257, -0.0020532361418706202, 0.00020293673591811182]
big = acm.KannalaBrandtModel(acm.Intrinsics(*[8 * v for v in KB[:4]]), acm.Resolution(4096, 4096), KB[4:], ctx=ctx)
uv, xyz = acm.sample_points(big, 10_000_000, device=True)
ds = acm.DoubleSphereModel(acm.Intrinsics(*[8 * v for v in KB[:4]]), acm.Resolution(4096, 4096), [0.59, -0.17], ctx=ctx)
print(acm.compute_image_quality_metrics(big, ds, xyz))
ctx.sync()
print("done")
