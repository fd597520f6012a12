"""Small invocation of every kernel family (for compute-sanitizer memcheck / racecheck runs)."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apex_camera_models_b200 as acm
KB = [190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434, 0.0007150348452162257, -0.0020532361418706202, 0.00020293673591811182]
ctx = acm.Context(0)
I = acm.Intrinsics(*KB[:4]); R = acm.Resolution(512, 512)
kb = acm.KannalaBrandtModel(I, R, KB[4:], ctx=ctx)
uv, xyz = acm.sample_points(kb, 60_001, device=True)
print("sampled", len(uv))
inits = {acm.DoubleSphereModel: [0.5, 0.1], acm.UcmModel: [0.5], acm.EucmModel: [0.5, 1.0], acm.KannalaBrandtModel: [0.0] * 4, acm.FovModel: [1.0],
         acm.RadTanModel: [0.0] * 5}
for cls, d in inits.items():
    m = cls(I, R, d, ctx=ctx)
    m.linear_estimation(xyz, uv)
    r = acm.OptimizationCost(m, xyz, uv).optimize()
    e = acm.compute_reprojection_error(m, xyz, uv)
    print(cls.__name__, r.iterations, r.status, f"{e.mean:.5f}")
    rays, st = m.unproject_batch(uv); ctx.device_free(st); rays.free()
    a, b, s1, s2 = m.round_trip_batch(xyz); a.free(); b.free(); ctx.device_free(s1); ctx.device_free(s2)
frames = np.random.default_rng(0).integers(0, 256, size=(6, 512, 512, 3), dtype=np.uint8)
for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):
    out = acm.undistort_images(frames, kb, None, interp)
    out2 = acm.undistort_images(frames, kb, acm.Intrinsics(100.0, 100.0, 256.0, 256.0), interp)  # zoom-out: list kernel
    print("undistort", int(interp), out.mean(), out2.mean())
ds = acm.DoubleSphereModel(acm.Intrinsics(150.0, 150.0, 192.3, 143.8), acm.Resolution(384, 288), [0.56, -0.24], ctx=ctx)
for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):  # remap plans: TMA + leftover gather, byte kernel
    with acm.RemapPlan(kb, ds, None, interp) as plan, acm.RemapPlan(ds, kb, None, interp) as back:
        print("remap", int(interp), plan.apply(frames).mean(), back.apply(frames[:, :288, :384]).mean(), acm.remap_map(kb, ds).shape)
c, s = np.cos(0.3), np.sin(0.3)
R1, R2, _, _ = acm.stereo_rectify([[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]], [-0.1, 0.01, 0.0])
with acm.RemapPlan(kb, ds, rotation=R1) as plan:  # rotated plan: map kernel with the rotation, leftover gather for the skewed boxes
    print("rotated remap", plan.apply(frames).mean(), acm.remap_map(kb, ds, rotation=R2).shape)
ctx.sync()
print("ok")
# round 2: scalar host path (mapped staging + completion flag), small batches, Jacobian kernels (vector and scalar forms)
p = kb.project([0.1, 0.2, 1.0]); r = kb.unproject(p)
uvb, stb = kb.project_batch(np.tile([0.1, 0.2, 1.0], (777, 1)))
rt = acm.RadTanModel(acm.Intrinsics(461.629, 460.152, 362.68, 246.049), acm.Resolution(752, 480), [-0.28340811, 0.07395907, 0.00019359, 1.76187114e-05, 0.0], ctx=ctx)
px = np.random.default_rng(1).uniform([0, 0], [752, 480], size=(50_001, 2))
rays, st = rt.unproject_batch(px)
for n in (4096, 4097):
    pts = np.random.default_rng(2).normal(size=(n, 3)) * [0.3, 0.3, 0.1] + [0, 0, 1.5]
    for m in (kb, rt):
        m.project_jacobian_batch(pts); m.project_point_jacobian_batch(pts)
print("round-2 paths ok", p, int((st == 0).sum()))
