"""Multi-GPU parity check of the converter pipeline (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 scripts/multi_gpu_check.py

Every rank runs sample_points(shard) -> linear_estimation -> LM -> compute_reprojection_error on its
shard with the communicator attached; rank 0 additionally runs the whole problem on a second,
single-rank context.  The sharded results must equal the single-GPU ones: kept points bit for
bit, parameters / statistics to rounding (count, min, max and median exactly)."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apex_camera_models_b200 as acm
from apex_camera_models_b200 import distributed as D
from apex_camera_models_b200.runtime import Context
from apex_camera_models_b200 import optimization as opt, util

KB = dict(params=[190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504, 0.0034823894022493434,
                  0.0007150348452162257, -0.0020532361418706202, 0.00020293673591811182], width=512, height=512)
N_REQ = int(os.environ.get("ACM_CHECK_POINTS", "2000000"))


def pipeline(ctx, shard, use_peer):
    res_ = acm.Resolution(KB["width"], KB["height"])
    kb = acm.KannalaBrandtModel(acm.Intrinsics(*KB["params"][:4]), res_, KB["params"][4:], ctx=ctx)
    uv, xyz = util.sample_points(kb, N_REQ, device=True, shard=shard)
    out = {"kept_local": len(uv)}
    for name, cls, cost_cls, init in [
        ("double_sphere", acm.DoubleSphereModel, opt.DoubleSphereOptimizationCost, [0.5, 0.1]),
        ("eucm", acm.EucmModel, opt.EucmOptimizationCost, [0.5, 1.0]),
        ("kannala_brandt", acm.KannalaBrandtModel, opt.KannalaBrandtOptimizationCost, [0.0, 0.0, 0.0, 0.0]),
        ("fov", acm.FovModel, opt.FovOptimizationCost, [1.0]),
    ]:
        m = cls(acm.Intrinsics(*KB["params"][:4]), res_, init, ctx=ctx)
        cost = cost_cls(m, xyz, uv)
        cost.linear_estimation()
        lin = [float(v) for v in m.params()]
        res = cost.optimize()
        err = util.compute_reprojection_error(m, xyz, uv)
        # image-quality diagnostics on the sharded points: every rank gets the metrics of the whole set
        q, img = acm.compute_image_quality_metrics(kb, m, xyz, return_image=True)
        out[name] = {"linear": lin, "params": [float(v) for v in m.params()], "iterations": int(res.iterations), "final_cost": float(res.final_cost),
                     "err": [err.rmse, err.min, err.max, err.mean, err.stddev, err.median, err.count],
                     "psnr": q.psnr, "ssim": q.ssim, "image_crc": int(np.bitwise_xor.reduce(np.frombuffer(img.tobytes(), np.uint32) * np.arange(1, img.size // 4 + 1, dtype=np.uint32)))}
    return out, uv, xyz


def main():
    rank, local, world = D.env_rank_world()
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    ok = True
    report = {}
    for mode in ("nccl", "peer"):
        ctx = Context(local)
        D.attach_communicator(ctx)
        if mode == "peer":
            D.attach_peers(ctx)
        got, uv, xyz = pipeline(ctx, (rank, world), mode == "peer")
        counts = [None] * world
        dist.all_gather_object(counts, got["kept_local"])
        uv_all = [None] * world
        xyz_all = [None] * world
        dist.all_gather_object(uv_all, uv.numpy())
        dist.all_gather_object(xyz_all, xyz.numpy())
        if rank == 0:
            single = Context(local)
            ref, uv1, xyz1 = pipeline(single, None, False)
            same_pts = np.array_equal(np.concatenate(uv_all), uv1.numpy()) and np.array_equal(np.concatenate(xyz_all), xyz1.numpy())
            report[mode] = {"kept": counts, "kept_single": ref["kept_local"], "points_bit_identical": bool(same_pts), "models": {}}
            ok &= same_pts and sum(counts) == ref["kept_local"]
            for name in ("double_sphere", "eucm", "kannala_brandt", "fov"):
                a, b = got[name], ref[name]
                rel = lambda x, y: float(np.max(np.abs(np.asarray(x) - np.asarray(y)) / np.maximum(np.abs(np.asarray(y)), 1e-300)))
                d = {"linear_rel": rel(a["linear"], b["linear"]), "params_rel": rel(a["params"], b["params"]),
                     "iterations": [a["iterations"], b["iterations"]], "err_rel": rel(a["err"][:6], b["err"][:6]),
                     "exact_count_min_max_median": a["err"][6] == b["err"][6] and a["err"][1] == b["err"][1] and a["err"][2] == b["err"][2]
                                                   and a["err"][5] == b["err"][5],
                     # absolute floor: `min` is a near-zero residual (~1e-6 px), where parameters that differ in the 15th digit
                     # already move it by 1e-8 relative
                     "err_close": bool(np.allclose(a["err"][:6], b["err"][:6], rtol=1e-9, atol=1e-11)),
                     "mean_px": a["err"][3], "psnr": [a["psnr"], b["psnr"]], "ssim": [a["ssim"], b["ssim"]],
                     "display_image_identical": a["image_crc"] == b["image_crc"]}
                report[mode]["models"][name] = d
                # bit-identical parameters must give bit-identical count / min / max / median; parameters that
                # differ in the last bits (different grouping of the sums) move the errors by as much
                ok &= d["linear_rel"] < 1e-9 and d["params_rel"] < 1e-9 and d["err_close"] and a["err"][6] == b["err"][6]
                ok &= d["exact_count_min_max_median"] or d["params_rel"] > 0.0
                # rendered images depend on the parameters only through rounded pixel positions: identical unless a
                # projection sits on a rounding tie; PSNR is integer arithmetic on the images, SSIM a fixed-order sum
                ok &= (a["psnr"] == b["psnr"] and abs(a["ssim"] - b["ssim"]) <= 1e-12 and d["display_image_identical"]) or d["params_rel"] > 0.0
        # every rank must hold identical results (rank-ordered sums)
        blob = json.dumps({k: v for k, v in got.items() if k != "kept_local"}, sort_keys=True)
        blobs = [None] * world
        dist.all_gather_object(blobs, blob)
        if rank == 0:
            report[mode]["rank_identical"] = all(b == blobs[0] for b in blobs)
            ok &= report[mode]["rank_identical"]
        dist.barrier()
    if rank == 0:
        report["world"] = world
        report["n_requested"] = N_REQ
        report["ok"] = bool(ok)
        print(json.dumps(report, indent=1))
    dist.destroy_process_group()
    sys.exit(0 if ok or rank != 0 else 1)


if __name__ == "__main__":
    main()
