"""`image_undistort` on the GPU path (reference bin/image_undistort.rs): same flags
(`-i/--input`, `-c/--calib`, `-o/--output`, `-m/--model` default fov, `--target-fx`, `--target-fy`),
bilinear interpolation as in the reference (:96-101).  Several inputs may be given (repeat `-i` / `-o`, or
pass directories): they are undistorted as ONE batch, which is what the GPU kernel is built for.

    python -m apex_camera_models_b200.image_undistort -i img.png -c calib.yaml -o out.png -m kb
"""
from __future__ import annotations

import argparse
import sys

import numpy as np

from ._image_cli import expand_inputs, load_model, load_rgb, pair_outputs, save_rgb
from .camera import Intrinsics
from .util import InterpolationMethod, undistort_images


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="image_undistort", description="Undistort images using camera calibration")
    ap.add_argument("-i", "--input", required=True, action="append", help="input image (repeatable) or a directory")
    ap.add_argument("-c", "--calib", required=True)
    ap.add_argument("-o", "--output", required=True, action="append", help="output image (one per input) or a directory")
    ap.add_argument("-m", "--model", default="fov")
    ap.add_argument("--target-fx", type=float, default=None)
    ap.add_argument("--target-fy", type=float, default=None)
    ap.add_argument("--nearest", action="store_true", help="nearest-neighbour instead of the reference's bilinear sampling")
    args = ap.parse_args(argv)

    model = load_model(args.model, args.calib)
    intr, res = model.get_intrinsics(), model.get_resolution()
    print("Image Undistortion Tool (B200 path)")
    print(f"Loaded {args.model} camera model: fx={intr.fx:.2f}, fy={intr.fy:.2f}, cx={intr.cx:.2f}, cy={intr.cy:.2f}, resolution {res.width}x{res.height}")

    inputs = expand_inputs(args.input)
    outputs = pair_outputs(inputs, args.output)

    frames = np.stack([load_rgb(p) for p in inputs])
    print(f"Loaded {len(inputs)} input image(s): {frames.shape[2]}x{frames.shape[1]}")
    target = None
    if args.target_fx is not None or args.target_fy is not None:  # image_undistort.rs:78-91
        target = Intrinsics(args.target_fx if args.target_fx is not None else intr.fx,
                            args.target_fy if args.target_fy is not None else intr.fy, intr.cx, intr.cy)
        print(f"Using custom target focal lengths: fx={target.fx:.2f}, fy={target.fy:.2f}")
    out = undistort_images(frames, model, target, InterpolationMethod.Nearest if args.nearest else InterpolationMethod.Bilinear)
    for p, a in zip(outputs, out):
        save_rgb(p, a)
        print(f"Saved undistorted image to: {p}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
