"""Rectify the frames of a calibrated stereo pair onto one pinhole camera, on the GPU path:

    python -m apex_camera_models_b200.image_rectify -l left.png -r right.png \\
        --left-calib cam0.yaml --left-model kb --right-calib cam1.yaml --right-model ds \\
        --rotation r00 r01 r02 r10 r11 r12 r20 r21 r22 --translation tx ty tz \\
        --size 640 480 --focal 300 --left-output rect0 --right-output rect1

R and t describe the pair as x_cam2 = R x_cam1 + t (OpenCV's stereoRectify convention).  Both views are rendered on the
same Pinhole camera (W x H, fx = fy = f, principal point at the image centre ((W-1)/2, (H-1)/2) unless --principal is given), so rows correspond
(columns for a vertically stacked pair).  As in `image_remap`, the model types come from the -m flags; several images per
side may be given (repeat the flag or pass directories) and are rectified as one batch.
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

from ._image_cli import expand_inputs, load_model, load_rgb, save_rgb
from .camera import Intrinsics, PinholeModel, Resolution
from .util import InterpolationMethod, StereoRectifier


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="image_rectify", description="Rectify stereo pairs of any two camera models")
    ap.add_argument("-l", "--left", required=True, action="append", help="left image (repeatable) or a directory")
    ap.add_argument("-r", "--right", required=True, action="append", help="right image (repeatable) or a directory")
    ap.add_argument("--left-calib", required=True, help="left camera calibration (YAML)")
    ap.add_argument("--left-model", required=True, help="left camera model type")
    ap.add_argument("--right-calib", required=True, help="right camera calibration (YAML)")
    ap.add_argument("--right-model", required=True, help="right camera model type")
    ap.add_argument("--rotation", required=True, nargs=9, type=float, metavar="R", help="R row-major: x_cam2 = R x_cam1 + t")
    ap.add_argument("--translation", required=True, nargs=3, type=float, metavar="T", help="t: x_cam2 = R x_cam1 + t")
    ap.add_argument("--size", required=True, nargs=2, type=int, metavar=("W", "H"), help="rectified image size")
    ap.add_argument("--focal", required=True, type=float, help="rectified focal length (pixels)")
    ap.add_argument("--principal", nargs=2, type=float, metavar=("CX", "CY"), help="rectified principal point (default: the centre, ((W-1)/2, (H-1)/2))")
    ap.add_argument("--interpolation", choices=["bilinear", "nearest"], default="bilinear")
    ap.add_argument("--left-output", required=True, help="output directory of the rectified left images")
    ap.add_argument("--right-output", required=True, help="output directory of the rectified right images")
    args = ap.parse_args(argv)

    left, right = load_model(args.left_model, args.left_calib), load_model(args.right_model, args.right_calib)
    W, H = args.size
    cx, cy = args.principal if args.principal else ((W - 1) / 2.0, (H - 1) / 2.0)
    rect = PinholeModel(Intrinsics(args.focal, args.focal, cx, cy), Resolution(W, H), ctx=left.ctx)
    left_paths, right_paths = expand_inputs(args.left), expand_inputs(args.right)
    if len(left_paths) != len(right_paths):
        raise SystemExit(f"need as many right images as left images ({len(right_paths)} != {len(left_paths)})")
    interp = InterpolationMethod.Nearest if args.interpolation == "nearest" else InterpolationMethod.Bilinear
    with StereoRectifier(left, right, np.reshape(args.rotation, (3, 3)), args.translation, rect, interp) as rig:
        print(f"Rectifying {len(left_paths)} pair(s) onto a {W}x{H} pinhole (f={args.focal}, c=({cx}, {cy})): "
              f"baseline {rig.baseline:.6g} along {'y' if rig.vertical else 'x'}")
        out_l, out_r = rig.apply(np.stack([load_rgb(p) for p in left_paths]), np.stack([load_rgb(p) for p in right_paths]))
    for d, paths, frames in ((args.left_output, left_paths, out_l), (args.right_output, right_paths, out_r)):
        os.makedirs(d, exist_ok=True)
        for p, a in zip(paths, frames):
            save_rgb(os.path.join(d, os.path.basename(p)), a)
    print(f"Saved rectified images to: {args.left_output}, {args.right_output}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
