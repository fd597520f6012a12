"""Render images as another camera model sees them, on the GPU path.  Together with the converter
(`camera_converter`), this shows a user's frames through the converted model:

    python -m apex_camera_models_b200.image_remap -i in.png -c in.yaml -m kb --output-calib out.yaml --output-model ds -o out.png

The input frames must have the input camera's resolution; the output has the output camera's.  As in the
reference's loaders, the model types come from `-m` / `--output-model` (the YAML `camera_model` key is not read).
Several inputs may be given (repeat `-i` / `-o`, or pass directories); they are remapped as one batch.
"""
from __future__ import annotations

import argparse
import sys

import numpy as np

from ._image_cli import expand_inputs, load_model, load_rgb, pair_outputs, save_rgb
from .util import InterpolationMethod, RemapPlan


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="image_remap", description="Remap images from one camera model to another")
    ap.add_argument("-i", "--input", required=True, action="append", help="input image (repeatable) or a directory")
    ap.add_argument("-c", "--calib", required=True, help="input camera calibration (YAML)")
    ap.add_argument("-m", "--model", required=True, help="input camera model type")
    ap.add_argument("--output-calib", required=True, help="output camera calibration (YAML)")
    ap.add_argument("--output-model", required=True, help="output camera model type")
    ap.add_argument("-o", "--output", required=True, action="append", help="output image (one per input) or a directory")
    ap.add_argument("--interpolation", choices=["bilinear", "nearest"], default="bilinear")
    args = ap.parse_args(argv)

    src, dst = load_model(args.model, args.calib), load_model(args.output_model, args.output_calib)
    ri, ro = src.get_resolution(), dst.get_resolution()
    print(f"Remapping {args.model} {ri.width}x{ri.height} -> {args.output_model} {ro.width}x{ro.height} ({args.interpolation})")

    inputs = expand_inputs(args.input)
    outputs = pair_outputs(inputs, args.output)

    frames = np.stack([load_rgb(p) for p in inputs])
    interp = InterpolationMethod.Nearest if args.interpolation == "nearest" else InterpolationMethod.Bilinear
    with RemapPlan(src, dst, None, interp) as plan:
        out = plan.apply(frames)
    for p, a in zip(outputs, out):
        save_rgb(p, a)
        print(f"Saved remapped image to: {p}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
