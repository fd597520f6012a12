"""Host-side glue shared by the image command-line tools (`image_undistort`, `image_remap`, `image_rectify`): image files
in and out, camera models by type alias, and the expansion of input directories."""
from __future__ import annotations

import os

import numpy as np

from .camera_converter import INPUT_ALIASES


def load_rgb(path: str) -> np.ndarray:
    if path.endswith(".npy"):
        return np.ascontiguousarray(np.load(path), dtype=np.uint8)
    from PIL import Image  # image decoding is host-side glue, like the `image` crate in the reference
    return np.asarray(Image.open(path).convert("RGB"), dtype=np.uint8)


def save_rgb(path: str, a: np.ndarray) -> None:
    if path.endswith(".npy"):
        np.save(path, a)
        return
    from PIL import Image
    Image.fromarray(a, "RGB").save(path)


def load_model(kind: str, calib: str):
    """The camera model of type `kind` (any of the converter's INPUT_ALIASES) loaded from the YAML file `calib`."""
    cls = INPUT_ALIASES.get(kind.lower())
    if cls is None:
        raise SystemExit(f"Unsupported model: {kind}")
    return cls.load_from_yaml(calib)


def expand_inputs(paths) -> list[str]:
    """Each path in turn; a directory stands for its entries in sorted order."""
    out = []
    for p in paths:
        out += sorted(os.path.join(p, f) for f in os.listdir(p)) if os.path.isdir(p) else [p]
    return out


def pair_outputs(inputs: list[str], outputs: list[str]) -> list[str]:
    """One output path per input: the given paths, or, for a single output that is a directory or that faces several
    inputs, the inputs' file names in that directory (created if missing)."""
    if len(outputs) == 1 and (os.path.isdir(outputs[0]) or len(inputs) > 1):
        os.makedirs(outputs[0], exist_ok=True)
        outputs = [os.path.join(outputs[0], os.path.basename(p)) for p in inputs]
    if len(outputs) != len(inputs):
        raise SystemExit("need one output per input (or one output directory)")
    return outputs
