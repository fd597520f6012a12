"""CPU-side checks of the drop-in boundary: libacm.so loads, exports every symbol include/acm.h
declares, the ctypes table covers the header, host-only logic (`new`, `validate_params`, YAML,
error mapping, shard ranges) behaves like the reference.  No compute calls here."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import apex_camera_models_b200 as acm
from apex_camera_models_b200 import _native as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "acm.h")


def _declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(acm_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    declared = _declared_functions()
    assert len(declared) >= 45
    out = subprocess.run(["nm", "-D", "--defined-only", N.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (acm_[a-z0-9_]+)", out))
    missing = [f for f in declared if f not in exported]
    assert not missing, f"declared in acm.h but not exported: {missing}"
    assert sorted(N.SIGNATURES) == declared, "ctypes table and header disagree"


def test_library_is_sm100a_cuda():
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-lelf", N.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_device_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(acm.AcmError, match="no CUDA device"):
        acm.Context(0)
    h = C.c_void_p()
    assert N.lib.acm_ctx_create(0, None, C.byref(h)) == N.ERR_NO_DEVICE


def test_abi_version_and_param_counts():
    assert N.lib.acm_abi_version() == 2
    assert [N.lib.acm_n_params(m) for m in range(7)] == [4, 9, 8, 5, 6, 6, 5]
    assert N.lib.acm_n_params(7) < 0


def test_new_rejects_wrong_length():
    """tests/model_conversions.rs:162-169 (test_parameter_bounds_checking)."""
    for cls, bad in [(acm.DoubleSphereModel, [500.0, 500.0]), (acm.KannalaBrandtModel, [500.0]), (acm.RadTanModel, [500.0, 500.0]),
                     (acm.UcmModel, [500.0]), (acm.EucmModel, [500.0]), (acm.PinholeModel, [500.0]), (acm.FovModel, [1.0])]:
        with pytest.raises(acm.InvalidParams):
            cls.new(bad)
    with pytest.raises(acm.InvalidParams, match=r"Expected 6 parameters \(fx, fy, cx, cy, alpha, xi\), got 2"):
        acm.DoubleSphereModel.new([500.0, 500.0])


def test_new_rejects_invalid_intrinsics():
    """tests/model_conversions.rs:172-184: only Pinhole / RadTan validate in `new`."""
    with pytest.raises(acm.FocalLengthMustBePositive):
        acm.PinholeModel.new([-500.0, 500.0, 320.0, 240.0])
    with pytest.raises(acm.FocalLengthMustBePositive):
        acm.PinholeModel.new([0.0, 500.0, 320.0, 240.0])
    with pytest.raises(acm.PrincipalPointMustBeFinite):
        acm.PinholeModel.new([500.0, 500.0, float("inf"), 240.0])
    with pytest.raises(acm.PrincipalPointMustBeFinite):
        acm.PinholeModel.new([500.0, 500.0, 320.0, float("nan")])
    with pytest.raises(acm.FocalLengthMustBePositive):
        acm.RadTanModel.new([-1.0, 500.0, 320.0, 240.0, 0, 0, 0, 0, 0])
    # DS / KB / UCM / EUCM / FOV `new` do not validate (double_sphere.rs:157-159)
    m = acm.DoubleSphereModel.new([-1.0, 500.0, 320.0, 240.0, 5.0, 0.0])
    with pytest.raises(acm.FocalLengthMustBePositive):
        m.validate_params()
    assert m.get_resolution() == acm.Resolution(0, 0)


def test_validate_params_messages(cameras):
    """double_sphere.rs:812-842, ucm.rs:695-708, eucm.rs:683-713, fov.rs:677-703."""
    def ds(alpha, xi):
        return acm.DoubleSphereModel(acm.Intrinsics(300.0, 300.0, 320.0, 240.0), acm.Resolution(640, 480), [alpha, xi])
    ds(0.5, 0.1).validate_params(); ds(1.0, -0.2).validate_params()
    for bad in (0.0, -0.1, 1.1):
        with pytest.raises(acm.InvalidParams, match=r"alpha must be in \(0, 1\]"):
            ds(bad, 0.0).validate_params()
    with pytest.raises(acm.InvalidParams, match="xi must be finite"):
        ds(0.5, float("nan")).validate_params()
    ucm = acm.UcmModel(acm.Intrinsics(300.0, 300.0, 1.0, 1.0), acm.Resolution(1, 1), [float("inf")])
    with pytest.raises(acm.InvalidParams, match="alpha must be finite"):
        ucm.validate_params()
    acm.UcmModel(acm.Intrinsics(300.0, 300.0, 1.0, 1.0), acm.Resolution(1, 1), [1.01674]).validate_params()
    with pytest.raises(acm.InvalidParams, match="beta must be finite"):
        acm.EucmModel(acm.Intrinsics(300.0, 300.0, 1.0, 1.0), acm.Resolution(1, 1), [0.5, float("nan")]).validate_params()
    for w in (0.0, 2.220446049250313e-16, 3.0000001, float("nan")):
        with pytest.raises(acm.InvalidParams, match=r"w must be in range \(epsilon, 3.0\]"):
            acm.FovModel(acm.Intrinsics(300.0, 300.0, 1.0, 1.0), acm.Resolution(1, 1), [w]).validate_params()
    acm.FovModel(acm.Intrinsics(300.0, 300.0, 1.0, 1.0), acm.Resolution(1, 1), [3.0]).validate_params()


def _write_sample_yaml(tmp_path, name, cam, key=None):
    p = cam["params"]
    lines = ["cam0:", f"  camera_model: {name}"]
    if key:
        lines += [f"  intrinsics: {p[:4]}", f"  {key}: {p[4:]}"]
    else:
        lines += [f"  intrinsics: {p}"]
    lines += ["  rostopic: /cam0/image_raw", f"  resolution: [{cam['width']}, {cam['height']}]"]
    f = tmp_path / f"{name}.yaml"
    f.write_text("\n".join(lines) + "\n")
    return str(f)


def test_yaml_load_exact_values(tmp_path, cameras):
    """double_sphere.rs:680-692, kannala_brandt.rs:865-884, rad_tan.rs:807-825, pinhole.rs:398-408,
    ucm.rs:536-547, fov.rs:526-537: loading the sample YAML gives exactly these parameters."""
    table = [("double_sphere", acm.DoubleSphereModel, None), ("kannala_brandt", acm.KannalaBrandtModel, "distortion"),
             ("rad_tan", acm.RadTanModel, "distortion"), ("pinhole", acm.PinholeModel, None), ("ucm", acm.UcmModel, None),
             ("eucm", acm.EucmModel, None), ("fov", acm.FovModel, None)]
    for name, cls, key in table:
        path = _write_sample_yaml(tmp_path, name, cameras[name], key)
        m = cls.load_from_yaml(path)
        assert m.params().tolist() == cameras[name]["params"]
        assert (m.resolution.width, m.resolution.height) == (cameras[name]["width"], cameras[name]["height"])
        assert m.get_model_name() == name
    ds = acm.DoubleSphereModel.load_from_yaml(_write_sample_yaml(tmp_path, "double_sphere", cameras["double_sphere"]))
    assert ds.alpha == 0.5657413673629862 and ds.xi == -0.24425190195168348
    assert ds.get_distortion() == [ds.alpha, ds.xi]  # code order wins over the doc-comment (SURVEY Appendix B)


def test_yaml_round_trip_and_kb_asymmetry(tmp_path, cameras):
    """tests/yaml_serialization.rs: save -> load equality; KB saves `distortion_coeffs` but loads
    `distortion` (kannala_brandt.rs:635 vs :737-741), so KB does not round-trip."""
    for name, cls in [("double_sphere", acm.DoubleSphereModel), ("pinhole", acm.PinholeModel), ("ucm", acm.UcmModel),
                      ("eucm", acm.EucmModel), ("fov", acm.FovModel), ("rad_tan", acm.RadTanModel)]:
        c = cameras[name]
        m = cls(acm.Intrinsics(*c["params"][:4]), acm.Resolution(c["width"], c["height"]), c["params"][4:])
        path = str(tmp_path / "out" / f"{name}.yaml")
        m.save_to_yaml(path)
        back = cls.load_from_yaml(path)
        assert back.params().tolist() == c["params"] and back.resolution == m.resolution
    c = cameras["kannala_brandt"]
    kb = acm.KannalaBrandtModel(acm.Intrinsics(*c["params"][:4]), acm.Resolution(512, 512), c["params"][4:])
    path = str(tmp_path / "kb.yaml")
    kb.save_to_yaml(path)
    assert "distortion_coeffs" in open(path).read()
    with pytest.raises(acm.InvalidParams):
        acm.KannalaBrandtModel.load_from_yaml(path)


def test_yaml_errors(tmp_path):
    with pytest.raises(acm.IOError_):
        acm.PinholeModel.load_from_yaml(str(tmp_path / "missing.yaml"))
    f = tmp_path / "bad.yaml"
    f.write_text("cam1: {}\n")
    with pytest.raises(acm.InvalidParams, match="Missing 'cam0'"):
        acm.PinholeModel.load_from_yaml(str(f))
    f.write_text("cam0:\n  intrinsics: [1.0, 2.0]\n  resolution: [1, 1]\n")
    with pytest.raises(acm.InvalidParams, match="at least 4"):
        acm.PinholeModel.load_from_yaml(str(f))
    f.write_text("cam0:\n  intrinsics: [-1.0, 2.0, 3.0, 4.0]\n  resolution: [1, 1]\n")
    with pytest.raises(acm.FocalLengthMustBePositive):
        acm.PinholeModel.load_from_yaml(str(f))


def test_point_status_maps_to_reference_error_variants():
    from apex_camera_models_b200.errors import raise_point_status
    raise_point_status(0)
    for code, exc in [(1, acm.PointIsOutSideImage), (2, acm.PointAtCameraCenter), (3, acm.ProjectionOutSideImage), (4, acm.NumericalError)]:
        with pytest.raises(exc):
            raise_point_status(code, 2)
    assert str(acm.PointAtCameraCenter()) == "z is close to zero, point is at camera center"
    assert str(acm.ProjectionOutSideImage()) == "Projection is outside the image"


def test_shard_ranges_cover_and_partition():
    for n in (0, 1, 7, 450, 10_000_000, 100_000_003):
        for world in (1, 2, 3, 4, 8):
            r = [acm.shard_range(n, k, world) for k in range(world)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(r[k][1] == r[k + 1][0] for k in range(world - 1))
            sizes = [b - a for a, b in r]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        acm.shard_range(10, 2, 2)


def test_converter_contract_tables():
    """bounds / tolerances copied from bin/camera_converter.rs:395-400, :410-415 (+ clones)."""
    assert acm.CONVERTER_BOUNDS[5] == [(1.0, 2000.0), (1.0, 2000.0), (0.0, 2000.0), (0.0, 2000.0), (1e-6, 1.0), (-5.0, 5.0)]
    assert acm.CONVERTER_BOUNDS[3][4] == (1e-6, 10.0) and acm.CONVERTER_BOUNDS[4][5] == (1e-6, 5.0) and acm.CONVERTER_BOUNDS[6][4] == (1e-6, 3.0)
    assert acm.CONVERTER_BOUNDS[1][6] == (-1.0, 1.0) and acm.CONVERTER_BOUNDS[2][7] == (-5.0, 5.0)
    cfg = N.LMConfig()
    assert N.lib.acm_lm_default_config(C.byref(cfg)) == 0
    assert (cfg.max_iterations, cfg.cost_tolerance, cfg.parameter_tolerance, cfg.gradient_tolerance) == (100, 1e-6, 1e-8, 1e-6)
    d = acm.LevenbergMarquardtConfig()
    assert (d.max_iterations, d.cost_tolerance, d.parameter_tolerance, d.gradient_tolerance) == (100, 1e-6, 1e-8, 1e-6)


def test_struct_sizes_match_header():
    # a C compiler's view of the header (guards the ctypes mirrors against layout drift)
    src = r'''
#include <stdio.h>
#include "acm.h"
int main(void){ printf("%zu %zu %zu %zu %zu\n", sizeof(acm_camera), sizeof(acm_normal_equations), sizeof(acm_lm_config), sizeof(acm_lm_result), sizeof(acm_projection_error)); return 0; }
'''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c"); exe = os.path.join(d, "s")
        open(c, "w").write(src)
        subprocess.run(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        sizes = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [C.sizeof(N.Camera), C.sizeof(N.NormalEquations), C.sizeof(N.LMConfig), C.sizeof(N.LMResult), C.sizeof(N.ProjectionError)]


# ------------------------------------------------------------------ report text (reporting.rs) ---
def test_rust_float_formatting_and_report_layout(tmp_path):
    """reporting.rs:225-413: the exported text file, with Rust's `{}` / `{:?}` / `{:.N}` float formatting."""
    from types import SimpleNamespace as NS
    from apex_camera_models_b200.reporting import (export_conversion_results, format_conversion_report, model_debug, rust_debug_f64,
                                                   rust_display_f64)
    assert [rust_display_f64(v) for v in (1.0, 0.5, 1e-7, 1e16, -0.28340811, 0.0)] == ["1", "0.5", "0.0000001", "10000000000000000", "-0.28340811", "0"]
    assert [rust_debug_f64(v) for v in (1.0, 1.76187114e-05, 0.00019359, 1e16, 2.5e-10, 0.0)] == ["1.0", "1.76187114e-5", "0.00019359", "1e16", "2.5e-10", "0.0"]
    assert rust_display_f64(float("nan")) == "NaN" and rust_debug_f64(float("inf")) == "inf"

    def model(name, intr, dist):
        return NS(get_model_name=lambda: name, get_intrinsics=lambda: NS(fx=intr[0], fy=intr[1], cx=intr[2], cy=intr[3]),
                  get_distortion=lambda: dist, get_resolution=lambda: NS(width=752, height=480))
    ds = model("double_sphere", (158.5, 158.25, 254.0, 256.125), [0.59, -0.17])
    rt = model("rad_tan", (461.629, 460.152, 362.68, 246.049), [-0.28340811, 0.07395907, 0.00019359, 1.76187114e-05, 0.0])
    assert model_debug(ds) == "DoubleSphere(DoubleSphere [fx: 158.5 fy: 158.25 cx: 254 cy: 256.125 alpha: 0.59 xi: -0.17])"
    assert model_debug(rt) == "RadTan(RadTan [fx: 461.629 fy: 460.152 cx: 362.68 cy: 246.049 distortions: [-0.28340811, 0.07395907, 0.00019359, 1.76187114e-5, 0.0]])"
    assert model_debug(model("pinhole", (500.0, 500.0, 320.0, 240.0), [])) == \
        "Pinhole(PinholeModel { intrinsics: Intrinsics { fx: 500.0, fy: 500.0, cx: 320.0, cy: 240.0 }, resolution: Resolution { width: 752, height: 480 } })"
    err = lambda mean: NS(mean=mean, rmse=mean * 1.5, min=0.0, max=mean * 9, stddev=mean, median=mean * 0.8)
    val = NS(average_error=0.00321, max_error=float("nan"), status="GOOD")
    metrics = [NS(model=ds, model_name="Double Sphere", final_reprojection_error=err(0.0077324), initial_reprojection_error=err(10.0321),
                  optimization_time_ms=1.2345, convergence_status="Converged", validation_results=val, image_quality=NS(psnr=float("inf"), ssim=0.99951)),
               NS(model=rt, model_name="Radial-Tangential", final_reprojection_error=err(184.95), initial_reprojection_error=err(34.5),
                  optimization_time_ms=0.5, convergence_status="Linear Only", validation_results=val, image_quality=None)]
    text = format_conversion_report(metrics, "kb")
    lines = text.split("\n")
    assert lines[0] == "FISHEYE CAMERA MODEL CONVERSION ANALYSIS REPORT - RUST IMPLEMENTATION" and lines[3] == "INPUT MODEL TYPE: KB"
    assert "Double Sphere                    |      0.007732   |     10.024368   |        1.23   | Converged      " in lines
    assert "Radial-Tangential                |    184.950000   |   -150.450000   |        0.50   | Linear Only    " in lines
    assert "🏆 Best Accuracy: Double Sphere (0.007732 pixels)" in lines and "⚡ Fastest Conversion: Radial-Tangential (0.50 ms)" in lines
    assert "DOUBLE SPHERE MODEL:" in lines and "-" * (len("Double Sphere") + 7) in lines
    assert "  Mean: 0.00773240 px" in lines and "  Max Error: NaN px" in lines and "  PSNR: inf dB" in lines and "  SSIM: 0.9995" in lines
    path = export_conversion_results(metrics, "KB", str(tmp_path))
    assert path.endswith("camera_conversion_results_kb.txt") and open(path, encoding="utf-8").read() == text
    assert "No conversions performed" in format_conversion_report([], "pinhole")


def test_rust_ffi_crate_declares_every_header_symbol():
    """rust/acm-sys (uncompiled here: no Rust toolchain) must bind exactly the functions include/acm.h declares,
    and the wrapper crate may only call functions acm-sys declares."""
    sys_rs = open(os.path.join(ROOT, "rust", "acm-sys", "src", "lib.rs")).read()
    declared = set(re.findall(r"pub fn (acm_[a-z0-9_]+)\s*\(", sys_rs))
    header = set(_declared_functions())
    assert header - declared == set(), f"in acm.h but not in acm-sys: {sorted(header - declared)}"
    assert declared - header == set(), f"in acm-sys but not in acm.h: {sorted(declared - header)}"
    wrapper = open(os.path.join(ROOT, "rust", "apex-camera-models-cuda", "src", "lib.rs")).read()
    used = set(re.findall(r"sys::(acm_[a-z0-9_]+)\s*\(", wrapper))
    assert used <= declared, sorted(used - declared)
    consts = set(re.findall(r"sys::(ACM_[A-Z0-9_]+)", wrapper))
    have = set(re.findall(r"pub const (ACM_[A-Z0-9_]+)", sys_rs))
    assert consts <= have, sorted(consts - have)
    # the drop-in: `impl CameraModel for GpuCamera<M>` with every method of the reference's trait (src/camera/mod.rs:241-340) ...
    m = re.search(r"impl<M: CameraModel \+ GpuModelId> CameraModel for GpuCamera<M> \{(.*?)\n\}\n", wrapper, re.S)
    assert m, "the wrapper crate must implement the reference's trait for GpuCamera"
    trait_methods = {"project", "unproject", "load_from_yaml", "save_to_yaml", "validate_params", "get_resolution", "get_intrinsics",
                     "get_distortion", "get_model_name"}
    assert set(re.findall(r"fn ([a-z_]+)\s*\(", m.group(1))) == trait_methods
    # ... a model id for each of the seven reference model types ...
    assert set(re.findall(r"impl GpuModelId for (\w+)", wrapper)) == {"PinholeModel", "RadTanModel", "KannalaBrandtModel", "UcmModel", "EucmModel",
                                                                      "DoubleSphereModel", "FovModel"}
    # ... the README-era facade (README.md:70-81), one newtype per target model with the five methods ...
    assert set(re.findall(r"optimization_cost!\((\w+),", wrapper)) == {"DoubleSphereOptimizationCost", "KannalaBrandtOptimizationCost", "RadTanOptimizationCost",
                                                                        "UcmOptimizationCost", "EucmOptimizationCost", "FovOptimizationCost"}
    macro = re.search(r"macro_rules! optimization_cost \{(.*?)\n\}\n", wrapper, re.S).group(1)
    assert {"new", "linear_estimation", "optimize", "get_intrinsics", "get_distortion"} <= set(re.findall(r"pub fn ([a-z_]+)", macro))
    # ... and the single-thread multi-GPU group over the *_multi entry points
    assert {"acm_comm_init_all", "acm_lm_solve_multi", "acm_linear_estimation_multi", "acm_reprojection_error_multi", "acm_sample_points_multi",
            "acm_linearize_multi", "acm_comm_destroy_all"} <= used


def test_export_point_correspondences_format(tmp_path):
    """point_sampling.rs:153-237: CSV + Rust-literal dump with `{:.15}` coordinates."""
    from apex_camera_models_b200.reporting import export_point_correspondences
    from apex_camera_models_b200.errors import UtilError
    p3 = np.array([[0.1, -0.2, 1.0], [1.0 / 3.0, 2.0, 3.5]]); p2 = np.array([[10.5, 20.25], [300.0, 400.125]])
    csv_path, rust_path = export_point_correspondences(p3, p2, "kb_points", str(tmp_path))
    lines = open(csv_path).read().split("\n")
    assert lines[:3] == ["# 3D-2D Point Correspondences from Rust Implementation", "# Format: x3d,y3d,z3d,x2d,y2d", "# Total points: 2"]
    assert lines[3] == "0.100000000000000,-0.200000000000000,1.000000000000000,10.500000000000000,20.250000000000000"
    assert lines[4].startswith("0.333333333333333,2.000000000000000,3.500000000000000,300.000000000000000,400.125")
    rust = open(rust_path).read()
    assert rust.startswith("// 3D-2D Point Correspondences for Rust Import\n// Generated from Rust fisheye-tools\nlet points_3d = Matrix3xX::from_columns(&[\n")
    assert "    Vector3::new(0.100000000000000, -0.200000000000000, 1.000000000000000),\n    Vector3::new(0.333333333333333, 2.000000000000000, 3.500000000000000)\n]);\n\nlet points_2d" in rust
    assert rust.endswith("    Vector2::new(300.000000000000000, 400.125000000000000)\n]);\n")
    with pytest.raises(UtilError):
        export_point_correspondences(p3, p2[:1], "bad", str(tmp_path))


def test_staging_frees_everything_and_keeps_the_body_error():
    """Staging.close() tries every free even when one fails; an error of the `with` body wins over a failed free, a failed
    free is raised when the body succeeded, and `keep` takes objects out of the staging.  A stand-in context, no device."""
    from apex_camera_models_b200.runtime import Staging

    class Ctx:
        def __init__(self):
            self.sizes, self.freed, self.bad = [], [], None

        def device_alloc(self, nbytes):
            self.sizes.append(nbytes)
            return 0x1000 * len(self.sizes)

        def device_free(self, ptr):
            self.freed.append(ptr)
            if ptr == self.bad:
                raise acm.AcmError("free failed")

    ctx = Ctx()
    with pytest.raises(acm.AcmError, match="free failed"):
        with Staging(ctx) as s:
            a, b, c = s.alloc(0), s.alloc(8), s.alloc(3)
            ctx.bad = a
            assert s.keep(c) == (c,)
    assert ctx.sizes == [1, 8, 3] and ctx.freed == [a, b]
    ctx.freed = []
    with pytest.raises(ValueError, match="body"):
        with Staging(ctx) as s:
            ctx.bad = s.alloc(1)
            d = s.alloc(1)
            raise ValueError("body")
    assert ctx.freed == [ctx.bad, d]
    s.close()  # a closed staging owns nothing
    assert ctx.freed == [ctx.bad, d]
