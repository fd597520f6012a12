"""Host logic of bench.py that runs without a GPU: the merge of the per-rank extras (maximum over ranks of every
timing, throughput of all ranks over that time, rank-0 samples passed through), the constants the roofline entries
are built from, the --dump-outputs files and the argument checks."""
import importlib.util
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_merge_extras_takes_the_slowest_rank_and_counts_every_ranks_points():
    b = _bench()
    n, world = 1_000_000, 2
    r0 = {"linearize_100M": {"kannala_brandt/pixel": {"ms": 1.0, "_bytes_per_point": 40, "sustained_ms": 1.25, "_r0_sm_mhz": 1700.0}},
          "project_unproject_100M_f64": {"ucm": {"project_ms": 0.5, "project_bytes_per_point": 41, "unproject_ms": 0.4, "unproject_bytes_per_point": 41}}}
    r1 = {"linearize_100M": {"kannala_brandt/pixel": {"ms": 2.0, "_bytes_per_point": 40, "sustained_ms": 1.0}},
          "project_unproject_100M_f64": {"ucm": {"project_ms": 0.25, "project_bytes_per_point": 41, "unproject_ms": 0.8, "unproject_bytes_per_point": 41}}}
    m = b.merge_extras([r0, r1], n, world)
    kb = m["linearize_100M"]["kannala_brandt/pixel"]
    assert kb["ms"] == 2.0 and kb["sustained_ms"] == 1.25          # maximum over ranks
    assert kb["sm_mhz"] == 1700.0                                  # sampled on rank 0 only
    assert kb["gpts_s"] == n * world / 2.0 / 1e6                   # all ranks' points over the slowest rank's time
    assert kb["gb_s"] == n * 40 / 2.0 / 1e6                        # per GPU
    assert kb["gb_s_all_gpus"] == world * kb["gb_s"]
    u = m["project_unproject_100M_f64"]["ucm"]
    assert u["project_ms"] == 0.5 and u["unproject_ms"] == 0.8
    assert u["unproject_gb_s"] == n * 41 / 0.8 / 1e6


def test_fp64_issue_constants():
    b = _bench()
    assert b.FP64_LANES_PER_CLOCK == 148 * 64
    assert set(b.FP64_INSTR_PER_POINT) == {"double_sphere/pixel", "kannala_brandt/pixel", "rad_tan/pixel", "fov/pixel"}
    # 102 FP64 instructions per point at 100 G points/s and 1.5 GHz is 72 % of the pipe
    frac = 102 * 100e9 / (b.FP64_LANES_PER_CLOCK * 1.5e9)
    assert 0.71 < frac < 0.73
    assert b.BYTES_PER_POINT == 40


def test_dump_outputs_writes_the_normal_equations_as_float64(tmp_path):
    from apex_camera_models_b200 import _native as N
    b = _bench()
    ne = N.NormalEquations()
    ne.n_params = 6
    for i in range(36):
        ne.H[i] = 0.5 * i
    for i in range(6):
        ne.g[i] = -1.0 - i
    ne.cost, ne.n_valid = 12.25, 99_999_937
    b.dump_outputs(str(tmp_path / "out"), *b.unpack_normal_equations(ne))
    got = {p.stem: np.load(p) for p in (tmp_path / "out").iterdir()}
    assert set(got) == {"H", "g", "cost", "n_valid"}
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["H"], 0.5 * np.arange(36.0).reshape(6, 6))
    assert np.array_equal(got["g"], -1.0 - np.arange(6.0))
    assert got["cost"].tolist() == [12.25] and got["n_valid"].tolist() == [99_999_937.0]


def test_steps_below_one_is_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_reference_arm_runs_exactly_the_requested_steps_and_dumps_its_last_pass(tmp_path, O):
    """--impl reference on the host: the JSON line reports the requested step count and --dump-outputs holds the normal
    equations of the oracle's pass over the arm's seeded 10 M-point sample."""
    import json
    b = _bench()
    out = tmp_path / "ref"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["steps"] == 2
    xyz = O.synth_points3(b.SEED, 0, 10_000_000, b.COS_MAX, False)
    uv, _ = O.project(O.make_model(O.KB, b.KB_SAMPLE, 512, 512), xyz, nthreads=os.cpu_count() or 1)
    H, g, cost, nv = O.linearize(O.make_model(O.DS, b.DS_START, 512, 512), O.RES_PIXEL, xyz, uv, nthreads=1)
    assert np.array_equal(np.load(out / "H.npy"), H) and np.array_equal(np.load(out / "g.npy"), g)
    assert np.load(out / "cost.npy").tolist() == [cost] and np.load(out / "n_valid.npy").tolist() == [float(nv)]
