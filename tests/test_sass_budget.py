"""Instruction budget of the Double Sphere linearize kernels, read from the SASS that nvcc makes for sm_100a (no GPU needed).

The headline pass (`lin_kernel<DOUBLE_SPHERE, PIXEL, 256, false>`) is bound by the FP64 issue rate at the clock the power cap
allows, so its FP64 instructions per point are the figure that matters; this pins them.  The algebraic-residual instantiations
share `Unified<DOUBLE_SPHERE>` with the bench's LM conversion and must not move at all when the pixel path is tuned.
"""
import hashlib
import importlib.util
import os
import re
import subprocess

import pytest

import __graft_entry__ as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("sass_loop_stats", os.path.join(ROOT, "scripts", "sass_loop_stats.py"))
S = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(S)

HEADLINE = "_Z10lin_kernelILi5ELi0ELi256ELb0EEv13LinKernelArgs"
DS_PIXEL = [HEADLINE, "_Z10lin_kernelILi5ELi0ELi128ELb1EEv13LinKernelArgs", "_Z10lin_kernelILi5ELi0ELi256ELb1EEv13LinKernelArgs"]
FP64_PER_POINT_MAX = 68          # the generic Unified/LinUnifiedPixel form compiled to 77.5
POINTS_PER_TRIP = 2
# SHA-1 of the opcode + operand text of every instruction, CUDA 12.9 (V12.9.86); FP64 instructions per trip of the streaming loop
ALGEBRAIC = {
    "_Z10lin_kernelILi5ELi1ELi128ELb1EEv13LinKernelArgs": ("a869b474650ad44202285c79ca40d5532813c728", 142),
    "_Z10lin_kernelILi5ELi1ELi256ELb1EEv13LinKernelArgs": ("b6bdd11926f7cbd0160ff76b8021d316f73b09a7", 142),
    "_Z10lin_kernelILi5ELi1ELi256ELb0EEv13LinKernelArgs": ("9b6c398f4840a6fc3597061f795e00ffa1eb6c85", 143),
}
HASH_RELEASE = "12.9"


@pytest.fixture(scope="module")
def cubin(tmp_path_factory):
    beside = os.path.join(os.path.dirname(G.NVCC), "cuobjdump")
    if os.path.exists(beside):
        S.CUOBJDUMP = beside
    if not os.path.exists(G.NVCC) or not os.path.exists(S.CUOBJDUMP):
        pytest.skip("nvcc / cuobjdump not available")
    out = str(tmp_path_factory.mktemp("sass") / "acm_solver.cubin")
    src = os.path.join(G.CSRC, "acm_solver.cu")
    cmd = [G.NVCC] + G.ARCH + G.COMMON + G.UNITS["acm_solver.cu"] + ["-Xptxas", "-v", "-cubin", src, "-o", out]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    release = re.search(r"release (\d+\.\d+)", subprocess.run([G.NVCC, "--version"], capture_output=True, text=True).stdout)
    return out, p.stdout + p.stderr, release.group(1) if release else None


def _ptxas_entries(log):
    """kernel -> (registers, spill store bytes, spill load bytes) from the -Xptxas -v log."""
    res, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res.setdefault(cur, [None, int(m.group(1)), int(m.group(2))])
        m = re.search(r"Used (\d+) registers", line)
        if m and cur in res:
            res[cur][0] = int(m.group(1))
    return res


def test_double_sphere_kernels_do_not_spill(cubin):
    _, log, _ = cubin
    entries = _ptxas_entries(log)
    ds = {k: v for k, v in entries.items() if k.startswith("_Z10lin_kernelILi5E")}
    assert len(ds) == 6, sorted(ds)
    for k, (regs, st, ld) in ds.items():
        assert st == 0 and ld == 0, (k, st, ld)
    # 256-thread one-pass blocks: two resident per SM (65536 registers); 128-thread solve blocks: MIN_BLOCKS = 2
    assert ds[HEADLINE][0] <= 128, ds[HEADLINE]


def test_double_sphere_pixel_loop_within_fp64_budget(cubin):
    obj, _, _ = cubin
    for fn in DS_PIXEL:
        st = S.loop_stats(obj, fn)
        assert st is not None, fn
        assert st["fp64"] <= FP64_PER_POINT_MAX * POINTS_PER_TRIP, (fn, st["fp64"], dict(st["ops"]))
        assert st["calls"] == 0, fn
        # the back edge and the guarded cp.async refill: nothing else branches inside the loop
        assert st["branches"] <= 2, (fn, st["branches"])


def test_algebraic_double_sphere_sass_unchanged(cubin):
    obj, _, release = cubin
    for fn, (sha, fp64) in ALGEBRAIC.items():
        ins = S.instructions(obj, fn)
        assert ins, fn
        assert S.loop_stats(obj, fn)["fp64"] == fp64, fn
        if release == HASH_RELEASE:
            assert hashlib.sha1("\n".join(op + rest for _, op, rest in ins).encode()).hexdigest() == sha, fn
