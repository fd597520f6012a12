"""Registers, spills and FP64 instruction counts of the 49 triangulate_kernel instantiations, read from what nvcc makes for
sm_100a (no GPU needed).

    python scripts/triangulate_sass.py

For KB -> Double Sphere and Pinhole -> Pinhole it prints the static FP64 instruction counts (DFMA, DMUL, DADD, DSETP) of
the per-pair loop body: the midpoint path (everything in the grid-stride loop outside the refinement loop) and one
Levenberg-Marquardt trial (the refinement loop body, which also rebuilds J^T J after an accepted step).  The IEEE division
and square-root slow paths are subroutines outside the loop and are not counted; nor are the iterations of a model's own
Newton loop beyond one pass (Kannala-Brandt's unproject).
"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import __graft_entry__ as G  # noqa: E402
import sass_loop_stats as S  # noqa: E402

NAMES = ["Pinhole", "RadTan", "KB", "UCM", "EUCM", "DS", "FOV"]


def loops(ins):
    out = []
    for a, op, rest in ins:
        m = re.search(r"(0x[0-9a-f]+)", rest) if op.startswith("BRA") else None
        if m and int(m.group(1), 16) < a:
            out.append((int(m.group(1), 16), a))
    return out


def fp64(ins, lo, hi):
    ops = collections.Counter(op.split(".")[0] for a, op, _ in ins if lo <= a <= hi)
    return sum(ops[k] for k in S.FP64)


def main():
    out = os.path.join(tempfile.mkdtemp(), "acm_triangulate.cubin")
    cmd = [G.NVCC] + G.ARCH + G.COMMON + G.UNITS["acm_triangulate.cu"] + ["-Xptxas", "-v", "-cubin",
                                                                          os.path.join(G.CSRC, "acm_triangulate.cu"), "-o", out]
    p = subprocess.run(cmd, capture_output=True, text=True, check=True)
    cur, res = None, {}
    for line in (p.stdout + p.stderr).splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res.setdefault(cur, {})["spill"] = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            res.setdefault(cur, {})["regs"] = int(m.group(1))
    table = {}
    for k, v in res.items():
        m = re.search(r"triangulate_kernelILi(\d)ELi(\d)E", k)
        table[(int(m.group(1)), int(m.group(2)))] = (k, v)
    print(f"{len(table)} instantiations")
    print("first \\ second " + " ".join(f"{n:>8}" for n in NAMES))
    for a in range(7):
        row = []
        for b in range(7):
            v = table[(a, b)][1]
            row.append(f"{v['regs']:>5}/{v['spill'][0] + v['spill'][1]:<2}")
        print(f"{NAMES[a]:>15} " + " ".join(f"{c:>8}" for c in row))
    print("(registers / spill bytes)")
    for a, b in ((2, 5), (0, 0)):
        fn = table[(a, b)][0]
        ins = S.instructions(out, fn)
        lp = sorted(loops(ins), key=lambda lp: lp[1] - lp[0], reverse=True)
        grid = lp[0]
        lm = next(lo_hi for lo_hi in lp[1:] if lo_hi[0] >= grid[0] and lo_hi[1] <= grid[1])
        print(f"  loops (start, end): {lp[:4]}")
        total = fp64(ins, *grid)
        trial = fp64(ins, *lm)
        print(f"{NAMES[a]} -> {NAMES[b]}: FP64 per pair, midpoint path {total - trial}; per LM trial {trial}; "
              f"kernel total (static) {fp64(ins, 0, 1 << 30)}")


if __name__ == "__main__":
    main()
