"""Count the instruction mix of the streaming loop of a kernel.

    python scripts/sass_loop_stats.py <cubin or .o> <kernel name regex>

The streaming loop is the innermost backward branch whose body both reads the cp.async ring (LDS.128) and refills it
(LDGSTS).  Picking the longest backward branch instead finds the reducer's polling loop in the one-pass kernels and the
whole pass loop in the solve kernels.  Kernels without a ring (register prefetch) fall back to the innermost loop with a
128-bit streaming (evict-first) global load; the hand-off cells are polled with strong loads.
"""
import collections
import os
import re
import shutil
import subprocess
import sys

CUOBJDUMP = os.environ.get("CUOBJDUMP") or shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"

FP64 = ("DFMA", "DMUL", "DADD", "DSETP")
_INS = re.compile(r"/\*([0-9a-f]{4,5})\*/\s+(@!?U?P\w+\s+)?([A-Z0-9_.]+)(.*?);")


def functions(obj):
    txt = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    return re.findall(r"Function : (\S+)", txt)


def instructions(obj, fn):
    """[(address, opcode with modifiers, operands)] of one function."""
    txt = subprocess.run([CUOBJDUMP, "-sass", "-fun", fn, obj], capture_output=True, text=True, check=True).stdout
    return [(int(m.group(1), 16), m.group(3), m.group(4)) for m in map(_INS.search, txt.splitlines()) if m]


def streaming_loop(ins):
    """(first, last) address of the streaming loop, or None."""
    loops = []
    for a, op, rest in ins:
        m = re.search(r"(0x[0-9a-f]+)", rest) if op.startswith("BRA") else None
        if m and int(m.group(1), 16) < a:
            loops.append((int(m.group(1), 16), a))
    for markers in ((r"LDS\.128", r"LDGSTS"), (r"LDG\.E\.EF\.128",)):
        inner = [lp for lp in loops if all(any(lp[0] <= a <= lp[1] and re.match(mk, op) for a, op, _ in ins) for mk in markers)]
        if inner:
            return min(inner, key=lambda lp: lp[1] - lp[0])
    return None


def loop_stats(obj, fn):
    """Instruction mix of the streaming loop of `fn`: {"instrs", "fp64", "branches", "calls", "ops": Counter}."""
    ins = instructions(obj, fn)
    lp = streaming_loop(ins)
    if lp is None:
        return None
    body = [op for a, op, _ in ins if lp[0] <= a <= lp[1]]
    ops = collections.Counter(op.split(".")[0] for op in body)
    return {"instrs": len(body), "fp64": sum(ops[k] for k in FP64), "branches": ops["BRA"], "calls": ops["CALL"], "ops": ops}


if __name__ == "__main__":
    obj, pat = sys.argv[1], sys.argv[2]
    for fn in functions(obj):
        if not re.search(pat, fn):
            continue
        s = loop_stats(obj, fn)
        if s is None:
            continue
        print(fn[:60], "loop instrs", s["instrs"], "fp64", s["fp64"], "bra", s["branches"], dict(s["ops"].most_common(12)))
