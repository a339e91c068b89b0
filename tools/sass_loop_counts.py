#!/usr/bin/env python3
"""
Opcode counts of every loop body of one kernel instantiation, from its SASS.

    python tools/sass_loop_counts.py ray_trace_pb_b200/_lib/obj/trace_lean.o "trace_lean_kernel<1,0,0,0,2>"

The first argument is an object file or cubin (anything `cuobjdump -sass` reads), the second a part of the kernel's
demangled name with `true` / `false` written 1 / 0 and no spaces or `(bool)` / `(int)` casts, so "trace_lean_kernel<1,0,0,0,2>"
picks trace_lean_kernel<true, false, false, false, (int)2>.  A loop body is the instructions from a backward branch's
target to the branch.  For each one the script prints its address range, its size, the FP64-pipe instructions (DADD,
DMUL, DFMA, DSETP, DMNMX, DSET) and everything else, and the count of every opcode; innermost loops (no other loop
inside) are marked; the lean kernel's surface-step loops are among them.  Opcodes are counted without modifiers
(DSETP.GEU.AND -> DSETP).
"""
from __future__ import annotations

import argparse
import collections
import os
import re
import shutil
import subprocess
import sys

FP64_PIPE = {"DADD", "DMUL", "DFMA", "DSETP", "DMNMX", "DSET"}

_INSTR = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(@!?U?P[0-9T]+\s+)?([A-Z][A-Z0-9_]*)(\.[A-Z0-9_.]+)?\s*([^;]*);")
_TARGET = re.compile(r"(0x[0-9a-f]+)\s*$")


def _tool(name: str) -> str:
    for d in (os.environ.get("CUDA_HOME"), "/usr/local/cuda"):
        if d and os.path.exists(os.path.join(d, "bin", name)):
            return os.path.join(d, "bin", name)
    found = shutil.which(name)
    if found is None:
        sys.exit(f"{name} not found (CUDA_HOME or PATH)")
    return found


def functions(path: str) -> dict[str, list[tuple[int, str, str]]]:
    """mangled name -> [(address, opcode, operands)] from cuobjdump -sass"""
    text = subprocess.run([_tool("cuobjdump"), "-sass", path], check=True, capture_output=True, text=True).stdout
    out: dict[str, list[tuple[int, str, str]]] = {}
    cur = None
    for line in text.splitlines():
        if "Function :" in line:
            cur = out.setdefault(line.split("Function :", 1)[1].strip(), [])
            continue
        m = _INSTR.match(line)
        if m and cur is not None:
            cur.append((int(m.group(1), 16), m.group(3), m.group(5).strip()))
    return out


def normalised(mangled: list[str]) -> dict[str, str]:
    """mangled -> demangled with 1 / 0 for true / false, no spaces, no casts"""
    dem = subprocess.run([_tool("cu++filt")], input="\n".join(mangled), check=True, capture_output=True,
                         text=True).stdout.splitlines()
    out = {}
    for m, d in zip(mangled, dem):
        d = re.sub(r"\((bool|int|unsigned int)\)", "", d.replace("true", "1").replace("false", "0"))
        out[m] = d.replace(" ", "")
    return out


def loops(code: list[tuple[int, str, str]]) -> list[tuple[int, int]]:
    """(first, last) instruction indices of every backward branch's body"""
    index = {addr: i for i, (addr, _, _) in enumerate(code)}
    out = []
    for i, (addr, op, args) in enumerate(code):
        if op != "BRA":
            continue
        t = _TARGET.search(args)
        if t and int(t.group(1), 16) <= addr and int(t.group(1), 16) in index:
            out.append((index[int(t.group(1), 16)], i))
    return sorted(out)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.strip().splitlines()[0])
    ap.add_argument("object", help="object file or cubin")
    ap.add_argument("kernel", help='part of the normalised demangled name, e.g. "trace_lean_kernel<1,0,0,0,2>"')
    ap.add_argument("--all", action="store_true", help="also print loops that contain other loops")
    args = ap.parse_args()

    funcs = functions(args.object)
    names = normalised(list(funcs))
    picked = [m for m in funcs if args.kernel.replace(" ", "") in names[m]]
    if not picked:
        sys.exit(f"no function matches {args.kernel!r}; functions: " + ", ".join(sorted(set(names.values()))))
    for m in picked:
        code = funcs[m]
        print(f"{names[m]}  ({len(code)} instructions)")
        ls = loops(code)
        for a, b in ls:
            inner = not any((c, d) != (a, b) and a <= c and d <= b for c, d in ls)
            if not (inner or args.all):
                continue
            ops = collections.Counter(op for _, op, _ in code[a:b + 1])
            fp64 = sum(n for op, n in ops.items() if op in FP64_PIPE)
            total = b - a + 1
            print(f"  loop 0x{code[a][0]:04x}-0x{code[b][0]:04x}{'  innermost' if inner else ''}: {total} instr, "
                  f"FP64-pipe {fp64} (" + ", ".join(f"{op} {ops[op]}" for op in sorted(FP64_PIPE) if ops[op]) +
                  f"), other {total - fp64}")
            print("    " + " ".join(f"{op}:{n}" for op, n in sorted(ops.items(), key=lambda kv: (-kv[1], kv[0]))))


if __name__ == "__main__":
    main()
