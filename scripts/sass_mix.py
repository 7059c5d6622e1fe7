#!/usr/bin/env python
"""Static SASS opcode counts per kernel of a built library (cuobjdump -sass), so that instruction-mix changes are
reviewable without a GPU.  Counts are of instructions in the binary, not of instructions executed.

    python scripts/sass_mix.py [LIB] [--filter REGEX] [--base OLD_LIB]

LIB defaults to graphnet_classifier_b200/libgnc.so; --filter (default "tc_chain") selects kernels by demangled name.
With --base, each kernel prints a second line with the counts of the same kernel in OLD_LIB.
"""
import argparse
import collections
import os
import re
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLUMNS = ["FFMA", "FADD", "FMUL", "FMNMX", "F2FP", "HADD2", "FFMA2", "FADD2", "FMUL2", "MOV", "LDS", "STS"]
_FUNC = re.compile(r"^\s*Function\s*:\s*(\S+)")
_INSN = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T0-9]\s+)?([A-Z][A-Z0-9_]*)")


def _tool(name):
    for cand in (shutil.which(name), os.path.join("/usr/local/cuda/bin", name)):
        if cand and os.path.exists(cand):
            return cand
    raise SystemExit(f"{name} not found")


def demangle(names):
    try:
        out = subprocess.run([_tool("c++filt")], input="\n".join(names), capture_output=True, text=True, check=True).stdout
        return dict(zip(names, out.splitlines()))
    except (SystemExit, subprocess.CalledProcessError):
        return {n: n for n in names}


def opcode_counts(lib):
    """{mangled kernel name: Counter(base opcode -> count)}; NOPs (alignment padding) are not counted."""
    sass = subprocess.run([_tool("cuobjdump"), "-sass", lib], capture_output=True, text=True, check=True).stdout
    kernels, cur = {}, None
    for line in sass.splitlines():
        m = _FUNC.match(line)
        if m:
            cur = kernels.setdefault(m.group(1), collections.Counter())
            continue
        m = _INSN.match(line)
        if m and cur is not None and m.group(1) != "NOP":
            cur[m.group(1)] += 1
    return kernels


def short(name):
    # "void gnc::chain::tc_chain2_kernel<1, false, true>(gnc::chain::Params)" -> "tc_chain2_kernel<1, false, true>"
    m = re.search(r"(\w+<[^()]*>|\w+)\(", name)
    return m.group(1) if m else name


def row(label, c):
    return f"{label:44s} {sum(c.values()):6d} " + " ".join(f"{c.get(k, 0):6d}" for k in COLUMNS)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib", nargs="?", default=os.path.join(ROOT, "graphnet_classifier_b200", "libgnc.so"))
    ap.add_argument("--filter", default="tc_chain")
    ap.add_argument("--base", default=None, help="a second build of the library to print beside LIB")
    a = ap.parse_args()
    new = opcode_counts(a.lib)
    old = opcode_counts(a.base) if a.base else {}
    names = demangle(sorted(set(new) | set(old)))
    pick = sorted((n for n in names if re.search(a.filter, names[n])), key=lambda n: short(names[n]))
    print(f"{'kernel':44s} {'total':>6s} " + " ".join(f"{k:>6s}" for k in COLUMNS))
    for n in pick:
        if a.base:
            if n in old:
                print(row(short(names[n]) + " [base]", old[n]))
            if n in new:
                print(row(short(names[n]) + " [new]", new[n]))
        elif n in new:
            print(row(short(names[n]), new[n]))


if __name__ == "__main__":
    main()
