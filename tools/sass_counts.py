#!/usr/bin/env python3
"""Per-kernel counts of the control instructions ptxas adds around warp-synchronous operations and divergent code, from the static SASS of a
built library (no GPU needed).  A shuffle, CREDUX or vote that ptxas cannot prove convergent is wrapped in WARPSYNC.COLLECTIVE ... ENDCOLLECTIVE
with a fallback path; every `if` it does not predicate is a BSSY/BSYNC region.  Counts are static (instructions in the binary, not executed).
Usage: python tools/sass_counts.py [path/to/libhcb200.so ...]   (default: the package's lib/libhcb200.so)"""
import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_LIB = os.path.join(ROOT, "trifocal_pose_estimation_using_improved_gpuhc_b200", "lib", "libhcb200.so")
COLUMNS = ("WARPSYNC.COLLECTIVE", "BRA.DIV", "BSSY", "BRA", "SHFL", "CREDUX", "VOTE", "total")
_INSN = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s+(@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_.]*)")


def kernel_name(mangled):
    """`hc_track_kernel<false,true,false>` style names, stable across builds (the anonymous-namespace hash is dropped)."""
    m = re.search(r"\d+(hc_[a-z_]+)(I(?:Lb[01]E)+E)?", mangled)
    if not m:
        return mangled
    name = m.group(1)
    if m.group(2):
        name += "<" + ",".join("true" if b == "1" else "false" for b in re.findall(r"Lb([01])E", m.group(2))) + ">"
    return name


def sass_counts(lib, cuobjdump="cuobjdump"):
    """{kernel name: {column: count}} for every kernel of `lib` (cuobjdump -sass)."""
    out = subprocess.run([cuobjdump, "-sass", lib], check=True, capture_output=True, text=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            cur = counts.setdefault(kernel_name(line.split("Function :", 1)[1].strip()), dict.fromkeys(COLUMNS, 0))
            continue
        m = _INSN.match(line) if cur is not None else None
        if not m:
            continue
        op = m.group(2)
        cur["total"] += 1
        if op.startswith("WARPSYNC.COLLECTIVE"):
            cur["WARPSYNC.COLLECTIVE"] += 1
        if op.startswith("BRA.DIV"):
            cur["BRA.DIV"] += 1
        base = op.split(".")[0]
        if base in cur and base != "total":
            cur[base] += 1
    return counts


def main(argv):
    if shutil.which("cuobjdump") is None:
        sys.exit("cuobjdump not found (CUDA toolkit bin/ on PATH)")
    for lib in argv or [DEFAULT_LIB]:
        print(lib)
        print("  %-40s" % "kernel" + "".join("%21s" % c if i == 0 else "%8s" % c for i, c in enumerate(COLUMNS)))
        for name, c in sass_counts(lib).items():
            print("  %-40s" % name + "".join("%21d" % c[k] if i == 0 else "%8d" % c[k] for i, k in enumerate(COLUMNS)))


if __name__ == "__main__":
    main(sys.argv[1:])
