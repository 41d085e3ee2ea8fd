#!/usr/bin/env python
"""Static SASS profile of the culled y scan at the cfg3 shape, k_sweep_y_cull<COORDS, 4, 512, BR>: registers, local memory (spills)
and instruction counts by opcode, from one or more builds of mp_sweep_fast_coords.o (one column per build and branch variant):
   python scripts/scan_sass.py                                  (after python -m midaspom_b200.build)
   python scripts/scan_sass.py OTHER_TREE/midaspom_b200/lib/obj/mp_sweep_fast_coords.o midaspom_b200/lib/obj/mp_sweep_fast_coords.o
Counts are static: instructions in the code, not executed ones.  They cover the whole kernel, set-up and write-back included."""
import collections, re, subprocess, sys
from pathlib import Path

# k_sweep_y_cull<COORDS, 4, 512> (builds before the branch sum) and k_sweep_y_cull<COORDS, 4, 512, false / true>
KERNEL = re.compile(r"_ZN2mp14k_sweep_y_cullILi1ELi4ELi512E(?:Lb([01])E)?EEvNS_9LandscapeIfEE\w+")
OPS = ("SHFL", "FADD", "FMUL", "FFMA", "FSEL", "SEL", "LDS", "STS", "MUFU", "CREDUX", "VOTE", "POPC", "FLO", "BRA", "BAR", "SYNCS", "LDL", "STL")
DEFAULT = Path(__file__).resolve().parents[1] / "midaspom_b200" / "lib" / "obj" / "mp_sweep_fast_coords.o"


def profile(obj):
    """One entry per instantiation of the kernel in obj: (label, registers, stack, local, opcode counts)."""
    res = subprocess.run(["cuobjdump", "-res-usage", str(obj)], capture_output=True, text=True, check=True).stdout
    out = []
    for kernel, branch in sorted({km.group(0): km.group(1) for km in KERNEL.finditer(res)}.items()):
        m = re.search(re.escape(kernel) + r":\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", res)
        if not m:
            continue
        sass = subprocess.run(["cuobjdump", "-sass", "-fun", kernel, str(obj)], capture_output=True, text=True, check=True).stdout
        ops = collections.Counter(re.sub(r"\..*", "", op) for op in
                                  re.findall(r"^\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T\d]\s+)?([A-Z][A-Z0-9_.]*)", sass, re.M))
        label = {None: "", "0": ", branch off", "1": ", branch on"}[branch]
        out.append(dict(label=f"`{obj}`{label}", REG=int(m.group(1)), STACK=int(m.group(2)), LOCAL=int(m.group(4)), ops=ops))
    if not out:
        sys.exit(f"{obj}: no k_sweep_y_cull<COORDS, 4, 512>")
    return out


def main():
    objs = [Path(a) for a in sys.argv[1:]] or [DEFAULT]
    prof = [p for o in objs for p in profile(o)]
    print("`k_sweep_y_cull<COORDS, 4, 512>` (cfg3: 512 threads per task as a cluster of 4 x 128), `cuobjdump` of sm_100a objects\n")
    for i, p in enumerate(prof):
        print(f"- ({i + 1}) {p['label']}")
    print("\n| | " + " | ".join(f"({i + 1})" for i in range(len(prof))) + " |")
    print("|---|" + "---|" * len(prof))
    for key in ("REG", "STACK", "LOCAL"):
        print(f"| {key} | " + " | ".join(str(p[key]) for p in prof) + " |")
    for op in OPS:
        print(f"| {op} | " + " | ".join(str(p['ops'].get(op, 0)) for p in prof) + " |")
    print("| total | " + " | ".join(str(sum(p['ops'].values()) - p['ops'].get('NOP', 0)) for p in prof) + " |")
    print("\nREG = registers per thread, STACK / LOCAL = stack frame / local memory bytes per thread (spills land there); total excludes NOP.")


if __name__ == "__main__":
    main()
