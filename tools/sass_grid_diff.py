#!/usr/bin/env python3
"""Instruction-for-instruction SASS comparison of two libvsiq.so builds (no GPU needed).

Kernels are matched by demangled name; a kernel that gained the value-grid template argument (``GRID``, csrc/common.cuh)
is matched with the grid set to the integer grid, i.e. ``fq_fwd_kernel<256, 8, true, 0>`` against the older
``fq_fwd_kernel<256, 8, true>``.  Addresses, encodings and per-build hashes of internal symbol names are ignored.

    python tools/sass_grid_diff.py OLD.so NEW.so      # exit status 1 when an old kernel is missing or differs
"""
import re
import subprocess
import sys

_GRID_KERNELS = ("fq_fwd_kernel", "fq_bwd_ste_kernel", "lsq_bwd_kernel", "lsq_bwd_pt_kernel", "lsq_bwd_pc_kernel",
                 "ci_fwd_kernel", "ci_bwd_kernel", "ci_bwd_tma_kernel")


def kernels(lib: str, drop_grid: bool) -> dict:
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and cur:
            ins = re.sub(r"_INTERNAL_[0-9a-f_]+_\w+?_cu_[0-9a-f]+", "_INTERNAL_", m.group(1))
            funcs[cur].append(re.sub(r"\s+", " ", ins))
    names = list(funcs)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    pat = re.compile(r"(%s)<([^<>]*), 0>" % "|".join(_GRID_KERNELS))
    return {re.sub(r"_INTERNAL_[0-9a-f_]+_\w+?_cu_[0-9a-f]+", "_INTERNAL_", pat.sub(r"\1<\2>", d) if drop_grid else d):
            funcs[n] for n, d in zip(names, dem)}


def main() -> int:
    old, new = kernels(sys.argv[1], False), kernels(sys.argv[2], True)  # only the new build has the grid argument
    bad = 0
    for name, sass in old.items():
        if name not in new:
            print("missing:", name)
            bad += 1
        elif new[name] != sass:
            print("differs:", name)
            bad += 1
    print(f"{len(old)} functions of {sys.argv[1]}: {bad} missing or different; {len(new) - len(old)} new in {sys.argv[2]}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
