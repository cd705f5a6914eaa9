"""Compares the SASS of two cubins kernel by kernel, e.g. the simulator unit before and after a change that must not
touch its kernels:

    nvcc -cubin -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false \\
         -o new.cubin spark-sched-sim_b200/csrc/ssb_api.cu        (same for the parent commit -> old.cubin)
    python profiles/sass_compare.py [--mask-cbank] old.cubin new.cubin

Normalisation: `cuobjdump -sass`, the instruction text of each function (addresses, encodings and comments dropped),
and the hash nvcc puts into the anonymous-namespace part of mangled names masked (it depends on the file's path).
--mask-cbank also masks the offsets of constant-bank 0 operands (`c[0x0][0x...]`): where the kernel arguments sit
there, which moves when a struct passed by value (Params) changes size while the code does not.
Prints one line per function (instruction count, digest, identical / DIFFERENT / only in one) and exits 1 unless
every function is identical in both."""
from __future__ import annotations

import argparse
import hashlib
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def normalised_sass(cubin: str, mask_cbank: bool = False) -> dict[str, list[str]]:
    out = subprocess.run([CUOBJDUMP, "-sass", cubin], capture_output=True, text=True, check=True).stdout
    funcs: dict[str, list[str]] = {}
    cur = None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]+", "ANON", m.group(1))
            cur = funcs.setdefault(name, [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if m and cur is not None:
            ins = m.group(1)
            cur.append(re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][CB]", ins) if mask_cbank else ins)
    return funcs


def main(old: str, new: str, mask_cbank: bool = False) -> int:
    a, b = normalised_sass(old, mask_cbank), normalised_sass(new, mask_cbank)
    same = True
    for name in sorted(set(a) | set(b)):
        if name not in a or name not in b:
            print(f"{name}: only in {'new' if name in b else 'old'}")
            same = False
            continue
        da = hashlib.sha256("\n".join(a[name]).encode()).hexdigest()[:16]
        db = hashlib.sha256("\n".join(b[name]).encode()).hexdigest()[:16]
        ok = da == db
        same &= ok
        print(f"{name}: {len(a[name])} -> {len(b[name])} instructions, {da} -> {db} {'identical' if ok else 'DIFFERENT'}")
    print("all functions identical" if same else "SASS differs")
    return 0 if same else 1


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description="kernel-by-kernel SASS comparison of two cubins")
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--mask-cbank", action="store_true", help="ignore the offsets of constant-bank 0 operands")
    args = ap.parse_args()
    sys.exit(main(args.old, args.new, args.mask_cbank))
