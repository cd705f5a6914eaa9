"""Compares the SASS of two cubins kernel by kernel, e.g. the simulator unit before and after a change that must not
touch its kernels:

    nvcc -cubin -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false \\
         -o new.cubin spark-sched-sim_b200/csrc/ssb_api.cu        (same for the parent commit -> old.cubin)
    python profiles/sass_compare.py old.cubin new.cubin

Normalisation: `cuobjdump -sass`, the instruction text of each function (addresses, encodings and comments dropped),
and the hash nvcc puts into the anonymous-namespace part of mangled names masked (it depends on the file's path).
Prints one line per function (instruction count, digest, identical / DIFFERENT / only in one) and exits 1 unless
every function is identical in both."""
from __future__ import annotations

import hashlib
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def normalised_sass(cubin: str) -> dict[str, list[str]]:
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
            cur.append(m.group(1))
    return funcs


def main(old: str, new: str) -> int:
    a, b = normalised_sass(old), normalised_sass(new)
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
    sys.exit(main(sys.argv[1], sys.argv[2]))
