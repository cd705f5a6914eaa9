"""Builds libssb.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension machinery).

`build()` produces the product library `_lib/libssb.so`.  `build(variant="x", extra=[...])` produces
`_lib/libssb_x.so` with extra nvcc flags -- a development aid for A/B timing on the GPU box
(`SSB_LIB=/path/to/libssb_x.so python bench.py`)."""
from __future__ import annotations

import os
import os.path as osp
import subprocess

PKG_DIR = osp.dirname(osp.abspath(__file__))
SRC = [osp.join(PKG_DIR, "csrc", "ssb_api.cu"), osp.join(PKG_DIR, "csrc", "ssb_policy.cu"),
       osp.join(PKG_DIR, "csrc", "ssb_backward.cu"), osp.join(PKG_DIR, "csrc", "ssb_learn.cu"),
       osp.join(PKG_DIR, "csrc", "ssb_random.cu")]
DEPS = SRC + [osp.join(PKG_DIR, "csrc", f) for f in ("ssb_sim.cuh", "ssb_rollout.cuh", "ssb_types.cuh", "ssb_env.cuh", "ssb_decima.cuh", "ssb_decima_tc.cuh", "ssb_decima_fused.cuh", "ssb_learn.cuh", "ssb_backward.cuh")] + [
    osp.join(osp.dirname(PKG_DIR), "include", "ssb.h")]
OUT = osp.join(PKG_DIR, "_lib", "libssb.so")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    # event times must be single IEEE f64 additions (spark_sched_sim.py:610,632): never contract
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared",
]


LAST: dict = {}  # what the last build() call did (path, compiled or up to date, seconds, the nvcc command line)


def build(force: bool = False, verbose: bool = False, variant: str | None = None,
          extra: list[str] | None = None) -> str:
    out = OUT if variant is None else osp.join(PKG_DIR, "_lib", f"libssb_{variant}.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (extra or []) + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + SRC
    if not force and osp.exists(out) and all(osp.getmtime(d) <= osp.getmtime(out) for d in DEPS):
        LAST.update(path=out, compiled=False, seconds=0.0, command=" ".join(cmd))
        return out
    os.makedirs(osp.dirname(out), exist_ok=True)
    import time

    t0 = time.time()
    subprocess.check_call(cmd)
    LAST.update(path=out, compiled=True, seconds=time.time() - t0, command=" ".join(cmd))
    return out


if __name__ == "__main__":
    print(build(force=True, verbose=True))
