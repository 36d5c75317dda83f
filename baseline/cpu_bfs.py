"""Builds and runs baseline/cpu_bfs.cpp (the benchmark's CPU arm) for one prebuilt lowered model.

Used by bench.py only (``--impl reference`` and the ``cpu_baseline`` leg), never by the product.  The model header
comes from build/models/<name>/model.h, so nothing here needs /root/reference at run time.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "build", "cpu_baseline")


def build(model: str, out_dir: str = OUT) -> str:
    hdr = os.path.join(ROOT, "build", "models", model, "model.h")
    src = os.path.join(HERE, "cpu_bfs.cpp")
    if not os.path.exists(hdr):
        raise RuntimeError(f"{hdr} is missing: build the model first")
    # -march=native: the cache key includes this machine's CPU flags, so a library built on the build host is never
    # reused on the GPU box (another CPU => illegal instruction)
    cpu = b""
    try:
        with open("/proc/cpuinfo", "rb") as f:
            cpu = next((l for l in f if l.startswith(b"flags")), b"")
    except OSError:
        pass
    tag = hashlib.sha256(open(hdr, "rb").read() + open(src, "rb").read() + cpu).hexdigest()[:12]
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"cpu_{model}_{tag}.so")
    if not os.path.exists(so):
        subprocess.check_call(["g++", "-O3", "-march=native", "-std=c++20", "-pthread", "-shared", "-fPIC",
                               f'-DKMC_MODEL_HEADER="{hdr}"', src, "-o", so])
    return so


def run(model: str, threads: int = 0, table_log2: int = 24, stop_after_states: int = 0, out_dir: str = OUT) -> dict:
    lib = ctypes.CDLL(build(model, out_dir))
    lib.kmc_cpu_bfs.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint64]
    st = np.zeros(320, dtype=np.uint64)
    rc = lib.kmc_cpu_bfs(st.ctypes.data, threads, table_log2, stop_after_states)
    depth = int(st[2])
    return {"rc": rc, "distinct": int(st[0]), "generated": int(st[1]), "depth": depth, "deadlocks": int(st[3]),
            "fail": int(st[4]), "complete": bool(st[5]), "out_of_model": int(st[6]), "seconds": int(st[7]) / 1e9,
            "threads": int(st[8]), "levels": [int(x) for x in st[64:64 + min(depth, 192)]],
            "violating": [int(x) for x in st[16:32]]}


if __name__ == "__main__":
    import json
    import sys
    r = run(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 0, int(sys.argv[3]) if len(sys.argv) > 3 else 24)
    r.pop("levels")
    print(json.dumps(r))
