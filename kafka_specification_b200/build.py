"""Ahead-of-time build: ``.tla`` + ``.cfg``  ->  lowered header  ->  ``libkmc_<model>.so`` (sm_100a).

    python -m kafka_specification_b200.build --all            # every model in models/MODELS.json
    python -m kafka_specification_b200.build Kip320 models/Kip320.cfg --name kip320

Artifacts go to ``build/`` (git-ignored):

    build/libkspecmc.so                 the C-ABI dispatcher (include/kspecmc.h)
    build/models/<name>/model.h         the lowered switch table
    build/models/<name>/model.json      layout / actions / invariants (for trace printing)
    build/models/<name>/libkmc_<name>.so

The ``.tla`` sources are read from the kafka-specification checkout (``KSPEC_TLA_PATH``, or the
default location in ``tla_search_dirs``) and from ``models/``; they are not copied into this
repository.  A build that can read them also saves each lowered model.h / model.json under
``oracle/_ref/models/<name>/`` (git-ignored: it is derived data of the specification); a build on a
machine without the specification (a GPU machine given that directory) compiles those saved headers.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "build")
CSRC = os.path.join(ROOT, "kafka_specification_b200", "csrc")
INCLUDE = os.path.join(ROOT, "include")
MODELS_DIR = os.path.join(ROOT, "models")
SPECS_DIR = os.path.join(ROOT, "tests", "specs")
SAVED_MODELS = os.path.join(ROOT, "oracle", "_ref", "models")
LOWERED_FILES = ("model.h", "model.json")

NVCC_ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def tla_search_dirs() -> list[str]:
    dirs = []
    env = os.environ.get("KSPEC_TLA_PATH")
    if env:
        dirs += env.split(os.pathsep)
    dirs += ["/root/reference", MODELS_DIR, os.path.join(ROOT, "tests", "specs")]
    return [d for d in dirs if os.path.isdir(d)]


def specification_reachable() -> bool:
    """True when a .tla search directory outside this repository (the kafka-specification checkout) exists."""
    return any(d not in (MODELS_DIR, SPECS_DIR) for d in tla_search_dirs())


def nvcc_path() -> str:
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _run(cmd: list[str], log: str | None = None):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log:
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + p.stdout)
    if p.returncode != 0:
        raise RuntimeError(f"command failed ({p.returncode}): {' '.join(cmd)}\n{p.stdout[-4000:]}")
    return p.stdout


def build_dispatcher(force: bool = False) -> str:
    os.makedirs(BUILD, exist_ok=True)
    out = os.path.join(BUILD, "libkspecmc.so")
    src = os.path.join(CSRC, "kspecmc.cpp")
    hdr = os.path.join(INCLUDE, "kspecmc.h")
    if not force and os.path.exists(out) and os.path.getmtime(out) >= max(os.path.getmtime(src), os.path.getmtime(hdr)):
        return out
    _run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", f"-I{INCLUDE}", src, "-o", out, "-ldl"])
    return out


def model_dir(name: str) -> str:
    return os.path.join(BUILD, "models", name)


# build variants: extra nvcc flags and a library-name suffix.  The default build carries the two-phase expand
# kernel only (-DKMC_NO_ONE_PHASE drops the one-phase form of the lowered Next from the translation unit);
# "1p" adds the round-1 one-phase kernel for A/B measurements (option "one_phase": true).
VARIANTS = {
    "": ["-DKMC_NO_ONE_PHASE"],
    "1p": ["-DKMC_ONE_PHASE"],
    "b512": ["-DKMC_NO_ONE_PHASE", "-DEXPAND_BLOCK_THREADS=512", "-DEXPAND_CTAS_PER_SM=2"],    # two 512-thread CTAs per SM
    "bs4": ["-DKMC_NO_ONE_PHASE", "-DKMC_BUCKET_SLOTS=4"],
    "b768": ["-DKMC_NO_ONE_PHASE", "-DEXPAND_BLOCK_THREADS=768"],      # 24 warps: leaves registers for K2 blocks (overlap)
    "b512x1": ["-DKMC_NO_ONE_PHASE", "-DEXPAND_BLOCK_THREADS=512"],                                   # 64-byte buckets of 16-byte keys
}


def model_lib_path(name: str, variant: str = "") -> str:
    return os.path.join(model_dir(name), f"libkmc_{name}{'.' + variant if variant else ''}.so")


def _engine_stamp() -> str:
    h = hashlib.sha256()
    for p in (os.path.join(CSRC, "kmc_engine.cu"), os.path.join(INCLUDE, "kspecmc.h")):
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def lower_to_dir(module: str, cfg_path: str, name: str, **lower_kw):
    """Lower and write model.h / model.json; returns the LoweredModel."""
    import time
    from .lower.model import lower_model
    with open(cfg_path) as f:
        cfg_text = f.read()
    t0 = time.time()
    m = lower_model(module, tla_search_dirs(), cfg_text, name=name, **lower_kw)
    lower_seconds = time.time() - t0
    d = model_dir(name)
    os.makedirs(d, exist_ok=True)
    hdr = os.path.join(d, "model.h")
    old = open(hdr).read() if os.path.exists(hdr) else None
    if old != m.header:
        with open(hdr, "w") as f:
            f.write(m.header)
    meta = m.meta()
    meta["cfg"] = os.path.relpath(cfg_path, ROOT)
    meta["lower_seconds"] = round(lower_seconds, 2)      # parse + lower on the build host (part of a cold start)
    with open(os.path.join(d, "model.json"), "w") as f:
        json.dump(meta, f, indent=1)
    return m


def compile_model(name: str, force: bool = False, verbose_ptxas: bool = True, variant: str = "",
                  extra_flags: list[str] | None = None) -> str:
    d = model_dir(name)
    hdr = os.path.join(d, "model.h")
    so = model_lib_path(name, variant)
    stamp_file = os.path.join(d, f"build{'.' + variant if variant else ''}.stamp")
    with open(hdr, "rb") as f:
        stamp = hashlib.sha256(f.read()).hexdigest()[:16] + ":" + _engine_stamp()
    if not force and os.path.exists(so) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return so
    cmd = [nvcc_path(), *NVCC_ARCH, "-lineinfo", "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC",
           "-diag-suppress", "177", *VARIANTS[variant], *(extra_flags or []),
           f"-I{INCLUDE}", "-include", hdr, os.path.join(CSRC, "kmc_engine.cu"), "-o", so]
    if verbose_ptxas:
        cmd[1:1] = ["-Xptxas", "-v"]
    import time
    t0 = time.time()
    _run(cmd, log=os.path.join(d, f"nvcc{'.' + variant if variant else ''}.log"))
    with open(os.path.join(d, f"nvcc{'.' + variant if variant else ''}.log"), "a") as f:
        f.write(f"nvcc wall time: {time.time() - t0:.1f} s\n")
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return so


def compile_model_to(name: str, out_so: str) -> str:
    """Plain nvcc of the prebuilt lowered header into `out_so` (no stamp, no log): the cold-start timing of bench.py."""
    hdr = os.path.join(model_dir(name), "model.h")
    _run([nvcc_path(), *NVCC_ARCH, "-lineinfo", "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-diag-suppress", "177",
          *VARIANTS[""], f"-I{INCLUDE}", "-include", hdr, os.path.join(CSRC, "kmc_engine.cu"), "-o", out_so])
    return out_so


def prepare_model(module: str, cfg_path: str, name: str) -> None:
    """Puts build/models/<name>/model.h and model.json in place.  With the specification reachable the model is
    lowered and saved under oracle/_ref/models/<name>/; without it the saved copy is used when there is one, else
    the model is lowered from this repository's own modules (a module that is not there raises ModuleError)."""
    saved = os.path.join(SAVED_MODELS, name)
    if specification_reachable():
        lower_to_dir(module, cfg_path, name)
        os.makedirs(saved, exist_ok=True)
        for f in LOWERED_FILES:
            shutil.copyfile(os.path.join(model_dir(name), f), os.path.join(saved, f))
    elif all(os.path.exists(os.path.join(saved, f)) for f in LOWERED_FILES):
        os.makedirs(model_dir(name), exist_ok=True)
        for f in LOWERED_FILES:
            shutil.copyfile(os.path.join(saved, f), os.path.join(model_dir(name), f))
    else:
        lower_to_dir(module, cfg_path, name)


def build_model(module: str, cfg_path: str, name: str, force: bool = False) -> str:
    """Lower (or take the saved lowering, see prepare_model) and compile; returns the library path."""
    prepare_model(module, cfg_path, name)
    return compile_model(name, force=force)


def registry() -> dict:
    with open(os.path.join(MODELS_DIR, "MODELS.json")) as f:
        return json.load(f)


def build_all(force: bool = False, only: list[str] | None = None, verbose: bool = True, jobs: int = 0) -> dict[str, str]:
    """Lower (sequentially, it is fast) and compile (in parallel: nvcc dominates) every registered model."""
    from concurrent.futures import ThreadPoolExecutor
    build_dispatcher(force)
    todo = []
    for name, spec in registry().items():
        if only and name not in only:
            continue
        prepare_model(spec["module"], os.path.join(ROOT, spec["cfg"]), name)
        todo.append(name)
    jobs = jobs or min(8, os.cpu_count() or 1)

    def one(name):
        so = compile_model(name, force=force)
        if verbose:
            print(f"[build] {name}: {so}", flush=True)
        return name, so

    with ThreadPoolExecutor(max_workers=jobs) as ex:
        return dict(ex.map(one, todo))


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("module", nargs="?")
    ap.add_argument("cfg", nargs="?")
    ap.add_argument("--name")
    ap.add_argument("--all", action="store_true")
    ap.add_argument("--force", action="store_true")
    a = ap.parse_args(argv)
    if a.all or not a.module:
        for n, p in build_all(force=a.force).items():
            print(n, p)
        return 0
    build_dispatcher(a.force)
    name = a.name or a.module
    print(build_model(a.module, a.cfg, name, force=a.force))
    return 0


if __name__ == "__main__":
    sys.exit(main())
