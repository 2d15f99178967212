"""In-tree build of libcgx_b200.so (sm_100a only) with plain nvcc.

    python -m new_cg_variants_b200.build [--force]

The shared library is written next to this file so that it travels to the GPU box with
the repository snapshot; it links only the CUDA runtime (no torch, no cuBLAS/cuSPARSE).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
import time

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libcgx_b200.so")
STAMP = LIB_PATH + ".stamp"

OBJ_DIR = os.path.join(PKG_DIR, "_obj")

# translation units: (object name, source, extra defines).  The stage launchers are compiled once
# per preconditioner mode and the persistent kernels once per operator kind, only so that the
# template instantiations build in parallel (one nvcc process per unit).
UNITS = [
    ("cgx_iter_pm0", "cgx_iter.cu", ["-DCGX_PM=0"]),
    ("cgx_iter_pm1", "cgx_iter.cu", ["-DCGX_PM=1"]),
    ("cgx_iter_pm2", "cgx_iter.cu", ["-DCGX_PM=2"]),
    *[(f"cgx_pers_{nm}_pm{pm}", "cgx_pers.cu", [f"-DCGX_PERS_OP={op}", f"-DCGX_PERS_PM={pm}"])
      for op, nm in ((2, "sten"), (1, "csr"), (3, "var")) for pm in (0, 1, 2)],
    ("cgx_fused", "cgx_fused.cu", []),
    ("cgx", "cgx.cu", []),
]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr", "--extended-lambda",
    "-Xptxas", "-v",
    "-Xfatbin", "-compress-all",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libcgx_b200.so cannot be built")


def _fingerprint() -> str:
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    h.update(repr(UNITS).encode())
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    files.append(os.path.join(ROOT, "include", "cgx.h"))
    for path in files:
        with open(path, "rb") as fh:
            h.update(os.path.basename(path).encode())      # (not the absolute path: the tree moves between boxes)
            h.update(fh.read())
    return h.hexdigest()


# device-code headers a kernel class (a key of profiles/traffic.json) is compiled from
_COMMON_CUH = ["cgx_common.cuh", "cgx_kernels.cuh"]
KERNEL_SOURCES = {
    "pr_fused": _COMMON_CUH + ["cgx_stencil_tma.cuh", "cgx_stencil_fused.cuh"],
    "ew_": _COMMON_CUH,
    "sp_": _COMMON_CUH + ["cgx_stencil_tma.cuh"],
    "csr_sp_pipe_r": _COMMON_CUH,                       # two right-hand sides: csr_stream_kernel (cgx_kernels.cuh)
    "csr_": _COMMON_CUH + ["cgx_csr_bulk.cuh"],         # one right-hand side: csr_bulk_kernel
}


def kernel_fingerprint(kernel_class: str | None = None) -> str:
    """sha256 over the device-code headers `kernel_class` is compiled from (all of them when the
    class is unknown or None); profiles/traffic.json entries are stamped with it."""
    files = None
    if kernel_class:
        for prefix, lst in KERNEL_SOURCES.items():
            if kernel_class.startswith(prefix):
                files = [f for f in lst if os.path.exists(os.path.join(CSRC, f))]
                break
    if files is None:
        files = [f for f in sorted(os.listdir(CSRC)) if f.endswith(".cuh")]
    h = hashlib.sha256()
    for f in sorted(files):
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode())
            h.update(fh.read())
    return h.hexdigest()[:16]


def build(force: bool = False, verbose: bool = False) -> str:
    fp = _fingerprint()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(STAMP):
        if open(STAMP).read().strip() == fp:
            return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)

    def compile_unit(unit):
        name, source, defs = unit
        obj = os.path.join(OBJ_DIR, name + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *defs, "-I", os.path.join(ROOT, "include"), "-c", "-o", obj,
               os.path.join(CSRC, source)]
        # incremental rebuilds: an object is reused when the PREPROCESSED unit is unchanged
        pre = subprocess.run([nvcc, "-E", "-std=c++17", "--expt-relaxed-constexpr", "--extended-lambda",
                              "-gencode", "arch=compute_100a,code=sm_100a", *defs,
                              "-I", os.path.join(ROOT, "include"), os.path.join(CSRC, source)],
                             capture_output=True, text=True)
        key = hashlib.sha256((" ".join(cmd[1:]) + pre.stdout).encode()).hexdigest() if pre.returncode == 0 else None
        keyfile = obj + ".key"
        if (not force and key and os.path.exists(obj) and os.path.exists(keyfile)
                and open(keyfile).read() == key):
            old = open(obj + ".log").read() if os.path.exists(obj + ".log") else ""
            return obj, old + f"[{name}: up to date]\n", 0
        if os.path.exists(keyfile):
            os.unlink(keyfile)
        t0 = time.time()
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if proc.returncode == 0 and key:
            with open(keyfile, "w") as fh:
                fh.write(key)
            with open(obj + ".log", "w") as fh:
                fh.write(" ".join(cmd) + "\n" + proc.stdout + proc.stderr)
        return obj, " ".join(cmd) + "\n" + proc.stdout + proc.stderr + f"\n[{name}: {time.time() - t0:.0f} s]\n", proc.returncode

    with ThreadPoolExecutor(max_workers=min(len(UNITS), os.cpu_count() or 1)) as pool:
        results = list(pool.map(compile_unit, UNITS))
    log = "\n".join(r[1] for r in results)
    failed = [r for r in results if r[2] != 0]
    if not failed:
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC",
               "-o", LIB_PATH, *[r[0] for r in results]]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        log += "\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr
        if proc.returncode != 0:
            failed = [(LIB_PATH, proc.stdout + proc.stderr, proc.returncode)]
    with open(os.path.join(PKG_DIR, "build.log"), "w") as fh:
        fh.write(log)
    if failed:
        raise RuntimeError("nvcc failed:\n" + "\n".join(f[1][-6000:] for f in failed))
    if verbose:
        print(log)
    with open(STAMP, "w") as fh:
        fh.write(fp)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
