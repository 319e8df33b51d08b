"""Build ``libscs_b200.so`` in-tree with nvcc for sm_100a.

    python -m spectralclustersupertree_b200.build [--force]

The library is plain CUDA C++ behind the C ABI of ``include/scs_b200.h``; it has no Python or
torch dependency.  nvcc cross-compiles without a GPU, so this also runs in the CPU-only build
container; the built ``.so`` is git-ignored but travels with the source tree.
"""

from __future__ import annotations

import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
INCLUDE = PKG.parent / "include"
LIB = PKG / "libscs_b200.so"

SOURCES = ["context.cu", "pcg.cu", "components.cu", "contract.cu", "spectral.cu", "medium.cu", "small.cu", "shard.cu", "driver.cu", "devforest.cu", "devdriver.cu", "support.cu", "triplets.cu", "pairwise.cu", "forest.cpp", "newick.cpp"]
HEADERS = ["common.cuh", "shard.cuh", "forest.hpp", "spectral_dev.cuh", "uf.cuh", "devforest.cuh", "driver.hpp", "supertree.cuh", "dominance.cuh"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "--fmad=true",  # contraction is wanted in the matvec; the graph build uses __dmul_rn/__dadd_rn
    "-Xcompiler", "-fPIC,-O2,-Wall,-fopenmp",
    "-shared",
    "-lgomp",
]  # fmt: skip


def find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).is_file():
        msg = "nvcc not found: the CUDA toolkit is required to build libscs_b200.so"
        raise RuntimeError(msg)
    return nvcc


OBJ_DIR = PKG.parent / "build" / "obj"


def _stale(target: Path, deps: list[Path]) -> bool:
    return not target.is_file() or any(d.stat().st_mtime > target.stat().st_mtime for d in deps)


def needs_build() -> bool:
    deps = [CSRC / s for s in SOURCES + HEADERS] + [INCLUDE / "scs_b200.h"]
    return _stale(LIB, deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    """Every source is compiled to its own object (in parallel, only when it or a header changed), then linked."""
    from concurrent.futures import ThreadPoolExecutor

    if not force and not needs_build():
        return LIB
    nvcc = find_nvcc()
    OBJ_DIR.mkdir(parents=True, exist_ok=True)
    headers = [CSRC / h for h in HEADERS] + [INCLUDE / "scs_b200.h"]
    compile_flags = [f for f in NVCC_FLAGS if f not in ("-shared", "-lgomp")]

    def compile_one(name: str):
        src = CSRC / name
        obj = OBJ_DIR / (name + ".o")
        if not force and not _stale(obj, [src, *headers]):
            return obj, None
        cmd = [nvcc, *compile_flags, f"-I{INCLUDE}", f"-I{CSRC}"]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        cmd += ["-c", str(src), "-o", str(obj)]
        return obj, subprocess.run(cmd, capture_output=True, text=True, check=False)

    with ThreadPoolExecutor(max_workers=8) as pool:
        done = list(pool.map(compile_one, SOURCES))
    failed = False
    for _obj, proc in done:
        if proc is not None and (verbose or proc.returncode != 0):
            sys.stderr.write(proc.stdout + proc.stderr)
        failed = failed or (proc is not None and proc.returncode != 0)
    if failed:
        msg = "nvcc failed"
        raise RuntimeError(msg)
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC,-fopenmp", "-lgomp",
            *[str(obj) for obj, _ in done], "-o", str(LIB)]  # fmt: skip
    proc = subprocess.run(link, capture_output=True, text=True, check=False)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        msg = f"link failed with exit code {proc.returncode}"
        raise RuntimeError(msg)
    return LIB


def build_fastflatten(force: bool = False) -> Path | None:
    """The CPython accelerator of ``Forest.from_trees`` (csrc/fastflatten.c): host-side glue, optional."""
    import sysconfig

    src = CSRC / "fastflatten.c"
    out = PKG / ("_fastflatten" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))
    if not force and not _stale(out, [src]):
        return out
    include = sysconfig.get_paths()["include"]
    cmd = ["gcc", "-O2", "-shared", "-fPIC", "-Wall", f"-I{include}", str(src), "-o", str(out), "-lm"]
    proc = subprocess.run(cmd, capture_output=True, text=True, check=False)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        return None
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_fastflatten(force="--force" in sys.argv))
