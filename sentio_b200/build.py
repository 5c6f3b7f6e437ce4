"""Build libsentio_b200.so in-tree with nvcc for sm_100a (and nothing else).

    python -m sentio_b200.build [--force] [--verbose]

The library is a plain C-ABI shared object (include/sentio_b200.h); it is loaded with ctypes by sentio_b200/_lib.py.
The built .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
OUT = PKG / "libsentio_b200.so"
OBJ = PKG / "build"

SOURCES = ["api.cu", "dense.cu", "bm25.cu", "bm25_build.cu", "fuse.cu", "mmr.cu", "cross_encoder.cu", "ce_gemm.cu", "dense_mma.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        h.update(str(p.name).encode())
        h.update(p.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _sources() -> list[Path]:
    return [CSRC / s for s in SOURCES if (CSRC / s).exists()]


def _compile_and_link(out: Path, obj_dir: Path, defines=(), verbose: bool = False) -> Path:
    """Compile every source into obj_dir with NVCC_FLAGS plus one -D flag per entry of `defines`, link them into `out`."""
    nvcc = _nvcc()
    obj_dir.mkdir(exist_ok=True)
    srcs = _sources()
    flags = [*NVCC_FLAGS, *[f"-D{d}" for d in defines]]

    def compile_one(src: Path) -> Path:
        obj = obj_dir / (src.stem + ".o")
        cmd = [nvcc, *flags, "-c", str(src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src.name}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(out), *map(str, objs),
            "-Xlinker", "--exclude-libs=ALL", "-lcudart_static", "-ldl", "-lrt", "-lpthread"]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return out


def build_variant(name: str, defines, verbose: bool = False) -> Path:
    """A second library `libsentio_b200_<name>.so` from the same sources with extra -D flags (kernel A/B measurements;
    loaded with SENTIO_B200_LIB=<path>)."""
    return _compile_and_link(PKG / f"libsentio_b200_{name}.so", PKG / f"build_{name}", defines, verbose)


def build(force: bool = False, verbose: bool = False) -> Path:
    deps = _sources() + sorted(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "sentio_b200.h"]
    stamp = OBJ / "stamp.txt"
    digest = _digest(deps)
    if not force and OUT.exists() and stamp.exists() and stamp.read_text() == digest:
        return OUT
    _compile_and_link(OUT, OBJ, verbose=verbose)
    stamp.write_text(digest)
    return OUT


if __name__ == "__main__":
    if "--variant" in sys.argv:   # python -m sentio_b200.build --variant NAME -DFOO -DBAR
        i = sys.argv.index("--variant")
        print(build_variant(sys.argv[i + 1], [a[2:] for a in sys.argv if a.startswith("-D")]))
        sys.exit(0)
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
