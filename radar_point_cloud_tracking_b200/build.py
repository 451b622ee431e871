"""Build ``libradarb200.so`` (hand-written CUDA for sm_100a + the C ABI) in-tree with nvcc."""
from __future__ import annotations

import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
INCLUDE = PKG.parent / "include"
LIB = PKG / "libradarb200.so"
SOURCES = ["context.cu", "spoke.cu", "land.cu", "dbscan.cu", "fuse.cu", "synth.cu", "pipeline.cu", "csv.cu", "plyfmt.cu", "clusters.cu", "comm.cu", "shard.cu", "recording.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--expt-extended-lambda",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "--fmad=false",            # no silent FMA contraction: the float32/float64 chains are bit-exact contracts
]


def nvcc_path() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(cand).exists():
        raise RuntimeError("nvcc not found; cannot build libradarb200.so")
    return cand


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = [CSRC / s for s in SOURCES] + [CSRC / "common.cuh", INCLUDE / "radarb200.h", Path(__file__)]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    """One nvcc process per source file (in parallel, objects under ``build/``; only stale ones are recompiled), then
    one link. ``build.log`` (git-ignored) keeps the ptxas -v output of the files compiled last."""
    if not force and not needs_build():
        return LIB
    from concurrent.futures import ThreadPoolExecutor

    obj_dir = PKG / "build"
    obj_dir.mkdir(exist_ok=True)
    common = [CSRC / "common.cuh", INCLUDE / "radarb200.h", Path(__file__)]
    nvcc = nvcc_path()

    def compile_one(name: str):
        src, obj = CSRC / name, obj_dir / (name + ".o")
        if not force and obj.exists() and all(obj.stat().st_mtime >= d.stat().st_mtime for d in [src, *common]):
            return name, 0, ""
        cmd = [nvcc, "-c", *NVCC_FLAGS, "-I", str(INCLUDE), "-I", str(CSRC), "-o", str(obj), str(src)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        return name, res.returncode, " ".join(cmd) + "\n" + res.stdout + res.stderr

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    log = "".join(r[2] for r in results)
    failed = [r[0] for r in results if r[1] != 0]
    if not failed:
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(LIB), *[str(obj_dir / (s + ".o")) for s in SOURCES], "-ldl"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        log += " ".join(cmd) + "\n" + res.stdout + res.stderr
        if res.returncode != 0:
            failed = ["link"]
    (PKG / "build.log").write_text(log)
    if failed:
        sys.stderr.write(log)
        raise RuntimeError(f"nvcc failed building libradarb200.so ({', '.join(failed)})")
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
