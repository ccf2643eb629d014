"""Build the C-ABI CUDA library in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_NAME = "librgbdslam_b200.so"

NVCC_FLAGS = [
    "-ldl",
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def library_path() -> Path:
    """In-tree library; RGBDSLAM_B200_LIB points tools/ at an A/B variant built by tools/build_variants.py."""
    override = os.environ.get("RGBDSLAM_B200_LIB")
    return Path(override) if override else PKG_DIR / LIB_NAME


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found")


def sources() -> list[Path]:
    return sorted(CSRC.glob("*.cu"))


def build_library(force: bool = False, verbose: bool = False) -> Path:
    """Compile csrc/*.cu into librgbdslam_b200.so (skipped if up to date)."""
    import fcntl
    out = PKG_DIR / LIB_NAME
    if not force and _up_to_date(out):  # nothing is written then: the tree may be read-only once built
        return out
    with open(PKG_DIR / ".build.lock", "w") as lk:  # several ranks may call build() at once
        fcntl.flock(lk, fcntl.LOCK_EX)
        return _build_locked(out, force, verbose)


def _up_to_date(out: Path) -> bool:
    deps = sources() + sorted(CSRC.glob("*.h")) + sorted(CSRC.glob("*.cuh")) + [PKG_DIR.parent / "include" / "rgbdslam_b200.h"]
    return out.exists() and out.stat().st_mtime >= max(p.stat().st_mtime for p in deps)


def _build_locked(out: Path, force: bool, verbose: bool) -> Path:
    if not force and _up_to_date(out):
        return out
    srcs = sources()
    cmd = [_nvcc(), *NVCC_FLAGS, "-o", str(out), *map(str, srcs)]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    env = dict(os.environ)
    # the image exports CC=/opt/gcc/bin/gcc; nvcc wants the system g++ as host compiler
    res = subprocess.run(cmd + ["-ccbin", shutil.which("g++") or "g++"], capture_output=True, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return out
