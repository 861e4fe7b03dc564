"""dcmrta_b200/build.py -- compile the CUDA libraries in-tree with nvcc for sm_100a (cross-compiles without a GPU):
libdcmrta_b200.so (the env step, include/dcmrta.h) and libdcmrta_policy.so (the policy's rollout-forward kernels, include/dcmrta_policy.h)."""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
SO = Path(os.environ["DCM_LIB"]).resolve() if os.environ.get("DCM_LIB") else PKG / "libdcmrta_b200.so"
SOURCES = [CSRC / "dcm_kernels.cu"]
HEADERS = [CSRC / "dcm_thread.cuh", CSRC / "dcm_philox.cuh", CSRC / "dcm_soa.h", CSRC / "dcm_layout.h", PKG.parent / "include" / "dcmrta.h"]

NVCC_FLAGS = [
    "-std=c++17", "-O3",
    "-fmad=false",                                   # fp64 event clock must round exactly like the reference (DESIGN.md)
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-Xcompiler", "-fPIC", "-shared",
]

# the policy kernels: bf16 activations, fp32 arithmetic with contraction allowed (nothing there has to round like NumPy)
POLICY_SO = PKG / "libdcmrta_policy.so"
POLICY_SOURCES = [CSRC / "policy_kernels.cu"]
POLICY_HEADERS = [CSRC / "dcm_philox.cuh", PKG.parent / "include" / "dcmrta_policy.h", PKG.parent / "include" / "dcmrta_sample.h"]
POLICY_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC", "-shared"]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(exe).exists():
        raise RuntimeError("nvcc not found: cannot build libdcmrta_b200.so")
    return exe


def source_hash(files=None, flags=None) -> str:
    """sha256 over the sources, headers and flags a library is built from (default: libdcmrta_b200.so)."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS if flags is None else flags).encode())
    for p in (SOURCES + HEADERS if files is None else files):
        h.update(p.name.encode()); h.update(p.read_bytes())
    return h.hexdigest()


HASH = Path(str(SO) + ".hash")


def stale() -> bool:
    """The library is rebuilt when the CONTENT of its sources changed since it was built (a hash written beside it), not when file
    times say so: a snapshot copied to another box (gpurun, a checkout) does not keep them, and N ranks recompiling for 70 s for
    nothing is not a start-up cost anybody wants."""
    if os.environ.get("DCM_LIB"):                    # development: load exactly this prebuilt library (A/B of build variants on one GPU visit)
        return False
    if not SO.exists():
        return True
    if not HASH.exists():                            # a library from before the hash file: fall back to file times
        t = SO.stat().st_mtime
        return any(p.stat().st_mtime > t for p in SOURCES + HEADERS)
    return HASH.read_text().strip() != source_hash()


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile to a temporary file and os.replace() it into place under an exclusive file lock: N ranks of one torchrun job
    that all find the library stale build it once, and nobody ever dlopens a half-written file."""
    if not (force or stale()):
        return SO
    import fcntl
    with open(PKG / ".build.lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not stale():            # another process built it while we waited
                return SO
            tmp = SO.with_name(f".{SO.name}.{os.getpid()}.tmp")
            cmd = [nvcc(), *NVCC_FLAGS, "-o", str(tmp), *map(str, SOURCES)]
            # DCM_BUILD_FAST=1 (development only): optimise the kernels of the one translation unit in parallel, 3 min -> under 1.
            # Not the default: register allocation then differs from build to build (k_step 0..64 B of spills, k_obs_tile 76..94 registers).
            if os.environ.get("DCM_BUILD_FAST") == "1":
                cmd[1:1] = ["--split-compile", "0"]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                tmp.unlink(missing_ok=True)
                raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
            os.replace(tmp, SO)
            HASH.write_text(source_hash() + "\n")
            if verbose:
                print(r.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return SO


def policy_stale() -> bool:
    h = Path(str(POLICY_SO) + ".hash")
    return not POLICY_SO.exists() or not h.exists() or h.read_text().strip() != source_hash(POLICY_SOURCES + POLICY_HEADERS, POLICY_FLAGS)


def build_policy(force: bool = False, verbose: bool = False) -> Path:
    """libdcmrta_policy.so, with the same discipline as build(): content hash, file lock, temporary file + os.replace()."""
    if not (force or policy_stale()):
        return POLICY_SO
    import fcntl
    with open(PKG / ".build.lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not policy_stale():
                return POLICY_SO
            tmp = POLICY_SO.with_name(f".{POLICY_SO.name}.{os.getpid()}.tmp")
            cmd = [nvcc(), *POLICY_FLAGS, "-o", str(tmp), *map(str, POLICY_SOURCES)]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                tmp.unlink(missing_ok=True)
                raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
            os.replace(tmp, POLICY_SO)
            Path(str(POLICY_SO) + ".hash").write_text(source_hash(POLICY_SOURCES + POLICY_HEADERS, POLICY_FLAGS) + "\n")
            if verbose:
                print(r.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return POLICY_SO


if __name__ == "__main__":
    print(build(force=True, verbose=True))
    print(build_policy(force=True, verbose=True))
