"""Build libmomlevel_b200.so in-tree with nvcc for sm_100a (no JIT cache, no pip install).

    python -m momlevel_b200._build [--force] [--verbose]

The built library is git-ignored but travels to the GPU box with the gpurun snapshot.
"""

import pathlib
import shutil
import subprocess
import sys

PKG = pathlib.Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libmomlevel_b200.so"
SOURCES = ["ml_api.cu", "ml_tma.cu", "ml_tma_flat.cu", "ml_tma3.cu", "ml_stream.cu", "ml_hostpath.cu", "ml_strat.cu", "ml_mean.cu",
           "ml_pack.cpp"]
NVCC_FLAGS = [
    "-gencode",
    "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-O3",
    "-std=c++17",
    "--threads",
    "0",
    "-shared",
    "-Xcompiler",
    "-fPIC,-pthread",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not pathlib.Path(exe).exists():
        raise RuntimeError("nvcc not found; libmomlevel_b200.so cannot be built")
    return exe


STAMP = PKG / "libmomlevel_b200.so.srchash"


def source_hash():
    """Hash of everything the library is built from (sources, headers, flags): the stamp next to the library says
    which sources it was built from, whatever a copy to another machine has done to the modification times."""
    import hashlib
    import os

    h = hashlib.sha256()
    files = sorted(list(CSRC.glob("*.c*")) + list(CSRC.glob("*.h")) + [PKG.parent / "include" / "momlevel_b200.h"])
    for f in files:
        h.update(f.name.encode())
        h.update(f.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    h.update(os.environ.get("MOMLEVEL_B200_NVCC_FLAGS", "").encode())
    return h.hexdigest()


def needs_build():
    if not LIB.exists() or not STAMP.exists():
        return True
    return STAMP.read_text().strip() != source_hash()


def build(force=False, verbose=False):
    """Compile every CUDA source into one shared library. Returns the library path.

    Safe when several processes get here at once (one rank per GPU under torchrun): the compile runs under an
    exclusive file lock, into a temporary file that is renamed over the library, so nobody ever loads half a file.
    """
    if not force and not needs_build():
        return LIB
    import fcntl
    import os
    import shlex

    lock_path = PKG / ".build.lock"
    with open(lock_path, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():  # another process built it while this one waited
                return LIB
            # extra flags for experiment builds, e.g. MOMLEVEL_B200_NVCC_FLAGS="-DML_TMA_FENCED_RELEASE" (csrc/ml_tma_dev.cuh)
            extra = shlex.split(os.environ.get("MOMLEVEL_B200_NVCC_FLAGS", ""))
            tmp = PKG / f".libmomlevel_b200.{os.getpid()}.tmp.so"
            cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else [])
            cmd += ["-o", str(tmp)] + [str(CSRC / s) for s in SOURCES if (CSRC / s).exists()]
            res = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
            if res.returncode != 0:
                tmp.unlink(missing_ok=True)
                raise RuntimeError("nvcc failed building libmomlevel_b200.so")
            os.replace(tmp, LIB)
            STAMP.write_text(source_hash() + "\n")
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
