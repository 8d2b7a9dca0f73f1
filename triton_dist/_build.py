"""In-tree native build for the B200 (sm_100a) backend.

Two shared libraries are produced under ``triton_dist/lib/``:

* ``libtd_b200.so``  -- every CUDA kernel + the device-side runtime (symmetric heap on CUDA VMM,
  multicast, stream mem-ops).  Compiled with ``nvcc -gencode arch=compute_100a,code=sm_100a``.
* ``libtd_host.so``  -- the CPU emulation runtime (POSIX shared-memory symmetric heap + atomic
  signal words + the host task-graph scheduler).  Plain g++.

Both expose a C ABI and are loaded with ctypes (see ``triton_dist/_C.py``) so that nvcc never has to
parse torch headers (seconds per file instead of minutes) and the libraries have no libtorch ABI
dependency.  The reference needs an LLVM/Triton source build plus NVSHMEM bitcode
(/root/reference/python/setup.py:236-285); ours is one nvcc invocation per translation unit.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "csrc"
LIBDIR = Path(__file__).resolve().parent / "lib"
OBJDIR = ROOT / "build" / "obj"

GENCODE = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-lineinfo", "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=hidden", "-cudart", "shared", "-DTD_BUILD=1",
    # ptxas: keep register info visible in the build log when TD_VERBOSE_BUILD=1
]
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-pthread", "-Wall"]


def _nvcc() -> str:
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(cand).exists():
        raise RuntimeError("nvcc not found (set NVCC=...)")
    return cand


def _digest(paths, extra: str) -> str:
    """Content hash that does not depend on where the repo is checked out (the GPU box uses a scratch path)."""
    h = hashlib.sha256(extra.replace(str(ROOT), "<root>").encode())
    for p in sorted(paths):
        h.update(str(Path(p).resolve().relative_to(ROOT)).encode())
        h.update(Path(p).read_bytes())
    return h.hexdigest()[:16]


class _BuildLock:
    """Inter-process lock: ranks launched together must not compile the same objects concurrently.

    The lock file is opened read-only (flock needs no write access) and created only when missing, so that loading an
    up-to-date build also works from a read-only checkout."""

    def __enter__(self):
        import fcntl
        LIBDIR.mkdir(parents=True, exist_ok=True)
        self.fd = os.open(LIBDIR / ".build.lock", os.O_RDONLY | os.O_CREAT, 0o644)
        fcntl.flock(self.fd, fcntl.LOCK_EX)
        return self

    def __exit__(self, *exc):
        import fcntl
        fcntl.flock(self.fd, fcntl.LOCK_UN)
        os.close(self.fd)


def _headers():
    return sorted(list(CSRC.rglob("*.cuh")) + list(CSRC.rglob("*.h")) + list(CSRC.rglob("*.hpp")))


def _run(cmd, verbose):
    if verbose:
        print(" ".join(map(str, cmd)), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError(f"build failed: {' '.join(map(str, cmd[:6]))} ...")
    if verbose and (r.stdout or r.stderr):
        print(r.stdout + r.stderr, flush=True)


def _compile_objects(sources, compiler_cmd, tag, verbose):
    OBJDIR.mkdir(parents=True, exist_ok=True)
    hdrs = _headers()
    jobs = []
    objs = []
    for src in sources:
        key = _digest([src] + hdrs, " ".join(compiler_cmd))
        obj = OBJDIR / f"{tag}_{src.stem}_{key}.o"
        objs.append(obj)
        if not obj.exists():
            for old in OBJDIR.glob(f"{tag}_{src.stem}_*.o"):
                old.unlink()
            jobs.append(compiler_cmd + ["-c", str(src), "-o", str(obj)])
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(lambda c: _run(c, verbose), jobs))
    return objs, bool(jobs)


def debug_wait_timeout_ns():
    """``TD_DEBUG_WAITS=<milliseconds>`` selects the hang-detection variant of the device code: every spin loop of the primitives
    (td::wait / wait_ge / barrier_all_block / grid_barrier / mbarrier waits / shmem waits) traps with a diagnostic after that long."""
    v = os.environ.get("TD_DEBUG_WAITS", "")
    if not v or v == "0":
        return None
    try:
        ms = float(v)
    except ValueError:
        ms = 5000.0
    return int(max(ms, 1.0) * 1e6)


def build_cuda(verbose: bool = False, force: bool = False) -> Path:
    """Compile every ``csrc/*.cu`` + ``csrc/runtime/*.cu`` into ``libtd_b200.so`` (sm_100a only).  With ``TD_DEBUG_WAITS`` set the
    hang-detection variant ``libtd_b200_dbg<ms>.so`` is built (and loaded by ``_C.cuda_lib``) instead; the default library is untouched."""
    with _BuildLock():
        return _build_cuda_locked(verbose, force)


def _build_cuda_locked(verbose: bool, force: bool) -> Path:
    LIBDIR.mkdir(parents=True, exist_ok=True)
    tmo = debug_wait_timeout_ns()
    out = LIBDIR / ("libtd_b200.so" if tmo is None else f"libtd_b200_dbg{tmo // 1000000}.so")
    cu = sorted(CSRC.glob("*.cu")) + sorted((CSRC / "runtime").glob("*.cu"))
    inc = ["-I", str(CSRC)]
    cmd = [_nvcc()] + GENCODE + NVCC_FLAGS + inc + ([] if tmo is None else [f"-DTD_WAIT_TIMEOUT_NS={tmo}ull"])
    if verbose or os.environ.get("TD_VERBOSE_BUILD") == "1":
        cmd = cmd + ["-Xptxas", "-v"]
    if force:
        shutil.rmtree(OBJDIR, ignore_errors=True)
    objs, rebuilt = _compile_objects(cu, cmd, "cu" if tmo is None else "cudbg", verbose)
    if rebuilt or not out.exists():
        link = [_nvcc(), "-shared", "-cudart", "shared", "-o", str(out)] + [str(o) for o in objs] + [
            "-Xlinker", "-rpath", "-Xlinker", "/usr/local/cuda/lib64", "-ldl", "-lpthread"]
        _run(link, verbose)
    return out


def build_host(verbose: bool = False, force: bool = False) -> Path:
    """Compile ``csrc/host/*.cpp`` into ``libtd_host.so`` (no CUDA dependency; runs on CPU-only boxes)."""
    with _BuildLock():
        return _build_host_locked(verbose, force)


def _build_host_locked(verbose: bool, force: bool) -> Path:
    LIBDIR.mkdir(parents=True, exist_ok=True)
    out = LIBDIR / "libtd_host.so"
    srcs = sorted((CSRC / "host").glob("*.cpp"))
    cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
    cmd = [cxx] + CXX_FLAGS + ["-I", str(CSRC)]
    objs, rebuilt = _compile_objects(srcs, cmd, "host", verbose)
    if rebuilt or not out.exists():
        _run([cxx, "-shared", "-o", str(out)] + [str(o) for o in objs] + ["-lrt", "-pthread"], verbose)
    return out


def build_all(verbose: bool = False, force: bool = False):
    return build_host(verbose, force), build_cuda(verbose, force)


if __name__ == "__main__":
    v = "-v" in sys.argv
    f = "-f" in sys.argv
    h, c = build_all(v, f)
    print(h)
    print(c)
