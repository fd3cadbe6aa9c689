"""In-tree build of the native core (C++ runtime + sm_100a kernels).

The reference builds one C++ TU through ``mpicc``/``mpicxx`` with ``-g`` only
(reference ``setup.py:22-58``, ``:90-106``).  Here the extension is a mix of
plain C++ (control plane, CPU backend, symmetric heap), torch-facing C++
(autograd layer, bindings) and CUDA compiled **only** for sm_100a.  The built
``.so`` lives in ``mpi4torch_b200/_lib`` so it travels with the source tree; a
content hash of sources + flags decides whether it is stale.
"""
from __future__ import annotations

import hashlib
import importlib.util
import os
import sys
from pathlib import Path

_PKG = Path(__file__).resolve().parent
_CSRC = _PKG / "csrc"
# M4T_LIB_DIR / M4T_EXTRA_CXXFLAGS / M4T_EXTRA_LDFLAGS: out-of-tree instrumented builds
# (scripts/asan_cpu.sh); the default is the in-tree release build.
_LIB = Path(os.environ["M4T_LIB_DIR"]) if os.environ.get("M4T_LIB_DIR") else _PKG / "_lib"
_NAME = "_m4t_C"

_SOURCES = [
    "runtime/control.cpp",
    "runtime/plan.cpp",
    "runtime/cpu_backend.cpp",
    "runtime/net_link.cpp",
    "runtime/net_backend.cpp",
    "runtime/symm_heap.cpp",
    "runtime/cuda_backend.cpp",
    "runtime/world.cpp",
    "kernels/allreduce.cu",
    "kernels/scan.cu",
    "kernels/slab.cu",
    "kernels/slab_push.cu",
    "kernels/rooted.cu",
    "kernels/p2p.cu",
    "kernels/gemm_tcgen05.cu",
    "kernels/gemm_tcgen05_2cta.cu",
    "kernels/wgrad_tcgen05_2cta.cu",
    "api/comm_raw.cpp",
    "api/autograd_ops.cpp",
    "api/fused_ops.cpp",
    "api/bindings.cpp",
]

CXX_FLAGS = ["-O3", "-std=c++17", "-fPIC", "-fopenmp", "-Wall", "-Wno-unused-function", "-Wno-sign-compare"]
CXX_FLAGS += os.environ.get("M4T_EXTRA_CXXFLAGS", "").split()
NVCC_FLAGS = [
    "-O3",
    "-std=c++17",
    "-gencode",
    "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "--expt-relaxed-constexpr",
    "-diag-suppress",
    "177",
]
LD_FLAGS = ["-lrt", "-lpthread", "-fopenmp"] + os.environ.get("M4T_EXTRA_LDFLAGS", "").split()


def _existing_sources() -> list[str]:
    return [str(_CSRC / s) for s in _SOURCES if (_CSRC / s).exists()]


def _stamp() -> str:
    h = hashlib.sha256()
    files = sorted(p for p in _CSRC.rglob("*") if p.suffix in {".cpp", ".cu", ".cuh", ".h"})
    for p in files:
        h.update(str(p.relative_to(_CSRC)).encode())
        h.update(p.read_bytes())
    h.update(" ".join(CXX_FLAGS + NVCC_FLAGS + LD_FLAGS).encode())
    try:
        import torch

        h.update(torch.__version__.encode())
    except Exception:  # pragma: no cover
        pass
    return h.hexdigest()


def so_path() -> Path:
    return _LIB / f"{_NAME}.so"


def is_fresh() -> bool:
    stamp = _LIB / ".stamp"
    return so_path().exists() and stamp.exists() and stamp.read_text().strip() == _stamp()


def _import_built():
    spec = importlib.util.spec_from_file_location(_NAME, so_path())
    if spec is None or spec.loader is None:  # pragma: no cover
        raise ImportError(f"cannot load {so_path()}")
    mod = importlib.util.module_from_spec(spec)
    sys.modules[_NAME] = mod
    spec.loader.exec_module(mod)
    return mod


def build(verbose: bool = False, force: bool = False):
    """Compile (if stale) and import the native module."""
    import torch  # noqa: F401  (must be imported before the extension)

    if _NAME in sys.modules:
        return sys.modules[_NAME]
    if not force and is_fresh():
        return _import_built()
    from torch.utils import cpp_extension

    _LIB.mkdir(exist_ok=True)
    os.environ.setdefault("MAX_JOBS", str(os.cpu_count() or 8))
    # The image presets CXX=/opt/gcc/bin/g++, a wrapper whose libstdc++.so symlink
    # dangles: it links libstdc++ statically, and a second iostream/locale copy
    # inside the extension crashes on the first ostringstream.  Use the distro g++.
    if os.path.exists("/usr/bin/g++") and os.environ.get("M4T_KEEP_CXX", "0") != "1":
        os.environ["CXX"] = "/usr/bin/g++"
        os.environ["CC"] = "/usr/bin/gcc"
    # stamp the inputs as they are now, and hand torch copies of the flag lists: cpp_extension appends its own
    # link flags to extra_ldflags in place, and a stamp taken from the extended list never matches the one a
    # fresh process computes (every import would rebuild, and fail in a read-only tree)
    stamp = _stamp()
    cpp_extension.load(
        name=_NAME,
        sources=_existing_sources(),
        extra_cflags=list(CXX_FLAGS),
        extra_cuda_cflags=list(NVCC_FLAGS),
        extra_ldflags=list(LD_FLAGS),
        extra_include_paths=[str(_CSRC)],
        build_directory=str(_LIB),
        with_cuda=True,
        is_python_module=True,
        verbose=verbose,
    )
    (_LIB / ".stamp").write_text(stamp)
    return sys.modules.get(_NAME) or _import_built()


def load():
    """Import the native module, building it first when missing or stale."""
    if os.environ.get("M4T_NO_BUILD", "0") == "1" and so_path().exists():
        return _import_built()
    return build(verbose=os.environ.get("M4T_BUILD_VERBOSE", "0") == "1")


if __name__ == "__main__":
    build(verbose=True, force="--force" in sys.argv)
    print("built", so_path())
