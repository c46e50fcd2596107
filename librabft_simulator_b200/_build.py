"""Build recipes for the native pieces (run by ``__graft_entry__.build()``).

* ``csrc/liblbft_b200.so`` — the product: sm_100a CUDA kernels + the C ABI of ``include/lbft.h``.
* ``oracle/liblbft_oracle.so`` and ``tests/hostcore/libhostcore.so`` — test infrastructure only.
These three are built in-tree (git-ignored) by ``build()``; nothing that runs later compiles into the tree.
"""
import os
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "librabft_simulator_b200", "csrc")
LIB_PATH = os.environ.get("LBFT_LIB_PATH") or os.path.join(CSRC, "liblbft_b200.so")
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_PATH = os.path.join(ORACLE_DIR, "liblbft_oracle.so")
HOSTCORE_DIR = os.path.join(ROOT, "tests", "hostcore")
HOSTCORE_PATH = os.path.join(HOSTCORE_DIR, "libhostcore.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
# Translation units of the product library: the host runtime (C ABI) and the kernel instantiations, one group per file so
# that they compile in parallel and the bench kernel (k_fixed.cu) can be rebuilt alone.
PRODUCT_UNITS = ["lbft_api.cu", "k_fixed.cu", "k_scan.cu", "k_calendar.cu", "k_heap.cu", "k_wide.cu"]
PRODUCT_HEADERS = ["kernels.cuh", "sim_core.cuh", "sim_params.h", "host_setup.hpp"]


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _run(cmd, cwd):
    proc = subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        raise RuntimeError("build failed: %s\n%s" % (" ".join(cmd), proc.stdout))
    return proc.stdout


def nvcc_path():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def build_product(force=False, verbose_ptxas=False, extra_flags=(), lib_path=None):
    """nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo on every unit (objects in csrc/build/, in parallel), then one
    shared library.  Only units older than their sources are recompiled."""
    from concurrent.futures import ThreadPoolExecutor
    lib_path = lib_path or LIB_PATH
    headers = [os.path.join(CSRC, f) for f in PRODUCT_HEADERS] + [os.path.join(ROOT, "include", "lbft.h")]
    sources = headers + [os.path.join(CSRC, u) for u in PRODUCT_UNITS]
    if not (force or verbose_ptxas or extra_flags) and _newer(lib_path, sources):
        return lib_path  # (the objects need not exist: on the GPU box only the library travels)
    objdir = os.path.join(CSRC, "build" if lib_path == LIB_PATH else "build_" + os.path.basename(lib_path))
    os.makedirs(objdir, exist_ok=True)
    jobs = []
    for unit in PRODUCT_UNITS:
        obj = os.path.join(objdir, unit.replace(".cu", ".o"))
        if force or verbose_ptxas or extra_flags or not _newer(obj, headers + [os.path.join(CSRC, unit)]):
            jobs.append((unit, obj))
    flags = NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose_ptxas else [])
    with ThreadPoolExecutor(max_workers=min(len(PRODUCT_UNITS), os.cpu_count() or 2)) as pool:
        outs = list(pool.map(lambda j: _run([nvcc_path()] + flags + ["-c", "-o", j[1], j[0]], CSRC), jobs))
    if verbose_ptxas:
        print("\n".join(outs))
    objs = [os.path.join(objdir, u.replace(".cu", ".o")) for u in PRODUCT_UNITS]
    if jobs or not _newer(lib_path, objs):
        _run([nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", lib_path] + objs, CSRC)
    return lib_path


def build_oracle(force=False):
    srcs = [os.path.join(ORACLE_DIR, f) for f in ("oracle_capi.cpp", "oracle_selftest.cpp", "lbft_oracle.hpp")]
    srcs.append(os.path.join(ROOT, "include", "lbft.h"))
    if not force and _newer(ORACLE_PATH, srcs):
        return ORACLE_PATH
    _run(["make", "-B", "liblbft_oracle.so"], ORACLE_DIR)
    return ORACLE_PATH


_NATIVE_ORACLE = {}


def build_oracle_native():
    """The CPU-baseline build of the oracle (-O3 -march=native), compiled on the machine that times it, once per process.
    It goes to a fresh private directory from tempfile.mkdtemp (this user's, mode 0700, unpredictable name) that is
    removed when the process exits: never into the source tree, which bench.py may find read-only, and never a library
    another user could have placed in a shared location.  Falls back to the portable build if no compiler is available.
    Returns (path, flags description)."""
    if "lib" not in _NATIVE_ORACLE:
        import atexit
        import tempfile
        outdir = tempfile.mkdtemp(prefix="lbft_oracle_native_")
        atexit.register(shutil.rmtree, outdir, True)
        path = os.path.join(outdir, "liblbft_oracle_native.so")
        try:
            _run(["make", "native", "NATIVE_OUT=" + path], ORACLE_DIR)
            _NATIVE_ORACLE["lib"] = path, "-O3 -march=native"
        except Exception:
            _NATIVE_ORACLE["lib"] = build_oracle(), "-O2 (portable build: native build failed)"
    return _NATIVE_ORACLE["lib"]


def build_hostcore(force=False):
    if os.environ.get("LBFT_HOSTCORE_PATH"):  # an alternatively built copy (A/B of compile-time switches)
        return os.environ["LBFT_HOSTCORE_PATH"]
    srcs = [os.path.join(HOSTCORE_DIR, "hostcore.cpp")] + [
        os.path.join(CSRC, f) for f in ("sim_core.cuh", "sim_params.h", "host_setup.hpp")]
    if not force and _newer(HOSTCORE_PATH, srcs):
        return HOSTCORE_PATH
    _run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-DLBFT_CHECK_C1",
          "-o", HOSTCORE_PATH, "hostcore.cpp"], HOSTCORE_DIR)
    return HOSTCORE_PATH


def build_all(force=False):
    return build_product(force), build_oracle(force), build_hostcore(force)
