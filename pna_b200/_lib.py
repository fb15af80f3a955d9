"""ctypes binding of ``libpna_sm100.so`` (the C ABI declared in ``include/pna_b200.h``).

The shared library is the product; this module only loads it, mirrors its structs and turns its status
codes into exceptions.  There is deliberately NO fallback: if the library is missing or a call fails the caller
gets an exception, never a silent PyTorch/CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("PNA_B200_LIB") or os.path.join(_HERE, "libpna_sm100.so")   # env override: tuning builds only
CUDA_SOURCES = [os.path.join(_HERE, "csrc", n) for n in
                ("pna_aggregate.cu", "pna_aggregate_f32_vec.cu", "pna_aggregate_f32_scalar.cu", "pna_aggregate_bf16_vec.cu",
                 "pna_aggregate_bf16_scalar.cu", "pna_aggregate_f32_fsplit.cu", "pna_aggregate_bwd.cu", "pna_linear.cu", "pna_csr.cu", "pna_peer.cu", "pna_misc.cu")]
CUDA_HEADERS = [os.path.join(_HERE, "csrc", n) for n in ("common.cuh", "pna_aggregate.cuh", "pna_aggregate_impl.cuh")] + [
    os.path.join(REPO_ROOT, "include", "pna_b200.h")]
BUILD_DIR = os.path.join(_HERE, "csrc", "build")

# sm_100a only: -gencode arch=compute_100a,code=sm_100a (no PTX for other targets, no multi-arch fat binary)
# -fmad=false: the accumulation must round the product m*m before adding it (reference: src * src, then scatter_add);
# ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 otherwise.  IEEE div/sqrt keep their explicit FMAs.
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false", "-Xcompiler", "-fPIC"]

# status codes / enums of include/pna_b200.h
ABI_VERSION = 8
PNA_OK = 0
PNA_F32, PNA_BF16 = 0, 1
AGGR_CODES = {"sum": 0, "mean": 1, "min": 2, "max": 3, "var": 4, "std": 5, "_skip": 15}
SCALER_CODES = {"identity": 0, "amplification": 1, "attenuation": 2, "linear": 3, "inverse_linear": 4}
FLAG_ZERO_ISOLATED, FLAG_SKIP_LIGHT, FLAG_SKIP_HUBS, FLAG_RELU_VAR, FLAG_GATHER_L1 = 1, 2, 4, 8, 16
(QUERY_ABI_VERSION, QUERY_SM_ARCH, QUERY_DEFAULT_SPLIT, QUERY_DEFAULT_CHUNK, QUERY_DEVICE_SM_COUNT,
 QUERY_MAX_FEATURES, QUERY_SIZEOF_CSR, QUERY_SIZEOF_AGG) = range(8)

# every symbol the header declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = ("pna_csr_workspace_bytes", "pna_csr_build", "pna_csr_light_view", "pna_csr_light_view_workspace_bytes", "pna_aggregate_fwd", "pna_aggregate_bwd",
                    "pna_aggregate_bwd_coef", "pna_aggregate_bwd_combine",
                    "pna_gather_rows", "pna_halo_pull", "pna_peer_barrier", "pna_linear_fwd", "pna_linear_scaled_fwd", "pna_row_scales", "pna_linear_workspace_bytes", "pna_query", "pna_last_error")


def cuda_tool(name: str) -> str:
    """Path of a CUDA toolkit program (nvcc, cuobjdump): PATH first, then $CUDA_HOME/bin (default /usr/local/cuda), so that
    the build does not depend on the caller's shell having the toolkit on PATH."""
    return shutil.which(name) or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", name)


class PnaError(RuntimeError):
    """A libpna_sm100 call returned a negative status; the message is pna_last_error()."""

    def __init__(self, status: int, message: str):
        super().__init__(f"libpna_sm100 status {status}: {message}")
        self.status = status


class CsrStruct(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_int64), ("n_edges", C.c_int64),
        ("split_threshold", C.c_int32), ("chunk_edges", C.c_int32),
        ("rowptr", C.c_void_p), ("col", C.c_void_p), ("perm", C.c_void_p),
        ("hub_info", C.c_void_p), ("chunk_items", C.c_void_p),
        ("cap_hubs", C.c_int64), ("cap_chunks", C.c_int64),
        ("n_hubs", C.c_int64), ("n_chunks", C.c_int64),
        ("max_degree", C.c_int32), ("n_part", C.c_int32),
        ("light_rowptr", C.c_void_p), ("light_deg", C.c_void_p), ("light_col", C.c_void_p), ("part", C.c_void_p),
        ("n_light_edges", C.c_int64), ("n_src_nodes", C.c_int64), ("hot_source_fraction", C.c_float), ("reserved", C.c_int32),
    ]


class AggStruct(C.Structure):
    _fields_ = [
        ("gathered", C.c_void_p), ("ld_gathered", C.c_int64),
        ("rowptr", C.c_void_p), ("col", C.c_void_p),
        ("row_bias", C.c_void_p), ("ld_row_bias", C.c_int64),
        ("self_feat", C.c_void_p), ("ld_self", C.c_int64), ("self_tower_stride", C.c_int64),
        ("out", C.c_void_p), ("ld_out", C.c_int64),
        ("n_rows", C.c_int64),
        ("n_feat", C.c_int32), ("n_towers", C.c_int32), ("dtype", C.c_int32),
        ("n_aggr", C.c_int32), ("aggr_codes", C.c_uint32),
        ("n_scalers", C.c_int32), ("scaler_codes", C.c_uint32),
        ("avg_log", C.c_float), ("avg_lin", C.c_float),
        ("flags", C.c_uint32),
        ("split_threshold", C.c_int32), ("chunk_edges", C.c_int32),
        ("hub_info", C.c_void_p), ("chunk_items", C.c_void_p),
        ("n_hubs", C.c_int64), ("n_chunks", C.c_int64),
        ("hub_partials", C.c_void_p),
        ("row_ids", C.c_void_p), ("n_row_ids", C.c_int64),
        ("light_rowptr", C.c_void_p), ("light_deg", C.c_void_p), ("light_col", C.c_void_p), ("part", C.c_void_p),
        ("n_part", C.c_int32), ("n_view_rows", C.c_int64), ("peer_gathered", C.c_void_p), ("peer_shift", C.c_int32),
        ("max_degree", C.c_int32), ("hub_done", C.c_void_p), ("scaler_degree", C.c_void_p), ("work_counter", C.c_void_p),
    ]


def build_library(force: bool = False, verbose: bool = False, extra_flags=()) -> str:
    """Compile libpna_sm100.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    Every .cu is compiled to an object file in parallel (they are independent translation units), then linked with
    ``nvcc -shared``.  Objects are rebuilt when their source or any header is newer.
    """
    from concurrent.futures import ThreadPoolExecutor
    srcs = [s for s in CUDA_SOURCES if os.path.exists(s)]
    hdrs = [h for h in CUDA_HEADERS if os.path.exists(h)]
    hdr_time = max(os.path.getmtime(h) for h in hdrs)
    os.makedirs(BUILD_DIR, exist_ok=True)
    jobs, objs = [], []
    for src in srcs:
        obj = os.path.join(BUILD_DIR, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        stale = force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_time)
        if stale:
            jobs.append([cuda_tool("nvcc")] + NVCC_FLAGS + list(extra_flags) + ["-c", src, "-o", obj])

    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed: {' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        logs = list(ex.map(run, jobs))
    if jobs or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(o) for o in objs):
        run([cuda_tool("nvcc"), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs)
    if verbose and extra_flags:
        print("\n".join(logs))
    return LIB_PATH


_lib = None
_lock = threading.Lock()


def lib() -> C.CDLL:
    """The loaded library.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  pna_b200 has no CPU or PyTorch fallback for its kernels.")
        L = C.CDLL(LIB_PATH)
        L.pna_last_error.restype = C.c_char_p
        L.pna_last_error.argtypes = []
        L.pna_query.restype = C.c_int
        L.pna_query.argtypes = [C.c_int]
        L.pna_csr_workspace_bytes.restype = C.c_int
        L.pna_csr_workspace_bytes.argtypes = [C.c_int64, C.c_int64, C.POINTER(C.c_size_t)]
        L.pna_csr_build.restype = C.c_int
        L.pna_csr_build.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(CsrStruct), C.c_void_p, C.c_size_t, C.c_void_p]
        L.pna_csr_light_view.restype = C.c_int
        L.pna_csr_light_view.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.pna_csr_light_view_workspace_bytes.restype = C.c_int
        L.pna_csr_light_view_workspace_bytes.argtypes = [C.c_int64, C.POINTER(C.c_size_t)]
        L.pna_aggregate_fwd.restype = C.c_int
        L.pna_aggregate_fwd.argtypes = [C.POINTER(AggStruct), C.c_void_p]
        L.pna_aggregate_bwd.restype = C.c_int
        L.pna_aggregate_bwd.argtypes = [C.POINTER(AggStruct), C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                        C.c_int64, C.c_void_p]
        L.pna_aggregate_bwd_coef.restype = C.c_int
        L.pna_aggregate_bwd_coef.argtypes = [C.POINTER(AggStruct), C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                             C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
        L.pna_aggregate_bwd_combine.restype = C.c_int
        L.pna_aggregate_bwd_combine.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64,
                                                C.c_int64, C.c_int32, C.c_void_p]
        L.pna_gather_rows.restype = C.c_int
        L.pna_gather_rows.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                                      C.c_int32, C.c_void_p]
        L.pna_halo_pull.restype = C.c_int
        L.pna_halo_pull.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                                    C.c_int32, C.c_void_p]
        L.pna_peer_barrier.restype = C.c_int
        L.pna_peer_barrier.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]
        L.pna_linear_workspace_bytes.restype = C.c_int
        L.pna_linear_workspace_bytes.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]
        L.pna_linear_fwd.restype = C.c_int
        L.pna_linear_fwd.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32,
                                     C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]
        L.pna_linear_scaled_fwd.restype = C.c_int
        L.pna_linear_scaled_fwd.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                            C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]
        L.pna_row_scales.restype = C.c_int
        L.pna_row_scales.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
        abi = L.pna_query(QUERY_ABI_VERSION)
        if abi != ABI_VERSION:
            raise ImportError(f"{LIB_PATH} has ABI version {abi}, this package needs {ABI_VERSION}: rebuild it")
        if L.pna_query(QUERY_SIZEOF_CSR) != C.sizeof(CsrStruct) or L.pna_query(QUERY_SIZEOF_AGG) != C.sizeof(AggStruct):
            raise ImportError("ctypes struct layout does not match include/pna_b200.h: rebuild libpna_sm100.so")
        _lib = L
    return _lib


def check(status: int) -> None:
    if status != PNA_OK:
        raise PnaError(status, lib().pna_last_error().decode("utf-8", "replace"))


def query(what: int) -> int:
    r = lib().pna_query(what)
    if r < 0:
        raise PnaError(r, lib().pna_last_error().decode("utf-8", "replace"))
    return r


def pack_codes(names, table, what) -> tuple[int, int]:
    """Pack an ordered list of aggregator/scaler names into (count, 4-bit codes) as the header defines."""
    if isinstance(names, str):
        names = names.split()
    names = list(names)
    if not names:
        raise ValueError(f"empty {what} list")
    codes = 0
    for i, n in enumerate(names):
        if n not in table:
            raise KeyError(f"unknown {what} {n!r}; known: {sorted(table)}")
        codes |= table[n] << (4 * i)
    return len(names), codes
