"""CPU-side checks of the C-ABI boundary: the library builds, loads and exports every symbol the header declares.
No compute call is made here (no GPU in the authoring container)."""
import ctypes as C
import os
import re

import pytest
import torch

import pna_b200
from pna_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pna_b200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"^\s*(?:int|const char\*)\s+(pna_\w+)\s*\(", src, flags=re.M)))


def test_library_is_built_and_loads():
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build()"
    L = _lib.lib()
    assert L.pna_query(_lib.QUERY_ABI_VERSION) == _lib.ABI_VERSION == 8
    assert L.pna_query(_lib.QUERY_SM_ARCH) == 100


def test_every_declared_symbol_is_exported():
    names = declared_functions()
    assert set(names) == set(_lib.EXPORTED_SYMBOLS)
    L = C.CDLL(_lib.LIB_PATH)
    for n in names:
        assert getattr(L, n) is not None


def test_struct_layouts_match_the_header():
    assert _lib.query(_lib.QUERY_SIZEOF_CSR) == C.sizeof(_lib.CsrStruct)
    assert _lib.query(_lib.QUERY_SIZEOF_AGG) == C.sizeof(_lib.AggStruct)


def test_library_targets_sm_100a_only():
    import subprocess
    out = subprocess.run([_lib.cuda_tool("cuobjdump"), "--list-elf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_queries_and_defaults_without_gpu():
    assert _lib.query(_lib.QUERY_DEFAULT_SPLIT) >= 2
    assert 1 <= _lib.query(_lib.QUERY_DEFAULT_CHUNK) <= _lib.query(_lib.QUERY_DEFAULT_SPLIT)
    assert _lib.query(_lib.QUERY_MAX_FEATURES) >= 1024
    with pytest.raises(pna_b200.PnaError) as ex:
        _lib.query(12345)
    assert ex.value.status == -1 and "selector" in str(ex.value)


def test_bad_arguments_return_status_codes_not_aborts():
    L = _lib.lib()
    assert L.pna_aggregate_fwd(None, None) == -1
    assert b"null descriptor" in L.pna_last_error()
    d = _lib.AggStruct(n_rows=4, n_feat=8, n_towers=3, n_aggr=4, n_scalers=3)
    assert L.pna_aggregate_fwd(C.byref(d), None) == -1            # 8 not divisible by 3 towers
    d = _lib.AggStruct(n_rows=4, n_feat=8, n_towers=1, n_aggr=9, n_scalers=3)
    assert L.pna_aggregate_fwd(C.byref(d), None) == -1
    d = _lib.AggStruct(n_rows=4, n_feat=8, n_towers=1, n_aggr=1, aggr_codes=7, n_scalers=1)
    assert L.pna_aggregate_fwd(C.byref(d), None) == -1            # aggregator code 7 does not exist
    d = _lib.AggStruct(n_rows=4, n_feat=8, n_towers=1, n_aggr=1, n_scalers=1, dtype=5)
    assert L.pna_aggregate_fwd(C.byref(d), None) == -2
    d = _lib.AggStruct(n_rows=0, n_feat=8, n_towers=1, n_aggr=1, n_scalers=1)
    assert L.pna_aggregate_fwd(C.byref(d), None) == 0             # empty problem: nothing to launch
    nb = C.c_size_t(0)
    assert L.pna_csr_workspace_bytes(-1, 0, C.byref(nb)) == -1
    assert L.pna_csr_workspace_bytes(1 << 40, 0, C.byref(nb)) == -2
    assert L.pna_gather_rows(None, 0, None, 0, None, 0, 8, 0, None) == 0
    assert L.pna_gather_rows(None, 0, None, 5, None, 0, 8, 0, None) == -1


def test_product_refuses_cpu_tensors():
    with pytest.raises(ValueError):
        pna_b200.build_csr(torch.zeros(2, dtype=torch.long), torch.zeros(2, dtype=torch.long), 2)


def test_header_is_plain_c():
    """The boundary is a C ABI: the header must compile as C99 (what a cgo / JNI / ctypes-generator binding consumes)."""
    import subprocess
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-fsyntax-only", "-x", "c", HEADER],
                       capture_output=True, text=True)
    assert r.returncode == 0 and not r.stderr.strip(), r.stderr


def test_post_linear_entry_points_validate_without_gpu():
    L = _lib.lib()
    fwd, scaled, scales = L.pna_linear_fwd, L.pna_linear_scaled_fwd, L.pna_row_scales
    assert fwd(None, 0, None, None, None, 0, 0, 64, 128, None, 0, None) == 0               # no rows: nothing to do
    assert fwd(None, 0, None, None, None, 0, 5, 60, 128, None, 0, None) == -2              # n_in % 32
    assert fwd(None, 0, None, None, None, 0, 5, 64, 100, None, 0, None) == -2              # n_out not 64/128/256
    assert fwd(None, 0, None, None, None, 0, 5, 64, 128, None, 0, None) == -1              # null pointers
    assert b"pna_linear_fwd" in L.pna_last_error()
    assert scaled(None, 0, None, 3, None, None, None, 0, 0, 96, 64, None, 0, None) == 0
    assert scaled(None, 0, None, 3, None, None, None, 0, 5, 96, 64, None, 0, None) == -1   # row_scale missing
    assert scaled(None, 0, None, 3, None, None, None, 0, 0, 100, 64, None, 0, None) == -2  # 100 / 3 is not a K width
    assert scaled(None, 0, None, 9, None, None, None, 0, 0, 288, 64, None, 0, None) == -1  # more scalers than exist
    assert b"pna_linear_scaled_fwd" in L.pna_last_error()
    assert scales(None, 0, 3, 0x210, 1.0, 1.0, None, None) == 0
    assert scales(None, 7, 3, 0x210, 1.0, 1.0, None, None) == -1                           # null pointers
    assert scales(None, 0, 2, 0x90, 1.0, 1.0, None, None) == -1                            # scaler code 9 does not exist
    assert scales(None, 0, 0, 0, 1.0, 1.0, None, None) == -1


def test_csr_build_rejects_inconsistent_capacities_before_touching_the_gpu():
    L = _lib.lib()
    dummy = 256                                                   # never dereferenced: validation fails first
    c = _lib.CsrStruct(n_nodes=10, n_edges=100, split_threshold=256, chunk_edges=128, rowptr=dummy, col=dummy, perm=dummy,
                       hub_info=dummy, chunk_items=dummy, cap_hubs=1, cap_chunks=2, light_rowptr=dummy)
    # consistent capacities pass the checks (the call then stops at the missing workspace / missing device)
    assert L.pna_csr_build(dummy, dummy, C.byref(c), None, 0, None) < 0 and b"cap_" not in L.pna_last_error()
    c.cap_chunks = 10_000                                          # > 2 * n_edges + 3: the view scan would overrun the workspace
    assert L.pna_csr_build(dummy, dummy, C.byref(c), None, 0, None) == -1
    assert b"cap_chunks" in L.pna_last_error()
    c.chunk_edges = 512                                            # chunk larger than the split threshold
    assert L.pna_csr_build(dummy, dummy, C.byref(c), None, 0, None) == -1


def test_plain_c_caller_compiles_and_links():
    """examples/c_caller.c drives the ABI from C99 with nothing but the header and the CUDA runtime."""
    import subprocess, tempfile
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    if not os.path.exists(os.path.join(cuda, "include", "cuda_runtime_api.h")):
        pytest.skip("CUDA toolkit headers not found")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "c_caller")
        r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                            os.path.join(ROOT, "examples", "c_caller.c"), "-o", exe, "-L", os.path.dirname(_lib.LIB_PATH),
                            "-l:" + os.path.basename(_lib.LIB_PATH), "-L", os.path.join(cuda, "lib64"), "-lcudart", "-lm",
                            "-Wl,-rpath," + os.path.dirname(_lib.LIB_PATH)], capture_output=True, text=True)
        assert r.returncode == 0 and not r.stderr.strip(), r.stderr
        assert os.path.exists(exe)
