"""The C-ABI library loads and exports every symbol include/spmm_b200.h declares (no GPU work)."""
import ctypes
import os
import re

from conftest import ROOT


def _declared():
    src = open(os.path.join(ROOT, "include", "spmm_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(spmm_b200_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
    names = _declared()
    assert len(names) >= 18
    lib = ctypes.CDLL(os.path.join(ROOT, "hpc_b200", "libspmm_b200.so"))
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_binding_table_matches_header():
    from hpc_b200._lib import SIGNATURES
    assert sorted(SIGNATURES) == _declared()


def test_status_codes_without_gpu():
    """Argument errors are reported as codes + message, never exit() (reference aborts: util.h:63-84)."""
    import hpc_b200
    from hpc_b200._lib import lib
    h = ctypes.c_void_p()
    rc = lib.spmm_b200_create(None, None, None, 5, 0, 32, ctypes.byref(h))   # num_v > 0 with NULL ptr
    assert rc == -1 and b"bad arguments" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_create(None, None, None, 0, 0, 32, ctypes.byref(h)) == 0
    assert lib.spmm_b200_set_option(h, b"nonsense", 1) == -1
    assert lib.spmm_b200_set_option(h, b"persistent", 1) == -1      # removed options are unknown names
    assert lib.spmm_b200_set_option(h, b"ticket_batch", 1) == -1
    assert lib.spmm_b200_set_option(h, b"kslice", 6) == -1          # not a multiple of 4
    assert lib.spmm_b200_run(h, None, None, None) == -2             # run before preprocess
    assert b"preprocess" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_destroy(h) == 0


def test_feat_zero_and_b_rows_without_gpu():
    """feat_in = 0 is accepted by create: preprocess must build an empty plan (no division by lanes = 0, no CUDA call)
    and run is a no-op; b_rows is part of the plan, so changing it afterwards invalidates it."""
    from hpc_b200._lib import lib
    h = ctypes.c_void_p()
    dummy = (ctypes.c_int * 6)()
    assert lib.spmm_b200_create(dummy, None, None, 5, 0, 0, ctypes.byref(h)) == 0
    assert lib.spmm_b200_preprocess(h, None, None, None) == 0
    assert lib.spmm_b200_run(h, None, None, None) == 0
    assert lib.spmm_b200_refresh_values(h, None) == 0
    assert lib.spmm_b200_set_option(h, b"b_rows", 7) == 0
    assert lib.spmm_b200_run(h, None, None, None) == -2
    assert lib.spmm_b200_destroy(h) == 0


def test_argument_errors_are_status_codes_without_gpu():
    """Entry points added in round 2 keep the ABI's contract — a status code and a message, never a crash or an exit —
    also on a machine without a device."""
    from hpc_b200._lib import lib
    out = ctypes.c_void_p()
    assert lib.spmm_b200_create_column_sorted(None, 32, None, ctypes.byref(out)) == -1
    assert b"create_column_sorted" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_create_transposed(None, 32, None, ctypes.byref(out)) == -1
    h = ctypes.c_void_p()
    dummy = (ctypes.c_int * 6)()
    assert lib.spmm_b200_create(dummy, None, None, 5, 0, 32, ctypes.byref(h)) == 0
    assert lib.spmm_b200_create_column_sorted(h, -1, None, ctypes.byref(out)) == -1
    assert lib.spmm_b200_destroy(h) == 0
    rc = lib.spmm_b200_trim_memory()             # 0 with a device; the CUDA error code (and its text) without one
    assert rc == 0 or lib.spmm_b200_last_error()


def test_mg_create_rejects_bad_csr_without_gpu():
    """spmm_b200_mg_create validates the host CSR before it slices it (status code, no crash, no GPU needed for that)."""
    from hpc_b200._lib import lib
    h = ctypes.c_void_p()
    ptr = (ctypes.c_int * 4)(0, 2, 1, 3)          # decreases at row 1
    idx = (ctypes.c_int * 3)(0, 1, 2)
    val = (ctypes.c_float * 3)(1, 2, 3)
    assert lib.spmm_b200_mg_create(ptr, idx, val, 3, 3, 4, 1, None, ctypes.byref(h)) == -1
    assert b"decreases" in lib.spmm_b200_last_error()
    ptr2 = (ctypes.c_int * 4)(0, 1, 2, 2)         # ptr[num_v] != num_e
    assert lib.spmm_b200_mg_create(ptr2, idx, val, 3, 3, 4, 1, None, ctypes.byref(h)) == -1
    assert b"inconsistent" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_mg_create(ptr2, idx, val, 3, 2, 4, 99, None, ctypes.byref(h)) == -1     # too many devices


def test_host_only_graph_library_matches():
    """libspmm_b200_graph.so (graph.cpp alone, what bench.py's CPU reference arm loads) has no CUDA dependency and
    generates the same graph as the main library."""
    import subprocess
    import numpy as np
    import hpc_b200 as H
    path = os.path.join(ROOT, "hpc_b200", "libspmm_b200_graph.so")
    needed = subprocess.run(["objdump", "-p", path], capture_output=True, text=True).stdout
    assert "libcudart" not in needed and "libcuda" not in needed
    g = ctypes.CDLL(path)
    nv, nnz, mx, tk, zp, lp, win = H.GRAPH_SHAPES["c0"]
    ptr, idx = np.empty(nv + 1, np.int32), np.empty(nnz, np.int32)
    g.spmm_b200_gen_graph.argtypes = [ctypes.c_int, ctypes.c_longlong] + [ctypes.c_int] * 5 + [ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]
    assert g.spmm_b200_gen_graph(nv, nnz, mx, tk, zp, lp, win, 123, ptr.ctypes.data, idx.ctypes.data) == 0
    p2, i2 = H.gen_named_graph("c0")
    assert np.array_equal(ptr, p2) and np.array_equal(idx, i2)


def test_product_does_not_import_oracle():
    """The product package never references oracle/ (no CPU fallback on the product path)."""
    pkg = os.path.join(ROOT, "hpc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cpp", ".h", ".hpp", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "liboracle" not in text and "oracle/_ref" not in text, f


def test_header_is_plain_c(tmp_path):
    """The boundary is a C ABI: the header compiles as C99 with -pedantic, no C++ or CUDA types."""
    import subprocess
    tu = tmp_path / "t.c"
    tu.write_text('#include "spmm_b200.h"\nint main(void) { spmm_b200_t h = 0; spmm_b200_plan_info_t i; (void)h; (void)i; return 0; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(tu)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_cpp_adapter_compiles_standalone_and_against_the_handout(tmp_path):
    """hpc_b200/cpp/spmm_b200.hpp: stand-alone mirror of class SpMM, and (where the reference is present) derived from
    the handout's own spmm_base.h — syntax check only, no GPU."""
    import shutil
    import subprocess
    if not shutil.which("nvcc"):
        import pytest
        pytest.skip("nvcc not on PATH")
    tu = tmp_path / "t.cu"
    tu.write_text('#include "spmm_b200.hpp"\n'
                  'SpMM *make(CSR *g, int k, const float *hb, float *hc) {\n'
                  '    SpMMB200 *a = new SpMMB200(g, k);\n'
                  '    a->set_option("seg_len", 256); a->refresh_values(); a->run_host(hb, hc); SpMMB200::trim_memory();\n'
                  '    SpMMB200 *t = a->transposed(); delete t; t = a->column_sorted(); delete t;\n'
                  '    return a;\n}\n')
    base = ["nvcc", "-std=c++14", "-w", "-c", "-o", str(tmp_path / "t.o"), "-I", os.path.join(ROOT, "include"),
            "-I", os.path.join(ROOT, "hpc_b200", "cpp")]
    r = subprocess.run(base + [str(tu)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    hand = "/root/reference/PA4/handout/include"
    if os.path.isdir(hand):
        r = subprocess.run(base + ["-DSPMM_B200_WITH_HANDOUT", "-I", hand, str(tu)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr


def test_plain_c_example_builds(tmp_path):
    """examples/minimal.c: the boundary used from C99 with only the CUDA runtime API (link check; it runs on the GPU box
    in tests/test_gpu_parity.py)."""
    import subprocess
    cuda = "/usr/local/cuda"
    if not os.path.isdir(os.path.join(cuda, "include")):
        import pytest
        pytest.skip("no CUDA toolkit headers")
    exe = str(tmp_path / "minimal")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                        os.path.join(ROOT, "examples", "minimal.c"), "-L", os.path.join(ROOT, "hpc_b200"), "-lspmm_b200",
                        "-L", os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.join(ROOT, "hpc_b200"), "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
