"""bench.py host-side pieces that need no GPU: the reference arm's JSON line and the byte/flop accounting."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def test_reference_arm_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c0_k32",
                        "--steps", "1", "--warmup", "3"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "spmm_gflops" and line["unit"] == "GFLOP/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["dtype"] == "f32"
    assert line["config"]["workload"] == "c0_k32" and line["config"]["nnz"] == 65536
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "c0_k32",
                        "--steps", "1", "--warmup", "3"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_argument_errors():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c0_k32", *extra], capture_output=True,
                           text=True, timeout=120, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-2000:])


def test_byte_accounting():
    sys.path.insert(0, ROOT)
    import bench
    m, nnz, k = 232965, 114615892, 256
    assert bench.bytes_min(m, nnz, k) == 4 * (m + 1) + 8 * nnz + 8 * m * k          # SURVEY.md 8d
    assert bench.bytes_gather(m, nnz, k) == 4 * (m + 1) + 8 * nnz + 4 * nnz * k + 4 * m * k
    assert bench.bytes_min(100, 10, 4, b_rows=1000) == 4 * 101 + 80 + 4 * 1000 * 4 + 4 * 100 * 4


def test_reference_arm_loads_no_product_kernel():
    """The CPU arm generates its graph from the host-only library: libspmm_b200.so (the product kernels) is never mapped."""
    code = ("import bench, numpy as np; p, i = bench.host_gen_named_graph('c0', 2); "
            "maps = open('/proc/self/maps').read(); "
            "assert 'libspmm_b200_graph.so' in maps and 'libspmm_b200.so' not in maps and 'hpc_b200/__init__' not in str(list(__import__('sys').modules)); "
            "c = bench.workload_config('c0_k32', p); print(sorted(c))")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "hpc_b200" not in [m for m in r.stdout.split()]
