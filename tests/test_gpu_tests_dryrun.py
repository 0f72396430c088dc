"""Dry run of the gpu-marked tests on a machine without a GPU: the C-ABI is answered by tests/cpp/tsgpu_oracle_double.cpp
(the oracle behind the tsgpu_* entry points, built here as a shared library and selected with TSGPU_LIB_PATH), so the
Python side of every GPU test — batch construction, calls, the reference expectations — executes before the code ever
reaches the GPU box. It proves nothing about the kernels (oracle is compared with oracle); tests that assert device
counters, device error codes or need CUDA tensors are left out."""
import os
import subprocess
import sys

import oracle_lib as ol

ROOT = ol.ROOT
GPU_ONLY = [
    "tests/test_cpp_host.py::test_cpp_host_scenarios",                            # links the real libtsgpu.so
    "tests/test_gpu_parity.py::test_large_scale_properties_and_sample_parity",    # generates its data on the device
    "tests/test_gpu_parity.py::test_keyword_single_token_large_lists",            # asserts device work counters
    "tests/test_gpu_parity.py::test_ids_setop",                                   # asserts the library's argument validation
    "tests/test_gpu_parity.py::test_edge_cases",                                  # asserts the library's capacity errors
    "tests/test_facets.py::test_gpu_all_result_ids_and_facets_of_a_search_batch",  # all_result_ids live in device memory
    "tests/test_gpu_parity.py::test_knn_selective_filters_long_walks",            # builds its graph on the device, asserts device counters
    "tests/test_gpu_parity.py::test_hnsw_load_rejects_malformed_graph_and_keeps_the_old_one",   # asserts the library's load-time validation
    "tests/test_incremental_mirror.py::test_append_lists_rejects_malformed_input",              # asserts the library's argument validation
    "tests/test_bench_contract.py::test_product_arm_dumps_the_same_outputs_every_run",          # runs bench.py's CUDA arm in a subprocess
]


def test_gpu_tests_execute_against_the_oracle_double():
    ol.build_oracle()
    so = os.path.join(ROOT, "tests", "cpp", "libtsgpu_double.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wno-unused", "-fPIC", "-shared", os.path.join(ROOT, "tests", "cpp", "tsgpu_oracle_double.cpp"),
                           "-o", so, "-L", os.path.join(ROOT, "oracle"), "-l:liboracle.so", f"-Wl,-rpath,{os.path.join(ROOT, 'oracle')}", "-pthread"])
    env = dict(os.environ, TSGPU_TEST_DOUBLE="1", TSGPU_LIB_PATH=so)
    cmd = [sys.executable, "-m", "pytest", os.path.join(ROOT, "tests"), "-q", "-m", "gpu", "-p", "no:cacheprovider",
           "--runxfail", "--ignore", os.path.join(ROOT, "tests", "test_hnsw_build_gpu.py")]      # the device build has no double
    for t in GPU_ONLY:
        cmd += ["--deselect", t]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, env=env, timeout=1500)
    tail = r.stdout[-3000:] + r.stderr[-1000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout, tail


def test_smoke_executes_against_the_oracle_double():
    """__graft_entry__.smoke() — the driver's first GPU step — with the same double behind the C-ABI."""
    so = os.path.join(ROOT, "tests", "cpp", "libtsgpu_double.so")
    if not os.path.exists(so):
        test_gpu_tests_execute_against_the_oracle_double()
    env = dict(os.environ, TSGPU_LIB_PATH=so)
    r = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], capture_output=True, text=True, cwd=ROOT, env=env, timeout=900)
    assert r.returncode == 0 and "smoke ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
