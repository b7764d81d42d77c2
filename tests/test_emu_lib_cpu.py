"""The LIBRARY on the CPU: cozo_b200/csrc/*.cu — host code and kernels — compiled by g++ against a fake CUDA runtime and
the CPU SIMT emulator (tests/emu/build_emu_lib.py -> libcozo_gpu_emu.so; test infrastructure, like oracle/), then driven
through the same ctypes binding and checked against the same oracle as the `-m gpu` tests, at emulator-sized inputs.

Why: gpurun closed mid-round (DESIGN.md §0) with several code paths never run on a GPU.  This runs ALL of them — the C ABI
entry points, their host logic (staging, CUB sorts, launch geometry, chunking, option handling) and the kernels — with
32-wide warps and real concurrency.  It is a logic check: no performance, no hardware memory model.  NCCL and CUDA IPC
are stand-ins whose ranks are threads of one process (tests/emu/fake_nccl.cpp), which is enough to run the sharded
operator — fused peer stores, flag barrier and all — at world sizes 1, 2, 3 and 8.  The product never loads this library (tests/emu/run_emu_lib.py points the binding at it by
hand, in a process of its own).  COZO_EMU_SANITIZE=1 builds with ASan + UBSan.

The `-m gpu` test files themselves run against it too (tests/conftest.py honours COZO_EMU_LIB): the host-layer file and
the quick graph tests in every CPU run, all of test_graph_gpu / test_hnsw_gpu / test_host_gpu / test_unverified_gpu with
COZO_EMU_LONG=1 (about 40 minutes; recorded in profiles/r02_emu_gpu_testfiles.txt)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu")
SANITIZE = os.environ.get("COZO_EMU_SANITIZE") == "1"


@pytest.fixture(scope="module")
def emu_lib(tmp_path_factory):
    sys.path.insert(0, EMU)
    try:
        import build_emu_lib
    finally:
        sys.path.remove(EMU)
    return build_emu_lib.build(str(tmp_path_factory.mktemp("emu_lib")), sanitize=SANITIZE)


def _run(lib, scenario, sm_count=4):
    env = dict(os.environ, UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1", ASAN_OPTIONS="detect_leaks=0",
               COZO_EMU_SM_COUNT=str(sm_count))       # the fake device's SM count: grids of persistent kernels follow it
    if SANITIZE:
        env["LD_PRELOAD"] = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    r = subprocess.run([sys.executable, os.path.join(EMU, "run_emu_lib.py"), lib, scenario], capture_output=True, text=True,
                       timeout=3000, env=env, cwd=ROOT)
    assert r.returncode == 0 and "EMU_OK" in r.stdout, r.stdout[-2500:] + r.stderr[-4000:]
    return r.stdout


def test_library_exports_every_abi_symbol(emu_lib):
    """the emulated build is the whole ABI: same symbols as include/cozo_gpu.h"""
    import ctypes

    from cozo_b200 import capi
    L = ctypes.CDLL(emu_lib)
    assert all(hasattr(L, s) for s in capi.EXPORTS)


@pytest.mark.parametrize("sm_count", [4, 148])
@pytest.mark.parametrize("scenario", ["graph", "pagerank", "hnsw", "hnsw_maintenance", "builder_fidelity"])
def test_library_scenario(emu_lib, scenario, sm_count):
    """graph: CSR staging, SSSP in three frontier forms, closeness, betweenness (+ zero-weight-cycle refusal), clustering,
    constrained paths, poison.  pagerank: both engines, blocking geometries, restaging on option change, edge cases.
    hnsw: build, three search modes (ids / distances / traversal counters == oracle), radius, k > ef, filter mask, re-staging,
    F64 indexes, device-pointer search + top-k merge.  hnsw_maintenance: insert / update / remove / exports, insert into a
    staged and into an empty staged handle.  builder_fidelity: max_batch = 1 and extend_candidates reproduce the oracle's
    sequential builder edge for edge."""
    out = _run(emu_lib, scenario, sm_count)
    print(out)


@pytest.mark.parametrize("scenario", ["fuzz_hnsw", "fuzz_graph", "fuzz_maintenance", "fuzz_sequences", "fuzz_sharded", "fuzz_csr"])
def test_differential_fuzzing(emu_lib, scenario):
    """random configurations against the oracle (COZO_EMU_FUZZ=<n> cases per family, default 40; 150 + 120 + 80 + 60 + 40 were run clean)"""
    print(_run(emu_lib, scenario))


def test_edge_cases_and_misuse(emu_lib):
    """k = 0, ef beyond shared memory, empty batches, out-of-range ids, duplicate updates, corrupt CSR (this found a crash:
    a decreasing row_ptr pair wrapped into an absurd stride in cozo_gpu_hnsw_stage), wrong dtype entry points, empty graphs,
    self loops, communicator misuse: an error code or a result, never a crash"""
    print(_run(emu_lib, "misuse"))


def test_sanitizer_workload(emu_lib):
    """tools/sanitize.py (every kernel on tiny inputs, option sweeps on one staged graph) runs to the end: this is the run
    that exposed the stale blocking state of a re-staged PageRank graph"""
    print(_run(emu_lib, "sanitize_workload"))


def test_sharded_operator_with_rank_threads(emu_lib):
    """cozo_gpu_shards_* / cozo_gpu_hnsw_*_sharded at world sizes 1, 2, 3, 8 (ranks = threads): both exchanges (one all-gather
    per list; peer stores fused into the search epilogue + flag barrier), tiles with double-buffered sets, host and device
    forms, broadcast roots, growth of the exchange buffers, radius == numpy merge of the per-shard lists == the oracle under
    the same sharding"""
    print(_run(emu_lib, "sharded"))


def _pytest_on_emu(lib, args, timeout):
    env = dict(os.environ, COZO_EMU_LIB=lib, COZO_RUN_UNVERIFIED="1", ASAN_OPTIONS="detect_leaks=0")
    if SANITIZE:
        env["LD_PRELOAD"] = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", *args], capture_output=True, text=True,
                       timeout=timeout, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    return r.stdout


def test_gpu_test_files_on_the_emulated_library(emu_lib):
    """the host-layer GPU tests (FixedRule / HnswSearchRA mirrors over the C ABI: PageRank, Dijkstra incl. keep_ties, Yen,
    centralities, clustering, index build / write-back / put / rm, device filter), the quick graph tests and the NaN
    ordering of zero-norm Cosine rows, unchanged, with the binding pointed at libcozo_gpu_emu.so"""
    out = _pytest_on_emu(emu_lib, ["-m", "gpu", "tests/test_host_gpu.py", "tests/test_graph_gpu.py",
                                   "tests/test_search_widths_gpu.py::test_nan_cosine_exhaustive",
                                   "tests/test_search_widths_gpu.py::test_nan_non_exhaustive_built_index",
                                   "-k", "not air_routes and not 17-5"], 2400)
    assert " passed" in out and "failed" not in out


@pytest.mark.skipif(os.environ.get("COZO_EMU_LONG") != "1", reason="about 40 minutes; COZO_EMU_LONG=1")
def test_all_gpu_test_files_on_the_emulated_library(emu_lib):
    """every -m gpu / gpu_unverified test that does not need torch CUDA tensors, several GPUs or a million vectors"""
    _pytest_on_emu(emu_lib, ["-m", "gpu or gpu_unverified", "-p", "no:timeout", "tests/test_graph_gpu.py", "tests/test_hnsw_gpu.py",
                             "tests/test_host_gpu.py", "tests/test_unverified_gpu.py", "tests/test_search_widths_gpu.py",
                             "-k", "not search_dev_and_merge"], 4 * 3600)
