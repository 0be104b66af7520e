"""Pod removal (kvb_index_remove_pods) checked against the oracle WITHOUT a GPU: csrc/index.cu compiled by g++ with
-DKVB_HOST_SIM (tests/cpp/sim_cuda.h) and driven through the product's Python binding.  The same scenarios run on the
real kernels in tests/test_gpu_index_remove_pods.py."""
import ctypes as C
import importlib
import os
import subprocess

import pytest

from tests import pod_removal as pr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SIM_NAMES = ["kvb_index_create", "kvb_index_destroy", "kvb_index_set_tier_weight", "kvb_index_add", "kvb_index_evict",
             "kvb_index_get_request_key", "kvb_index_num_keys", "kvb_index_flush", "kvb_index_get_stats",
             "kvb_index_lookup", "kvb_index_host_peek", "kvb_index_remove_pods"]


@pytest.fixture(scope="module")
def sim():
    spec = importlib.util.spec_from_file_location("build_index_sim", os.path.join(ROOT, "tests", "cpp", "build_index_sim.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    lib = C.CDLL(mod.build())
    kvb = importlib.import_module("llm-d-kv-cache_b200")
    kvb._lib.bind(lib, SIM_NAMES)
    lib.kvb_last_error = lambda: b"(host simulation)"
    return kvb.kvblock, lib


def test_known_answer(sim):
    pr.known_answer(*sim)


def test_queued_ops_apply_in_call_order(sim):
    pr.queue_ordering(*sim)


def test_recency_is_not_touched(sim):
    pr.recency_untouched(*sim)


@pytest.mark.parametrize("batch", [8, 400])
def test_purge_at_capacity_then_add_batches(sim, batch):
    """batch 8: the one-thread replay; batch 400: planned parallel batches."""
    st = pr.purge_at_capacity_then_adds(*sim, batch=batch)
    if batch > 16:
        assert st["flushes_planned"] > 5
    else:
        assert st["flushes_sequential"] > 5
    assert st["lru_evictions"] > 1000


@pytest.mark.parametrize("size,n_keys,max_batch", [(3, 60, 40), (300, 500, 5), (10 ** 8, 6000, 400)])
def test_random_traffic_with_purges(sim, size, n_keys, max_batch):
    st = pr.random_traffic(*sim, seed=size % 1000 + 1, size=size, ppk=3, n_keys=n_keys, steps=500, max_batch=max_batch)
    if size == 10 ** 8:
        assert st["rehashes"] >= 1 and st["lru_evictions"] == 0
    else:
        assert st["lru_evictions"] > 0


def test_invalid_arguments(sim):
    K, lib = sim
    idx = K.Index(size=10, pod_cache_size=2, expected_keys=16, lib=lib)
    pods = (C.c_uint16 * 1)(0)
    assert lib.kvb_index_remove_pods(None, pods, 1, None, 0, None, None) == -1
    assert lib.kvb_index_remove_pods(idx._h, pods, 0, None, 0, None, None) == -1
    assert lib.kvb_index_remove_pods(idx._h, None, 1, None, 0, None, None) == -1
    assert lib.kvb_index_remove_pods(idx._h, pods, 1, None, -1, None, None) == -1
    assert lib.kvb_index_remove_pods(idx._h, pods, 1, None, 0, None, None) == 0   # NULL outputs are allowed
    idx.close()


def test_cpp_mirror_compiles(tmp_path):
    """tests/cpp/test_remove_pods.cpp (run on the GPU by tests/test_gpu_index_remove_pods.py): compile only."""
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c",
                        os.path.join(ROOT, "tests", "cpp", "test_remove_pods.cpp"), "-o", str(tmp_path / "t.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
