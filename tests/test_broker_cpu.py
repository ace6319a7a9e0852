"""The broker (pgvector_b200/ext/vb_broker.c, INTEGRATION.md section 6): many requesters, one scan each, answered from
batched vb_ivf_search calls.  Run here against the oracle-backed mock ABI (tests/harness/mock_abi.c): every scan gets
exactly what a direct single-query call returns, the scans of concurrent requesters share calls, a full queue blocks
instead of dropping, and a lone requester is not held longer than the window."""
import ctypes as C
import time

import numpy as np
import pytest

import oracle as O
from tests.harness import build as hbuild
from tests.util import build_ivf_arrays, mixture


@pytest.fixture(scope="module")
def lib():
    L = C.CDLL(hbuild.build_broker())
    L.vb_ivf_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    L.vb_ivf_load.argtypes = [C.c_void_p] * 5
    L.vb_ivf_free.argtypes = [C.c_void_p]
    L.vb_ivf_search.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.hb_broker_run.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p]
    L.hb_broker_run_fork.argtypes = L.hb_broker_run.argtypes
    L.mock_ivf_search_calls.restype = C.c_int
    return L


@pytest.fixture(scope="module")
def index(lib):
    rows, centers = mixture(4000, 32, 16, seed=71)
    queries, _ = mixture(600, 32, 16, seed=72)
    assign = O.ivf_assign(O.VECTOR, O.L2_SQUARED, rows, centers, threads=4)
    grouped, ids, offsets = build_ivf_arrays(rows, assign, 16)
    h = C.c_void_p()
    assert lib.vb_ivf_create(O.VECTOR, O.L2, 32, 16, C.byref(h)) == 0
    keep = [np.ascontiguousarray(centers), np.ascontiguousarray(offsets, dtype=np.int64), np.ascontiguousarray(grouped),
            np.ascontiguousarray(ids, dtype=np.int64)]
    assert lib.vb_ivf_load(h, *[a.ctypes.data_as(C.c_void_p) for a in keep]) == 0
    yield h, np.ascontiguousarray(queries)
    lib.vb_ivf_free(h)


def direct(lib, h, queries, probes, k):
    ids = np.empty((len(queries), k), dtype=np.int64)
    dist = np.empty((len(queries), k), dtype=np.float64)
    for i in range(len(queries)):      # one call per scan: what the glue does without a broker
        assert lib.vb_ivf_search(h, queries[i].ctypes.data_as(C.c_void_p), 1, probes, k, ids[i].ctypes.data_as(C.c_void_p),
                                 dist[i].ctypes.data_as(C.c_void_p)) == 0
    return ids, dist


def through_broker(lib, h, queries, threads, probes, k, max_batch, window_us, processes=False):
    ids = np.full((len(queries), k), -7, dtype=np.int64)
    dist = np.full((len(queries), k), np.nan)
    stats = np.zeros(4, dtype=np.int64)
    run = lib.hb_broker_run_fork if processes else lib.hb_broker_run
    rc = run(h, queries.ctypes.data_as(C.c_void_p), len(queries), queries.shape[1] * 4, threads, probes, k, max_batch,
                           window_us, ids.ctypes.data_as(C.c_void_p), dist.ctypes.data_as(C.c_void_p), stats.ctypes.data_as(C.c_void_p))
    assert rc == 0
    return ids, dist, dict(requests=int(stats[0]), batches=int(stats[1]), largest=int(stats[2]), failed=int(stats[3]))


@pytest.mark.parametrize("threads,max_batch,window_us", [(1, 64, 0), (8, 64, 200), (32, 16, 2000), (64, 4, 0), (16, 1, 0)])
def test_every_scan_gets_the_result_of_a_direct_call(lib, index, threads, max_batch, window_us):
    h, queries = index
    want_i, want_d = direct(lib, h, queries, 3, 10)
    ids, dist, st = through_broker(lib, h, queries, threads, 3, 10, max_batch, window_us)
    assert np.array_equal(ids, want_i) and np.array_equal(dist, want_d)
    assert st["requests"] == len(queries) and st["failed"] == 0
    assert 1 <= st["largest"] <= min(max_batch, threads)
    assert st["batches"] >= (len(queries) + min(max_batch, threads) - 1) // min(max_batch, threads)


def test_concurrent_scans_share_calls(lib, index):
    """32 requesters with a 5 ms window: the 600 scans arrive in far fewer than 600 library calls"""
    h, queries = index
    before = lib.mock_ivf_search_calls()
    _, _, st = through_broker(lib, h, queries, 32, 3, 10, 64, 5000)
    calls = lib.mock_ivf_search_calls() - before
    assert calls == st["batches"]
    assert st["batches"] <= len(queries) // 8, st
    assert st["largest"] >= 16, st


def test_a_lone_requester_is_not_held_much_longer_than_the_window(lib, index):
    h, queries = index
    t0 = time.perf_counter()
    _, _, st = through_broker(lib, h, queries[:20], 1, 3, 10, 64, 1000)
    dt = time.perf_counter() - t0
    assert st["batches"] == 20 and st["largest"] == 1
    assert dt < 20 * 0.03, dt          # 1 ms of window per scan + the scan itself (CPU mock), generous for a loaded machine


def test_k_larger_than_the_candidates_pads_like_the_library(lib, index):
    h, queries = index
    want_i, want_d = direct(lib, h, queries[:40], 1, 600)
    ids, dist, st = through_broker(lib, h, queries[:40], 8, 1, 600, 8, 100)
    assert np.array_equal(ids, want_i) and np.array_equal(dist, want_d)
    assert (ids == -1).any() and np.isinf(dist[ids == -1]).all()


@pytest.mark.timeout(120)
@pytest.mark.parametrize("procs,max_batch,window_us", [(1, 8, 0), (6, 64, 500), (12, 4, 0)])
def test_requesters_in_other_processes(lib, index, procs, max_batch, window_us):
    """backends are processes: the request block sits in shared memory, the requesters are forked children that never
    touch the library; only the broker (this process) does"""
    h, queries = index
    q = queries[:240]
    want_i, want_d = direct(lib, h, q, 3, 10)
    before = lib.mock_ivf_search_calls()
    ids, dist, st = through_broker(lib, h, q, procs, 3, 10, max_batch, window_us, processes=True)
    assert np.array_equal(ids, want_i) and np.array_equal(dist, want_d)
    assert st["requests"] == len(q) and st["failed"] == 0
    assert lib.mock_ivf_search_calls() - before == st["batches"]       # every library call was made by the broker, here
    assert 1 <= st["largest"] <= min(max_batch, procs)
    if procs >= 6 and window_us > 0:
        assert st["batches"] < len(q)
