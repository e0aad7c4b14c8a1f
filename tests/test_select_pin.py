"""Pins the product's select post-processing (reindexer_b200/host/knn_select.h: selectPostprocess, reached through
rxgpu_select_postprocess) and the oracle port (oracle/knn_port.c: port_select_postprocess) to the REFERENCE'S OWN code of
HnswIndexBase<Map>::select + removeOverK + removeDuplicateRowId: oracle/Makefile extracts that text from
cpp_src/core/index/float_vector/hnsw_index.cc / float_vector_index.h where it lies and compiles it behind duck-typed stand-ins
(oracle/ref_select_facade.cc -> oracle/_ref/liboracle_ref_select.so), whose answers are stored in tests/golden/ref_tapes/.
Host logic only: no GPU."""
import ctypes as C
import os

import numpy as np

from helpers import digest

from reindexer_b200 import binding as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "liboracle_ref_select.so")


def ref_select(metric, is_bf, need_sort, is_array, k, radius, index_radius, dist, label):
    lib = C.CDLL(LIB)
    fn = lib.ref_select_postprocess
    fn.restype = C.c_int64
    fn.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_float, C.c_int, C.c_float, C.c_uint64,
                   C.POINTER(C.c_float), C.POINTER(C.c_uint64), C.POINTER(C.c_int32), C.POINTER(C.c_float)]
    d = np.ascontiguousarray(dist, np.float32)
    l = np.ascontiguousarray(label, np.uint64)
    ids = np.zeros(max(len(d), 1), np.int32)
    ranks = np.zeros(max(len(d), 1), np.float32)
    n = fn(metric, int(is_bf), int(need_sort), int(is_array), int(k is not None), k or 0, int(radius is not None), radius or 0.0,
           int(index_radius is not None), index_radius or 0.0, len(d), d.ctypes.data_as(C.POINTER(C.c_float)),
           l.ctypes.data_as(C.POINTER(C.c_uint64)), ids.ctypes.data_as(C.POINTER(C.c_int32)), ranks.ctypes.data_as(C.POINTER(C.c_float)))
    assert n >= 0
    return ids[:n], ranks[:n]


def test_select_postprocess_equals_the_references_own_select_code(ref_tape):
    rng = np.random.default_rng(11)
    cases = 0
    for trial in range(600):
        metric = int(rng.integers(0, 3))
        n = int(rng.integers(0, 40))
        is_array = bool(rng.integers(0, 2))
        need_sort = bool(rng.integers(0, 2))
        has_k = bool(rng.integers(0, 2))
        has_radius = (not has_k) or bool(rng.integers(0, 2))
        k = int(rng.integers(1, 25)) if has_k else None
        # few distinct distances: runs of bit-equal ranks (the reference sorts row ids inside them); array fields: several labels per row
        dist = np.sort(rng.integers(-3, 4, size=n).astype(np.float32) * np.float32(0.5))
        rows = rng.integers(0, 12 if is_array else 1000, size=n)
        if not is_array:
            rows = rng.permutation(1000)[:n]
        label = (rows.astype(np.uint64) << np.uint64(32)) | rng.integers(0, 5 if is_array else 1, size=n).astype(np.uint64)
        # a map's answer: best first under (dist, label)
        order = np.lexsort((label, dist))
        dist, label = dist[order], label[order]
        args = (metric, True, need_sort, is_array, k, 1.0 if has_radius else None, None, dist, label)
        # the reference's ids and rank bits, as a digest: equal digests <=> identical ids and identical rank bits
        want, n_ids = ref_tape(lambda: (lambda ids, ranks: (digest(ids, ranks), len(ids)))(*ref_select(*args)), *args)
        got_ids, got_ranks = B.select_postprocess(metric, dist, label, k=k, has_radius=has_radius, need_sort=need_sort, is_array=is_array)
        assert digest(np.asarray(got_ids, np.int32), np.asarray(got_ranks, np.float32)) == want, \
            (trial, metric, is_array, need_sort, k, has_radius, got_ids, got_ranks)
        cases += n_ids > 1
    assert cases > 300


def test_port_select_postprocess_equals_the_references_own_select_code(ref_tape):
    from oracle import oracle as O

    rng = np.random.default_rng(12)
    for trial in range(300):
        metric = int(rng.integers(0, 3))
        n = int(rng.integers(1, 30))
        is_array = bool(rng.integers(0, 2))
        need_sort = bool(rng.integers(0, 2))
        k = int(rng.integers(1, 20))
        has_radius = bool(rng.integers(0, 2))
        dist = np.sort(rng.integers(-3, 4, size=n).astype(np.float32))
        rows = rng.integers(0, 9 if is_array else 500, size=n) if is_array else rng.permutation(500)[:n]
        label = (rows.astype(np.uint64) << np.uint64(32)) | rng.integers(0, 4 if is_array else 1, size=n).astype(np.uint64)
        order = np.lexsort((label, dist))
        dist, label = dist[order], label[order]
        args = (metric, True, need_sort, is_array, k, 1.0 if has_radius else None, None, dist, label)
        want_ids, want_ranks = ref_tape(lambda: ref_select(*args), *args)
        got_ids, got_ranks = O.select_postprocess(metric, dist, label, need_sort=need_sort, is_array=is_array, k=k, has_radius=has_radius)
        assert (want_ids == np.asarray(got_ids)).all() and np.array_equal(want_ranks, np.asarray(got_ranks, np.float32)), trial
