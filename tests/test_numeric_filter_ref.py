"""The comparator semantics tsgpu_filter_numeric is held to (tests/test_filters_device.py::expect_ids, SURVEY 8 f-2) against the
reference's OWN numeric index: src/num_tree.cpp compiled in place into oracle/_ref (oracle/ref_numtree_wrap.cpp) — `=`, `<`, `<=`,
`>`, `>=` through num_tree_t::search, `[a..b]` through range_inclusive_search, `!=` as the complement of the equal ids; a document
without a value is in no leaf. Live where oracle/_ref is built, otherwise against its answers stored under tests/golden/ref_answers
(oracle_lib.RefAnswers)."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
from test_filters_device import MISSING, expect_ids

OPS = {"=": 0, "!=": 1, "<": 2, "<=": 3, ">": 4, ">=": 5, "range": 6}


def _num_tree_search(col, code, v1, v2):
    L = C.CDLL(ol.REF_SO)
    L.ref_num_tree_search.restype = C.c_size_t
    L.ref_num_tree_search.argtypes = [C.POINTER(C.c_int64), C.c_uint32, C.c_int, C.c_int64, C.c_int64, C.POINTER(C.c_uint32)]
    out = np.zeros(len(col) + 1, np.uint32)
    k = L.ref_num_tree_search(col.ctypes.data_as(C.POINTER(C.c_int64)), len(col), code, v1, v2, out.ctypes.data_as(C.POINTER(C.c_uint32)))
    return out[:k]


@pytest.mark.parametrize("seed", range(5))
def test_numpy_expectation_equals_the_reference_num_tree(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(200, 3000))
    col = rng.integers(-50, 200, n).astype(np.int64)                      # few distinct values: long id lists per value
    col[rng.random(n) < 0.15] = MISSING
    if seed == 0:
        col[:] = MISSING                                                   # an empty tree
    with ol.RefAnswers("test_numeric_filter_ref", f"num_tree[{seed}]") as answers:
        for op, code in OPS.items():
            for _ in range(12):
                v1 = int(rng.integers(-60, 210))
                v2 = v1 + int(rng.integers(0, 40))
                assert answers.same(expect_ids(col, op, v1, v2), lambda: _num_tree_search(col, code, v1, v2)), (op, v1, v2)
