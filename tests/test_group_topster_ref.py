"""The host layer's Topsters against the reference's OWN Topster<KV> (include/topster.h compiled in place into oracle/_ref,
oracle/ref_topster_wrap.cpp): plain top-K with de-duplication by key, and group_by — Topster<KV>(capacity, distinct = group_limit) +
the distinct branch of Index::populate_result_kvs (src/index.cpp:8968-9013). Live where oracle/_ref is built, otherwise against its
answers stored under tests/golden/ref_answers (oracle_lib.RefAnswers)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as ol

SO = os.path.join(ol.ROOT, "tests", "cpp", "libgrouptopster.so")
u64p, i64p, u32p = C.POINTER(C.c_uint64), C.POINTER(C.c_int64), C.POINTER(C.c_uint32)


@pytest.fixture(scope="module")
def libs():
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", os.path.join(ol.ROOT, "tests", "cpp", "group_topster_capi.cpp"), "-o", SO])
    host = C.CDLL(SO)
    ref = C.CDLL(ol.REF_SO) if ol.have_ref() else None
    for L, pre in ((host, "host"), (ref, "ref")):
        if L is None:
            continue
        f = getattr(L, pre + "_topster")
        f.restype = C.c_size_t
        f.argtypes = [u64p, i64p, C.c_size_t, C.c_uint32, u64p]
        g = getattr(L, pre + "_group_topster")
        g.restype = C.c_size_t
        g.argtypes = [u64p, u64p, i64p, C.c_size_t, C.c_uint32, C.c_uint32, u64p, u64p, u32p]
    return host, ref


def _group(fn, keys, distinct, scores, capacity, limit):
    n = len(keys)
    ok, od, gs = np.zeros(n + 1, np.uint64), np.zeros(n + 1, np.uint64), np.zeros(n + 1, np.uint32)
    ng = fn(keys.ctypes.data_as(u64p), distinct.ctypes.data_as(u64p), scores.ctypes.data_as(i64p), n, capacity, limit,
            ok.ctypes.data_as(u64p), od.ctypes.data_as(u64p), gs.ctypes.data_as(u32p))
    out, w = [], 0
    for g in range(ng):
        out.append([[int(od[w + j]), int(ok[w + j])] for j in range(int(gs[g]))])
        w += int(gs[g])
    return out


def test_distinct_int_values_table(libs):
    """the table of TEST(TopsterTest, DistinctIntValues), test/topster_test.cpp:181-262, through the reference's compiled Topster and
    populate_result_kvs' group branch: groups by their best KV, each group's two best"""
    host, ref = libs
    data = [(1, 11, 20, 30), (1, 12, 20, 32), (2, 4, 20, 30), (3, 7, 20, 30), (4, 14, 20, 30), (5, 9, 20, 30), (5, 10, 20, 32),
            (5, 9, 20, 30), (6, 6, 20, 30), (7, 6, 22, 30), (7, 6, 22, 30), (8, 9, 20, 30), (9, 8, 20, 30), (10, 5, 20, 30)]
    keys = np.arange(100, 114, dtype=np.uint64)
    distinct = np.asarray([d[0] for d in data], np.uint64)
    scores = np.ascontiguousarray([[d[1], d[2], d[3]] for d in data], np.int64)
    with ol.RefAnswers("test_group_topster_ref", "distinct_int_values_table") as answers:
        want = answers(lambda: _group(ref.ref_group_topster, keys, distinct, scores, 5, 2))
    assert [g[0][0] for g in want] == [4, 1, 5, 8, 9]
    assert want[1] == [[1, 101], [1, 100]] and want[2] == [[5, 106], [5, 107]]
    assert _group(host.host_group_topster, keys, distinct, scores, 5, 2) == want


@pytest.mark.parametrize("seed", range(6))
def test_group_topster_equals_the_reference(libs, seed):
    host, ref = libs
    rng = np.random.default_rng(seed)
    with ol.RefAnswers("test_group_topster_ref", f"group_topster[{seed}]") as answers:
        for _ in range(40):
            n = int(rng.integers(1, 400))
            keys = rng.integers(0, max(2, n // 2), n).astype(np.uint64)                 # repeated keys: the greatest KV per key survives
            distinct = (keys % np.uint64(int(rng.integers(1, 40)))).astype(np.uint64)   # a key always belongs to the same group
            scores = np.ascontiguousarray(rng.integers(0, 4, (n, 3)), np.int64)         # few values: ties down to the key
            capacity, limit = int(rng.integers(1, 30)), int(rng.integers(1, 5))
            got = _group(host.host_group_topster, keys, distinct, scores, capacity, limit)
            assert answers.same(got, lambda: _group(ref.ref_group_topster, keys, distinct, scores, capacity, limit))


@pytest.mark.parametrize("seed", range(4))
def test_plain_topster_equals_the_reference(libs, seed):
    host, ref = libs
    rng = np.random.default_rng(100 + seed)
    with ol.RefAnswers("test_group_topster_ref", f"plain_topster[{seed}]") as answers:
        for _ in range(40):
            n = int(rng.integers(1, 600))
            keys = rng.integers(0, max(2, n // 2), n).astype(np.uint64)
            scores = np.ascontiguousarray(rng.integers(0, 5, (n, 3)), np.int64)
            capacity = int(rng.integers(1, 300))
            assert answers.same(_topster(host.host_topster, keys, scores, capacity), lambda: _topster(ref.ref_topster, keys, scores, capacity))


def _topster(fn, keys, scores, capacity):
    n = len(keys)
    a = np.zeros(n + 1, np.uint64)
    na = fn(keys.ctypes.data_as(u64p), scores.ctypes.data_as(i64p), n, capacity, a.ctypes.data_as(u64p))
    return a[:na].tolist()


@pytest.mark.parametrize("seed", range(4))
def test_oracle_topster_equals_the_reference(libs, seed):
    """tso_topster_run — the restatement every GPU top-k is compared with — against the reference's compiled Topster<KV>"""
    from typesense_b200.structs import KV_DTYPE
    host, ref = libs
    rng = np.random.default_rng(200 + seed)
    with ol.RefAnswers("test_group_topster_ref", f"oracle_topster[{seed}]") as answers:
        for _ in range(40):
            n = int(rng.integers(1, 600))
            keys = rng.integers(0, max(2, n // 2), n).astype(np.uint64)
            scores = np.ascontiguousarray(rng.integers(0, 5, (n, 3)), np.int64)
            capacity = int(rng.integers(1, 300))
            rows = np.zeros(n, KV_DTYPE)
            rows["key"] = keys; rows["distinct_key"] = keys; rows["scores"] = scores
            out = np.zeros(max(capacity, 1), KV_DTYPE)
            no = ol.oracle().tso_topster_run(capacity, rows.ctypes.data_as(C.c_void_p), n, out.ctypes.data_as(C.c_void_p))
            assert answers.same(out["key"][:no], lambda: _topster(ref.ref_topster, keys, scores, capacity))
