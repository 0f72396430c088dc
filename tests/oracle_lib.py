"""TEST INFRASTRUCTURE: ctypes bindings of the CPU oracle (oracle/liboracle.so) and, when built, of the
reference's own compiled posting-list sources (oracle/_ref/liboracle_ref.so).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline/--impl reference legs import this.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import lzma
import os
import subprocess
from typing import List, Optional, Sequence

import numpy as np

from typesense_b200.structs import (FieldStruct, FlatField, HnswGraph, HnswStruct, KV_DTYPE, KwBatch, KwBatchStruct,
                                    VecParamsStruct, f32p, i32p, u8p, u16p, u32p, u64p)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "liboracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "liboracle_ref.so")


def build_oracle(force: bool = False):
    srcs = [os.path.join(ORACLE_DIR, f) for f in ("ts_oracle.cpp", "ts_oracle.h", "ts_oracle_vec.inc")]
    if force or not os.path.exists(ORACLE_SO) or any(os.path.getmtime(s) > os.path.getmtime(ORACLE_SO) for s in srcs):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "liboracle.so"])
    if os.path.isdir("/root/reference/src"):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "ref"])


_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        build_oracle()
        L = C.CDLL(ORACLE_SO)
        L.tso_intersect.restype = C.c_size_t
        L.tso_merge.restype = C.c_size_t
        L.tso_contains_atleast_one.argtypes = [u32p, C.c_size_t, u32p, C.c_size_t]
        L.tso_facet_counts.restype = C.c_size_t
        L.tso_facet_counts.argtypes = [C.c_uint32, C.c_uint32, u64p, u32p, u32p, C.c_size_t, C.c_uint32, C.c_void_p, C.c_size_t, u32p]
        for n in ("tso_and_scalar", "tso_or_scalar", "tso_exclude_scalar"):
            getattr(L, n).restype = C.c_size_t
            getattr(L, n).argtypes = [u32p, C.c_size_t, u32p, C.c_size_t, u32p]
        L.tso_match.argtypes = [C.c_uint32, u32p, u16p, u8p, C.c_int, u8p]
        L.tso_match_score.restype = C.c_uint64
        L.tso_match_score.argtypes = [C.c_uint8] * 4 + [C.c_uint32, C.c_uint32, C.c_uint8]
        L.tso_has_phrase_match.argtypes = [C.c_uint32, u32p, u16p]
        L.tso_index_new.restype = C.c_void_p
        L.tso_index_new.argtypes = [C.c_uint32]
        L.tso_index_free.argtypes = [C.c_void_p]
        L.tso_index_add_field.argtypes = [C.c_void_p, C.POINTER(FieldStruct)]
        L.tso_index_add_sort_column.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.tso_index_set_hnsw.argtypes = [C.c_void_p, C.POINTER(HnswStruct)]
        L.tso_keyword_combo.restype = C.c_size_t
        L.tso_keyword_combo.argtypes = [C.c_void_p, C.POINTER(KwBatchStruct), C.c_uint32, C.c_uint32, u32p, u64p,
                                        C.c_size_t, u64p]
        L.tso_keyword_search_batch.argtypes = [C.c_void_p, C.POINTER(KwBatchStruct), C.c_void_p, C.c_uint32, u32p, u32p,
                                               C.c_uint32]
        L.tso_wildcard_search_batch.argtypes = [C.c_void_p, C.POINTER(KwBatchStruct), C.c_void_p, C.c_uint32, u32p, u32p,
                                                C.c_uint32]
        L.tso_topster_run.restype = C.c_uint32
        L.tso_topster_run.argtypes = [C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]
        for n in ("tso_phrase_matches", "tso_exact_matches", "tso_prefix_matches"):
            getattr(L, n).restype = C.c_size_t
            getattr(L, n).argtypes = [C.c_void_p, C.c_uint32, u32p, C.c_uint32, u32p, C.c_size_t, u32p]
        L.tso_ip_distance.restype = C.c_float
        L.tso_ip_distance.argtypes = [f32p, f32p, C.c_uint32]
        L.tso_normalize.argtypes = [f32p, f32p, C.c_uint32]
        L.tso_hnsw_build.restype = C.c_void_p
        L.tso_hnsw_build.argtypes = [f32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.tso_hnsw_build_info.argtypes = [C.c_void_p, u32p, u32p, u64p]
        L.tso_hnsw_build_fetch.argtypes = [C.c_void_p, u8p, u32p, u64p, u32p]
        L.tso_hnsw_build_free.argtypes = [C.c_void_p]
        L.tso_hnsw_search.restype = C.c_uint32
        L.tso_hnsw_search.argtypes = [C.POINTER(HnswStruct), f32p, C.c_uint32, C.c_uint32, u32p, C.c_size_t, u32p,
                                      C.c_size_t, f32p, u32p, u64p]
        L.tso_hnsw_search_batch.argtypes = [C.POINTER(HnswStruct), f32p, C.c_uint32, C.c_uint32, C.c_uint32, i32p, u64p,
                                            u32p, f32p, u32p, u32p, u64p, C.c_uint32]
        L.tso_flat_distances.argtypes = [C.POINTER(HnswStruct), f32p, u32p, C.c_size_t, f32p]
        for n in ("tso_hybrid_search_batch", "tso_vector_search_batch"):
            getattr(L, n).argtypes = [C.c_void_p, C.POINTER(KwBatchStruct), f32p, C.POINTER(VecParamsStruct), C.c_void_p,
                                      C.c_uint32, u32p, u32p, C.c_uint32]
        L.tso_float_to_int64.restype = C.c_int64
        L.tso_float_to_int64.argtypes = [C.c_float]
        L.tso_int64_to_float.restype = C.c_float
        L.tso_int64_to_float.argtypes = [C.c_int64]
        _oracle = L
    return _oracle


def have_ref() -> bool:
    if not os.path.exists(REF_SO) and os.path.isdir("/root/reference/src"):
        build_oracle()
    return os.path.exists(REF_SO)


REF_ANSWERS_DIR = os.path.join(ROOT, "tests", "golden", "ref_answers")


def _plain(v):
    if isinstance(v, np.ndarray):
        return v.tolist()
    if isinstance(v, (list, tuple)):
        return [_plain(x) for x in v]
    if isinstance(v, dict):
        return {str(k): _plain(x) for k, x in v.items()}
    if isinstance(v, np.generic):
        return v.item()
    return v


class RefAnswers:
    """What the reference's own compiled sources answered in one test, in call order, stored under
    tests/golden/ref_answers/<group>.json.xz so the comparison runs where oracle/_ref cannot be built.

    `ref(fn)` returns fn()'s answer as plain lists / numbers / strings; `ref.same(got, fn)` says whether `got` equals it, and
    stores a long answer as a 128-bit SHA-256 digest only. With oracle/_ref built, fn runs and its answer must equal the stored one
    (TSGPU_REF_RECORD=1 stores the live answers instead); without it, the stored answer is used and fn is not called, so fn
    alone may touch ol.ref()."""

    def __init__(self, group: str, name: str):
        self.path = os.path.join(REF_ANSWERS_DIR, group + ".json.xz")
        self.name = name
        self.live = have_ref()
        self.record = self.live and os.environ.get("TSGPU_REF_RECORD") == "1"
        self.stored = _load_answers(self.path).get(name)
        assert self.record or self.stored is not None, \
            f"no stored reference answers for {group}/{name}: record them with TSGPU_REF_RECORD=1 where oracle/_ref is built"
        self.got = []

    def __call__(self, fn):
        i = len(self.got)
        if self.live:
            v = _plain(fn())
            if not self.record:
                assert i < len(self.stored) and v == self.stored[i], f"{self.name}: reference answer {i} differs from the stored one"
        else:
            assert i < len(self.stored), f"{self.name}: more reference calls than stored answers"
            v = self.stored[i]
        self.got.append(v)
        return v

    def same(self, got, fn) -> bool:
        return _compact(got) == self(lambda: _compact(fn()))

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is not None:
            return False
        if self.record:
            data = _load_answers(self.path)
            data[self.name] = self.got
            os.makedirs(REF_ANSWERS_DIR, exist_ok=True)
            with open(self.path, "wb") as f:
                f.write(lzma.compress(json.dumps(data, sort_keys=True, separators=(",", ":")).encode(), preset=9 | lzma.PRESET_EXTREME))
        else:
            assert len(self.got) == len(self.stored), f"{self.name}: {len(self.got)} reference calls, {len(self.stored)} stored answers"
        return False


def _compact(v):
    v = _plain(v)
    s = json.dumps(v, sort_keys=True, separators=(",", ":"))
    return v if len(s) <= 64 else "sha256:" + hashlib.sha256(s.encode()).hexdigest()[:32]


def _load_answers(path: str) -> dict:
    if not os.path.exists(path):
        return {}
    with open(path, "rb") as f:
        return json.loads(lzma.decompress(f.read()))


class RefParams(C.Structure):
    _fields_ = [("n_tokens", C.c_uint32), ("n_dropped", C.c_uint32), ("n_fields", C.c_uint32),
                ("total_cost", C.c_uint32), ("num_query_tokens", C.c_uint32), ("syn_orig_num_tokens", C.c_int32),
                ("orig_num_tokens", C.c_int32), ("is_synonym_query", C.c_uint8), ("demote_synonym_match", C.c_uint8),
                ("prioritize_exact_match", C.c_uint8), ("prioritize_token_position", C.c_uint8),
                ("prioritize_num_matching_fields", C.c_uint8), ("match_type", C.c_uint8), ("pad", C.c_uint8 * 2),
                ("field_weight", C.c_int64 * 32), ("field_is_array", C.c_uint8 * 32)]


def ref():
    global _ref
    if _ref is None:
        assert have_ref(), "oracle/_ref not built"
        L = C.CDLL(REF_SO)
        vp = C.c_void_p
        L.ref_sorted_array_new.restype = vp
        L.ref_array_new.restype = vp
        L.ref_plist_new.restype = vp
        L.ref_plist_new.argtypes = [C.c_uint32]
        L.ref_plist_free.argtypes = [vp]
        L.ref_plist_upsert.argtypes = [vp, C.c_uint32, u32p, C.c_uint32]
        L.ref_plist_erase.argtypes = [vp, C.c_uint32]
        L.ref_plist_num_ids.argtypes = [vp]
        L.ref_plist_num_ids.restype = C.c_uint32
        L.ref_plist_num_blocks.argtypes = [vp]
        L.ref_plist_num_blocks.restype = C.c_uint32
        L.ref_plist_bulk.argtypes = [vp, u32p, u32p, u32p, C.c_uint32]
        L.ref_plist_dump.restype = C.c_size_t
        L.ref_plist_dump.argtypes = [vp, u32p, u32p, u32p, C.c_size_t, C.c_size_t]
        for n in ("ref_plist_intersect", "ref_plist_merge"):
            getattr(L, n).restype = C.c_size_t
            getattr(L, n).argtypes = [C.POINTER(vp), C.c_uint32, u32p, C.c_size_t]
        L.ref_plist_contains_atleast_one.argtypes = [vp, u32p, C.c_size_t]
        L.ref_plist_block_intersect.restype = C.c_size_t
        L.ref_plist_block_intersect.argtypes = [C.POINTER(vp), C.c_uint32, u32p, C.c_size_t, u32p, C.c_size_t, u32p,
                                                C.c_size_t]
        for n in ("ref_plist_phrase_matches", "ref_plist_exact_matches", "ref_plist_prefix_matches"):
            getattr(L, n).restype = C.c_size_t
            getattr(L, n).argtypes = [C.POINTER(vp), C.c_uint32, C.c_int, u32p, C.c_uint32, u32p]
        L.ref_match.argtypes = [C.c_uint32, u32p, u16p, u8p, C.c_int, u8p]
        L.ref_match_score.restype = C.c_uint64
        L.ref_match_score.argtypes = [C.c_uint8] * 4 + [C.c_uint32, C.c_uint32, C.c_uint8]
        L.ref_has_phrase_match.argtypes = [C.c_uint32, u32p, u16p]
        for n in ("ref_and_scalar", "ref_or_scalar", "ref_exclude_scalar"):
            getattr(L, n).restype = C.c_size_t
            getattr(L, n).argtypes = [u32p, C.c_size_t, u32p, C.c_size_t, u32p]
        L.ref_keyword_combo.restype = C.c_size_t
        L.ref_keyword_combo.argtypes = [C.POINTER(RefParams), C.POINTER(vp), u32p, C.c_size_t, u32p, C.c_size_t, C.c_int,
                                        u32p, u64p, C.c_size_t, u64p]
        for n in ("ref_sorted_array_free", "ref_array_free"):
            getattr(L, n).argtypes = [vp]
        L.ref_sorted_array_append.argtypes = [vp, C.c_uint32]
        L.ref_sorted_array_append.restype = C.c_uint32
        L.ref_sorted_array_load.argtypes = [vp, u32p, C.c_uint32]
        L.ref_sorted_array_at.argtypes = [vp, C.c_uint32]
        L.ref_sorted_array_at.restype = C.c_uint32
        L.ref_sorted_array_length.argtypes = [vp]
        L.ref_sorted_array_length.restype = C.c_uint32
        L.ref_sorted_array_contains.argtypes = [vp, C.c_uint32]
        L.ref_sorted_array_index_of.argtypes = [vp, C.c_uint32]
        L.ref_sorted_array_index_of.restype = C.c_uint32
        L.ref_sorted_array_bulk_index_of.argtypes = [vp, u32p, C.c_uint32, u32p]
        L.ref_sorted_array_num_found_of.argtypes = [vp, u32p, C.c_uint32]
        L.ref_sorted_array_num_found_of.restype = C.c_uint32
        L.ref_sorted_array_remove_value.argtypes = [vp, C.c_uint32]
        L.ref_sorted_array_uncompress.argtypes = [vp, u32p]
        L.ref_array_append.argtypes = [vp, C.c_uint32]
        L.ref_array_at.argtypes = [vp, C.c_uint32]
        L.ref_array_at.restype = C.c_uint32
        L.ref_array_length.argtypes = [vp]
        L.ref_array_length.restype = C.c_uint32
        L.ref_array_index_of.argtypes = [vp, C.c_uint32]
        L.ref_array_index_of.restype = C.c_uint32
        L.ref_array_remove_index.argtypes = [vp, C.c_uint32, C.c_uint32]
        if hasattr(L, "ref_art_new"):          # the reference's ART (src/art.cpp)
            L.ref_art_new.restype = vp
            L.ref_art_free.argtypes = [vp]
            L.ref_art_insert.argtypes = [vp, C.c_char_p, C.c_uint32, C.c_int64, u32p, C.c_uint32]
            L.ref_art_export.restype = C.c_size_t
            L.ref_art_export.argtypes = [vp, C.c_char_p, C.c_size_t]
            L.ref_art_fuzzy.restype = C.c_size_t
            L.ref_art_fuzzy.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_char_p, u32p, C.c_size_t,
                                        C.c_int, C.c_char_p, C.c_char_p, C.c_size_t]
        _ref = L
    return _ref


def p32(a: np.ndarray):
    return a.ctypes.data_as(u32p)


class OracleIndex:
    """Oracle-side index over the same flat arrays the CUDA mirror is loaded from."""

    def __init__(self, n_docs: int, fields: Sequence[FlatField], sort_cols: Sequence[np.ndarray] = (),
                 hnsw: Optional[HnswGraph] = None):
        self.L = oracle()
        self.n_docs = n_docs
        self.fields = list(fields)
        self.sort_cols = [np.ascontiguousarray(c, np.int64) for c in sort_cols]
        self.hnsw = hnsw
        self.h = C.c_void_p(self.L.tso_index_new(n_docs))
        self._keep = []
        for f in self.fields:
            s = f.struct()
            self._keep.append(s)
            self.L.tso_index_add_field(self.h, C.byref(s))
        for c in self.sort_cols:
            self.L.tso_index_add_sort_column(self.h, c.ctypes.data_as(C.POINTER(C.c_int64)))
        if hnsw is not None:
            self.hs = hnsw.struct()
            self.L.tso_index_set_hnsw(self.h, C.byref(self.hs))

    def __del__(self):
        try:
            self.L.tso_index_free(self.h)
        except Exception:
            pass

    def keyword_combo(self, b: KwBatch, q: int, c: int, cap: int = 1 << 22):
        ids = np.zeros(cap, np.uint32)
        sc = np.zeros(cap, np.uint64)
        nkm = C.c_uint64(0)
        s = b.struct()
        n = self.L.tso_keyword_combo(self.h, C.byref(s), q, c, p32(ids), sc.ctypes.data_as(u64p), cap, C.byref(nkm))
        assert n != C.c_size_t(-1).value
        return ids[:n].copy(), sc[:n].copy(), nkm.value

    def _run(self, fn, b: KwBatch, stride: int, threads: int, extra=()):
        out = np.zeros((b.n_queries, stride), KV_DTYPE)
        cnt = np.zeros(b.n_queries, np.uint32)
        found = np.zeros(b.n_queries, np.uint32)
        s = b.struct()
        rc = fn(self.h, C.byref(s), *extra, out.ctypes.data_as(C.c_void_p), stride, p32(cnt), p32(found), threads)
        assert rc == 0
        return out, cnt, found

    def keyword_search(self, b: KwBatch, stride: int = 256, threads: int = 1):
        return self._run(self.L.tso_keyword_search_batch, b, stride, threads)

    def wildcard_search(self, b: KwBatch, stride: int = 256, threads: int = 1):
        return self._run(self.L.tso_wildcard_search_batch, b, stride, threads)

    def hybrid_search(self, b: KwBatch, qvecs: np.ndarray, vp: VecParamsStruct, stride: int = 256, threads: int = 1):
        qv = np.ascontiguousarray(qvecs, np.float32)
        return self._run(self.L.tso_hybrid_search_batch, b, stride, threads, (qv.ctypes.data_as(f32p), C.byref(vp)))

    def vector_search(self, b: KwBatch, qvecs: np.ndarray, vp: VecParamsStruct, stride: int = 256, threads: int = 1):
        qv = np.ascontiguousarray(qvecs, np.float32)
        return self._run(self.L.tso_vector_search_batch, b, stride, threads, (qv.ctypes.data_as(f32p), C.byref(vp)))

    def flat_distances(self, query: np.ndarray, ids: np.ndarray) -> np.ndarray:
        """tso_flat_distances: process_results_bruteforce's loop (src/index.cpp:3345-3374), fp32, in id order."""
        q = np.ascontiguousarray(query, np.float32)
        ids = np.ascontiguousarray(ids, np.uint32)
        out = np.zeros(max(len(ids), 1), np.float32)
        self.L.tso_flat_distances(C.byref(self.hs), q.ctypes.data_as(f32p), p32(ids), len(ids), out.ctypes.data_as(f32p))
        return out[:len(ids)]

    def knn(self, queries: np.ndarray, k: int, ef: int, q_filter=None, filters=(), threads: int = 1):
        q = np.ascontiguousarray(queries, np.float32)
        nq = q.shape[0]
        d = np.zeros((nq, k), np.float32)
        l = np.zeros((nq, k), np.uint32)
        n = np.zeros(nq, np.uint32)
        st = np.zeros(2, np.uint64)
        off = [0]
        for f in filters:
            off.append(off[-1] + len(f))
        foff = np.asarray(off, np.uint64)
        fids = np.concatenate([np.asarray(f, np.uint32) for f in filters]) if filters and off[-1] else np.zeros(1, np.uint32)
        qf = None if q_filter is None else np.ascontiguousarray(q_filter, np.int32)
        self.L.tso_hnsw_search_batch(C.byref(self.hs), q.ctypes.data_as(f32p), nq, k, ef,
                                     qf.ctypes.data_as(i32p) if qf is not None else C.cast(None, i32p),
                                     foff.ctypes.data_as(u64p), p32(fids), d.ctypes.data_as(f32p), p32(l), p32(n),
                                     st.ctypes.data_as(u64p), threads)
        return d, l, n, st


def hnsw_build(vectors: np.ndarray, M: int = 16, ef_construction: int = 200, seed: int = 100, metric: int = 0) -> HnswGraph:
    """hnswlib-equivalent single-threaded construction by the oracle (exported graph is shared with the GPU)."""
    L = oracle()
    v = np.ascontiguousarray(vectors, np.float32)
    n, dim = v.shape
    b = C.c_void_p(L.tso_hnsw_build(v.ctypes.data_as(f32p), n, dim, M, ef_construction, seed))
    ml, ep, nup = C.c_uint32(0), C.c_uint32(0), C.c_uint64(0)
    L.tso_hnsw_build_info(b, C.byref(ml), C.byref(ep), C.byref(nup))
    levels = np.zeros(n, np.uint8)
    links0 = np.zeros(n * (2 * M + 1), np.uint32)
    upper_off = np.zeros(n + 1, np.uint64)
    links_up = np.zeros(max(1, nup.value * (M + 1)), np.uint32)
    L.tso_hnsw_build_fetch(b, levels.ctypes.data_as(u8p), p32(links0), upper_off.ctypes.data_as(u64p), p32(links_up))
    L.tso_hnsw_build_free(b)
    return HnswGraph(v, levels, links0, upper_off, links_up, M, ml.value, ep.value, metric)


class RefPlist:
    """posting_list_t of the reference (oracle/_ref)."""

    def __init__(self, block_max: int = 256):
        self.L = ref()
        self.h = C.c_void_p(self.L.ref_plist_new(block_max))

    def upsert(self, sid: int, offsets: Sequence[int]):
        a = np.asarray(list(offsets) if len(offsets) else [0], np.uint32)
        self.L.ref_plist_upsert(self.h, sid, p32(a), len(offsets))

    def __del__(self):
        try:
            self.L.ref_plist_free(self.h)
        except Exception:
            pass


def ref_plists_of(field: FlatField, lists: Sequence[int], block_max: int = 256) -> List[RefPlist]:
    out = []
    for l in lists:
        pl = RefPlist(block_max)
        a, b = int(field.list_off[l]), int(field.list_off[l + 1])
        ids = np.ascontiguousarray(field.ids[a:b])
        po = field.pos_off[a:b + 1]
        base = int(po[0])
        offs = np.ascontiguousarray(field.positions[base:int(po[-1])]) if int(po[-1]) > base else np.zeros(1, np.uint32)
        oi = np.ascontiguousarray((po - base).astype(np.uint32))
        pl.L.ref_plist_bulk(pl.h, p32(ids), p32(oi), p32(offs), len(ids))
        out.append(pl)
    return out


def facet_counts(n_docs: int, n_values: int, doc_off: np.ndarray, value_ids: np.ndarray, ids, cap: int, sample_mod: int = 0):
    """tso_facet_counts: (entries as the FACET_DTYPE of typesense_b200.capi, distinct values with a count)."""
    from typesense_b200.capi import FACET_DTYPE
    a = np.ascontiguousarray(ids, np.uint32)
    out = np.zeros(max(cap, 1), FACET_DTYPE)
    dis = C.c_uint32(0)
    n = oracle().tso_facet_counts(n_docs, n_values, doc_off.ctypes.data_as(u64p), value_ids.ctypes.data_as(u32p), a.ctypes.data_as(u32p), len(a), sample_mod,
                                  out.ctypes.data, cap, C.byref(dis))
    return out[:n], dis.value
