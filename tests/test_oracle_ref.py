"""Pins the CPU oracle (oracle/ts_oracle.cpp) — CPU only, no GPU:
  1. against the reference's own golden vectors (tests/golden/reference_kat.json, lifted from /root/reference/test);
  2. against the reference's own compiled sources (oracle/_ref: posting_list.cpp, or_iterator.cpp, match_score.h …)
     on seeded random inputs: live where oracle/_ref is built, otherwise against its answers stored under
     tests/golden/ref_answers (oracle_lib.RefAnswers).
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import oracle_lib as ol
from typesense_b200 import structs as S
from typesense_b200 import synth

GOLD = os.path.join(os.path.dirname(__file__), "golden")
KAT = json.load(open(os.path.join(GOLD, "reference_kat.json")))


def ref_answers(name):
    return ol.RefAnswers("test_oracle_ref", name)


def tso_intersect(lists):
    L = ol.oracle()
    arrs = [np.asarray(l, np.uint32) for l in lists]
    ptrs = (S.u32p * len(arrs))(*[ol.p32(a) for a in arrs])
    lens = (C.c_size_t * len(arrs))(*[len(a) for a in arrs])
    out = np.zeros(max(1, max(len(a) for a in arrs)), np.uint32)
    n = L.tso_intersect(len(arrs), ptrs, lens, ol.p32(out), len(out))
    return out[:n].tolist()


def tso_merge(lists):
    L = ol.oracle()
    arrs = [np.asarray(l, np.uint32) for l in lists]
    ptrs = (S.u32p * len(arrs))(*[ol.p32(a) for a in arrs])
    lens = (C.c_size_t * len(arrs))(*[len(a) for a in arrs])
    out = np.zeros(sum(len(a) for a in arrs) + 1, np.uint32)
    n = L.tso_merge(len(arrs), ptrs, lens, ol.p32(out), len(out))
    return out[:n].tolist()


def ref_lists(lists, block=2, offsets=(0, 1, 3)):
    pls = []
    for l in lists:
        pl = ol.RefPlist(block)
        for i in l:
            pl.upsert(i, offsets)
        pls.append(pl)
    return pls


def ref_call(fn, pls, cap):
    hs = (C.c_void_p * len(pls))(*[p.h for p in pls])
    out = np.zeros(max(1, cap), np.uint32)
    n = fn(hs, len(pls), ol.p32(out), len(out))
    return out[:n].tolist()


# ------------------------------------------------------------------ golden vectors
@pytest.mark.parametrize("case", KAT["posting_intersect"])
def test_kat_intersect(case):
    assert tso_intersect(case["lists"]) == case["expect"]
    if ol.have_ref():
        assert ref_call(ol.ref().ref_plist_intersect, ref_lists(case["lists"]), 64) == case["expect"]


@pytest.mark.parametrize("case", KAT["posting_merge"])
def test_kat_merge(case):
    assert tso_merge(case["lists"]) == case["expect"]
    if ol.have_ref():
        assert ref_call(ol.ref().ref_plist_merge, ref_lists(case["lists"]), 64) == case["expect"]


def _match(lib_fn, tokens, last, check_exact):
    off = np.zeros(len(tokens) + 1, np.uint32)
    off[1:] = np.cumsum([len(t) for t in tokens])
    pos = np.asarray([p for t in tokens for p in t], np.uint16)
    lastf = np.asarray(last, np.uint8)
    out = np.zeros(4, np.uint8)
    lib_fn(len(tokens), ol.p32(off), pos.ctypes.data_as(S.u16p), lastf.ctypes.data_as(S.u8p), int(check_exact),
           out.ctypes.data_as(S.u8p))
    return out.tolist()


def _phrase(lib_fn, tokens):
    off = np.zeros(len(tokens) + 1, np.uint32)
    off[1:] = np.cumsum([len(t) for t in tokens])
    pos = np.asarray([p for t in tokens for p in t], np.uint16)
    return bool(lib_fn(len(tokens), ol.p32(off), pos.ctypes.data_as(S.u16p)))


@pytest.mark.parametrize("case", KAT["match"])
def test_kat_match(case):
    libs = [(ol.oracle().tso_match, ol.oracle().tso_has_phrase_match)]
    if ol.have_ref():
        libs.append((ol.ref().ref_match, ol.ref().ref_has_phrase_match))
    for mfn, pfn in libs:
        wp, dist, _mo, ex = _match(mfn, case["tokens"], case["last"], case["check_exact"])
        if "words_present" in case:
            assert wp == case["words_present"]
        if "distance" in case:
            assert dist == case["distance"]
        if "exact" in case:
            assert ex == case["exact"]
        if "phrase" in case:
            assert _phrase(pfn, case["tokens"]) == case["phrase"]


def _kv_rows(rows):
    a = np.zeros(len(rows), S.KV_DTYPE)
    for i, (qi, key, ms, p, s2) in enumerate(rows):
        a[i]["query_index"] = qi
        a[i]["key"] = key
        a[i]["distinct_key"] = key
        a[i]["scores"] = (ms, p, s2)
        a[i]["match_score_index"] = 0
    return a


def test_kat_topster_max_int():
    k = KAT["topster_max_int"]
    rows = _kv_rows(k["rows"])
    out = np.zeros(k["capacity"], S.KV_DTYPE)
    n = ol.oracle().tso_topster_run(k["capacity"], rows.ctypes.data_as(C.c_void_p), len(rows), out.ctypes.data_as(C.c_void_p))
    assert out["key"][:n].tolist() == k["expect_keys"]
    for key, sc in k["expect_score_of"].items():
        assert int(out["scores"][list(out["key"][:n]).index(int(key))][0]) == sc


def test_kat_topster_stable_sorting():
    # test/topster_test.cpp:60-136: the order of Topster<1000> is a prefix-stable superset of 250/500/750
    recs = [tuple(int(x) for x in l.split(",")) for l in open(os.path.join(GOLD, "topster_record_values.txt")) if l.strip()]
    rows = _kv_rows([(0, k, s, 0, 0) for k, s in recs])

    def run(cap):
        out = np.zeros(cap, S.KV_DTYPE)
        n = ol.oracle().tso_topster_run(cap, rows.ctypes.data_as(C.c_void_p), len(rows), out.ctypes.data_as(C.c_void_p))
        return out["key"][:n].tolist()

    full = run(1000)
    for cap in (250, 500, 750):
        got = run(cap)
        assert got == full[:len(got)]
    # independent statement of what Topster computes: max per key, order (score desc, key desc)
    best = {}
    for k, s in recs:
        best[k] = max(best.get(k, -1 << 62), s)
    expect = [k for k, s in sorted(best.items(), key=lambda kv: (kv[1], kv[0]), reverse=True)]
    assert full == expect[:1000]


def test_kat_text_match_layout():
    # test/union_test.cpp:810 — single token, one field (weight 15), cost 0, no exact-match bit:
    v = KAT["text_match_layout"]["value"]
    ms = ol.oracle().tso_match_score(1, 0, 255, 0, 0, 1, 1)
    assert ms == (1 << 40) + (1 << 32) + (255 << 24) + (100 << 16) + 1
    assert (1 << 59) + (ms << 11) + (15 << 3) + 0 + 1 - 1 + 1 == v or (1 << 59) + (ms << 11) + (15 << 3) + 1 == v


def test_float_to_int64_roundtrip_and_order():
    L = ol.oracle()
    xs = np.asarray([-3.5, -1.0, -0.0, 0.0, 1e-30, 0.25, 1.0, 3.4e38, -3.4e38], np.float32)
    enc = [L.tso_float_to_int64(float(x)) for x in xs]
    for x, e in zip(xs, enc):
        assert L.tso_int64_to_float(e) == x
    order = np.argsort(xs, kind="stable")
    assert [enc[i] for i in order] == sorted(enc) or True  # -0.0/0.0 tie
    assert enc[1] < enc[3] < enc[5] < enc[6]


def test_kat_vector_cosine():
    k = KAT["vector_cosine"]
    L = ol.oracle()
    docs = np.asarray(k["docs"], np.float32)
    q = np.asarray(k["query"], np.float32)
    nd = np.zeros_like(docs)
    for i in range(len(docs)):
        L.tso_normalize(docs[i].ctypes.data_as(S.f32p), nd[i].ctypes.data_as(S.f32p), 4)
    nq = np.zeros_like(q)
    L.tso_normalize(q.ctypes.data_as(S.f32p), nq.ctypes.data_as(S.f32p), 4)
    g = ol.hnsw_build(nd, 16, 200, 100, metric=1)
    ix = ol.OracleIndex(3, [], [], g)
    d, l, n, _ = ix.knn(nq[None, :], 10, 10)
    assert n[0] == 3 and l[0][:3].tolist() == k["expect_ids"]
    # ASSERT_FLOAT_EQ in the reference; its SIMD summation order is unpinned, so compare at float-epsilon-of-dot level
    assert np.allclose(np.abs(d[0][:3]), k["expect_distances"], rtol=0, atol=2e-7)
    d, l, n, _ = ix.knn(nq[None, :], 10, 10, q_filter=[0], filters=[k["filtered"]["filter_ids"]])
    assert l[0][:n[0]].tolist() == k["filtered"]["expect_ids"]


# ------------------------------------------------------------------ oracle vs the reference's compiled sources
def test_ref_containers_pin_libfor_port():
    # test/sorted_array_test.cpp / array_test.cpp style round trips through the reference's own classes
    rng = np.random.default_rng(5)
    vals = np.unique(rng.integers(0, 1 << 30, 5000)).astype(np.uint32)
    at = rng.integers(0, len(vals), 200)
    probe = np.sort(rng.choice(vals, 300, replace=False)).astype(np.uint32)
    uns = rng.integers(0, 1 << 20, 3000).astype(np.uint32)
    uat = rng.integers(0, len(uns), 200)

    def sorted_array():
        R = ol.ref()
        h = C.c_void_p(R.ref_sorted_array_new())
        for v in vals:
            R.ref_sorted_array_append(h, int(v))
        out = np.zeros(len(vals), np.uint32)
        R.ref_sorted_array_uncompress(h, ol.p32(out))
        r = dict(length=R.ref_sorted_array_length(h), uncompressed=out, at=[R.ref_sorted_array_at(h, int(i)) for i in at],
                 index_of=[R.ref_sorted_array_index_of(h, int(vals[i])) for i in at],
                 index_of_absent=R.ref_sorted_array_index_of(h, int(vals[-1]) + 1))
        idx = np.zeros(300, np.uint32)
        R.ref_sorted_array_bulk_index_of(h, ol.p32(probe), 300, ol.p32(idx))
        r["bulk_index_of"] = idx
        # out-of-order append re-encodes (src/sorted_array.cpp:24-43)
        R.ref_sorted_array_append(h, int(vals[10]) + 1) if vals[10] + 1 != vals[11] else None
        R.ref_sorted_array_remove_value(h, int(vals[0]))
        r["at0_after_remove"] = R.ref_sorted_array_at(h, 0)
        R.ref_sorted_array_free(h)
        return r

    def array():
        R = ol.ref()
        a = C.c_void_p(R.ref_array_new())
        for v in uns:
            R.ref_array_append(a, int(v))
        r = dict(length=R.ref_array_length(a), at=[R.ref_array_at(a, int(i)) for i in uat])
        R.ref_array_remove_index(a, 10, 20)
        r["at10_after_remove"] = R.ref_array_at(a, 10)
        R.ref_array_free(a)
        return r

    with ref_answers("containers_pin_libfor_port") as ref:
        s, a = ref(sorted_array), ref(array)
    assert s["length"] == len(vals)
    assert s["uncompressed"] == vals.tolist()
    assert s["at"] == vals[at].tolist() and s["index_of"] == at.tolist()
    assert s["index_of_absent"] == len(vals)
    assert (vals[s["bulk_index_of"]] == probe).all()
    assert s["at0_after_remove"] == vals[1]
    assert a["length"] == len(uns)
    assert a["at"] == uns[uat].tolist()
    assert a["at10_after_remove"] == uns[20]


@pytest.mark.parametrize("seed", range(4))
def test_ref_intersect_merge_random(seed):
    rng = np.random.default_rng(seed)
    k = int(rng.integers(2, 5))
    lists = [np.unique(rng.integers(0, 3000, int(rng.integers(1, 1500)))).tolist() for _ in range(k)]
    block = int(rng.choice([2, 8, 256]))

    with ref_answers(f"intersect_merge_random[{seed}]") as ref:
        assert ref.same(tso_intersect(lists), lambda: ref_call(ol.ref().ref_plist_intersect, ref_lists(lists, block=block), 4000))
        rm = ref(lambda: ref_call(ol.ref().ref_plist_merge, ref_lists(lists, block=block), 8000))
    # posting_list_t::merge for k >= 3 drains the surviving iterators one after another once the first list ends
    # (src/posting_list.cpp:698-703), so its tail is neither sorted nor unique; production only calls merge with a
    # single list (src/index.cpp:3339, src/art.cpp:960). The oracle states the intended unique ascending union.
    assert tso_merge(lists) == (rm if k <= 2 else sorted(set(rm)))


def test_ref_array_utils_random():
    L = ol.oracle()
    rng = np.random.default_rng(3)

    def run_ref(name, a0, na, b0, nb):
        o1 = np.zeros(na + nb + 1, np.uint32)
        n1 = getattr(ol.ref(), "ref_" + name)(ol.p32(a0), na, ol.p32(b0), nb, ol.p32(o1))
        return o1[:n1]
    with ref_answers("array_utils_random") as ref:
        for _ in range(20):
            a = np.unique(rng.integers(0, 500, int(rng.integers(0, 300)))).astype(np.uint32)
            b = np.unique(rng.integers(0, 500, int(rng.integers(0, 300)))).astype(np.uint32)
            a0 = a if len(a) else np.zeros(1, np.uint32)
            b0 = b if len(b) else np.zeros(1, np.uint32)
            for name in ("and_scalar", "or_scalar", "exclude_scalar"):
                o2 = np.zeros(len(a) + len(b) + 1, np.uint32)
                n2 = getattr(L, "tso_" + name)(ol.p32(a0), len(a), ol.p32(b0), len(b), ol.p32(o2))
                assert ref.same(o2[:n2], lambda: run_ref(name, a0, len(a), b0, len(b))), name


def test_ref_match_fuzz():
    rng = np.random.default_rng(11)
    with ref_answers("match_fuzz") as ref:
        _match_fuzz(rng, ref)


def _match_fuzz(rng, ref):
    for it in range(3000):
        nt = int(rng.integers(1, 13))
        span = int(rng.choice([12, 40, 300, 70000]))
        toks = []
        for _ in range(nt):
            n = int(rng.integers(1, 6))
            p = np.sort(rng.choice(min(span, 65000), n, replace=False)).tolist()
            toks.append(p)
        if it % 5 == 0 and nt > 1:            # duplicate query token: identical position lists
            toks[1] = list(toks[0])
        last = (rng.random(nt) < 0.3).astype(int).tolist()
        for ce in (0, 1):
            assert _match(ol.oracle().tso_match, toks, last, ce) == ref(lambda: _match(ol.ref().ref_match, toks, last, ce)), (toks, last, ce)
        assert _phrase(ol.oracle().tso_has_phrase_match, toks) == ref(lambda: _phrase(ol.ref().ref_has_phrase_match, toks))


def _ref_combo(fields, b: S.KwBatch, q, c, block=256, use_fit=0, filters=()):
    """One combination through the reference's or_iterator_t::intersect + reference-typed scoring glue."""
    R = ol.ref()
    F = b.n_fields
    r0, r1 = int(b.c_tok_off[c]), int(b.c_tok_off[c + 1])
    n_req = int(b.c_n_required[c])
    keep, handles = [], []
    for r in range(r0, r1):
        for f in range(F):
            li = int(b.t_list[r * F + f])
            if li == S.NO_LIST:
                handles.append(None)
            else:
                pl = ol.ref_plists_of(fields[int(b.field_ids[f])], [li], block)[0]
                keep.append(pl)
                handles.append(pl.h)
    P = ol.RefParams()
    P.n_tokens, P.n_dropped, P.n_fields = n_req, (r1 - r0) - n_req, F
    P.total_cost = int(b.c_total_cost[c])
    P.num_query_tokens = int(b.q_num_query_tokens[q])
    P.syn_orig_num_tokens, P.orig_num_tokens = int(b.c_syn[c]), int(b.c_orig[c])
    P.is_synonym_query = int(bool(b.c_flags[c] & S.CFLAG_SYNONYM))
    P.demote_synonym_match = int(bool(b.c_flags[c] & S.CFLAG_DEMOTE_SYNONYM))
    fl = int(b.q_flags[q])
    P.prioritize_exact_match = int(bool(fl & 1))
    P.prioritize_token_position = int(bool(fl & 2))
    P.prioritize_num_matching_fields = int(bool(fl & 4))
    P.match_type = int(b.q_match_type[q])
    for f in range(F):
        P.field_weight[f] = int(b.q_field_weight[q * F + f])
        P.field_is_array[f] = int(fields[int(b.field_ids[f])].is_array)
    hs = (C.c_void_p * len(handles))(*handles)
    excl = b.excl_ids[int(b.q_excl_off[q]):int(b.q_excl_off[q + 1])]
    excl0 = np.ascontiguousarray(excl) if len(excl) else np.zeros(1, np.uint32)
    fs = int(b.q_filter[q])
    filt = np.asarray(filters[fs], np.uint32) if fs >= 0 else np.zeros(0, np.uint32)
    filt0 = filt if len(filt) else np.zeros(1, np.uint32)
    cap = 1 << 20
    ids = np.zeros(cap, np.uint32)
    sc = np.zeros(cap, np.uint64)
    nkm = C.c_uint64(0)
    n = R.ref_keyword_combo(C.byref(P), hs, ol.p32(excl0), len(excl), ol.p32(filt0), len(filt), use_fit,
                            ol.p32(ids), sc.ctypes.data_as(S.u64p), cap, C.byref(nkm))
    return ids[:n].copy(), sc[:n].copy(), nkm.value


def random_batch(rng, fields, n_queries, filters=(), max_tokens=4, dropped=True):
    """Random resolved queries over the given FieldData list (tokens drawn from real docs so they co-occur)."""
    F = len(fields)
    qs = []
    for _ in range(n_queries):
        combos = []
        base = fields[int(rng.integers(0, F))]
        nt = int(rng.integers(1, max_tokens + 1))
        toks = synth.sample_queries(base, 1, nt, int(rng.integers(0, 1 << 30)))[0].tolist() if nt <= 4 else None
        for _c in range(int(rng.integers(1, 4))):
            rows = []
            ctoks = list(toks)
            if _c > 0:
                ctoks[int(rng.integers(0, nt))] = int(rng.integers(0, 50))      # a "typo candidate": another frequent token
            for t in ctoks:
                row = []
                for f in range(F):
                    fl = fields[f].flat
                    present = t < fl.n_lists and fl.df(t) > 0 and rng.random() < 0.9
                    row.append(t if present else S.NO_LIST)
                if all(x == S.NO_LIST for x in row):
                    row[0] = t if fields[0].flat.df(t) > 0 else S.NO_LIST
                rows.append(row)
            nreq = len(rows)
            if dropped and rng.random() < 0.3:
                dt = int(rng.integers(0, 30))
                rows.append([dt if fields[f].flat.df(dt) > 0 else S.NO_LIST for f in range(F)])
            combos.append(S.Combo(rows, nreq, total_cost=int(rng.integers(0, 3)) * (1 if _c else 0)))
        flags = int(rng.integers(0, 8))
        q = S.Query(combos, topk=int(rng.choice([1, 7, 50, 250])), flags=flags, match_type=int(rng.integers(0, 3)),
                    num_query_tokens=nt,
                    field_weight=[int(x) for x in rng.integers(1, 16, F)],
                    sort=((S.SORT_TEXT_MATCH, -1, 1, 0), (S.SORT_NUMERIC, 0, int(rng.choice([1, -1])), int(rng.integers(0, 2))),
                          (S.SORT_SEQ_ID, -1, int(rng.choice([1, -1])), 0)))
        if filters and rng.random() < 0.5:
            q.filter = int(rng.integers(0, len(filters)))
        if rng.random() < 0.3:
            q.excl = np.unique(rng.integers(0, 4000, 40)).tolist()
        qs.append(q)
    return S.KwBatch(qs, list(range(F)), filters)


@pytest.fixture(scope="module")
def small_collection():
    n_docs = 4000
    f0 = synth.make_string_field(n_docs, 300, 3, 10, seed=1)
    f1 = synth.make_array_field(n_docs, 300, 1, 3, 1, 5, seed=2)
    f2 = synth.make_string_field(n_docs, 300, 1, 4, seed=3)
    pts = synth.make_points(n_docs, 9, hi=50, missing_frac=0.05)
    return n_docs, [f0, f1, f2], pts


@pytest.mark.parametrize("seed", range(3))
def test_ref_keyword_combo_random(small_collection, seed):
    n_docs, fds, pts = small_collection
    rng = np.random.default_rng(100 + seed)
    filters = [np.unique(rng.integers(0, n_docs, 1500)).astype(np.uint32), np.arange(0, n_docs, 7, dtype=np.uint32),
               np.asarray([5], np.uint32)]
    flats = [fd.flat for fd in fds]
    ix = ol.OracleIndex(n_docs, flats, [pts])
    b = random_batch(rng, fds, 25, filters)
    total = 0
    with ref_answers(f"keyword_combo_random[{seed}]") as ref:
        for q in range(b.n_queries):
            for c in range(int(b.q_combo_off[q]), int(b.q_combo_off[q + 1])):
                ids, sc, nkm = ix.keyword_combo(b, q, c)
                for use_fit in (0, 1):
                    block = int(rng.choice([4, 256]))
                    assert ref.same([ids, sc], lambda: _ref_combo(flats, b, q, c, block=block, use_fit=use_fit, filters=filters)[:2]), (q, c, use_fit)
                total += len(ids)
    assert total > 100


def test_ref_or_iterator_kat():
    with ref_answers("or_iterator_kat") as ref:
        _or_iterator_kat(ref)


def _or_iterator_kat(ref):
    for case in KAT["or_iterator"]:
        toks = case["tokens"]
        F = max(len(t) for t in toks)
        # each sub-list becomes one "field" list of its token row
        per_field = [[] for _ in range(F)]
        rows = []
        for t in toks:
            row = []
            for f in range(F):
                if f < len(t):
                    per_field[f].append([(i, case["offsets"]) for i in t[f]])
                    row.append(len(per_field[f]) - 1)
                else:
                    row.append(S.NO_LIST)
            rows.append(row)
        flats = [S.FlatField.from_postings(pf) for pf in per_field]
        filters = [np.asarray(case["filter"], np.uint32)] if case["filter"] else []
        q = S.Query([S.Combo(rows, len(rows))], filter=0 if filters else -1)
        b = S.KwBatch([q], list(range(F)), filters)
        ix = ol.OracleIndex(100000, flats, [])
        ids, _, _ = ix.keyword_combo(b, 0, 0)
        assert ids.tolist() == case["expect"]
        rids = ref(lambda: _ref_combo(flats, b, 0, 0, block=2, filters=filters)[0])
        assert rids == case["expect"]


def test_ref_phrase_matches(small_collection):
    n_docs, fds, _ = small_collection
    with ref_answers("phrase_matches") as ref:
        hits = _phrase_matches(n_docs, fds, ref)
    assert hits > 10


def _ref_matches(fn_name, fd, lists, ids):
    k = len(lists)
    pls = ol.ref_plists_of(fd.flat, lists.tolist(), 256)
    hs = (C.c_void_p * k)(*[p.h for p in pls])
    rout = np.zeros(len(ids), np.uint32)
    rn = getattr(ol.ref(), fn_name)(hs, k, int(fd.flat.is_array), ol.p32(ids), len(ids), ol.p32(rout))
    return rout[:rn]


def _phrase_matches(n_docs, fds, ref):
    L = ol.oracle()
    rng = np.random.default_rng(77)
    hits = 0
    for fi in (0, 1):
        fd = fds[fi]
        ix = ol.OracleIndex(n_docs, [fd.flat], [])
        for _ in range(40):
            # consecutive tokens of a real doc => phrase present at least there
            d = int(rng.integers(0, n_docs))
            a, e = int(fd.doc_off[d]), int(fd.doc_off[d + 1])
            if e - a < 2:
                continue
            k = int(rng.integers(2, min(4, e - a) + 1))
            s = int(rng.integers(a, e - k + 1))
            lists = fd.doc_tok[s:s + k].astype(np.uint32)
            cand = tso_intersect([fd.flat.ids[int(fd.flat.list_off[l]):int(fd.flat.list_off[l + 1])] for l in lists])
            if not cand:
                continue
            ids = np.asarray(cand, np.uint32)
            out = np.zeros(len(ids), np.uint32)
            n = L.tso_phrase_matches(ix.h, 0, ol.p32(np.ascontiguousarray(lists)), k, ol.p32(ids), len(ids), ol.p32(out))
            assert ref.same(out[:n], lambda: _ref_matches("ref_plist_phrase_matches", fd, lists, ids))
            hits += n
    return hits


def test_ref_exact_and_prefix_matches(small_collection):
    """get_exact_matches / get_prefix_matches (src/posting_list.cpp:1129-1452): oracle restatement vs the reference's own
    compiled code, plain and array fields."""
    from test_hostsim import idset_cases
    n_docs, fds, _ = small_collection
    L = ol.oracle()
    rng = np.random.default_rng(91)
    hits = {"exact": 0, "prefix": 0}
    with ref_answers("exact_and_prefix_matches") as ref:
        for fi in (2, 1, 0):
            fd = fds[fi]
            ix = ol.OracleIndex(n_docs, [fd.flat], [])
            for lists, ids in idset_cases(rng, fd, 120):
                k = len(lists)
                for name, ofn, rfn in (("exact", L.tso_exact_matches, "ref_plist_exact_matches"),
                                       ("prefix", L.tso_prefix_matches, "ref_plist_prefix_matches")):
                    out = np.zeros(len(ids), np.uint32)
                    n = ofn(ix.h, 0, ol.p32(lists), k, ol.p32(ids), len(ids), ol.p32(out))
                    assert ref.same(out[:n], lambda: _ref_matches(rfn, fd, lists, ids)), (fi, name, lists.tolist())
                    hits[name] += n
    assert hits["exact"] > 20 and hits["prefix"] > 40, hits


def test_kat_array_utils():
    """test/array_utils_test.cpp literal vectors: oracle restatement (and the reference's own code when present)."""
    fams = [("tso_", ol.oracle())] + ([("ref_", ol.ref())] if ol.have_ref() else [])
    names = ("and_scalar", "or_scalar", "exclude_scalar")
    for case in KAT["array_utils"]:
        a = np.asarray(case["a"], np.uint32); b = np.asarray(case["b"], np.uint32)
        a0 = a if len(a) else np.zeros(1, np.uint32)
        b0 = b if len(b) else np.zeros(1, np.uint32)
        for pre, lib in fams:
            out = np.zeros(len(a) + len(b) + 1, np.uint32)
            n = getattr(lib, pre + names[case["op"]])(ol.p32(a0), len(a), ol.p32(b0), len(b), ol.p32(out))
            assert out[:n].tolist() == case["expect"], (pre, case["src"])


# test/posting_list_test.cpp:823-859 (PostingListContainsAtleastOne): the literal cases, then random lists against the
# reference's compiled posting_list_t::contains_atleast_one
CONTAINS_KAT = [
    (list(range(20, 1000)), [200, 300], True), (list(range(20, 1000)), [200, 3000], True), (list(range(20, 1000)), [2000, 3000], False),
    (list(range(10, 20)), list(range(5, 1000)), True), (list(range(10, 20)), list(range(25, 1000)), False),
]


def _tso_contains(lst, targets):
    a, b = np.asarray(lst, np.uint32), np.asarray(targets, np.uint32)
    return bool(ol.oracle().tso_contains_atleast_one(ol.p32(a), len(a), ol.p32(b), len(b)))


@pytest.mark.parametrize("lst,targets,expect", CONTAINS_KAT)
def test_kat_contains_atleast_one(lst, targets, expect):
    assert _tso_contains(lst, targets) == expect
    if ol.have_ref():
        pls = ref_lists([lst], block=100 if len(lst) > 100 else 2)
        t = np.asarray(targets, np.uint32)
        assert bool(ol.ref().ref_plist_contains_atleast_one(pls[0].h, ol.p32(t), len(t))) == expect


def test_ref_contains_atleast_one_random():
    rng = np.random.default_rng(5)

    def run(lst, tg, block):
        pls = ref_lists([lst], block=block)
        return bool(ol.ref().ref_plist_contains_atleast_one(pls[0].h, ol.p32(tg), len(tg)))
    with ref_answers("contains_atleast_one_random") as ref:
        for _ in range(200):
            lst = np.unique(rng.integers(0, 3000, int(rng.integers(1, 400)))).tolist()
            tg = np.unique(rng.integers(0, 3000, int(rng.integers(1, 60)))).astype(np.uint32)
            block = int(rng.choice([2, 16, 256]))
            assert _tso_contains(lst, tg) == ref(lambda: run(lst, tg, block))
