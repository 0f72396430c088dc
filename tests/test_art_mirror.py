"""SURVEY §8 f-1: the ART mirror (typesense_b200/host/art_mirror.hpp) against the reference's own src/art.cpp compiled in
oracle/_ref. A reference tree is filled with art_insert document by document (as the reference's tests index), exported
(ref_art_export) and loaded into the mirror; art_fuzzy_search_i and art_mirror_t::fuzzy_search must then return the SAME
tokens in the SAME order — typos 0..2, prefix and whole-word search, both token orders, max_words truncation, pre-excluded
tokens, the previous-token restriction and a filter; ties included. A second check covers the mirror BUILT from a
vocabulary (no live tree): same candidates up to the order of equal-score tokens. Without oracle/_ref the reference's exported
trees and answers come from tests/golden/ref_answers (oracle_lib.RefAnswers)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as ol
import refflow

ROOT = ol.ROOT
SO = os.path.join(ROOT, "tests", "cpp", "libartmirror.so")


@pytest.fixture(scope="module")
def am():
    src = os.path.join(ROOT, "tests", "cpp", "art_mirror_capi.cpp")
    hdr = os.path.join(ROOT, "typesense_b200", "host", "art_mirror.hpp")
    if not os.path.exists(SO) or max(os.path.getmtime(src), os.path.getmtime(hdr)) > os.path.getmtime(SO):
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", src, "-o", SO])
    L = C.CDLL(SO)
    vp = C.c_void_p
    L.am_load.restype = vp
    L.am_load.argtypes = [C.c_char_p, C.c_size_t]
    L.am_build.restype = vp
    L.am_build.argtypes = [C.c_char_p, C.POINTER(C.c_int64), ol.u32p, C.c_uint32]
    L.am_free.argtypes = [vp]
    L.am_bind.argtypes = [vp, C.c_char_p, C.POINTER(C.c_uint64), ol.u32p]
    L.am_num_nodes.restype = C.c_size_t
    L.am_num_nodes.argtypes = [vp]
    L.am_num_leaves.restype = C.c_size_t
    L.am_num_leaves.argtypes = [vp]
    L.am_fuzzy.restype = C.c_size_t
    L.am_fuzzy.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_char_p, ol.u32p, C.c_size_t, C.c_int, C.c_char_p,
                           C.c_char_p, C.c_size_t]
    return L


def rand_word(rng, alpha, lo, hi):
    return "".join(rng.choice(list(alpha), int(rng.integers(lo, hi))))


def make_collection(rng, trial):
    alpha = ["abcde", "abcdefghij", "ab", "abcdefghijklmnopqrstuvwxyz"][trial % 4]
    n_words = int(rng.integers(5, 160)) if trial % 6 != 5 else int(rng.integers(800, 2500))     # large: 48/256-way nodes, deep heaps
    words = {rand_word(rng, alpha, 1, 8) for _ in range(n_words)}
    if trial % 3 == 0:            # long shared prefixes: compressed paths beyond the 8 stored bytes
        stem = rand_word(rng, alpha, 9, 14)
        words |= {stem + rand_word(rng, alpha, 1, 5) for _ in range(12)} | {stem}
    words = sorted(words)
    n_docs = int(rng.integers(5, 80)) if n_words < 800 else int(rng.integers(300, 900))
    docs = [{"title": " ".join(rng.choice(words, int(rng.integers(1, 9)))), "points": int(rng.integers(0, 40))} for _ in range(n_docs)]
    return refflow.Collection(docs)


def ref_tree(R, coll):
    t = R.ref_art_new()
    fl = coll.flat
    order = np.argsort(fl.ids, kind="stable")               # document by document, as Collection::add does
    post_list = np.repeat(np.arange(len(fl.list_off) - 1), np.diff(fl.list_off.astype(np.int64)))
    toks = {l: t_ for t_, l in coll.vocab.items()}
    for i in order:
        sid = int(fl.ids[i])
        offs = np.ascontiguousarray(fl.positions[int(fl.pos_off[i]):int(fl.pos_off[i + 1])], np.uint32)
        R.ref_art_insert(t, toks[int(post_list[i])].encode(), sid, int(coll.points[sid]), ol.p32(offs), len(offs))
    return t


def export(R, t):
    n = R.ref_art_export(t, None, 0)
    buf = C.create_string_buffer(n)
    assert R.ref_art_export(t, buf, n) == n
    return buf.raw


def stored_export(ref, t):
    """the reference tree's export, through the stored answers (hex text)"""
    return bytes.fromhex(ref(lambda: export(ol.ref(), t).hex()))


def ref_answers(name):
    return ol.RefAnswers("test_art_mirror", name)


def bind(am, h, coll):
    toks = sorted(coll.vocab, key=coll.vocab.get)
    lo = np.ascontiguousarray(coll.flat.list_off, np.uint64)
    ids = np.ascontiguousarray(coll.flat.ids, np.uint32)
    am.am_bind(h, "\n".join(toks).encode(), lo.ctypes.data_as(C.POINTER(C.c_uint64)), ol.p32(ids))
    return lo, ids          # keep alive


def queries(rng, coll, n):
    vw = list(coll.vocab)
    alpha = sorted({ch for w in vw for ch in w})
    for _ in range(n):
        term = str(rng.choice(vw)) if rng.random() < 0.7 else rand_word(rng, alpha, 1, 9)
        if rng.random() < 0.5 and len(term) > 1:
            i = int(rng.integers(0, len(term)))
            op = int(rng.integers(0, 4))
            if op == 0:
                term = term[:i] + term[i + 1:]
            elif op == 1:
                term = term[:i] + str(rng.choice(alpha)) + term[i:]
            elif op == 2:
                term = term[:i] + str(rng.choice(alpha)) + term[i + 1:]
            elif i + 1 < len(term):
                term = term[:i] + term[i + 1] + term[i] + term[i + 2:]
        if rng.random() < 0.4:
            term = term[:max(1, int(rng.integers(1, len(term) + 1)))]
        if not term:
            continue
        excl = sorted({str(x) for x in rng.choice(vw, int(rng.integers(1, 4)))}) if rng.random() < 0.3 else []
        prev = str(rng.choice(vw)) if rng.random() < 0.3 else ""
        filt = np.unique(rng.integers(0, coll.n_docs, int(rng.integers(1, coll.n_docs)))).astype(np.uint32) if rng.random() < 0.25 else None
        yield dict(term=term, cost=int(rng.integers(0, 3)), prefix=int(rng.integers(0, 2)), order=int(rng.integers(0, 2)),
                   max_words=int(rng.choice([1, 2, 4, 10, 100])), excl=excl, prev=prev, filt=filt)


def run_ref(R, t, q):
    buf = C.create_string_buffer(1 << 16)
    f = q["filt"]
    R.ref_art_fuzzy(t, q["term"].encode(), q.get("min_cost", q["cost"]), q["cost"], q["max_words"], q["order"], q["prefix"], 1 if q["prev"] else 0, q["prev"].encode(),
                    ol.p32(f) if f is not None else None, 0 if f is None else len(f), 0 if f is None else 1, "\n".join(q["excl"]).encode(), buf, len(buf))
    return [x for x in buf.value.decode().split("\n") if x]


def run_am(am, h, q):
    buf = C.create_string_buffer(1 << 16)
    f = q["filt"]
    am.am_fuzzy(h, q["term"].encode(), q.get("min_cost", q["cost"]), q["cost"], q["max_words"], q["order"], q["prefix"], q["prev"].encode(),
                ol.p32(f) if f is not None else None, 0 if f is None else len(f), 0 if f is None else 1, "\n".join(q["excl"]).encode(), buf, len(buf))
    return [x for x in buf.value.decode().split("\n") if x]


def test_loaded_mirror_returns_the_references_candidates_in_order(am):
    rng = np.random.default_rng(77)
    n = hits = 0
    with ref_answers("loaded_mirror") as ref:
        for trial in range(48):
            coll = make_collection(rng, trial)
            t = ref_tree(ol.ref(), coll) if ref.live else None
            blob = stored_export(ref, t)
            h = am.am_load(blob, len(blob))
            assert h, "export did not parse"
            assert am.am_num_leaves(h) == len(coll.vocab)
            keep = bind(am, h, coll)
            for q in queries(rng, coll, 80):
                got = run_am(am, h, q)
                assert ref.same(got, lambda: run_ref(ol.ref(), t, q)), (trial, {k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in q.items()}, got)
                n += 1
                hits += len(got)
            am.am_free(h)
            if ref.live:
                ol.ref().ref_art_free(t)
            del keep
    assert n > 3000 and hits > 4000, (n, hits)


def test_reference_fixture_tokens(am):
    """test/documents.jsonl (the collection_test.cpp fixture): prefix / typo candidates of the scenario queries."""
    coll = refflow.Collection.from_jsonl(os.path.join(ROOT, "tests", "golden", "documents.jsonl"))
    with ref_answers("fixture_tokens") as ref:
        t = ref_tree(ol.ref(), coll) if ref.live else None
        blob = stored_export(ref, t)
        h = am.am_load(blob, len(blob))
        keep = bind(am, h, coll)
        for term, cost, prefix in [("loox", 1, 0), ("lau", 0, 1), ("launch", 0, 0), ("rocket", 1, 0), ("ro", 0, 1), ("t", 0, 1), ("kind", 1, 1),
                                   ("the", 0, 0), ("laun", 1, 1), ("ex", 0, 1), ("what", 0, 1), ("rokket", 2, 0), ("lauch", 1, 0)]:
            for order in (0, 1):
                q = dict(term=term, cost=cost, prefix=prefix, order=order, max_words=4, excl=[], prev="", filt=None)
                assert run_am(am, h, q) == ref(lambda: run_ref(ol.ref(), t, q)), q
        q = dict(term="loox", cost=1, prefix=0, order=0, max_words=4, excl=[], prev="", filt=None)
        assert ref(lambda: run_ref(ol.ref(), t, q)) == ["look", "loop"]            # QueryWithTypo's candidates, most frequent first
        am.am_free(h)
        if ref.live:
            ol.ref().ref_art_free(t)
        del keep


def test_built_mirror_matches_up_to_tie_order(am):
    """No live tree to export (this repository's harness): the mirror built from the vocabulary finds the same candidates;
    tokens of equal rank may come in another order (the reference's inner-node scores depend on its insertion history)."""
    with ref_answers("built_mirror") as ref:
        _built_mirror_matches(am, ref)


def _built_mirror_matches(am, ref):
    rng = np.random.default_rng(5)
    n = 0
    for trial in range(20):
        coll = make_collection(rng, trial)
        t = ref_tree(ol.ref(), coll) if ref.live else None
        toks = sorted(coll.vocab, key=coll.vocab.get)
        fl = coll.flat
        df = np.diff(fl.list_off.astype(np.int64)).astype(np.uint32)
        ms = np.asarray([max(int(coll.points[int(i)]) for i in fl.ids[int(fl.list_off[l]):int(fl.list_off[l + 1])]) for l in range(len(toks))], np.int64)
        h = am.am_build("\n".join(toks).encode(), ms.ctypes.data_as(C.POINTER(C.c_int64)), ol.p32(df), len(toks))
        keep = bind(am, h, coll)
        rank = [dict(zip(toks, df.tolist())), dict(zip(toks, ms.tolist()))]
        for q in queries(rng, coll, 60):
            q["max_words"] = 100000               # truncation would make membership depend on the tie order
            got = run_am(am, h, q)
            assert ref.same(sorted(got), lambda: sorted(run_ref(ol.ref(), t, q))), (trial, q, got)
            exact_first = q["cost"] == 0 and q["term"] in coll.vocab and q["term"] not in q["excl"]
            body = got[1:] if exact_first and got and got[0] == q["term"] else got
            ranks = [rank[q["order"]][x] for x in body]
            assert ranks == sorted(ranks, reverse=True), (trial, q, got)
            n += 1
        am.am_free(h)
        if ref.live:
            ol.ref().ref_art_free(t)
        del keep
    assert n > 800


# ---- the reference's own ART tests (test/art_test.cpp) with inline keys or the two small word lists it ships
class _RefTree:
    """a reference tree (live only) and its export (live or stored)"""

    def __init__(self, ref, keys, scores=None):
        self.t = _tree_of(ol.ref(), keys, scores) if ref.live else None
        self.blob = stored_export(ref, self.t)

    def free(self):
        if self.t is not None:
            ol.ref().ref_art_free(self.t)


def _tree_of(R, keys, scores=None):
    """art_insert(key, get_document(id)): id = score = position (1-based) unless scores are given (art_test.cpp:18-21)."""
    t = R.ref_art_new()
    off = np.zeros(1, np.uint32)
    for i, k in enumerate(keys):
        kb = k if isinstance(k, bytes) else k.encode()
        R.ref_art_insert(t, kb, i + 1 if scores is None else i, (i + 1) if scores is None else scores[i], ol.p32(off), 1)
    return t


def _both(ref, am, tree, term, lo, hi, max_words, order, prefix):
    h = am.am_load(tree.blob, len(tree.blob))
    assert h
    tb = term if isinstance(term, bytes) else term.encode()

    def fuzzy(fn, handle, *rest):
        buf = C.create_string_buffer(1 << 16)
        fn(handle, tb, lo, hi, max_words, order, prefix, *rest, buf, len(buf))
        return [x.decode() for x in buf.value.split(b"\n") if x]
    want = ref(lambda: fuzzy(ol.ref().ref_art_fuzzy, tree.t, 0, b"", None, 0, 0, b""))
    got = fuzzy(am.am_fuzzy, h, b"", None, 0, 0, b"")
    am.am_free(h)
    assert want == got, (term, lo, hi, want, got)
    return got


def test_reference_art_tests(am):
    with ref_answers("reference_art_tests") as ref:
        _reference_art_tests(am, ref)


def _reference_art_tests(am, ref):
    FREQ, SCORE = 0, 1
    # test_art_fuzzy_search_single_leaf :579
    t = _RefTree(ref, ["implement"])
    assert len(_both(ref, am, t, "implement", 0, 0, 10, FREQ, 0)) == 1
    assert len(_both(ref, am, t, "implment", 0, 0, 10, FREQ, 0)) == 0
    assert len(_both(ref, am, t, "implment", 0, 1, 10, FREQ, 0)) == 1
    assert len(_both(ref, am, t, "implwnent", 0, 2, 10, FREQ, 0)) == 1
    t.free()
    # test_art_fuzzy_search_single_leaf_prefix :617
    t = _RefTree(ref, ["application"])
    assert len(_both(ref, am, t, "aplication", 0, 1, 10, FREQ, 1)) == 1
    assert len(_both(ref, am, t, "aplication", 0, 2, 10, FREQ, 1)) == 1
    t.free()
    # ..._qlen_greater_than_key :643, ..._non_prefix :661, test_art_prefix_larger_than_key :684
    t = _RefTree(ref, ["storka"])
    assert _both(ref, am, t, "starkbin", 0, 2, 10, FREQ, 1) == []
    t.free()
    t = _RefTree(ref, ["spz005"])
    assert _both(ref, am, t, "spz", 0, 1, 10, FREQ, 0) == []
    assert _both(ref, am, t, "spz", 0, 1, 10, FREQ, 1) == ["spz005"]
    t.free()
    t = _RefTree(ref, ["arvin"])
    assert _both(ref, am, t, "earrings", 0, 2, 10, FREQ, 0) == []
    t.free()
    # test_art_fuzzy_search_prefix_token_ordering :702 — score = 12 - i; the exact token comes first
    keys = ["enter", "elephant", "enamel", "ercot", "enyzme", "energy", "epoch", "epyc", "express", "everest", "end", "e"]
    t = _RefTree(ref, keys, scores=[len(keys) - i for i in range(len(keys))])
    assert _both(ref, am, t, "e", 0, 0, 3, SCORE, 1) == ["e", "enter", "elephant"]
    assert _both(ref, am, t, "enter", 1, 1, 3, SCORE, 1) == []
    t.free()
    # test_art_fuzzy_search_unicode_chars :864
    keys = ["роман", "обладать", "роисхождения", "без", "பஞ்சமம்", "சுதந்திரமாகவே", "அல்லது", "அடிப்படையில்"]
    t = _RefTree(ref, keys)
    for k in keys:
        assert _both(ref, am, t, k, 0, 0, 10, FREQ, 1) == [k]
    t.free()
    # test_art_fuzzy_search_extra_chars :891, roche_chews :1083, raspberry :1118, highliving :1152, ill_like_tokens2 :1035
    t = _RefTree(ref, ["abbviation"])
    assert len(_both(ref, am, t, "abbreviation", 0, 2, 10, FREQ, 1)) == 1
    t.free()
    t = _RefTree(ref, ["roche"])
    assert _both(ref, am, t, "chews", 0, 2, 10, FREQ, 1) == []
    assert _both(ref, am, t, "roche", 0, 0, 10, FREQ, 0) == ["roche"]
    assert _both(ref, am, t, "xxroche", 0, 2, 10, FREQ, 0) == ["roche"]
    t.free()
    t = _RefTree(ref, ["raspberry", "raspberries"])
    assert len(_both(ref, am, t, "raspberries", 0, 2, 10, FREQ, 1)) == 2
    assert len(_both(ref, am, t, "raspberry", 0, 2, 10, FREQ, 1)) == 2
    t.free()
    t = _RefTree(ref, ["highliving"])
    assert len(_both(ref, am, t, "higghliving", 0, 1, 10, FREQ, 0)) == 1
    assert len(_both(ref, am, t, "higghliving", 0, 2, 10, FREQ, 1)) == 1
    t.free()
    keys = ["input", "illustrations", "illustration"]
    t = _RefTree(ref, keys)
    for k in keys:
        assert len(_both(ref, am, t, k, 0, 0, 10, FREQ, 1)) == (2 if k == "illustration" else 1)
        assert _both(ref, am, t, k, 0, 0, 10, FREQ, 0) == [k]
    t.free()
    # test_art_search_sku_like_tokens :914 and test_art_search_ill_like_tokens :964 (test/skus.txt, test/ill.txt: byte copies in tests/golden)
    skus = [l.rstrip("\n") for l in open(os.path.join(ROOT, "tests", "golden", "art_skus.txt"))]
    t = _RefTree(ref, skus)
    for k in skus:
        assert _both(ref, am, t, k, 0, 0, 10, FREQ, 1) == [k]
        assert _both(ref, am, t, k, 0, 0, 10, FREQ, 0) == [k]
    t.free()
    ill = [l.rstrip("\n") for l in open(os.path.join(ROOT, "tests", "golden", "art_ill.txt"))]
    counts = {"input": 2, "illustration": 2, "image": 7, "instrument": 2, "in": 10, "info": 2, "inventor": 2, "imageresize": 2, "id": 5,
              "insect": 2, "ice": 2}
    t = _RefTree(ref, ill)
    for k in ill:
        got = _both(ref, am, t, k, 0, 0, 10, FREQ, 1)
        assert len(got) == counts.get(k, 1) and (k in counts or got == [k]), (k, got)
        assert _both(ref, am, t, k, 0, 0, 10, FREQ, 0) == [k]
    t.free()


def test_device_walk_function_equals_the_host_walk(am):
    """art_walk() of typesense_b200/csrc/art_device.cuh — the explicit-stack, fixed-size-row form the CUDA kernel runs per
    thread — compiled for the host: same hit list (same subtrees, same order) as art_mirror_t::walk_hits on random
    vocabularies, typos 0..2 (exact costs and ranges), prefix and whole-word searches."""
    am.am_walk.restype = C.c_size_t
    am.am_walk.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_size_t, C.POINTER(C.c_int)]
    rng = np.random.default_rng(909)
    n = n_hits = 0
    cap = 1 << 14
    a, b = np.zeros(cap, np.int32), np.zeros(cap, np.int32)
    so = C.c_int(0)
    for trial in range(36):
        coll = make_collection(rng, trial)
        toks = sorted(coll.vocab, key=coll.vocab.get)
        df = np.diff(coll.flat.list_off.astype(np.int64)).astype(np.uint32)
        ms = np.zeros(len(toks), np.int64)
        h = am.am_build("\n".join(toks).encode(), ms.ctypes.data_as(C.POINTER(C.c_int64)), ol.p32(df), len(toks))
        for q in queries(rng, coll, 70):
            lo = q["cost"] if rng.random() < 0.7 else int(rng.integers(0, q["cost"] + 1))
            na = am.am_walk(h, 0, q["term"].encode(), lo, q["cost"], q["prefix"], a.ctypes.data_as(C.POINTER(C.c_int32)), cap, C.byref(so))
            nb = am.am_walk(h, 1, q["term"].encode(), lo, q["cost"], q["prefix"], b.ctypes.data_as(C.POINTER(C.c_int32)), cap, C.byref(so))
            assert so.value == 0 and na == nb and a[:na].tolist() == b[:nb].tolist(), (trial, q["term"], lo, q["cost"], q["prefix"], na, nb)
            n += 1
            n_hits += na
        am.am_free(h)
    assert n > 2000 and n_hits > 3000, (n, n_hits)


def test_frontier_walk_with_preorder_ranks_equals_the_recursion(am):
    """The breadth-first form (art_enter() per frontier item, level by level — the shape of the parallel device walk) finds the
    same hits, and sorting them by the tree's static pre-order rank gives the recursion's order."""
    am.am_walk.restype = C.c_size_t
    am.am_walk.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_size_t, C.POINTER(C.c_int)]
    am.am_walk_frontier.restype = C.c_size_t
    am.am_walk_frontier.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_size_t)]
    rng = np.random.default_rng(31337)
    cap = 1 << 14
    a, b = np.zeros(cap, np.int32), np.zeros(cap, np.int32)
    so, lv, pk = C.c_int(0), C.c_int(0), C.c_size_t(0)
    n = n_hits = max_levels = 0
    for trial in range(30):
        coll = make_collection(rng, trial)
        toks = sorted(coll.vocab, key=coll.vocab.get)
        df = np.diff(coll.flat.list_off.astype(np.int64)).astype(np.uint32)
        ms = np.zeros(len(toks), np.int64)
        h = am.am_build("\n".join(toks).encode(), ms.ctypes.data_as(C.POINTER(C.c_int64)), ol.p32(df), len(toks))
        for q in queries(rng, coll, 60):
            if len(q["term"]) + (0 if q["prefix"] else 1) > 31:
                continue
            na = am.am_walk(h, 0, q["term"].encode(), q["cost"], q["cost"], q["prefix"], a.ctypes.data_as(C.POINTER(C.c_int32)), cap, C.byref(so))
            nb = am.am_walk_frontier(h, q["term"].encode(), q["cost"], q["cost"], q["prefix"], b.ctypes.data_as(C.POINTER(C.c_int32)), cap, C.byref(lv), C.byref(pk))
            assert na == nb and a[:na].tolist() == b[:nb].tolist(), (trial, q["term"], q["cost"], q["prefix"])
            n += 1
            n_hits += na
            max_levels = max(max_levels, lv.value)
        am.am_free(h)
    assert n > 1500 and n_hits > 2000 and max_levels >= 4, (n, n_hits, max_levels)
