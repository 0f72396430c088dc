"""SURVEY §8 f-4, posting half: tsgpu_index_append_lists / tsgpu_index_set_sort_values — the device side of posting_t::upsert / erase
(src/posting.cpp:247-333). A mirror that was loaded from an early state of a collection and then patched must answer exactly like a
mirror (and the oracle) loaded from the final state: same ids, scores, found — for inserted documents, updated documents (new offsets
under an old seq_id) and removed ones."""
import numpy as np
import pytest

import oracle_lib as ol
from typesense_b200 import capi, structs as S, synth

pytestmark = pytest.mark.gpu


def _lists_of(flat: S.FlatField):
    """per list: [(seq_id, [offsets])]"""
    out = []
    for l in range(flat.n_lists):
        a, b = int(flat.list_off[l]), int(flat.list_off[l + 1])
        out.append([(int(flat.ids[i]), flat.positions[int(flat.pos_off[i]):int(flat.pos_off[i + 1])].tolist()) for i in range(a, b)])
    return out


def _subset(lists, keep_doc):
    return [[p for p in pl if keep_doc(p[0])] for pl in lists]


@pytest.mark.parametrize("is_array", [False, True])
def test_patched_mirror_equals_fresh_mirror(is_array):
    n_docs, vocab = 6000, 400
    fd = synth.make_array_field(n_docs, vocab, 1, 3, 2, 5, seed=21) if is_array else synth.make_string_field(n_docs, vocab, 3, 9, seed=21)
    final_lists = _lists_of(fd.flat)
    L = len(final_lists)
    pts_final = synth.make_points(n_docs, 5)
    rng = np.random.default_rng(3)
    # state 0: documents < 4000 only, and 300 of them with other offsets (they will be "updated"), 200 extra documents that will be removed
    changed = set(rng.choice(4000, 300, replace=False).tolist())
    removed = set(rng.choice(np.arange(4000, 4500), 200, replace=False).tolist())

    def early(pl):
        out = []
        for sid, offs in pl:
            if sid < 4000 or sid in removed:
                o = list(offs)
                if sid in changed and not is_array and len(o) and o[0] > 1:
                    o[0] -= 1                                  # an older version of the document had the token one position earlier
                out.append((sid, o))
        return out
    lists0 = [early(pl) for pl in final_lists]
    # the final state has no `removed` documents
    final_lists = [[p for p in pl if p[0] not in removed] for pl in final_lists]
    flat0 = S.FlatField.from_postings(lists0, is_array)
    flat_final = S.FlatField.from_postings(final_lists, is_array)
    pts0 = pts_final.copy()
    pts0[4000:] = np.iinfo(np.int64).min
    gi = capi.GpuIndex(n_docs, 0)
    f = gi.load_field(flat0)
    col = gi.load_sort_column(pts0)
    # patch in two batches: every list whose content differs between state 0 and the final state is handed over in full
    touched = [l for l in range(L) if lists0[l] != final_lists[l]]
    assert len(touched) > L // 2
    remap = np.arange(L, dtype=np.int64)
    half = len(touched) // 2
    for part in (touched[:half], touched[half:]):
        delta = S.FlatField.from_postings([final_lists[l] for l in part], is_array)
        first = gi.append_lists(f, delta)
        for k, l in enumerate(part):
            remap[l] = first + k
    ids_new = np.arange(4000, n_docs, dtype=np.uint32)
    vals_new = pts_final[4000:].copy()
    vals_new[[i - 4000 for i in removed]] = np.iinfo(np.int64).min
    gi.set_sort_values(col, ids_new, vals_new)
    pts_expect = pts_final.copy()
    pts_expect[list(removed)] = np.iinfo(np.int64).min
    oi = ol.OracleIndex(n_docs, [flat_final], [pts_expect])
    gf = capi.GpuIndex(n_docs, 0)
    gf.load_field(flat_final); gf.load_sort_column(pts_expect)
    sort = ((S.SORT_TEXT_MATCH, -1, 1, 0), (S.SORT_NUMERIC, 0, 1, 0), (S.SORT_NONE, -1, 1, 0))
    df = np.diff(flat_final.list_off.astype(np.int64))
    live = np.nonzero(df > 0)[0]
    for seed in range(3):
        r = np.random.default_rng(100 + seed)
        qs_final, qs_patched = [], []
        for i in range(80):
            nt = int(r.integers(1, 4))
            toks = [int(t) for t in r.choice(live, nt, replace=False)]
            if i % 4 == 0:                                   # tokens of one document: guaranteed hits
                d = int(r.integers(0, n_docs))
                cand = [l for l in live[:200] if any(p[0] == d for p in final_lists[l])]
                if len(cand) >= nt:
                    toks = [int(t) for t in cand[:nt]]
            qs_final.append(S.Query([S.Combo([[t] for t in toks], nt)], topk=int(r.choice([10, 250])), sort=sort, num_query_tokens=nt))
            qs_patched.append(S.Query([S.Combo([[int(remap[t])] for t in toks], nt)], topk=qs_final[-1].topk, sort=sort, num_query_tokens=nt))
        bf, bp = S.KwBatch(qs_final, [0]), S.KwBatch(qs_patched, [0])
        okv, ocnt, ofound = oi.keyword_search(bf, 256)
        fkv, fcnt, ffound = gf.keyword_search(bf, 256)
        pkv, pcnt, pfound = gi.keyword_search(bp, 256)
        assert int(ocnt.sum()) > 50
        for kv, cnt, found in ((fkv, fcnt, ffound), (pkv, pcnt, pfound)):
            assert cnt.tolist() == ocnt.tolist() and found.tolist() == ofound.tolist()
            for q in range(len(cnt)):
                n = int(cnt[q])
                assert kv["key"][q, :n].tolist() == okv["key"][q, :n].tolist(), f"query {q}: ids"
                assert kv["scores"][q, :n].tolist() == okv["scores"][q, :n].tolist(), f"query {q}: scores"
                assert kv["text_match_score"][q, :n].tolist() == okv["text_match_score"][q, :n].tolist()
    # the id-set primitives follow the new lists too
    a, b = int(live[0]), int(live[1])
    assert gi.intersect(f, [int(remap[a]), int(remap[b])], n_docs).tolist() == gf.intersect(0, [a, b], n_docs).tolist()
    gi.close(); gf.close()


def test_append_lists_rejects_malformed_input():
    n_docs = 1000
    fd = synth.make_string_field(n_docs, 50, 3, 6, seed=2)
    gi = capi.GpuIndex(n_docs, 0)
    f = gi.load_field(fd.flat)
    bad = S.FlatField.from_postings([[(5, [1]), (3, [2])]])                      # not ascending
    with pytest.raises(capi.TsgpuError):
        gi.append_lists(f, bad)
    with pytest.raises(capi.TsgpuError):
        gi.append_lists(f, S.FlatField.from_postings([[(n_docs + 3, [1])]]))     # beyond the index's capacity
    with pytest.raises(capi.TsgpuError):
        gi.append_lists(f + 7, S.FlatField.from_postings([[(1, [1])]]))
    # the field is unchanged
    assert gi.intersect(f, [0], n_docs).tolist() == fd.flat.ids[int(fd.flat.list_off[0]):int(fd.flat.list_off[1])].tolist()
    gi.close()


@pytest.mark.skipif(__import__("os").environ.get("TSGPU_TEST_DOUBLE") != "1",
                    reason="a check of the DATA PATH reference posting_list_t -> mirror: runs in the dry run against the oracle double "
                           "(tests/test_gpu_tests_dryrun.py); the device side of the same calls is test_patched_mirror_equals_fresh_mirror")
def test_mirror_follows_the_reference_posting_lists():
    """The write side as the reference keeps it: one posting_list_t per token — the reference's OWN src/posting_list.cpp, compiled in
    oracle/_ref — receives posting_t::upsert / erase for every written document; after each batch of writes the touched tokens' lists
    are read back through the reference's iterator (what the binding of INTEGRATION.md §1 does) and handed to tsgpu_index_append_lists.
    The patched mirror must answer exactly like the oracle over the reference's lists as they stand. Each list read back must equal
    the list the writes describe, which is what the mirror is loaded with; without oracle/_ref that equality is checked against the
    reference's answers stored in tests/golden/ref_answers (oracle_lib.RefAnswers)."""
    with ol.RefAnswers("test_incremental_mirror", "reference_posting_lists") as ref:
        _mirror_follows_the_reference_posting_lists(ref)


def _mirror_follows_the_reference_posting_lists(ref):
    import ctypes as C
    R = ol.ref() if ref.live else None
    rng = np.random.default_rng(11)
    vocab, n_docs = 80, 3000
    zipf = np.arange(1, vocab + 1, dtype=np.float64) ** -1.0
    zipf /= zipf.sum()
    plists = [C.c_void_p(R.ref_plist_new(256)) for _ in range(vocab)] if ref.live else None
    doc_tokens, doc_offsets = {}, {}

    def offsets_of(tokens):
        """Index::tokenize_string (src/index.cpp:1323-1349): 1-based positions per token, a trailing 0 on the document's last token"""
        per = {}
        for pos, t in enumerate(tokens):
            per.setdefault(int(t), []).append(pos + 1)
        per[int(tokens[-1])].append(0)
        return per

    def write(doc, tokens, touched):
        if doc in doc_tokens:                                   # an update: Index::remove_field first
            for t in offsets_of(doc_tokens[doc]):
                if ref.live:
                    R.ref_plist_erase(plists[t], doc)
                touched.add(t)
        if tokens is None:
            doc_tokens.pop(doc, None)
            doc_offsets.pop(doc, None)
            return
        for t, offs in offsets_of(tokens).items():
            a = np.asarray(offs, np.uint32)
            if ref.live:
                R.ref_plist_upsert(plists[t], doc, ol.p32(a), len(a))
            touched.add(t)
        doc_tokens[doc] = tokens
        doc_offsets[doc] = offsets_of(tokens)

    def read_back(t):
        n = R.ref_plist_num_ids(plists[t])
        ids = np.zeros(n + 1, np.uint32); oi = np.zeros(n + 2, np.uint32); offs = np.zeros(8 * n + 16, np.uint32)
        k = R.ref_plist_dump(plists[t], ol.p32(ids), ol.p32(oi), ol.p32(offs), len(ids), len(offs))
        assert k == n
        return [(int(ids[i]), offs[int(oi[i]):int(oi[i + 1])].tolist()) for i in range(n)]

    def dump(t):
        want = [(d, per[t]) for d, per in sorted(doc_offsets.items()) if t in per]
        assert ref.same(want, lambda: read_back(t)), t
        return want

    def random_doc():
        return rng.choice(vocab, int(rng.integers(2, 7)), p=zipf).tolist()

    touched = set()
    for d in range(2000):
        write(d, random_doc(), touched)
    flat0 = S.FlatField.from_postings([dump(t) for t in range(vocab)])
    pts = synth.make_points(n_docs, 9)
    gi = capi.GpuIndex(n_docs, 0)
    f = gi.load_field(flat0)
    gi.load_sort_column(pts)
    remap = np.arange(vocab, dtype=np.int64)
    sort = ((S.SORT_TEXT_MATCH, -1, 1, 0), (S.SORT_NUMERIC, 0, 1, 0), (S.SORT_NONE, -1, 1, 0))

    def check(seed):
        final = S.FlatField.from_postings([dump(t) for t in range(vocab)])
        oi_ = ol.OracleIndex(n_docs, [final], [pts])
        live = [t for t in range(vocab) if final.df(t) > 0]
        r = np.random.default_rng(seed)
        qf, qp = [], []
        for _ in range(60):
            nt = int(r.integers(1, 4))
            toks = [int(t) for t in r.choice(live, nt, replace=False)]
            qf.append(S.Query([S.Combo([[t] for t in toks], nt)], topk=50, sort=sort, num_query_tokens=nt))
            qp.append(S.Query([S.Combo([[int(remap[t])] for t in toks], nt)], topk=50, sort=sort, num_query_tokens=nt))
        okv, ocnt, ofound = oi_.keyword_search(S.KwBatch(qf, [0]), 64)
        kv, cnt, found = gi.keyword_search(S.KwBatch(qp, [0]), 64)
        assert cnt.tolist() == ocnt.tolist() and found.tolist() == ofound.tolist() and int(ocnt.sum()) > 100
        for q in range(len(qf)):
            n = int(cnt[q])
            assert kv["key"][q, :n].tolist() == okv["key"][q, :n].tolist() and kv["scores"][q, :n].tolist() == okv["scores"][q, :n].tolist()

    check(1)
    for batch in range(3):
        touched = set()
        if batch == 0:
            for d in range(2000, 2600):                         # new documents
                write(d, random_doc(), touched)
        elif batch == 1:
            for d in rng.choice(2600, 150, replace=False):      # rewritten documents
                write(int(d), random_doc(), touched)
        else:
            for d in rng.choice(2600, 200, replace=False):      # removed documents
                write(int(d), None, touched)
        part = sorted(touched)
        first = gi.append_lists(f, S.FlatField.from_postings([dump(t) for t in part]))
        for k, t in enumerate(part):
            remap[t] = first + k
        check(10 + batch)
    if ref.live:
        for h in plists:
            R.ref_plist_free(h)
    gi.close()
