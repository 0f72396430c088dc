#!/usr/bin/env python
"""bench.py — queries/sec of the Typesense query hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # CUDA path through the tsgpu C-ABI / the C++ host layer
    python bench.py --impl reference --gpus N --steps K ...  # the CPU implementation of the same path (same host layer over the oracle)

Workload (config.workload = "hybrid10m"): BASELINE.json configs[3] — 10 M docs, one `title` string field (Zipf 1.07 over 1 M words,
4-12 tokens), int64 `points`, int `cat` in [0,10) mirrored as 10 persistent filters, 10 M x 768 fp32 unit vectors with an HNSW graph
built BY THE LIBRARY on the device (hnswlib's insertion, M=16, ef_construction=200); a step is ONE multi_search request of 4096 hybrid
queries (3 terms, 30 % of the queries with one misspelt token, half with `cat:=c`, vector k=100 ef=100, alpha 0.3, sort _text_match
desc, points desc, Topster 250, 100 hits returned). Synthetic, seeded. Every rank holds a full replica; with N > 1 every rank answers
its slice of the SAME request and the slices' records are gathered by the library's NCCL exchange (strong scaling).

`value`  : queries/s of the device pipeline: the request's RESOLVED combinations, query vectors and result buffers resident in HBM, one
           tsgpu_hybrid_search_batch per step (wall clock of K steps, synchronised on both sides, max over ranks).
`e2e`    : the same metric end to end: query STRINGS in host memory -> C++ host layer (tokens, typo / prefix / drop-token control flow,
           candidate walks on the device ART) -> device rounds -> KV records in host memory; `--e2e-depth` requests in flight.
`roofline`: dominant kernel, algorithmic bytes / CUDA-event time measured inside the library on its own stream (isolated pass).
`cpu_baseline`: the same host layer over the CPU oracle (a port of the reference algorithm, see oracle/) on all host cores, bounded sample.
`other_configs`: BASELINE.json's other configurations + the tensor-core flat scan, measured next to the headline.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


_RESULT_FD = None


def claim_stdout():
    """stdout carries exactly one JSON line: libraries that print there (NCCL's version banner does) go to stderr."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, line)


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="tsgpu", choices=["tsgpu", "reference"])
    ap.add_argument("--docs", type=int, default=10_000_000)
    ap.add_argument("--vocab", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--cpu-sample", type=int, default=1024, help="queries per CPU-baseline sample")
    ap.add_argument("--workload", default="hybrid10m", choices=["hybrid10m", "keyword10m"])
    ap.add_argument("--recall-queries", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graph", default="hnsw", choices=["hnsw", "bulk"], help="hnsw: built by tsgpu_index_build_hnsw; bulk: r01's harness stand-in")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the secondary BASELINE.json configurations (other_configs)")
    ap.add_argument("--e2e-threads", type=int, default=32, help="host threads of one multi_search call's control-flow passes (capped at the core count)")
    ap.add_argument("--e2e-depth", type=int, default=6, help="multi_search calls in flight in the end-to-end leg (1 = strictly one after the other; measured best of 4 / 6 / 8 / 12 / 16: profiles/r02n_e2e_depth.md)")
    ap.add_argument("--no-graph-cache", action="store_true", help="always rebuild the HNSW graph (default: reuse /tmp/tsgpu_bench_cache)")
    ap.add_argument("--exp-sorted-vectors", action="store_true",
                    help="experiment only: store vectors in cluster order (seq_id locality) to measure what row locality is worth")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last timed step to DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, kv, cnt, found):
    """The results a caller of the timed path receives for its last step: per query its hit count and found count, per hit the
    fields of the KV record. Every array is float64 (vector_distance stays float32); int64 fields are split into exact high
    (signed) and low 32-bit halves, and records past a query's count are zeroed. Above DUMP_LIMIT bytes in all, a fixed, seeded
    sample of the queries is written; query_rows.npy names the rows written, in order."""
    nq, stride = kv.shape
    cnt = np.asarray(cnt, np.int64)
    kv = np.ascontiguousarray(kv).copy()
    kv.view(np.uint8).reshape(nq, stride, kv.dtype.itemsize)[np.arange(stride)[None, :] >= cnt[:, None]] = 0
    per_query = stride * 13 * 8 + 3 * 8
    rows = np.arange(nq)
    if nq * per_query > DUMP_LIMIT:
        rows = np.sort(np.random.default_rng(0).choice(nq, DUMP_LIMIT // per_query, replace=False))
    kv = kv[rows]
    f64 = lambda a: np.asarray(a, np.float64)
    arrays = {"query_rows": f64(rows), "count": f64(cnt[rows]), "found": f64(np.asarray(found)[rows]),
              "key": f64(kv["key"]), "distinct_key": f64(kv["distinct_key"]),
              "scores_hi": f64(kv["scores"] >> 32), "scores_lo": f64(kv["scores"] & 0xFFFFFFFF),
              "text_match_score_hi": f64(kv["text_match_score"] >> 32), "text_match_score_lo": f64(kv["text_match_score"] & 0xFFFFFFFF),
              "vector_distance": np.asarray(kv["vector_distance"], np.float32), "match_score_index": f64(kv["match_score_index"]),
              "query_index": f64(kv["query_index"])}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"outputs of the last timed step: {len(rows)} of {nq} queries, {sum(a.nbytes for a in arrays.values()) / 1e6:.1f} MB in {out_dir}")


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for l in self.lines:
            p = [x.strip() for x in l.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smax = float(p[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ workload
class Workload:
    pass


def build_workload(args, device, rank, need_host_copy):
    """Seeded synthetic collection. Returns host-side flat postings (always: the loader packs on the host and the
    oracle reads them) and device-side vectors/graph."""
    import torch
    from typesense_b200 import synth
    t0 = time.time()
    w = Workload()
    w.n_docs, w.dim = args.docs, args.dim
    fd = synth.make_string_field(args.docs, args.vocab, 4, 12, seed=7, device=device)
    w.fd = fd
    w.points = synth.make_points(args.docs, seed=13)
    g = torch.Generator(device="cpu"); g.manual_seed(17)
    w.cat = torch.randint(0, 10, (args.docs,), generator=g).numpy().astype(np.int32)
    w.filters = [np.nonzero(w.cat == c)[0].astype(np.uint32) for c in range(10)]
    w.words = synth.vocab_words(args.vocab)               # token rank -> its string (the host layer searches strings)
    log(f"rank{rank}: postings {len(fd.flat.ids)/1e6:.1f}M in {time.time()-t0:.1f}s")
    w.graph_host = None
    w.vec_dev = None
    if args.workload != "keyword10m":
        t1 = time.time()
        w.n_clusters = max(8, args.docs // 2000)
        vec, cid = synth.make_vectors_clustered(args.docs, args.dim, w.n_clusters, seed=1234, device=device, spread=0.35)
        if args.exp_sorted_vectors:
            perm = torch.argsort(cid)
            vec = vec[perm]; cid = cid[perm]
            del perm
        # brute-force ground truth for the recall report (outside every timed region)
        R = args.recall_queries
        w.recall_q = synth.make_vectors_clustered(R, args.dim, w.n_clusters, seed=555, device=device, centers_seed=1234, spread=0.35)[0] if R else None
        w.recall_exact = None
        if R:
            ex = torch.empty(R, 100, dtype=torch.int64, device=device)
            best = torch.full((R, 100), -2.0, device=device)
            step = 1 << 20
            for s0 in range(0, args.docs, step):
                sims = w.recall_q @ vec[s0:s0 + step].T
                cat_s = torch.cat([best, sims], 1)
                cat_i = torch.cat([ex, torch.arange(s0, min(args.docs, s0 + step), device=device)[None, :].expand(R, -1)], 1)
                best, pos = torch.topk(cat_s, 100, dim=1)
                ex = torch.gather(cat_i, 1, pos)
            w.recall_exact = ex.cpu().numpy()
            w.recall_q = w.recall_q.cpu().numpy()
        w.vec_dev = vec
        w.graph_note = None
        if args.graph == "bulk" or device == "cpu":
            # r01's stand-in (windowed exact kNN keyed on the generating cluster): kept for A/B and for machines without a GPU
            lv, l0, uo, lu, ml, ep = synth.build_graph_bulk(vec, 16, 100, order_key=cid)
            w.graph_dev = (lv, l0.to(torch.int32), uo, lu.to(torch.int32), ml, ep)
            w.graph_note = "bulk windowed-kNN build (harness)"
        else:
            w.graph_dev = None                  # built by the library itself: tsgpu_index_build_hnsw (see attach_vector_index)
        if device != "cpu":
            torch.cuda.synchronize()
        log(f"rank{rank}: vectors ({args.docs/1e6:.1f}M x {args.dim}) in {time.time()-t1:.1f}s")
    return w


_GRAPH_NOTE = [None]
GRAPH_PARAMS = {"M": 16, "ef_construction": 200, "seed": 100, "max_batch": 8192}


def attach_vector_index(args, w, gi, rank, need_host_copy):
    """Vector index of the workload inside `gi`. Default: hnswlib's insertion algorithm (heuristic neighbour selection, M 16,
    ef_construction 200, level seed 100) run by the library on the device over ALL vectors — tsgpu_index_build_hnsw; no
    locality hint, nothing but the vectors goes in. The built graph is cached on local disk (same seeds => same graph), so
    the driver's back-to-back bench runs on one box build it once. Returns the host copy for the CPU arm when asked."""
    import torch
    from typesense_b200.structs import HnswGraph
    t0 = time.time()
    n, dim, M = w.n_docs, w.dim, GRAPH_PARAMS["M"]
    if w.graph_dev is not None:
        lv, l0, uo, lu, ml, ep = w.graph_dev
        gi.load_hnsw_raw(n, dim, M, ml, ep, 0, w.vec_dev, lv, l0, uo, lu)
        host = None
        if need_host_copy:
            host = HnswGraph(w.vec_dev.cpu().numpy(), lv.cpu().numpy(), l0.cpu().numpy().astype(np.uint32), uo.cpu().numpy().astype(np.uint64),
                             lu.cpu().numpy().astype(np.uint32), M, ml, ep)
        w.vec_dev = None; w.graph_dev = None
        _GRAPH_NOTE[0] = w.graph_note
        torch.cuda.empty_cache()
        return host
    cache_dir = os.environ.get("TSGPU_BENCH_CACHE", "/tmp/tsgpu_bench_cache")
    key = f"hnsw_n{n}_d{dim}_M{M}_efc{GRAPH_PARAMS['ef_construction']}_s{GRAPH_PARAMS['seed']}_b{GRAPH_PARAMS['max_batch']}_v1234"
    path = os.path.join(cache_dir, key + ".npz")
    g = None
    if os.path.exists(path) and not args.no_graph_cache:
        try:
            z = np.load(path)
            g = HnswGraph(None, z["levels"], z["links0"], z["upper_off"], z["links_up"], M, int(z["max_level"]), int(z["entry_point"]))
            gi.load_hnsw_raw(n, dim, M, g.max_level, g.entry_point, 0, w.vec_dev, g.levels, g.links0, g.upper_off, g.links_up)
            w.graph_note = f"tsgpu_index_build_hnsw (device build; graph reloaded from {path})"
            w.build_info = {"cached": True}
            log(f"rank{rank}: HNSW graph reloaded from the local cache in {time.time()-t0:.1f}s")
        except Exception as e:             # a torn cache file: rebuild
            log(f"rank{rank}: graph cache unreadable ({e}); rebuilding")
            g = None
    if g is None:
        info = gi.build_hnsw(w.vec_dev, M, GRAPH_PARAMS["ef_construction"], GRAPH_PARAMS["seed"], max_batch=GRAPH_PARAMS["max_batch"])
        w.build_info = {"cached": False, "seconds": time.time() - t0, **info["build"]}
        w.graph_note = "tsgpu_index_build_hnsw (device build of all vectors)"
        log(f"rank{rank}: HNSW graph built on the device in {time.time()-t0:.1f}s ({info['build']['rounds']} rounds, max level {info['max_level']})")
        if need_host_copy or not args.no_graph_cache:
            g = gi.export_hnsw(np.zeros((0, dim), np.float32))
            g.vectors = None
            if not args.no_graph_cache and rank == 0:
                try:
                    os.makedirs(cache_dir, exist_ok=True)
                    tmp = path + f".tmp{os.getpid()}.npz"
                    np.savez(tmp, levels=g.levels, links0=g.links0, upper_off=g.upper_off, links_up=g.links_up, max_level=g.max_level, entry_point=g.entry_point)
                    os.replace(tmp, path)
                except Exception as e:
                    log(f"rank{rank}: graph cache not written ({e})")
    _GRAPH_NOTE[0] = w.graph_note
    host = None
    if need_host_copy:
        t2 = time.time()
        g.vectors = w.vec_dev.cpu().numpy()
        host = g
        log(f"rank{rank}: host copy of the vectors for the CPU baseline in {time.time()-t2:.1f}s")
    w.vec_dev = None
    torch.cuda.empty_cache()
    return host


TYPO_FRACTION = 0.30


def make_batches(args, w, n_batches, rank):
    """Query batches in both forms. STRINGS (what a client sends, what the end-to-end leg and the CPU arm search): three tokens of
    a random document, in 30 % of the queries one token misspelt by one substituted letter (never a vocabulary word itself), half of
    the queries with `cat:=c`, plus a query vector. RESOLVED (what the device-resident leg times: the C-ABI's input after the host's
    tokenising and candidate search): the same queries as one combination of the corrected tokens, total_cost 2 where a typo was
    fixed — the combination the reference's fuzzy_search_fields arrives at for these strings."""
    from typesense_b200 import hostapi, structs as S, synth
    rng = np.random.default_rng(1000 + rank)
    out = []
    taken = set(w.words)
    sort = ((S.SORT_TEXT_MATCH, -1, 1, 0), (S.SORT_NUMERIC, 0, 1, 0), (S.SORT_NONE, -1, 1, 0))
    for bi in range(n_batches):
        toks = synth.sample_queries(w.fd, args.batch, 3, int(rng.integers(0, 1 << 30)))
        qs, strings, filt = [], [], np.full(args.batch, -1, np.int32)
        for i in range(args.batch):
            row = [int(t) for t in toks[i]]
            words = [w.words[t] for t in row]
            cost = 0
            if rng.random() < TYPO_FRACTION:
                j = int(rng.integers(0, 3))
                words[j] = synth.misspell(words[j], rng, taken)
                cost = 2                                  # next_suggestion2: 2 * typo cost of the corrected token
            q = S.Query([S.Combo([[t] for t in row], 3, total_cost=cost)], topk=250, num_query_tokens=3, sort=sort)
            if i % 2 == 1:
                q.filter = int(rng.integers(0, 10))
                filt[i] = q.filter
            qs.append(q); strings.append(words)
        b = S.KwBatch(qs, [0], w.filters)
        qv = (synth.make_vectors_clustered(args.batch, args.dim, w.n_clusters, seed=4321 + 97 * rank + bi, centers_seed=1234, spread=0.35)[0].numpy()
              if args.workload != "keyword10m" else None)
        out.append((b, qv, {"strings": strings, "packed": hostapi.pack_queries(strings), "filter": filt}))
    return out


def kw_algorithmic_bytes(b, flat, matches):
    """SURVEY §8(d): 4*sum df over every executed (combination, token) + per match [T*(8+4p) + 8S] + 36*K per query."""
    df = np.diff(flat.list_off.astype(np.int64))
    lists = b.t_list[b.t_list != 0xFFFFFFFF]
    return int(4 * df[lists].sum() + matches * (3 * (8 + 4 * 1.3) + 8) + 36 * 250 * b.n_queries)


# ------------------------------------------------------------------------------------------------ the CPU path
HOST_OPTIONS = dict(num_typos=2, prefix=1, max_candidates=4, typo_tokens_threshold=1, drop_tokens_threshold=1, topster_size=250,
                    vec_k=0, vec_ef=10, vec_flat_search_cutoff=0, vec_fetch_size=100, vec_alpha=0.3)


def build_cpu_host(args, w, cores):
    """The reference's CPU path for this workload: the SAME C++ host layer (tokens -> ART candidate search -> typo / prefix /
    drop-token control flow of Index::search -> rank fusion) with every C-ABI call answered by the CPU oracle (the port of
    posting-list intersection, scoring, Topster, HNSW walk: oracle/), one query per thread on all host cores. ART walks run on the
    host (the mirror's walk, pinned on the reference's compiled art.cpp)."""
    import hostlib
    from typesense_b200 import hostapi
    os.environ["TSGPU_DOUBLE_THREADS"] = str(cores)            # read once by the double when it is loaded
    t0 = time.time()
    hc = hostapi.HostIndex(w.n_docs, 0, hostlib.build_host_cpu())
    hc.add_field_flat("title", w.words, w.fd.flat)
    hc.add_sort_column("points", w.points)
    handles = [hc.add_filter(f) for f in w.filters]
    if w.graph_host is not None:
        hc.device_index().load_hnsw(w.graph_host)
    log(f"CPU arm: host layer over the oracle double ready in {time.time()-t0:.1f}s")
    return hc, handles


def cpu_search(args, hc, handles, batch, n, cores, out=None):
    from typesense_b200 import hostapi
    b, qv, qs = batch
    blob, tok_off, q_off = qs["packed"]
    packed = (blob, tok_off, q_off[:n + 1])
    qf = np.asarray([handles[f] if f >= 0 else -1 for f in qs["filter"][:n]], np.int32)
    opt = hostapi.Options(device_art_walk=0, n_threads=cores, **HOST_OPTIONS)
    hybrid = args.workload != "keyword10m"
    return hc.multi_search("title", "points", None, 100, qf, qv[:n] if hybrid else None, opt, packed=packed, out=out)


def run_reference(args, rank, world):
    if rank != 0:
        return
    import oracle_lib as ol
    import torch
    ol.build_oracle()
    device = "cuda" if torch.cuda.is_available() else "cpu"
    w = build_workload(args, device, 0, True)
    if w.vec_dev is not None:
        if device == "cuda":              # the graph both arms search is the one the library builds (outside any timed region)
            from typesense_b200 import capi
            gtmp = capi.GpuIndex(w.n_docs, 0)
            w.graph_host = attach_vector_index(args, w, gtmp, 0, True)
            gtmp.close()
            torch.cuda.empty_cache()
        else:
            from typesense_b200.structs import HnswGraph
            lv, l0, uo, lu, ml, ep = w.graph_dev
            w.graph_host = HnswGraph(w.vec_dev.numpy(), lv.numpy(), l0.numpy().astype(np.uint32), uo.numpy().astype(np.uint64),
                                     lu.numpy().astype(np.uint32), 16, ml, ep)
            w.vec_dev = None
    cores = os.cpu_count() or 1
    hc, handles = build_cpu_host(args, w, cores)
    batches = make_batches(args, w, min(args.steps + args.warmup, 4), 0)
    S_n = min(args.cpu_sample, args.batch)

    def step(i):
        return cpu_search(args, hc, handles, batches[i % len(batches)], S_n, cores)
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        res = step(args.warmup + i)
    dt = time.perf_counter() - t0
    st = res[3]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res[0], res[1], res[2])
    qps = S_n * args.steps / dt
    out = {"impl": "reference", "metric": "queries/sec", "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": SCALING,
           "vs_baseline": None, "dtype": "u32+f32", "data": "synthetic",
           "config": workload_config(args, args.batch),
           "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                            "sample": f"{S_n} queries of the batch per step, {args.steps} steps, query strings through the C++ host layer over the CPU oracle",
                            "host_rounds_last_step": st},
           "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)
    hc.close()


SCALING = "strong"


def workload_config(args, batch):
    return {"workload": args.workload, "docs": args.docs, "vocab": args.vocab, "dim": args.dim, "batch": batch,
            "terms": 3, "typo": {"executed": True, "misspelt_queries": TYPO_FRACTION, "num_typos": 2, "prefix": True, "max_candidates": 4,
                                 "typo_tokens_threshold": 1, "drop_tokens_threshold": 1,
                                 "where": "e2e and the CPU arm: query STRINGS through the C++ host layer (ART candidate search + Index::search control flow); "
                                          "value: the same queries in resolved form through the C-ABI"},
            "filtered_queries": 0.5, "topster": 250, "hits": 100,
            "vector": {"k": 100, "ef_param": 10, "ef_effective": 100, "alpha": 0.3, "M": 16, "ef_construction": GRAPH_PARAMS["ef_construction"],
                       "data": "clustered unit vectors, latent dim 8, ~2000 per cluster",
                       "graph": (_GRAPH_NOTE[0] or "tsgpu_index_build_hnsw (device build of all vectors)") + "; the CPU arm walks the exported copy"},
            "cache": "index working set (>= 30 GB vectors + postings) >> 126 MB L2; query batches cycle through min(steps+warmup, 6) distinct batches",
            "parallelism": f"replica x{args.gpus}, queries sharded",
            "kw_scoring": "r01 local-array scorer (TSGPU_REG_SCORE=0)" if os.environ.get("TSGPU_REG_SCORE") == "0" else "register-resident (default)"}


# ------------------------------------------------------------------------------------------------ secondary configurations
def other_configs(args, w, hi, gi, sl, qv_pin, host_opt, hbm_peak):
    """BASELINE.json's other configurations, measured on the same box next to the headline (rank 0, N = 1, outside its timed
    regions): parity for each is in tests/; these are the timings.
      configs[0]  3-way posting-list AND in the reference's own DISABLED_BenchmarkIntersection shape (tools/bench_intersect.py)
      configs[1]  10 M-doc 3-term keyword search with typo tolerance, Topster 250 -> 100 hits: query strings through the host layer
      configs[2]  HNSW k=100 (ef 10 -> effective 100), inner product, batch 1024, no filter — on THIS index (10 M x 768; the named one is 5 M)
      configs[4]-shaped  faceted keyword search: all_result_ids kept on the device + facet counts over a 50 K-value facet (1-5 values per doc)"""
    import torch
    from typesense_b200 import capi, hostapi, synth, structs as S
    out = {}
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_intersect
        out["intersect_3way_100k"] = bench_intersect.run(cpu_reps=5)
    except Exception as e:
        out["intersect_3way_100k"] = {"error": str(e)[:200]}
    try:        # configs[1]: keyword + typo through the host layer
        sb, _, packed, qf = sl[0]
        nl = sb.n_queries
        kvb = (np.zeros((nl, 100), S.KV_DTYPE), np.zeros(nl, np.uint32), np.zeros(nl, np.uint32))
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            _, _, _, st = hi.multi_search("title", "points", None, 100, qf, None, host_opt, packed=packed, out=kvb)
            ts.append(time.perf_counter() - t0)
        out["keyword10m_typo"] = {"queries": nl, "ms_per_batch": 1000 * min(ts), "queries_per_s": nl / min(ts), "host_rounds": st,
                                  "path": "query strings (30 % misspelt, half filtered) -> host layer -> device; keyword only"}
    except Exception as e:
        out["keyword10m_typo"] = {"error": str(e)[:200]}
    try:        # configs[2]: pure kNN
        nqv = min(1024, qv_pin[0].shape[0])
        qv = qv_pin[0].numpy()[:nqv]
        gi.knn(qv, 100, 10)
        ts, sts = [], []
        for _ in range(3):
            t0 = time.perf_counter()
            gi.knn(qv, 100, 10)
            ts.append(time.perf_counter() - t0)
            sts.append(gi.stats())
        st = sts[-1]
        algo = st["knn_dist"] * 4 * w.dim + st["knn_expanded"] * 4 * 33
        out["hnsw_knn_batch1024"] = {"queries": nqv, "nodes": w.n_docs, "ms_per_batch": 1000 * min(ts), "queries_per_s": nqv / min(ts), "kernel_ms": st["ms_knn"],
                                     "dist_per_query": st["knn_dist"] / nqv, "expanded_per_query": st["knn_expanded"] / nqv,
                                     "roofline_frac": algo / (st["ms_knn"] * 1e-3) / 1e9 / hbm_peak if st["ms_knn"] > 0 else None}
    except Exception as e:
        out["hnsw_knn_batch1024"] = {"error": str(e)[:200]}
    try:        # K7: the flat scan (process_results_bruteforce) of the queries of a batch that share one filter, on the tensor cores
        nqf = min(256, qv_pin[0].shape[0])
        ids = np.ascontiguousarray(w.filters[0][:200000])
        qf_ = qv_pin[0].numpy()[:nqf]
        gi.flat_distances_batch(qf_[:16], ids[:1024])
        ts = []
        for _ in range(3):
            dtc = gi.flat_distances_batch(qf_, ids)
            ts.append(gi.stats()["ms_knn"])
        tc_q = gi.stats()["flat_tc_queries"]
        d0 = gi.flat_distances(qf_[0], ids[:8192])                 # the fp32 pair-by-pair kernel (bit-equal to the CPU loop)
        ms = min(ts)
        flops = 2.0 * nqf * len(ids) * w.dim
        tf32_peak = None
        try:
            tf32_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"]) / 2
        except Exception:
            pass
        out["flat_scan_tensor"] = {"queries": nqf, "candidates": int(len(ids)), "dim": w.dim, "kernel_ms": ms, "tensor_core_queries": int(tc_q),
                                   "fp32_equivalent_tflops": flops / (ms * 1e-3) / 1e12 if ms > 0 else None,
                                   "tf32_mma_tflops": 3 * flops / (ms * 1e-3) / 1e12 if ms > 0 else None,
                                   "roofline": {"bound": "tensor", "achieved": 3 * flops / (ms * 1e-3) / 1e12 if ms > 0 else None, "peak": tf32_peak, "unit": "TFLOP/s",
                                                "frac": (3 * flops / (ms * 1e-3) / 1e12 / tf32_peak) if (ms > 0 and tf32_peak) else None,
                                                "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (tf32 runs at half the bf16 rate); 3 tf32 MMAs per fp32 product"},
                                   "rows_gbs": len(ids) * w.dim * 4 / (ms * 1e-3) / 1e9 if ms > 0 else None,
                                   "max_abs_dev_vs_fp32_kernel": float(np.abs(dtc[0, :len(d0)] - d0).max()),
                                   "path": "tsgpu_flat_distances_batch: tcgen05 kind::tf32, 3-term split (csrc/flat_tc.cu); kernel time only, outputs copied to the host outside it"}
    except Exception as e:
        out["flat_scan_tensor"] = {"error": str(e)[:200]}
    try:        # configs[4]-shaped: facets over all_result_ids
        n_values = 50000
        rng = np.random.default_rng(99)
        per = rng.integers(1, 6, w.n_docs)
        off = np.zeros(w.n_docs + 1, np.uint64); off[1:] = np.cumsum(per)
        cdf = np.cumsum(np.arange(1, n_values + 1, dtype=np.float64) ** -1.07); cdf /= cdf[-1]
        vals = np.minimum(np.searchsorted(cdf, rng.random(int(off[-1]))), n_values - 1).astype(np.uint32)
        fac = gi.load_facet(n_values, off, vals)
        sb = sl[0][0]
        nf = min(512, sb.n_queries)                         # 512 faceted queries per call: 512 x 1.25 MB of all_result_ids bitmaps, 512 x 50 K histograms
        hb = sb.head(nf)
        flags0 = hb.q_flags.copy()
        hb.q_flags = hb.q_flags.copy(); hb.q_flags[:nf] |= capi.QFLAG_KEEP_ALL_IDS
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            gi.keyword_search(hb, 100)
            t1 = time.perf_counter()
            fc, fn, fdis = gi.facet_counts_last(fac, nf, 10)
            ts.append((t1 - t0, time.perf_counter() - t1, gi.stats()["ms_total"]))
        best = min(ts, key=lambda x: x[0] + x[1])
        out["faceted_keyword"] = {"queries": nf, "facet_values": n_values, "values_per_doc": "1-5", "search_ms": 1000 * best[0], "facet_ms": 1000 * best[1],
                                  "facet_device_ms": best[2], "queries_per_s": nf / (best[0] + best[1]), "mean_distinct_values": float(fdis.mean())}
    except Exception as e:
        out["faceted_keyword"] = {"error": str(e)[:200]}
    return out


# ------------------------------------------------------------------------------------------------ tsgpu arm
def run_tsgpu(args, rank, world, local_rank):
    """One process per GPU, a full replica each. STRONG scaling (BASELINE config 4 literally): every step is ONE multi_search batch
    of `--batch` queries — the same batch on every rank — of which rank r answers its contiguous slice; the slices' result
    records are gathered on rank 0 by the library's own NCCL exchange (tsgpu_comm_gather) inside the timed region."""
    import torch
    import torch.distributed as dist
    from typesense_b200 import capi, hostapi, shard, structs as S
    assert torch.cuda.is_available(), "bench.py --impl tsgpu needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    device = f"cuda:{local_rank}"
    want_cpu = (rank == 0 and world == 1 and not args.no_cpu_baseline)
    w = build_workload(args, device, rank, want_cpu)
    t0 = time.time()
    hi = hostapi.HostIndex(w.n_docs, local_rank)                    # the C++ host layer (libtshost.so) owns the device index
    hi.add_field_flat("title", w.words, w.fd.flat)
    hi.add_sort_column("points", w.points)
    handles = [hi.add_filter(f) for f in w.filters]
    gi = hi.device_index()
    if w.vec_dev is not None:
        w.graph_host = attach_vector_index(args, w, gi, rank, want_cpu)
    log(f"rank{rank}: mirror loaded in {time.time()-t0:.1f}s")
    if world > 1:                                                   # the library's communicator: id made on rank 0, shared through torch.distributed
        ident = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            ident = torch.from_numpy(gi.comm_unique_id().copy())
        ident = ident.to(device)
        dist.broadcast(ident, src=0)
        gi.comm_init(rank, world, ident.cpu().numpy())
    n_b = min(args.steps + args.warmup, 6)
    batches = make_batches(args, w, n_b, 0)                         # the same batches on every rank
    vp = S.vec_params(k=0, ef=10, alpha=0.3, fetch_size=100)
    stride = 100
    nq = args.batch
    lo, hi_q = shard.shard_range(nq, world, rank)
    nl = hi_q - lo                                                  # this rank's slice
    max_nl = max(b_ - a_ for a_, b_ in (shard.shard_range(nq, world, r) for r in range(world)))
    hybrid = args.workload != "keyword10m"

    def slice_batch(bt):
        b, qv, qs = bt
        sb = S.KwBatch(b.queries[lo:hi_q], [0], w.filters).with_filter_handles(handles) if world > 1 else b.with_filter_handles(handles)
        blob, tok_off, q_off = qs["packed"]
        packed = (blob, tok_off, (q_off[lo:hi_q + 1]).copy())
        return sb, (qv[lo:hi_q] if qv is not None else None), packed, np.asarray([handles[f] if f >= 0 else -1 for f in qs["filter"][lo:hi_q]], np.int32)
    sl = [slice_batch(bt) for bt in batches]
    structs = [x[0].struct() for x in sl]
    rec = stride * 56

    # device-resident inputs/outputs (value) and pinned host ones (e2e)
    kv_dev = torch.zeros(max_nl * rec, dtype=torch.uint8, device=device)
    cnt_dev = torch.zeros(max_nl, dtype=torch.int32, device=device)
    fnd_dev = torch.zeros(max_nl, dtype=torch.int32, device=device)
    qv_dev = [torch.from_numpy(np.ascontiguousarray(x[1])).to(device) for x in sl] if hybrid else [None] * n_b
    kv_pin = torch.zeros(max_nl * rec, dtype=torch.uint8).pin_memory()
    cnt_pin = torch.zeros(max_nl, dtype=torch.int32).pin_memory()
    fnd_pin = torch.zeros(max_nl, dtype=torch.int32).pin_memory()
    qv_pin = [torch.from_numpy(np.ascontiguousarray(x[1])).pin_memory() for x in sl] if hybrid else [None] * n_b
    all_dev = torch.zeros(world * max_nl * rec, dtype=torch.uint8, device=device) if (world > 1 and rank == 0) else None
    all_pin = torch.zeros(world * max_nl * rec, dtype=torch.uint8).pin_memory() if (world > 1 and rank == 0) else None
    E2E_DEPTH = max(1, args.e2e_depth)              # multi_search calls in flight in the end-to-end leg (client threads of a server)
    host_bufs = [(np.zeros((max_nl, stride), S.KV_DTYPE), np.zeros(max_nl, np.uint32), np.zeros(max_nl, np.uint32)) for _ in range(E2E_DEPTH)]
    host_kv, host_cnt, host_fnd = host_bufs[0]
    host_opt = hostapi.Options(device_art_walk=1, n_threads=max(2, min((os.cpu_count() or 1) // max(1, world), args.e2e_threads)), **HOST_OPTIONS)      # the ranks of one node share its cores
    comm_ms = []

    def step(i, mode):
        """mode 0: resolved queries, device-resident buffers (value); 1: resolved queries, pinned host buffers; 2: query strings
        through the C++ host layer (e2e)."""
        j = i % n_b
        sb, _, packed, qf = sl[j]
        if mode == 2:
            _, _, _, hst = hi.multi_search("title", "points", None, stride, qf, qv_pin[j].numpy() if hybrid else None, host_opt, packed=packed,
                                           out=(host_kv[:nl], host_cnt[:nl], host_fnd[:nl]))
            if world > 1:
                gi.comm_gather(host_kv, max_nl * rec, all_pin, 0)
                comm_ms.append(gi.comm_last_ms())
            return hst
        out = (kv_dev, cnt_dev, fnd_dev) if mode == 0 else (kv_pin, cnt_pin, fnd_pin)
        if hybrid:
            gi.hybrid_search(sb, qv_dev[j] if mode == 0 else qv_pin[j], vp, stride, out=out, bstruct=structs[j])
        else:
            gi.keyword_search(sb, stride, out=out, bstruct=structs[j])
        st = gi.stats()
        if world > 1:
            gi.comm_gather(kv_dev if mode == 0 else kv_pin, max_nl * rec, all_dev if mode == 0 else all_pin, 0)
            comm_ms.append(gi.comm_last_ms())
        return st

    def timed(mode):
        for i in range(args.warmup):
            step(i, mode)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sts = []
        for i in range(args.steps):
            t1 = time.perf_counter()
            sts.append(step(args.warmup + i, mode))                 # the calls are synchronous: results are final on return
            sts[-1]["wall_ms"] = 1000 * (time.perf_counter() - t1)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt, sts

    def timed_e2e():
        """The end-to-end leg: K multi_search calls of query strings through the host layer, E2E_DEPTH of them in flight (a server's
        request threads: while one call's device round runs, another call's host pass does; the library serialises device calls).
        Every call's results land in host buffers; with several ranks each call is followed, in call order, by the NCCL gather."""
        import concurrent.futures as cf

        def run(i, slot):
            j = i % n_b
            sb, _, packed, qf = sl[j]
            t1 = time.perf_counter()
            kvb, cb, fb = host_bufs[slot]
            _, _, _, hst = hi.multi_search("title", "points", None, stride, qf, qv_pin[j].numpy() if hybrid else None, host_opt, packed=packed,
                                           out=(kvb[:nl], cb[:nl], fb[:nl]))
            hst["wall_ms"] = 1000 * (time.perf_counter() - t1)
            return hst
        for i in range(args.warmup):
            step(i, 2)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sts, futs, nxt = [], {}, 0
        with cf.ThreadPoolExecutor(E2E_DEPTH) as pool:
            t0 = time.perf_counter()
            for i in range(args.steps):
                while nxt < args.steps and nxt < i + E2E_DEPTH:
                    futs[nxt] = pool.submit(run, args.warmup + nxt, nxt % E2E_DEPTH)
                    nxt += 1
                sts.append(futs.pop(i).result())
                if world > 1:
                    gi.comm_gather(host_bufs[i % E2E_DEPTH][0], max_nl * rec, all_pin, 0)
                    comm_ms.append(gi.comm_last_ms())
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt, sts

    def xfer():
        s_ = gi.stats()
        return s_["h2d_total"] + s_["h2d_bytes"], s_["d2h_total"] + s_["d2h_bytes"], s_["calls_total"]

    launches0 = gi.stats()["launches_total"]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dt_res, sts = timed(0)
    launches = gi.stats()["launches_total"] - launches0
    if args.dump_outputs and rank == 0:            # this rank's slice; copied before the later legs reuse the buffers
        dump_outputs(args.dump_outputs, np.frombuffer(kv_dev[:nl * rec].cpu().numpy().tobytes(), S.KV_DTYPE).reshape(nl, stride),
                     cnt_dev[:nl].cpu().numpy(), fnd_dev[:nl].cpu().numpy())
    dt_pin, sts_pin = timed(1)
    x0 = xfer()
    dt_e2e, sts_e2e = timed_e2e()
    x1 = xfer()
    clocks = sampler.stop() if rank == 0 else None
    e2e_steps = args.steps + args.warmup
    # per-kernel durations for the roofline: the timed region overlaps the graph walk with the keyword kernels on two
    # streams, which stretches each kernel's own wall time; measure them once more back to back (same batches, CUDA
    # events on the library's stream) with the overlap switched off. Not part of `value`.
    os.environ["TSGPU_KNN_OVERLAP_BLOCKS"] = "0"
    sts_iso = [step(args.warmup + i, 0) for i in range(min(args.steps, 4))]
    os.environ.pop("TSGPU_KNN_OVERLAP_BLOCKS", None)
    knn_work = gi.knn_work(nl) if hybrid else None
    launches_per_region = (launches * args.steps) // (args.steps + args.warmup)
    # latency of a small multi_search (64 query strings through the host layer), the p50/p99 half of BASELINE.json's metric
    lat_small = []
    if rank == 0:
        ns = min(64, nl)
        for i in range(40):
            sb, _, packed, qf = sl[i % n_b]
            pk = (packed[0], packed[1], packed[2][:ns + 1])
            t1 = time.perf_counter()
            hi.multi_search("title", "points", None, stride, qf[:ns], qv_pin[i % n_b].numpy()[:ns] if hybrid else None, host_opt, packed=pk,
                            out=(host_kv[:ns], host_cnt[:ns], host_fnd[:ns]))
            lat_small.append(1000 * (time.perf_counter() - t1))
        lat_small = lat_small[8:]

    # parity spot check + recall on rank 0 (outside the timed region)
    extra = {}
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        ms_kw = statistics.mean(s["ms_kw_search"] for s in sts_iso)
        ms_knn = statistics.mean(s["ms_knn"] for s in sts_iso)
        ms_fuse = statistics.mean(s["ms_fuse"] for s in sts)
        ms_dev = statistics.mean(s["ms_total"] for s in sts)
        n_dist = statistics.mean(s["knn_dist"] for s in sts_iso)
        n_exp = statistics.mean(s["knn_expanded"] for s in sts_iso)
        matches = statistics.mean(s["kw_matches"] for s in sts_iso)
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            pass
        knn_bytes = n_dist * 4 * args.dim + n_exp * 4 * 33
        iso_ids = [(args.warmup + i) % n_b for i in range(min(args.steps, 4))]            # the batches the isolated pass ran
        kw_bytes = statistics.mean(kw_algorithmic_bytes(sl[j][0], w.fd.flat, s_["kw_matches"]) for j, s_ in zip(iso_ids, sts_iso))
        roof = []
        if hybrid and ms_knn > 0:
            a = knn_bytes / (ms_knn * 1e-3) / 1e9
            roof.append({"kernel": "hnsw_walk_kernel", "bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s",
                         "frac": a / hbm_peak, "traffic": traffic.get("hnsw_walk_kernel"), "ms": ms_knn, "algorithmic_bytes": knn_bytes,
                         "n_dist_per_query": n_dist / nl, "n_expanded_per_query": n_exp / nl, "peak_source": peak_src})
        if ms_kw > 0:
            a = kw_bytes / (ms_kw * 1e-3) / 1e9
            roof.append({"kernel": "kw_search_kernel", "bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s",
                         "frac": a / hbm_peak, "traffic": traffic.get("kw_search_kernel"), "ms": ms_kw, "algorithmic_bytes": kw_bytes,
                         "matches_per_query": matches / nl, "peak_source": peak_src})
        for r in roof:          # what the kernel really moves over the HBM pins (one ncu --set full launch of this build, see profiles/)
            r["achieved_dram_gbs"] = (r["traffic"] / (r["ms"] * 1e-3) / 1e9) if r.get("traffic") else None
            r["note"] = ("achieved = ALGORITHMIC bytes (SURVEY 8d: 4*sum(df) + per-match offsets + K*36; n_dist*4d + n_exp*4*(2M+1)) / live kernel time; "
                         "achieved_dram_gbs = DRAM bytes of one ncu-profiled launch / live kernel time: block skipping and L2 hits keep it far below")
        roof.sort(key=lambda r: -r["ms"])
        extra["roofline"] = roof[0] if roof else None
        extra["roofline_other"] = roof[1:]
        extra["device_ms_per_step"] = {"total": ms_dev, "note": "value leg: vector stage on its own stream, overlapped",
                                       "keyword": statistics.mean(s["ms_keyword"] for s in sts),
                                       "knn_overlapped": statistics.mean(s["ms_knn"] for s in sts), "fuse": ms_fuse,
                                       "host_plan": statistics.mean(s["ms_host_plan"] for s in sts)}
        extra["device_ms_isolated"] = {"kw_search": ms_kw, "kw_merge": statistics.mean(s["ms_kw_merge"] for s in sts_iso),
                                       "knn": ms_knn, "total": statistics.mean(s["ms_total"] for s in sts_iso)}
        extra["work_per_step"] = {k: float(statistics.mean(s_[k] for s_ in sts_iso)) for k in
                                  ("kw_driver_ids", "kw_probe_ids", "kw_matches", "knn_dist", "knn_expanded", "knn_spec_hits", "knn_table_probes")}
        if knn_work is not None and len(knn_work):
            ex = np.sort(knn_work[:, 0])
            filt = (sl[(args.warmup + min(args.steps, 4) - 1) % n_b][0].q_filter != -1)[:len(knn_work)]
            extra["knn_walks"] = {"expanded_mean": float(ex.mean()), "expanded_p50": int(ex[len(ex) // 2]), "expanded_p99": int(ex[int(0.99 * (len(ex) - 1))]),
                                  "expanded_max": int(ex[-1]), "expanded_mean_filtered": float(knn_work[filt, 0].mean()) if filt.any() else None,
                                  "expanded_mean_unfiltered": float(knn_work[~filt, 0].mean()) if (~filt).any() else None,
                                  "dist_max": int(knn_work[:, 1].max())}
        if traffic:
            extra["roofline_traffic_source"] = traffic.get("source")
        extra["host_rounds_per_step"] = {k: float(statistics.mean(s_[k] for s_ in sts_e2e)) for k in
                                         ("passes", "kw_batches", "kw_queries", "walk_batches", "walks", "host_walk_fallbacks", "fuse_queries",
                                          "ms_host_passes", "ms_kw_calls", "ms_walk_calls", "ms_fuse_calls")}
        if getattr(w, "build_info", None):
            extra["hnsw_build"] = w.build_info
        if want_cpu:
            cores = os.cpu_count() or 1
            S_n = min(args.cpu_sample, nq)
            hc, chandles = build_cpu_host(args, w, cores)
            passes = []
            for _ in range(3):                    # one pass is ~1 s of all cores: too short to be stable, so median of three
                t0 = time.perf_counter()
                okv, ocnt, ofound, ost = cpu_search(args, hc, chandles, batches[0], S_n, cores)
                passes.append(time.perf_counter() - t0)
            dt_cpu = statistics.median(passes)
            extra["cpu_baseline"] = {"value": S_n / dt_cpu, "unit": "queries/s", "cores": cores, "kind": "port",
                                     "sample": f"first {S_n} query strings of batch 0 through the C++ host layer over the CPU oracle, all {cores} host threads, median of 3 passes",
                                     "passes_qps": [S_n / p for p in passes], "host_rounds": ost}
            # parity on that sample: the end-to-end GPU path against the CPU path, query by query (identical top-k ids is the bar)
            sb, _, packed, qf = sl[0]
            pk = (packed[0], packed[1], packed[2][:S_n + 1])
            kv, cnt, found, _ = hi.multi_search("title", "points", None, stride, qf[:S_n], batches[0][1][:S_n] if hybrid else None, host_opt, packed=pk)
            same = sum(int(cnt[q] == ocnt[q] and (kv["key"][q, :cnt[q]] == okv["key"][q, :ocnt[q]]).all()) for q in range(S_n))
            score_same = sum(int(cnt[q] == ocnt[q] and (kv["scores"][q, :cnt[q]] == okv["scores"][q, :ocnt[q]]).all()) for q in range(S_n))
            extra["parity_sample"] = {"queries": S_n, "identical_topk": same, "identical_scores": score_same, "found_equal": int((found[:S_n] == ofound[:S_n]).sum()),
                                      "what": "end-to-end GPU path (host layer + device ART walks + device rounds) vs the CPU arm, same query strings"}
            # and the resolved form through the C-ABI against the same CPU answers (what `value` times)
            kv2, cnt2, found2 = gi.hybrid_search(sl[0][0], batches[0][1], vp, stride) if hybrid else gi.keyword_search(sl[0][0], stride)
            same2 = sum(int(cnt2[q] == ocnt[q] and (kv2["key"][q, :cnt2[q]] == okv["key"][q, :ocnt[q]]).all()) for q in range(S_n))
            extra["parity_resolved_vs_cpu"] = {"queries": S_n, "identical_topk": same2,
                                               "note": "differences = queries whose resolved single combination is not where the reference's flow ends (no match under the filter -> typo / drop-token rounds)"}
            hc.close()
        if world == 1 and not args.no_other_configs:
            extra["other_configs"] = other_configs(args, w, hi, gi, sl, qv_pin, host_opt, hbm_peak)
        if hybrid and w.recall_exact is not None:
            R = len(w.recall_q)
            d, l, n = gi.knn(w.recall_q, 100, 100)
            extra["knn_recall_at_100"] = float(np.mean([len(set(l[i][:n[i]].tolist()) & set(w.recall_exact[i].tolist())) / 100 for i in range(R)]))
            extra["knn_recall_note"] = "GPU kNN (k=100, ef=100) vs brute force over all vectors; the CPU oracle returns the same ids on the same graph"
        if not want_cpu:
            extra["cpu_baseline"] = None

    if rank == 0:
        value = nq * args.steps / dt_res
        e2e = nq * args.steps / dt_e2e
        out = {"metric": "queries/sec", "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": 1000 * dt_res / args.steps, "higher_is_better": True, "scaling": SCALING, "vs_baseline": None,
               "dtype": "u32+f32", "data": "synthetic", "config": workload_config(args, nq),
               "e2e": {"value": e2e, "unit": "queries/s", "ms_per_step": 1000 * dt_e2e / args.steps,
                       "h2d_bytes_per_step": int((x1[0] - x0[0]) / e2e_steps), "d2h_bytes_per_step": int((x1[1] - x0[1]) / e2e_steps),
                       "device_calls_per_step": (x1[2] - x0[2]) / e2e_steps, "calls_in_flight": E2E_DEPTH, "host_threads_per_call": int(host_opt.n_threads),
                       "path": "query strings -> C++ host layer (libtshost.so: tokens, ART candidate walks on the device, typo / prefix / drop-token control flow) -> "
                               "C-ABI rounds with host buffers -> tsgpu_hybrid_fuse_batch; rank 0's slice per step" + (" + NCCL gather" if world > 1 else "")},
               "e2e_resolved": {"value": nq * args.steps / dt_pin, "unit": "queries/s", "ms_per_step": 1000 * dt_pin / args.steps,
                                "h2d_bytes_per_step": int(sts_pin[-1]["h2d_bytes"]), "d2h_bytes_per_step": int(sts_pin[-1]["d2h_bytes"]),
                                "path": "resolved queries, ONE tsgpu_hybrid_search_batch with pinned host buffers (r01's e2e)"},
               "gpu_launches": int(launches_per_region), "clocks": clocks}
        lat_b = sorted(s_["wall_ms"] for s_ in sts_e2e)
        pct = lambda xs, p: float(xs[min(len(xs) - 1, int(round(p * (len(xs) - 1))))]) if xs else None
        ls = sorted(lat_small)
        out["latency_ms"] = {"note": "wall time of one synchronous multi_search of query strings through the host layer (this rank's slice); every query of a call completes with it",
                             "batch": {"queries": nl, "p50": pct(lat_b, 0.5), "p99": pct(lat_b, 0.99), "calls": len(lat_b)},
                             "small": {"queries": min(64, nl), "p50": pct(ls, 0.5), "p99": pct(ls, 0.99), "calls": len(ls)}}
        if world > 1 and comm_ms:
            out["collective"] = {"what": "tsgpu_comm_gather (in-library NCCL send/recv group, device to device) of the slices' KV records to rank 0",
                                 "bytes_per_rank": max_nl * rec, "ms_median_rank0": float(statistics.median(comm_ms)), "ms_max_rank0": float(max(comm_ms)), "calls": len(comm_ms)}
        out.update(extra)
        emit(out)
    if world > 1:
        gi.comm_destroy()
    hi.close()


def main():
    args = parse()
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        run_tsgpu(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
