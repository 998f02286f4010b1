#!/usr/bin/env python
"""bench.py -- RAG /retrieve queries/sec on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[2] "hybrid dense+BM25+RRF /retrieve, 10M docs
(768-d fp32 vectors + postings), top-10" -- the largest single-GPU configuration (the 100M x 768
headline corpus is 307 GB in fp32 and does not fit one B200).  A step = one batch of 256 queries
through dense top-P + BM25 top-P + fuse.  N GPUs shard the SAME corpus by document (strong
scaling): local candidates, one NCCL all-gather, merge + fuse on every rank.

One JSON line on rank 0:
  value   : queries/s with the batch already resident in HBM (device pipeline, CUDA events)
  e2e     : queries/s through the public host-buffer API, H2D + D2H inside the timed region
  batch1  : the same two numbers at batch 1
  roofline: dominant kernel (dense scan) algorithmic GB/s against MEASURED_PEAKS.json
  cpu_baseline / --impl reference: the CPU oracle (restated reference path; faiss/bm25s are not
            installable offline) on all host cores over a bounded sample, extrapolated linearly in N.

--dump-outputs DIR writes the /retrieve result of the last timed step of `value` as DIR/<name>.npy (float32 / float64;
integer outputs as exact float64; a missing score, NaN in the result, as 0 with <name>_present.npy = 0 beside it).  The
inputs depend only on the arguments, so two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VOCAB = 1 << 20
BGE = {  # BertConfig of BAAI/bge-*-en-v1.5 (random-init weights here: no checkpoints offline)
    "bge-small": dict(num_hidden_layers=12, hidden_size=384, num_attention_heads=12, intermediate_size=1536, vocab_size=30522),
    "bge-base": dict(num_hidden_layers=12, hidden_size=768, num_attention_heads=12, intermediate_size=3072, vocab_size=30522),
    "bge-large": dict(num_hidden_layers=24, hidden_size=1024, num_attention_heads=16, intermediate_size=4096, vocab_size=30522),
}


def pick_embedding(name, dim):
    if name == "none":
        return None
    if name == "auto":
        name = {384: "bge-small", 768: "bge-base", 1024: "bge-large"}.get(dim)
    if name is None or BGE[name]["hidden_size"] != dim:
        return None
    return name


def random_bert_state(cfg, seed=0):
    """Hugging Face BertModel tensor names with N(0, 0.02) weights (the init of an untrained BERT)."""
    g = np.random.default_rng(seed)
    d, i, v = cfg["hidden_size"], cfg["intermediate_size"], cfg["vocab_size"]
    n = lambda *s: (0.02 * g.standard_normal(s, dtype=np.float32))  # noqa: E731
    st = {"embeddings.word_embeddings.weight": n(v, d), "embeddings.position_embeddings.weight": n(512, d),
          "embeddings.token_type_embeddings.weight": n(2, d), "embeddings.LayerNorm.weight": np.ones(d, np.float32),
          "embeddings.LayerNorm.bias": np.zeros(d, np.float32)}
    for l in range(cfg["num_hidden_layers"]):
        p = f"encoder.layer.{l}."
        for nm in ("attention.self.query", "attention.self.key", "attention.self.value", "attention.output.dense"):
            st[p + nm + ".weight"] = n(d, d); st[p + nm + ".bias"] = np.zeros(d, np.float32)
        st[p + "intermediate.dense.weight"] = n(i, d); st[p + "intermediate.dense.bias"] = np.zeros(i, np.float32)
        st[p + "output.dense.weight"] = n(d, i); st[p + "output.dense.bias"] = np.zeros(d, np.float32)
        for nm in ("attention.output.LayerNorm", "output.LayerNorm"):
            st[p + nm + ".weight"] = np.ones(d, np.float32); st[p + nm + ".bias"] = np.zeros(d, np.float32)
    return st


def bert_flops(cfg, seq):
    """SURVEY.md section 8d: L * (24 S d^2 + 4 S^2 d) per sequence of S tokens"""
    L, d = cfg["num_hidden_layers"], cfg["hidden_size"]
    return L * (24 * seq * d * d + 4 * seq * seq * d)
WORKLOADS = {
    # name: (docs, dim, hybrid)
    "c3": (10_000_000, 768, True),
    "c2": (1_000_000, 768, False),
    "headline": (100_000_000, 768, True),    # BASELINE.json metric corpus: needs >= 4 GPUs in fp32 (8 recommended)
    "c4": (100_000_000, 1024, False),        # BASELINE.json configs[3]: 100M x 1024 dense, 8 GPUs (51.2 GB fp32 per GPU)
    "tiny": (200_000, 768, True),            # functional check of the harness
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("KRAG_BENCH_WORKLOAD", "c3"), choices=list(WORKLOADS))
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--dense-mode", type=int, default=0, help="0 auto, 1 scan (K1), 2 tensor-core TF32 (K2), 3 K2 pruning on a bf16 shadow (opt-in, +50%% memory)")
    ap.add_argument("--embedding", default="auto", choices=["auto", "none", "bge-small", "bge-base", "bge-large"],
                    help="query embedding forward (K5) inside the step; auto = the bge model whose width is the corpus dim")
    ap.add_argument("--query-tokens", type=int, default=32, help="WordPiece tokens per query incl. [CLS]/[SEP]")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-optin", action="store_true", help="skip the extra OPT-IN measurement (bf16 shadow prune pass) after the default one")
    ap.add_argument("--cpu-sample-rows", type=int, default=40_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the last timed step returned to DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """arrays: name -> [B, ...] results of one step.  The fuse kernel marks a score that does not exist (a candidate only
    one list found, a slot past count) with NaN: every float array is stored with those entries as 0 and a 0/1 mask
    <name>_present.npy, so all files are finite.  Integer arrays are stored as float64 (exact below 2^53).  Above
    DUMP_LIMIT bytes in all, a fixed seeded sample of the B rows is stored, with its row indices as rows.npy."""
    out = {}
    for n, a in arrays.items():
        if a.dtype.kind == "f":
            ok = np.isfinite(a)
            out[n], out[n + "_present"] = np.where(ok, a, 0).astype(a.dtype), ok.astype(np.float32)
        else:
            out[n] = a.astype(np.float64)
    arrays = out
    B = len(next(iter(arrays.values())))
    per_row = sum(a.nbytes for a in arrays.values()) / B
    if per_row * B > DUMP_LIMIT:
        rows = np.sort(np.random.default_rng(0).choice(B, int((DUMP_LIMIT - 65536) // (per_row + 8)), replace=False))   # .npy headers
        arrays = {n: a[rows] for n, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(out_dir, n + ".npy"), a)


# ------------------------------------------------------------------------- helpers
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synth_query_terms(batch, seed, vocab=VOCAB, s=1.07, rank_offset=100):
    """3-8 power-law terms per query, skipping the stop-word-like head (SURVEY.md section 8d)."""
    g = np.random.default_rng(seed)
    out = []
    lo, hi = float(rank_offset + 1) ** (1 - s), float(vocab + 1) ** (1 - s)
    for _ in range(batch):
        m = int(g.integers(3, 9))
        x = (lo + g.random(m) * (hi - lo)) ** (1.0 / (1 - s))
        out.append(np.clip(x.astype(np.int64) - 1, 0, vocab - 1).astype(np.uint32))
    return out


# ------------------------------------------------------------------ CPU baseline (oracle)
class CpuReference:
    """Restated reference path (oracle: FAISS-flat scan + bm25s-lucene + _fuse) on all host cores, on a bounded SAMPLE of the
    workload: the same number of queries per step as the GPU arm (global_batch), a row sample of the corpus.  Both stages
    are O(N) per query, so the per-query time on the full corpus is the sample's time scaled by n_docs / sample_rows; the
    line reports the MEASURED step time of the sample (ms_per_step, measured.*) and the extrapolated queries/s (value).
    Postings are prebuilt (the reference rebuilds them on every query -- slower still, reported separately as
    bm25_rebuild_per_query_s_extrapolated)."""

    def __init__(self, n_docs, dim, hybrid, k, sample_rows, n_queries=256, seed=0, embedding=None, query_tokens=32):
        from oracle import oracle as o
        o.build()
        self.threads = o.set_threads(os.cpu_count() or 1)       # torchrun pins OMP_NUM_THREADS=1 for its children
        self.embed_s = 0.0
        self.embedding = embedding
        if embedding:
            # the reference embeds every query with torch BertModel on the CPU (huggingface_local_embedding.py:34-53)
            import torch
            from transformers import BertConfig, BertModel
            if os.environ.get("OMP_NUM_THREADS") == "1" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
                # torchrun pins OMP_NUM_THREADS=1 for its children: give torch what it takes by default in a plain process
                # (one thread per physical core), so the reference arm does not depend on how it was launched
                torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))
            self.torch_threads = torch.get_num_threads()
            torch.manual_seed(0)
            m = BertModel(BertConfig(**BGE[embedding]), add_pooling_layer=False).eval()
            ne = min(16, n_queries)
            ids = torch.randint(0, 30522, (ne, query_tokens))
            with torch.no_grad():
                m(input_ids=ids[:1])
                t0 = time.perf_counter()
                for b in range(ne):             # one query per request, as the service receives them
                    torch.nn.functional.normalize(m(input_ids=ids[b:b + 1]).last_hidden_state[:, 0], dim=1)
                self.embed_s = (time.perf_counter() - t0) / ne
            del m
        self.o, self.n_docs, self.dim, self.hybrid, self.k, self.nq = o, n_docs, dim, hybrid, k, n_queries
        self.n = int(min(sample_rows, n_docs))
        g = np.random.default_rng(seed + 1)                      # unit-norm Gaussian rows (the statistics of the GPU arm's corpus)
        self.x = g.standard_normal((self.n, dim), dtype=np.float32)
        self.x /= np.linalg.norm(self.x, axis=1, keepdims=True)
        self.q = o.synth_queries(self.x, n_queries, seed + 2)
        self.P = o.pool_size(k)
        self.rebuild_s = None
        if hybrid:
            vocab = 1 << 16
            self.ns = min(self.n, 20_000)
            off, ids, tf, dl = o.synth_sparse(self.ns, vocab, seed + 3)
            t0 = time.perf_counter()
            self.post = o.bm25_build(off, ids, tf, dl, vocab)
            self.rebuild_s = (time.perf_counter() - t0) * (n_docs / self.ns)
            self.qs = o.synth_query_terms(vocab, n_queries, seed + 4)
        o.dense_topk(self.x, self.q[:1], self.P)  # warm: page-touch the sample, start the OpenMP team
        self.last_step_s = None

    def step(self):
        """one pass of n_queries queries over the sample; returns extrapolated seconds per query at n_docs"""
        o = self.o
        t00 = t0 = time.perf_counter()
        dd, do = o.dense_topk(self.x, self.q, self.P)
        t_dense = (time.perf_counter() - t0) / self.nq
        t_sparse = 0.0
        if self.hybrid:
            t0 = time.perf_counter()
            for b in range(self.nq):
                bs, bo = o.bm25_query(self.post, self.qs[b], self.P)
                o.fuse(dd[b], do[b], bs, bo, self.k)
            t_sparse = (time.perf_counter() - t0) / self.nq * (self.n_docs / self.ns)
        self.last_step_s = time.perf_counter() - t00 + self.embed_s * self.nq      # what this step cost on the SAMPLE (+ embedding)
        return t_dense * (self.n_docs / self.n) + t_sparse + self.embed_s

    def describe(self, per_query, step_s=None):
        return {"value": 1.0 / per_query, "unit": "queries/s", "cores": self.threads, "kind": "port",
                "sample": f"oracle (restated FAISS-flat + bm25s + _fuse; the real wheels are not installable offline) on "
                          f"{self.n} of {self.n_docs} rows x {self.dim} fp32 (BM25: {getattr(self, 'ns', 0)} docs), {self.nq} queries per "
                          f"step, {self.threads} host threads, prebuilt postings; value is extrapolated linearly in N, measured.* is not",
                "measured": {"rows": self.n, "queries_per_step": self.nq, "step_s": step_s,
                             "queries_per_s_on_sample": None if not step_s else self.nq / step_s},
                "per_query_s_extrapolated": per_query,
                "query_embedding_s": self.embed_s if self.embedding else None,
                "query_embedding": f"torch CPU BertModel {self.embedding} shapes on {getattr(self, 'torch_threads', '?')} threads, measured per query, not extrapolated" if self.embedding else "excluded",
                "bm25_rebuild_per_query_s_extrapolated": self.rebuild_s}


def cpu_reference_qps(n_docs, dim, hybrid, k, sample_rows, embedding=None, query_tokens=32, n_queries=256):
    ref = CpuReference(n_docs, dim, hybrid, k, sample_rows, n_queries=n_queries, embedding=embedding, query_tokens=query_tokens)
    ref.step()
    ts, ss = [], []
    for _ in range(3):
        ts.append(ref.step()); ss.append(ref.last_step_s)
    return ref.describe(float(np.median(ts)), float(np.median(ss)))


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) timed on the host cores, same queries per step as the GPU arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    docs, dim, hybrid = WORKLOADS[args.workload]
    ref = CpuReference(docs, dim, hybrid, args.k, args.cpu_sample_rows, n_queries=args.batch, embedding=pick_embedding(args.embedding, dim),
                       query_tokens=args.query_tokens)
    for _ in range(args.warmup):
        ref.step()
    pq, st = [], []
    for _ in range(args.steps):
        pq.append(ref.step()); st.append(ref.last_step_s)
    per_query, step_s = float(np.mean(pq)), float(np.mean(st))
    v = 1.0 / per_query
    line = {"impl": "reference", "metric": "rag_retrieve_queries_per_sec", "value": v, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * step_s,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {docs} docs x {dim} fp32" + (" + BM25 postings, hybrid weighted fusion" if hybrid else ", dense only"),
                       "top_k": args.k, "global_batch": ref.nq, "parallelism": f"{ref.threads} host threads",
                       "timed_sample": f"ms_per_step is the MEASURED time of one step on the sample ({ref.n} rows); value = queries/s "
                                       f"extrapolated to {docs} rows (x{docs / ref.n:.0f} on the O(N) stages)",
                       "query_embedding": ref.describe(per_query)["query_embedding"]},
            "cpu_baseline": ref.describe(per_query, step_s),
            "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ in-bench correctness check (every N)
def _key_values(keys, desc):
    """u64 candidate keys (include/kaito_rag.h) -> (fp32 values, ordinals); KRAG_KEY_PAD entries come back as ordinal -1"""
    keys = np.asarray(keys).astype(np.uint64)
    hi = (keys >> np.uint64(32)).astype(np.uint32)
    if desc:
        hi = ~hi
    u = np.where(hi & np.uint32(0x80000000), hi & np.uint32(0x7FFFFFFF), ~hi).astype(np.uint32)
    vals = u.view(np.float32)
    ords = (keys & np.uint64(0xFFFFFFFF)).astype(np.int64)
    ords[keys == np.uint64(0xFFFFFFFFFFFFFFFF)] = -1
    return vals, ords


def _host_fuse(dd, do, bs, bo, k, w_v=0.7, w_t=0.3):
    """HybridRetriever._fuse (hybrid_retriever.py:132-166) in numpy doubles: final = w_v*L2^2 + w_t/(1+rank), sorted by
    (final desc, ordinal asc), cut to k.  Checker only."""
    tot = w_v + w_t
    w_v, w_t = w_v / tot, w_t / tot
    vec = {int(o): float(np.float32(d)) for d, o in zip(dd, do) if o >= 0}
    rank = {}
    for r, o in enumerate(int(o) for o in bo if o >= 0):
        rank.setdefault(o, r)
    ids = sorted(set(vec) | set(rank))
    fin = [(w_v * vec.get(i, 0.0) + (w_t * (1.0 / (1.0 + rank[i])) if i in rank else 0.0), i) for i in ids]
    fin.sort(key=lambda t: (-t[0], t[1]))
    return fin[:k]


def sharded_check(ix, sr, stages, qh, qpad, terms_list, d_terms, d_toff, offs, k, P, hybrid, world, rank, dev, n_check=16):
    """Independent of the exchange: every rank runs the EXACT fp32 scan (K1, batch < 16) and its BM25 kernel on its own shard
    through the host-buffer C ABI; the per-shard lists are gathered as Python objects and merged on the host; numpy fuses.
    The pipeline under test (K2 prune/rescore -> P2P or NCCL exchange -> merge -> fuse kernel) must return the same ids and the
    same fp64 scores for the checked queries.  recall@10 = overlap of the pipeline's dense top-10 with the exact top-10."""
    import torch
    import torch.distributed as dist
    B = qh.shape[0]
    half = max(1, n_check // 2)
    sel = sorted(set(list(range(min(half, B))) + [min(B - 1, B // 2 + i) for i in range(half)]))
    dl, ol = [], []
    for i in range(0, len(sel), 8):                       # batches of 8: below the tensor-core threshold -> K1
        d_, o_ = ix.search_dense(qh[sel[i:i + 8]], P)
        dl.append(d_); ol.append(o_)
    mine = {"dd": np.concatenate(dl), "do": np.concatenate(ol)}
    if hybrid:
        mine["bs"], mine["bo"] = ix.search_bm25([terms_list[i] for i in sel], P)
    parts = [None] * world
    if world > 1:
        dist.all_gather_object(parts, mine)
    else:
        parts = [mine]
    out = sr.retrieve_dev(qpad, d_terms, d_toff, k, toff_host=offs if hybrid else None)
    torch.cuda.synchronize()
    merged = sr.last_lists
    got_ord = out["ordinal"].cpu().numpy(); got_fin = out["final"].cpu().numpy(); got_cnt = out["count"].cpu().numpy()
    dense_keys = merged[0].cpu().numpy()
    if rank != 0:
        return None
    ids_ok = fin_ok = dense_ok = True
    rec = []
    for j, qi in enumerate(sel):
        cd = np.concatenate([p["dd"][j] for p in parts]); co = np.concatenate([p["do"][j] for p in parts])
        keep = co >= 0
        order = np.lexsort((co[keep], cd[keep]))[:P]
        ex_d, ex_o = cd[keep][order], co[keep][order]
        pv, po = _key_values(dense_keys[qi], desc=False)
        dense_ok &= bool(np.array_equal(po[: len(ex_o)], ex_o) and np.array_equal(pv[: len(ex_o)], ex_d))
        rec.append(len(set(po[:10].tolist()) & set(ex_o[:10].tolist())) / float(min(10, len(ex_o)) or 1))
        if hybrid:
            cs = np.concatenate([p["bs"][j] for p in parts]); cb = np.concatenate([p["bo"][j] for p in parts])
            kb = cb >= 0
            ob = np.lexsort((cb[kb], -cs[kb].astype(np.float64)))[:P]
            want = _host_fuse(ex_d, ex_o, cs[kb][ob], cb[kb][ob], k)
        else:
            want = [(float(np.float32(d)), int(o)) for d, o in zip(ex_d[:k], ex_o[:k])]
        c = int(got_cnt[qi])
        ids_ok &= (c == len(want)) and [int(x) for x in got_ord[qi, :c]] == [w[1] for w in want]
        fin_ok &= (c == len(want)) and [float(x) for x in got_fin[qi, :c]] == [w[0] for w in want]
    return {"queries": len(sel), "dense_lists_equal_exact_scan": bool(dense_ok), "fused_ids_equal": bool(ids_ok),
            "fused_scores_equal": bool(fin_ok), "recall_at_10": float(np.mean(rec)),
            "method": "per-shard exact fp32 scan (K1) + BM25 through the host-buffer C ABI, host merge + numpy fuse, vs the "
                      "timed pipeline (K2 -> exchange -> merge -> fuse kernel) on the same queries"}


# --------------------------------------------------------------------------- our arm
def trace(msg):
    """phase markers on stderr (KRAG_BENCH_TRACE=1): which phase a rank was in when a run dies"""
    if os.environ.get("KRAG_BENCH_TRACE", "1") != "0":
        sys.stderr.write(f"[bench rank {os.environ.get('RANK', '0')} +{time.perf_counter() - _T0:7.2f}s] {msg}\n")
        sys.stderr.flush()


_T0 = time.perf_counter()


def run_ours(args):
    import faulthandler
    faulthandler.enable(all_threads=True)      # a SIGABRT/SIGSEGV inside a native library prints the Python stacks
    import torch
    import torch.distributed as dist
    from kaito_b200 import _native
    from kaito_b200.sharded import NativeStages, ShardedRetriever, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    docs, dim, hybrid = WORKLOADS[args.workload]
    lo, hi = shard_range(docs, world, rank)
    n_local = hi - lo
    k, B = args.k, args.batch
    P = int(k * 3.0)

    ctx = _native.Context(device_id=local_rank, rank=rank, world_size=world, dense_mode=args.dense_mode)
    ix = ctx.create_index("bench", dim)
    t_build = time.perf_counter()
    ix.synth_fill(n_local, row_base=lo, seed=20260921, vocab=VOCAB if hybrid else 0)
    stages = NativeStages(ctx, ix)
    st = ix.stats()
    sr = ShardedRetriever(stages, dev, st.dim_padded)
    if hybrid:
        free_b, total_b = torch.cuda.mem_get_info(dev)
        trace(f"rows + raw term lists resident: {free_b / 1e9:.1f} of {total_b / 1e9:.1f} GB free before the postings build")
        sr.commit(VOCAB, n_local)
        free_b, _ = torch.cuda.mem_get_info(dev)
        trace(f"postings built: {free_b / 1e9:.1f} GB free")
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t_build
    trace(f"index built in {t_build:.1f}s")
    st = ix.stats()

    # queries: half planted (perturbed corpus rows of rank 0's shard), half random; same on every rank
    g = np.random.default_rng(7)
    qh = g.standard_normal((B, dim)).astype(np.float32)
    planted = np.sort(g.integers(0, min(n_local, shard_range(docs, world, 0)[1]), B // 2))
    if rank == 0 and B >= 2:
        rows = np.concatenate([ix.read_rows(int(r), 1) for r in planted])
        qh[: B // 2] = rows + 0.1 * qh[: B // 2] / np.sqrt(dim)
    qh /= np.linalg.norm(qh, axis=1, keepdims=True)
    qt = torch.from_numpy(qh).to(dev)
    if world > 1:
        dist.broadcast(qt, 0)
        qh = qt.cpu().numpy()
    terms_list = synth_query_terms(B, 11) if hybrid else None
    qpad = torch.zeros((B, st.dim_padded), dtype=torch.float32, device=dev)
    qpad[:, :dim] = qt
    if hybrid:
        offs = np.zeros(B + 1, np.int32)
        for i, t in enumerate(terms_list):
            offs[i + 1] = offs[i] + len(t)
        flat = np.concatenate(terms_list)
        d_terms = torch.from_numpy(flat.view(np.int32)).to(dev)
        d_toff = torch.from_numpy(offs).to(dev)
        n_terms = int(offs[-1])
    else:
        d_terms = d_toff = None
        n_terms = 0

    emb_name = pick_embedding(args.embedding, dim)
    embedder = flat_tok = tok_off = None
    if emb_name:
        ecfg = BGE[emb_name]
        embedder = _native.Embedder(ctx, ecfg["num_hidden_layers"], ecfg["hidden_size"], ecfg["num_attention_heads"],
                                    ecfg["intermediate_size"], ecfg["vocab_size"])
        embedder.load_state_dict(random_bert_state(ecfg))
        tok_lists = [np.random.default_rng(100 + b).integers(1000, 30000, args.query_tokens) for b in range(B)]
        flat_tok, tok_off = _native.Embedder.pack(tok_lists)
        flat_tok1, tok_off1 = _native.Embedder.pack(tok_lists[:1])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_dev():   # token ids (host, 32 KB) -> K5 embeddings on the device -> candidates -> merge -> fuse
        if embedder:
            sr.embed_into(embedder, flat_tok, tok_off, qpad)      # queries split across ranks + one all-gather
        return sr.retrieve_dev(qpad, d_terms, d_toff, k, toff_host=offs if hybrid else None)

    def step_e2e():   # host buffers in (token ids or vectors, term ids), host results out
        if embedder:
            return sr.retrieve(None, terms_list, k, embedder=embedder, tokens=(flat_tok, tok_off))
        return sr.retrieve(qh, terms_list, k)

    last = {}

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last["out"] = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count()
    trace("timed ms_dev")
    ms_dev = timed(step_dev, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:          # the result buffers are reused by the legs below: copy them out now
        dump_outputs(args.dump_outputs, {n: t.cpu().numpy() for n, t in last["out"].items()})
    launches = (ctx.launch_count() - l0) // (args.steps + args.warmup) * args.steps
    trace("timed ms_e2e")
    ms_e2e = timed(step_e2e, args.steps, args.warmup)
    # batch-1 (latency mode)
    q1, t1 = qpad[:1], None
    if hybrid:
        d_t1 = torch.from_numpy(terms_list[0].view(np.int32)).to(dev)
        offs1 = np.array([0, len(terms_list[0])], np.int32)
        d_o1 = torch.from_numpy(offs1).to(dev)
    def step_b1():
        if embedder:
            embedder.embed_dev(flat_tok1, tok_off1, q1.data_ptr(), st.dim_padded, stages.stream())
        return sr.retrieve_dev(q1, d_t1 if hybrid else None, d_o1 if hybrid else None, k, toff_host=offs1 if hybrid else None)

    def step_b1_e2e():
        if embedder:
            return sr.retrieve(None, terms_list[:1] if hybrid else None, k, embedder=embedder, tokens=(flat_tok1, tok_off1))
        return sr.retrieve(qh[:1], terms_list[:1] if hybrid else None, k)

    trace("timed ms_b1")
    ms_b1 = timed(step_b1, args.steps * 4, args.warmup)
    trace("timed ms_b1_e2e")
    ms_b1_e2e = timed(step_b1_e2e, args.steps * 4, args.warmup)
    ms_embed = ms_embed1 = None
    if embedder:
        trace("timed ms_embed")
        ms_embed = timed(lambda: sr.embed_into(embedder, flat_tok, tok_off, qpad), args.steps, args.warmup)
        trace("timed ms_embed1")
        ms_embed1 = timed(lambda: embedder.embed_dev(flat_tok1, tok_off1, q1.data_ptr(), st.dim_padded, stages.stream()), args.steps * 4, args.warmup)
        qpad[:, :dim] = qt      # restore the planted/random query vectors for the stage timings below
    # dominant kernel: the dense candidate stage alone; the library brackets the kernel itself with
    # CUDA events on the launching stream (krag_last_dense_kernel), read after each timed region
    keys = torch.empty((B, P), dtype=torch.int64, device=dev)
    trace("timed ms_dense")
    ms_dense = timed(lambda: stages.dense_candidates(qpad, P, keys), args.steps, args.warmup)
    kern_ms, kern_id, kern_bytes, kern_flops = _native.last_dense_kernel()
    trace("timed ms_dense1")
    ms_dense1 = timed(lambda: stages.dense_candidates(q1, P, keys[:1]), args.steps * 4, args.warmup)
    kern1_ms, kern1_id, kern1_bytes, _ = _native.last_dense_kernel()
    ms_bm25 = None
    if hybrid:
        trace("timed ms_bm25")
        ms_bm25 = timed(lambda: stages.bm25_candidates(d_terms, d_toff, B, P, keys, offs), args.steps, args.warmup)
    # K3 roofline: algorithmic bytes per batch = 8 * sum over the query terms of df_local(t) (SURVEY.md section 8d: u32 doc + f32
    # score per posting); the stage time is CUDA-event bracketed above (resolve + sample pass + select + main pass + select + fill)
    k3 = None
    if hybrid:
        sum_df = 0
        for t in np.unique(np.concatenate(terms_list)):
            sum_df += int(ix.read_postings(int(t), cap=1)[2]) * int(sum(int((tl == t).sum()) for tl in terms_list))
        k3 = {"sum_df_local": sum_df, "algorithmic_bytes_per_batch": 8 * sum_df, "stage_ms": ms_bm25 / args.steps}
    fallbacks = int(_native.load().krag_tc_fallback_queries())
    clocks = sampler.stop() if rank == 0 else None

    # OPT-IN leg, reported beside (never instead of) the default: the same step with K2's prune pass reading a bf16
    # shadow of the corpus (+50% memory, built here by one conversion pass); returned distances stay exact fp32.
    trace("default legs done")
    optin = None
    if args.dense_mode == 0 and not args.no_optin and kern_id in (2, 3, 5):
        t_sh = time.perf_counter()
        ix.set_dense_mode(_native.DENSE_TC_BF16)
        t_sh = time.perf_counter() - t_sh
        trace("timed ms_opt")
        ms_opt = timed(step_dev, args.steps, args.warmup)
        trace("timed ms_opt_dense")
        ms_opt_dense = timed(lambda: stages.dense_candidates(qpad, P, keys), args.steps, args.warmup)
        ko_ms, ko_id, ko_bytes, _ = _native.last_dense_kernel()
        optin = {"what": "KRAG_DENSE_TC_BF16: K2 prune pass over a bf16 shadow of the fp32 corpus (+50% memory); exact fp32 rescoring "
                         "and certificate unchanged, ids/scores bit-identical to the default",
                 "value": B * args.steps / (ms_opt * 1e-3), "unit": "queries/s", "ms_per_step": ms_opt / args.steps,
                 "dense_stage_ms": ms_opt_dense / args.steps, "dense_kernel_ms": ko_ms,
                 "dense_kernel_gbs": ko_bytes / (ko_ms * 1e-3) / 1e9, "shadow_build_s": t_sh,
                 "tc_certificate_fallback_queries": int(_native.load().krag_tc_fallback_queries()) - fallbacks}
        ix.set_dense_mode(args.dense_mode, release_shadow=True)

    # correctness inside the bench, at every N: the sharded pipeline against per-shard exact scans merged on the host
    trace("sharded check")
    qpad[:, :dim] = qt                              # the embedding legs left K5 outputs in qpad: check with the planted/random vectors
    chk = sharded_check(ix, sr, stages, qh, qpad, terms_list, d_terms, d_toff, offs if hybrid else None, k, P, hybrid, world, rank, dev)
    recall = None
    if rank == 0 and B >= 2:                       # planted rows (rank 0's shard) come back as nearest neighbour
        m = min(8, B // 2)
        _, ord_b = ix.search_dense(qh[:m], k)
        recall = float(np.mean(ord_b[:, 0] == planted[:m] + lo))

    if rank == 0:
        peak, peak_src = load_peaks()
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
        gbs = kern_bytes / (kern_ms * 1e-3) / 1e9
        gbs1 = kern1_bytes / (kern1_ms * 1e-3) / 1e9
        tflops = kern_flops / (kern_ms * 1e-3) / 1e12
        tf32_peak = float(peaks.get("bf16_tflops", 1590.0)) / 2.0   # TF32 dense = half the measured bf16 rate
        if kern_id in (4, 5):     # kind::f16 prune pass (bf16 operands), timed back to back: the sustained bf16 figure
            tensor_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
            tensor_peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kind::f16 MMAs)"
        else:
            tensor_peak, tensor_peak_src = tf32_peak, "MEASURED_PEAKS.json bf16_tflops / 2 (TF32 dense rate)"
        # dram__bytes_read.sum + dram__bytes_write.sum of the same kernel on the same workload from the committed
        # ncu --set full capture (profiles/traffic.json names the report); null when no capture matches this run
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath) and world == 1:
            traffic = json.load(open(tpath)).get(args.workload, {}).get(str(kern_id))
        kname = {1: "K1 dense_scan_kernel (exact fp32 L2^2 scan + fused top-P)",
                 2: "K2 dense_tc_kernel (tcgen05 cta_group::1 TF32 prune pass; exact fp32 rescoring follows)",
                 3: "K2 dense_tc2_kernel (tcgen05 cta_group::2 TF32 prune pass, CTA pairs; exact fp32 rescoring follows)",
                 5: "K2 dense_tc2cvt_kernel (tcgen05 cta_group::2 kind::f16 prune pass; fp32 corpus rows staged by TMA and rounded to bf16 in shared memory -- no shadow copy, 4 B/element from HBM; exact fp32 rescoring follows)",
                 4: "K2 dense_tc2_kernel<bf16> (OPT-IN: prune pass over a bf16 shadow of the corpus, kind::f16; exact fp32 rescoring of the fp32 corpus follows)"}
        qps = B * args.steps / (ms_dev * 1e-3)
        qps_e2e = B * args.steps / (ms_e2e * 1e-3)
        h2d, d2h = ShardedRetriever.io_bytes(B, dim, n_terms, k)
        embed_info = None
        if embedder:
            h2d = int(flat_tok.nbytes + tok_off.nbytes + n_terms * 4 + (B + 1) * 4)   # token ids replace the query vectors
            fl = bert_flops(BGE[emb_name], args.query_tokens) * B
            etf = fl / (ms_embed / args.steps * 1e-3) / 1e12
            embed_info = {"model_shape": emb_name, "weights": "random init N(0, 0.02) (no checkpoints offline)", "tokens_per_query": args.query_tokens,
                          "batch_ms": ms_embed / args.steps, "batch1_ms": ms_embed1 / (args.steps * 4), "flops_per_batch": fl,
                          "tflops": etf, "tflops_per_gpu": etf / world,
                          "arithmetic": "split-fp16 operands (hi + lo*2^-11), 3 kind::f16 MMAs per step: fp32-accurate products; "
                                        "tflops counts the fp32-equivalent flops L(24 S d^2 + 4 S^2 d), the tensor pipe executes 3x the GEMM part",
                          "tensor_frac_of_f16_peak_per_gpu": 3.0 * etf / world / float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0))),
                          "queries_per_s": B / (ms_embed / args.steps * 1e-3)}
        line = {
            "metric": "rag_retrieve_queries_per_sec", "value": qps, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {docs} docs x {dim} fp32 resident" + (" (+ bf16 shadow for the prune pass: OPT-IN mode, not the default)" if args.dense_mode == 3 else "") +
                                   (f" + BM25 postings nnz={st.nnz} (local), vocab 2^20, hybrid weighted fusion" if hybrid else ", dense only"),
                       "global_batch": B, "top_k": k, "candidate_pool": P, "parallelism": f"doc-shard x{world}",
                       "rows_per_gpu": n_local, "cache": "inputs larger than L2 (corpus >> 126 MB); no explicit flush",
                       "query_embedding": (f"K5 BERT forward ({emb_name} shapes, {args.query_tokens} tokens/query, random-init weights) "
                                           "INSIDE the timed region of value, e2e and batch1") if embedder else
                                          "precomputed query vectors (embedding forward not in the timed region)",
                       "dense_kernel": kname[kern_id], "dense_kernel_batch1": kname[kern1_id],
                       "tc_certificate_fallback_queries": fallbacks,
                       "index_build_s": t_build},
            "e2e": {"value": qps_e2e, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "batch1": {"value": args.steps * 4 / (ms_b1 * 1e-3), "e2e": args.steps * 4 / (ms_b1_e2e * 1e-3), "unit": "queries/s",
                       "ms_per_query": ms_b1 / (args.steps * 4), "dense_kernel_ms": kern1_ms, "dense_kernel_gbs": gbs1, "dense_frac": gbs1 / peak},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "traffic": traffic,
                         "kernel": kname[kern_id], "peak_source": peak_src, "kernel_ms": kern_ms,
                         "algorithmic_bytes_per_launch": kern_bytes, "flops_per_launch": kern_flops,
                         "tensor_tflops": tflops, "tensor_peak": tensor_peak, "tensor_frac": tflops / tensor_peak,
                         "tensor_peak_source": tensor_peak_src,
                         "dense_stage_ms": ms_dense / args.steps, "bm25_stage_ms": None if ms_bm25 is None else ms_bm25 / args.steps},
            "roofline_k3": None if k3 is None else {
                "bound": "hbm", "kernel": "K3 bm25_warp_kernel (sampled-threshold pass + main pass; stage = resolve + 2 passes + 2 selects + fill)",
                "achieved": k3["algorithmic_bytes_per_batch"] / (k3["stage_ms"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": k3["algorithmic_bytes_per_batch"] / (k3["stage_ms"] * 1e-3) / 1e9 / peak, "stage_ms": k3["stage_ms"],
                "algorithmic_bytes_per_batch": k3["algorithmic_bytes_per_batch"], "postings_per_batch": k3["sum_df_local"],
                "note": "algorithmic bytes = 8 B x sum of df_local over the batch's query terms; the whole stage time is the denominator"},
            "embed": embed_info, "optin_bf16_shadow": optin,
            "clocks": clocks, "planted_top1_hit": recall, "recall_at_10": chk["recall_at_10"], "check": chk,
            "recall_note": "computed: overlap of the pipeline's dense top-10 with the exact per-shard fp32 scan merged on the host (check.queries queries)",
        }
        if not args.no_cpu_baseline and world == 1:      # the CPU leg is reported at N = 1 only (rank 0 would stall the other ranks)
            line["cpu_baseline"] = cpu_reference_qps(docs, dim, hybrid, k, args.cpu_sample_rows, emb_name, args.query_tokens, n_queries=B)
        print(json.dumps(line), flush=True)
    trace("line printed; teardown")
    barrier()
    if embedder:
        embedder.destroy()
    ix.drop()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
