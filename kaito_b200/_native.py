"""ctypes binding of libkaito_rag.so (include/kaito_rag.h).

The CUDA library IS the product path: there is no CPU or PyTorch fallback.  Importing this
module without the built library, or initialising it without an sm_100 GPU, raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkaito_rag.so")

KRAG_OK = 0
KRAG_E_INVALID, KRAG_E_NO_DEVICE, KRAG_E_CUDA, KRAG_E_OOM = -1, -2, -3, -4
KRAG_E_NOT_FOUND, KRAG_E_STATE, KRAG_E_IO, KRAG_E_UNSUPPORTED = -5, -6, -7, -8
KRAG_KEY_PAD = 0xFFFFFFFFFFFFFFFF
KRAG_MAX_TOP_K = 300
KRAG_MAX_POOL = 1024
FUSION_REFERENCE, FUSION_SIMILARITY = 0, 1
FILTER_PUSHDOWN = 0x100   # OR into fusion_mode: the allow bitmap restricts the dense and BM25 scans themselves
DENSE_AUTO, DENSE_SCAN, DENSE_TC, DENSE_TC_BF16, DENSE_TC_TF32 = 0, 1, 2, 3, 4

# every symbol include/kaito_rag.h declares (tests check the export table against this)
SYMBOLS = [
    "krag_version", "krag_last_error", "krag_init", "krag_shutdown", "krag_launch_count", "krag_ctx_stream",
    "krag_index_create", "krag_index_drop", "krag_index_reserve", "krag_index_add", "krag_index_remove",
    "krag_index_commit", "krag_index_commit_local", "krag_index_commit_global", "krag_index_stats",
    "krag_index_node_ids", "krag_index_set_ordinal_map", "krag_index_persist", "krag_index_load", "krag_search_dense", "krag_search_bm25",
    "krag_retrieve", "krag_dev_dense_candidates", "krag_dev_bm25_candidates", "krag_dev_merge", "krag_dev_fuse",
    "krag_synth_fill", "krag_index_read_rows", "krag_index_read_postings", "krag_index_read_rank_scores", "krag_tc_fallback_queries",
    "krag_debug_tc_dump", "krag_last_dense_kernel", "krag_embedder_create", "krag_embedder_load_tensor",
    "krag_embedder_finalize", "krag_embed", "krag_embed_dev", "krag_embedder_destroy", "krag_debug_gemm_tf32",
    "krag_debug_linear_ln", "krag_index_set_dense_mode", "krag_text_analyze", "krag_wordpiece_create",
    "krag_wordpiece_encode_batch", "krag_wordpiece_destroy", "krag_p2p_create", "krag_p2p_connect", "krag_dev_exchange_merge", "krag_p2p_destroy",
]


class KragError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libkaito_rag error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("device_id", C.c_int32), ("rank", C.c_int32), ("world_size", C.c_int32), ("dense_mode", C.c_int32),
                ("search_slots", C.c_int32), ("reserved", C.c_int32 * 3)]


class Stats(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_live", C.c_int64), ("nnz", C.c_int64), ("n_docs_global", C.c_int64),
                ("total_len_global", C.c_int64), ("vocab", C.c_int64), ("ordinal_base", C.c_int64), ("dim", C.c_int32),
                ("dim_padded", C.c_int32), ("committed", C.c_int32), ("reserved", C.c_int32),
                ("device_bytes", C.c_int64)]


class BertConfig(C.Structure):
    _fields_ = [("layers", C.c_int32), ("hidden", C.c_int32), ("heads", C.c_int32), ("intermediate", C.c_int32),
                ("vocab", C.c_int32), ("max_position", C.c_int32), ("type_vocab", C.c_int32), ("ln_eps", C.c_float)]


_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library; fail loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(make -C kaito_b200/csrc). kaito_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_double
    L.krag_version.restype = i32
    L.krag_last_error.restype = C.c_char_p
    L.krag_init.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.krag_shutdown.argtypes = [vp]
    L.krag_launch_count.argtypes = [vp]
    L.krag_launch_count.restype = i64
    L.krag_ctx_stream.argtypes = [vp]
    L.krag_ctx_stream.restype = vp
    L.krag_index_create.argtypes = [vp, C.c_char_p, i32, C.POINTER(vp)]
    L.krag_index_drop.argtypes = [vp]
    L.krag_index_reserve.argtypes = [vp, i64, i64]
    L.krag_index_add.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp]
    L.krag_index_remove.argtypes = [vp, i64, vp, C.POINTER(i64)]
    L.krag_index_commit.argtypes = [vp, i64]
    L.krag_index_commit_local.argtypes = [vp, i64, vp, C.POINTER(i64), C.POINTER(i64)]
    L.krag_index_commit_global.argtypes = [vp, i64, vp, i64, i64, i64]
    L.krag_index_stats.argtypes = [vp, C.POINTER(Stats)]
    L.krag_index_set_ordinal_map.argtypes = [vp, i64, i64]
    L.krag_index_node_ids.argtypes = [vp, i64, vp, vp]
    L.krag_index_persist.argtypes = [vp, C.c_char_p]
    L.krag_index_load.argtypes = [vp, C.c_char_p, C.c_char_p, C.POINTER(vp)]
    L.krag_search_dense.argtypes = [vp, i32, vp, i32, vp, vp]
    L.krag_search_bm25.argtypes = [vp, i32, vp, vp, i32, vp, vp]
    L.krag_retrieve.argtypes = [vp, i32, vp, vp, vp, i32, f64, f64, f64, i32, vp, i64, vp, vp, vp, vp, vp, vp]
    L.krag_dev_dense_candidates.argtypes = [vp, i32, vp, i32, vp, vp]
    L.krag_dev_bm25_candidates.argtypes = [vp, i32, vp, vp, vp, i32, vp, vp]
    L.krag_dev_merge.argtypes = [vp, i32, i32, i32, vp, vp, vp]
    L.krag_dev_fuse.argtypes = [vp, i32, i32, i32, vp, vp, f64, f64, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.krag_synth_fill.argtypes = [vp, i64, i64, C.c_uint64, i64]
    L.krag_index_read_rows.argtypes = [vp, i64, i64, vp]
    L.krag_index_read_postings.argtypes = [vp, u32, i64, vp, vp, C.POINTER(i64)]
    L.krag_index_read_rank_scores.argtypes = [vp, u32, vp]
    L.krag_embedder_create.argtypes = [vp, C.POINTER(BertConfig), C.POINTER(vp)]
    L.krag_embedder_load_tensor.argtypes = [vp, C.c_char_p, vp, i64]
    L.krag_embedder_finalize.argtypes = [vp]
    L.krag_embed.argtypes = [vp, i32, vp, vp, vp]
    L.krag_embed_dev.argtypes = [vp, i32, vp, vp, vp, i32, vp]
    L.krag_embedder_destroy.argtypes = [vp]
    L.krag_debug_gemm_tf32.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, i32, vp]
    L.krag_debug_linear_ln.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, C.c_float, vp]
    L.krag_index_set_dense_mode.argtypes = [vp, i32, i32]
    L.krag_text_analyze.argtypes = [C.c_char_p, i64, vp, i64, C.POINTER(i64), C.POINTER(i32)]
    L.krag_wordpiece_create.argtypes = [C.c_char_p, i64, i32, C.POINTER(vp)]
    L.krag_wordpiece_encode_batch.argtypes = [vp, i64, C.c_char_p, vp, i32, vp, vp]
    L.krag_wordpiece_destroy.argtypes = [vp]
    L.krag_p2p_create.argtypes = [vp, i32, i32, i32, i32, C.POINTER(vp), vp]
    L.krag_p2p_connect.argtypes = [vp, vp]
    L.krag_dev_exchange_merge.argtypes = [vp, i32, i32, i32, vp, vp, vp]
    L.krag_p2p_destroy.argtypes = [vp]
    L.krag_tc_fallback_queries.restype = i64
    L.krag_last_dense_kernel.argtypes = [C.POINTER(C.c_float), C.POINTER(i32), C.POINTER(i64), C.POINTER(i64)]
    L.krag_debug_tc_dump.argtypes = [vp, i32, vp, vp, i64, C.POINTER(i64), C.POINTER(i32)]
    for name in SYMBOLS:
        fn = getattr(L, name)
        if fn.restype is C.c_int:  # default: every remaining call returns an int32 status
            fn.restype = i32
    _lib = L
    return L


def check(rc: int):
    if rc != KRAG_OK:
        raise KragError(rc, load().krag_last_error().decode("utf-8", "replace"))


def ptr(a):
    """numpy array / int address / None -> void*"""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.c_void_p(int(a))


def last_dense_kernel():
    """(ms, kernel_id, algorithmic_bytes, flops) of the dominant dense kernel of the last search."""
    ms, kid, by, fl = C.c_float(0), C.c_int32(0), C.c_int64(0), C.c_int64(0)
    check(load().krag_last_dense_kernel(C.byref(ms), C.byref(kid), C.byref(by), C.byref(fl)))
    return ms.value, kid.value, by.value, fl.value


class Context:
    """krag_ctx: one per process per GPU."""

    def __init__(self, device_id: int = 0, rank: int = 0, world_size: int = 1, dense_mode: int = DENSE_AUTO,
                 search_slots: int = 0):
        L = load()
        cfg = Config(device_id=device_id, rank=rank, world_size=world_size, dense_mode=dense_mode,
                     search_slots=search_slots)
        h = C.c_void_p()
        check(L.krag_init(C.byref(cfg), C.byref(h)))
        self._h, self._L = h, L
        self.device_id, self.rank, self.world_size = device_id, rank, world_size

    def close(self):
        if self._h:
            check(self._L.krag_shutdown(self._h))
            self._h = None

    def launch_count(self) -> int:
        return int(self._L.krag_launch_count(self._h))

    def stream(self) -> int:
        return int(self._L.krag_ctx_stream(self._h) or 0)

    def create_index(self, name: str, dim: int) -> "Index":
        h = C.c_void_p()
        check(self._L.krag_index_create(self._h, name.encode(), dim, C.byref(h)))
        return Index(self, h, name, dim)

    def load_index(self, name: str, path: str) -> "Index":
        h = C.c_void_p()
        check(self._L.krag_index_load(self._h, name.encode(), path.encode(), C.byref(h)))
        ix = Index(self, h, name, 0)
        ix.dim = ix.stats().dim
        return ix

    # ---- device-pointer stage API (multi-GPU host) ----
    def dev_merge(self, n_lists, batch, P, d_in, d_out, stream=0):
        check(self._L.krag_dev_merge(self._h, n_lists, batch, P, ptr(d_in), ptr(d_out), ptr(stream)))

    def dev_fuse(self, batch, P, k, d_dense, d_bm25, vw, tw, mode, d_allow, d_final, d_dense_out, d_sparse_out, d_rank,
                 d_ord, d_count, stream=0):
        check(self._L.krag_dev_fuse(self._h, batch, P, k, ptr(d_dense), ptr(d_bm25), vw, tw, mode, ptr(d_allow),
                                    ptr(d_final), ptr(d_dense_out), ptr(d_sparse_out), ptr(d_rank), ptr(d_ord),
                                    ptr(d_count), ptr(stream)))


class P2PExchange:
    """krag_p2p: candidate-list all-gather + merge over NVLink peer memory (our kernels, not NCCL)."""

    def __init__(self, ctx: "Context", rank: int, world: int, max_batch: int, max_P: int):
        self._L = ctx._L
        h = C.c_void_p()
        self.handle = np.zeros(64, np.uint8)
        check(self._L.krag_p2p_create(ctx._h, rank, world, max_batch, max_P, C.byref(h), ptr(self.handle)))
        self._h, self.world = h, world

    def connect(self, handles: np.ndarray):
        handles = np.ascontiguousarray(handles, np.uint8).reshape(self.world, 64)
        check(self._L.krag_p2p_connect(self._h, ptr(handles)))

    def exchange_merge(self, n_lists, batch, P, d_local, d_merged, stream=0):
        check(self._L.krag_dev_exchange_merge(self._h, n_lists, batch, P, ptr(d_local), ptr(d_merged), ptr(stream)))

    def destroy(self):
        if self._h:
            check(self._L.krag_p2p_destroy(self._h))
            self._h = None


class Embedder:
    """krag_embedder: BERT-family encoder forward on the GPU (K5)."""

    def __init__(self, ctx: "Context", layers, hidden, heads, intermediate, vocab, max_position=512, type_vocab=2,
                 ln_eps=1e-12):
        self.ctx, self._L, self.hidden = ctx, ctx._L, hidden
        cfg = BertConfig(layers, hidden, heads, intermediate, vocab, max_position, type_vocab, ln_eps)
        h = C.c_void_p()
        check(self._L.krag_embedder_create(ctx._h, C.byref(cfg), C.byref(h)))
        self._h = h

    def load_state_dict(self, state: dict):
        """state: Hugging Face BertModel names -> numpy fp32 arrays (pooler / position_ids entries are ignored)"""
        for name, arr in state.items():
            if name.startswith("pooler.") or name.endswith("position_ids"):
                continue
            a = np.ascontiguousarray(arr, np.float32)
            check(self._L.krag_embedder_load_tensor(self._h, name.encode(), ptr(a), a.size))
        check(self._L.krag_embedder_finalize(self._h))

    def embed(self, token_lists) -> np.ndarray:
        offs = np.zeros(len(token_lists) + 1, np.int32)
        for i, t in enumerate(token_lists):
            offs[i + 1] = offs[i] + len(t)
        flat = np.ascontiguousarray(np.concatenate([np.asarray(t, np.int32) for t in token_lists]), np.int32)
        out = np.empty((len(token_lists), self.hidden), np.float32)
        check(self._L.krag_embed(self._h, len(token_lists), ptr(flat), ptr(offs), ptr(out)))
        return out

    def embed_flat(self, flat_tokens: np.ndarray, offsets: np.ndarray) -> np.ndarray:
        """embed() for tokens that are already packed (int32 ids, int32 offsets [batch + 1])"""
        flat_tokens = np.ascontiguousarray(flat_tokens, np.int32); offsets = np.ascontiguousarray(offsets, np.int32)
        out = np.empty((len(offsets) - 1, self.hidden), np.float32)
        check(self._L.krag_embed(self._h, len(offsets) - 1, ptr(flat_tokens), ptr(offsets), ptr(out)))
        return out

    @staticmethod
    def pack(token_lists):
        offs = np.zeros(len(token_lists) + 1, np.int32)
        for i, t in enumerate(token_lists):
            offs[i + 1] = offs[i] + len(t)
        return np.ascontiguousarray(np.concatenate([np.asarray(t, np.int32) for t in token_lists]), np.int32), offs

    def embed_dev(self, flat_tokens: np.ndarray, offsets: np.ndarray, d_out: int, ld_out: int, stream: int = 0):
        """embeddings written to device memory (row stride ld_out floats); `stream` waits for them"""
        check(self._L.krag_embed_dev(self._h, len(offsets) - 1, ptr(flat_tokens), ptr(offsets), ptr(d_out), ld_out, ptr(stream)))

    def destroy(self):
        if self._h:
            check(self._L.krag_embedder_destroy(self._h))
            self._h = None


def debug_gemm_tf32(ctx: "Context", A, B, bias, residual=None, gelu=False) -> np.ndarray:
    A = np.ascontiguousarray(A, np.float32); B = np.ascontiguousarray(B, np.float32)
    bias = np.ascontiguousarray(bias, np.float32)
    if residual is not None:
        residual = np.ascontiguousarray(residual, np.float32)
    out = np.empty((A.shape[0], B.shape[0]), np.float32)
    check(load().krag_debug_gemm_tf32(ctx._h, A.shape[0], B.shape[0], A.shape[1], ptr(A), ptr(B), ptr(bias), ptr(residual),
                                      1 if gelu else 0, ptr(out)))
    return out


def debug_linear_ln(ctx: "Context", A, B, bias, residual, gamma, beta, eps=1e-12) -> np.ndarray:
    A = np.ascontiguousarray(A, np.float32); B = np.ascontiguousarray(B, np.float32)
    bias = np.ascontiguousarray(bias, np.float32); gamma = np.ascontiguousarray(gamma, np.float32)
    beta = np.ascontiguousarray(beta, np.float32)
    if residual is not None:
        residual = np.ascontiguousarray(residual, np.float32)
    out = np.empty((A.shape[0], B.shape[0]), np.float32)
    check(load().krag_debug_linear_ln(ctx._h, A.shape[0], B.shape[0], A.shape[1], ptr(A), ptr(B), ptr(bias), ptr(residual),
                                      ptr(gamma), ptr(beta), eps, ptr(out)))
    return out


class Index:
    """krag_index: one document shard (dense rows + BM25 postings) resident on one GPU."""

    def __init__(self, ctx: Context, handle, name: str, dim: int):
        self.ctx, self._h, self.name, self.dim = ctx, handle, name, dim
        self._L = ctx._L

    def drop(self):
        if self._h:
            check(self._L.krag_index_drop(self._h))
            self._h = None

    def reserve(self, rows: int, nnz: int = 0):
        check(self._L.krag_index_reserve(self._h, rows, nnz))

    def add(self, node_ids, vecs, term_offsets=None, term_ids=None, term_tf=None, doc_len=None):
        node_ids = np.ascontiguousarray(node_ids, np.uint64)
        vecs = np.ascontiguousarray(vecs, np.float32).reshape(len(node_ids), self.dim)
        if term_offsets is not None:
            term_offsets = np.ascontiguousarray(term_offsets, np.int64)
            term_ids = np.ascontiguousarray(term_ids, np.uint32)
            term_tf = np.ascontiguousarray(term_tf, np.uint16)
            doc_len = np.ascontiguousarray(doc_len, np.uint32)
        check(self._L.krag_index_add(self._h, len(node_ids), ptr(node_ids), ptr(vecs), ptr(term_offsets), ptr(term_ids),
                                     ptr(term_tf), ptr(doc_len)))

    def remove(self, node_ids) -> int:
        node_ids = np.ascontiguousarray(node_ids, np.uint64)
        n = C.c_int64(0)
        check(self._L.krag_index_remove(self._h, len(node_ids), ptr(node_ids), C.byref(n)))
        return n.value

    def commit(self, vocab: int):
        check(self._L.krag_index_commit(self._h, vocab))

    def commit_local(self, vocab: int):
        df = np.zeros(vocab, np.uint32)
        n_live, total = C.c_int64(0), C.c_int64(0)
        check(self._L.krag_index_commit_local(self._h, vocab, ptr(df), C.byref(n_live), C.byref(total)))
        return df, n_live.value, total.value

    def commit_global(self, vocab: int, df_global, n_docs_global: int, total_len_global: int, ordinal_base: int):
        df_global = np.ascontiguousarray(df_global, np.uint32)
        check(self._L.krag_index_commit_global(self._h, vocab, ptr(df_global), n_docs_global, total_len_global,
                                               ordinal_base))

    def set_ordinal_map(self, base: int, stride: int):
        """global ordinal of local row r = base + r * stride (round-robin shards: base = shard, stride = n_shards)"""
        check(self._L.krag_index_set_ordinal_map(self._h, base, stride))

    def stats(self) -> Stats:
        s = Stats()
        check(self._L.krag_index_stats(self._h, C.byref(s)))
        return s

    def node_ids(self, ordinals) -> np.ndarray:
        ordinals = np.ascontiguousarray(ordinals, np.int64)
        out = np.empty(ordinals.shape, np.uint64)
        check(self._L.krag_index_node_ids(self._h, ordinals.size, ptr(ordinals), ptr(out)))
        return out

    def persist(self, path: str):
        check(self._L.krag_index_persist(self._h, path.encode()))

    def set_dense_mode(self, dense_mode: int, release_shadow: bool = False):
        """KRAG_DENSE_*; DENSE_TC_BF16 builds the bf16 shadow on first use (results stay exact fp32 in every mode)"""
        check(self._L.krag_index_set_dense_mode(self._h, dense_mode, 1 if release_shadow else 0))

    def search_dense(self, q, k: int):
        q = np.ascontiguousarray(q, np.float32).reshape(-1, self.dim)
        b = q.shape[0]
        dist = np.empty((b, k), np.float32)
        ordn = np.empty((b, k), np.int64)
        check(self._L.krag_search_dense(self._h, b, ptr(q), k, ptr(dist), ptr(ordn)))
        return dist, ordn

    @staticmethod
    def _pack_terms(q_terms_list):
        offs = np.zeros(len(q_terms_list) + 1, np.int32)
        for i, t in enumerate(q_terms_list):
            offs[i + 1] = offs[i] + len(t)
        flat = (np.concatenate([np.asarray(t, np.uint32) for t in q_terms_list]) if offs[-1] > 0
                else np.zeros(1, np.uint32))
        return np.ascontiguousarray(flat, np.uint32), offs

    def search_bm25(self, q_terms_list, k: int):
        flat, offs = self._pack_terms(q_terms_list)
        b = len(q_terms_list)
        score = np.empty((b, k), np.float32)
        ordn = np.empty((b, k), np.int64)
        check(self._L.krag_search_bm25(self._h, b, ptr(flat), ptr(offs), k, ptr(score), ptr(ordn)))
        return score, ordn

    def retrieve(self, q, q_terms_list, k: int, cand_mult: float = 3.0, vector_weight: float = 0.7,
                 text_weight: float = 0.3, fusion_mode: int = FUSION_REFERENCE, keyword_allow_bitmap=None):
        """HybridRetriever._aretrieve for a batch. q_terms_list=None -> vector-only fallback."""
        q = np.ascontiguousarray(q, np.float32).reshape(-1, self.dim)
        b = q.shape[0]
        flat = offs = None
        if q_terms_list is not None:
            flat, offs = self._pack_terms(q_terms_list)
        if keyword_allow_bitmap is not None:
            keyword_allow_bitmap = np.ascontiguousarray(keyword_allow_bitmap, np.uint32)
        out = {
            "final": np.empty((b, k), np.float64), "dense": np.empty((b, k), np.float32),
            "sparse": np.empty((b, k), np.float32), "rank": np.empty((b, k), np.int32),
            "ordinal": np.empty((b, k), np.int64), "count": np.empty(b, np.int32),
        }
        check(self._L.krag_retrieve(self._h, b, ptr(q), ptr(flat), ptr(offs), k, cand_mult, vector_weight, text_weight,
                                    fusion_mode, ptr(keyword_allow_bitmap),
                                    0 if keyword_allow_bitmap is None else keyword_allow_bitmap.size, ptr(out["final"]), ptr(out["dense"]),
                                    ptr(out["sparse"]), ptr(out["rank"]), ptr(out["ordinal"]), ptr(out["count"])))
        return out

    # ---- device-pointer stage API ----
    def dev_dense_candidates(self, batch, d_q, P, d_keys, stream=0):
        check(self._L.krag_dev_dense_candidates(self._h, batch, ptr(d_q), P, ptr(d_keys), ptr(stream)))

    def dev_bm25_candidates(self, batch, d_terms, d_toff, P, d_keys, stream=0, h_toff=None):
        """h_toff: optional host copy (int32 [batch+1]) of the offsets; saves a 4-byte device read-back"""
        check(self._L.krag_dev_bm25_candidates(self._h, batch, ptr(d_terms), ptr(d_toff), ptr(h_toff), P, ptr(d_keys),
                                               ptr(stream)))

    # ---- synthetic / inspection ----
    def synth_fill(self, n: int, row_base: int = 0, seed: int = 1, vocab: int = 0):
        check(self._L.krag_synth_fill(self._h, n, row_base, seed, vocab))

    def read_rows(self, row0: int, n: int) -> np.ndarray:
        out = np.empty((n, self.dim), np.float32)
        check(self._L.krag_index_read_rows(self._h, row0, n, ptr(out)))
        return out

    def debug_tc_dump(self, q) -> np.ndarray:
        """K2 raw output a[j, r] = |x_r|^2 - 2 x_r.q_j for all rows (test hook)."""
        q = np.ascontiguousarray(q, np.float32).reshape(-1, self.dim)
        S, nqp = C.c_int64(0), C.c_int32(0)
        check(self._L.krag_debug_tc_dump(self._h, q.shape[0], ptr(q), None, 0, C.byref(S), C.byref(nqp)))
        out = np.empty((nqp.value, S.value), np.float32)
        check(self._L.krag_debug_tc_dump(self._h, q.shape[0], ptr(q), ptr(out), out.size, C.byref(S), C.byref(nqp)))
        return out

    def read_postings(self, term: int, cap: int = 1 << 22):
        cnt = C.c_int64(0)
        docs = np.empty(cap, np.uint32)
        scores = np.empty(cap, np.float32)
        check(self._L.krag_index_read_postings(self._h, term, cap, ptr(docs), ptr(scores), C.byref(cnt)))
        m = min(cnt.value, cap)
        return docs[:m], scores[:m], cnt.value

    def read_rank_scores(self, term: int) -> np.ndarray:
        """rank-table row of a term: [i] = its 2^i-th best posting score (i = 0..10), 0 below df"""
        out = np.empty(11, np.float32)
        check(self._L.krag_index_read_rank_scores(self._h, term, ptr(out)))
        return out
