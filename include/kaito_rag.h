/*
 * kaito_rag.h -- C ABI of libkaito_rag.so, the B200 (sm_100a) retrieval engine behind
 * KAITO's RAGService /retrieve and /index.
 *
 * The reference has no in-process FFI seam: its service is Python calling pip wheels
 * (faiss-cpu, bm25s) -- SURVEY.md section 8(b).  This header is the seam a Go (cgo) or
 * Python (ctypes) RAGService host binds instead of those wheels.  Each entry point
 * names the reference call it replaces (paths relative to presets/ragengine/).
 *
 * Conventions
 *   - every call returns int32 status: 0 = KRAG_OK, negative = KRAG_E_*;
 *     krag_last_error() returns a thread-local UTF-8 message for the last failure.
 *   - caller owns host buffers; the library owns device memory; handles are opaque.
 *   - NO CPU FALLBACK: without an sm_100 device krag_init fails with KRAG_E_NO_DEVICE.
 *   - thread-safety mirrors the reference's aiorwlock (vector_store/base.py:77-79):
 *     searches on one index may run concurrently, mutations are exclusive.
 *   - "ordinal" = position of a node in insertion order (global across shards:
 *     shard base + local row).  Ties everywhere break by ascending ordinal.
 *   - candidate keys are u64: high 32 bits = order-preserving bits of the fp32 value
 *     (dense: L2^2 ascending; bm25: complemented, so ascending key == descending
 *     score), low 32 bits = global ordinal.  KRAG_KEY_PAD (all ones) pads short lists.
 */
#ifndef KAITO_RAG_H_
#define KAITO_RAG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KRAG_OK 0
#define KRAG_E_INVALID (-1)     /* bad argument */
#define KRAG_E_NO_DEVICE (-2)   /* no sm_100 CUDA device / driver */
#define KRAG_E_CUDA (-3)        /* CUDA runtime error (message has details) */
#define KRAG_E_OOM (-4)         /* device or host allocation failed */
#define KRAG_E_NOT_FOUND (-5)   /* unknown index / node id */
#define KRAG_E_STATE (-6)       /* call not valid in the current state (e.g. search before commit) */
#define KRAG_E_IO (-7)          /* persist / load failure */
#define KRAG_E_UNSUPPORTED (-8) /* feature compiled out or not available on this device */

#define KRAG_KEY_PAD 0xFFFFFFFFFFFFFFFFull
#define KRAG_MAX_TOP_K 300   /* config.py:127 RAG_MAX_TOP_K */
#define KRAG_MAX_POOL 1024   /* >= int(300 * 3.0) = 900, hybrid_retriever.py:97-98 */

#define KRAG_FUSION_REFERENCE 0  /* vec_score = L2^2 itself (hybrid_retriever.py:139-142,158-166) */
#define KRAG_FUSION_SIMILARITY 1 /* vec_score = 1 - L2^2/2 (not the reference) */
/* OR-ed into fusion_mode: apply krag_retrieve's allow bitmap INSIDE the dense and BM25 kernels (every one of the P
 * candidates of both lists satisfies the filter) instead of the reference's post-filter of the keyword list only
 * (hybrid_retriever.py:227-235; its dense side cannot filter at all, SURVEY.md section 8 a9).  Not the reference. */
#define KRAG_FILTER_PUSHDOWN 0x100

#define KRAG_DENSE_AUTO 0   /* exact fp32 scan for small batches, tensor-core path for large */
#define KRAG_DENSE_SCAN 1   /* K1: exact fp32 CUDA-core scan */
#define KRAG_DENSE_TC 2     /* K2: tcgen05 prune pass (fp32 rows rounded to bf16 in shared memory, kind::f16; TF32 when the
                               padded dimension is not a multiple of 64) + exact fp32 rescoring */
#define KRAG_DENSE_TC_BF16 3 /* K2 pruning on a bf16 SHADOW copy of the corpus (+50% memory); the returned distances are
                               still exact fp32 re-scores of the fp32 corpus and carry the same exactness certificate */

#define KRAG_DENSE_TC_TF32 4 /* K2 with the fp32 rows consumed directly as TF32 (kind::tf32): the earlier default, kept for comparison */

typedef struct krag_ctx krag_ctx;
typedef struct krag_index krag_index;

typedef struct krag_config {
    int32_t device_id;      /* CUDA device ordinal */
    int32_t rank;           /* shard rank of this process (0 when single GPU) */
    int32_t world_size;     /* number of shards (1 when single GPU) */
    int32_t dense_mode;     /* KRAG_DENSE_* */
    int32_t search_slots;   /* concurrent search workspaces (0 = default 4) */
    int32_t reserved[3];
} krag_config;

typedef struct krag_stats_t {
    int64_t n_rows;         /* local dense rows (incl. tombstoned) */
    int64_t n_live;         /* local live rows */
    int64_t nnz;            /* local postings */
    int64_t n_docs_global;  /* BM25 N used for idf */
    int64_t total_len_global;
    int64_t vocab;
    int64_t ordinal_base;   /* global ordinal of local row 0 */
    int32_t dim;            /* logical dimension */
    int32_t dim_padded;     /* row stride in floats (multiple of 32) */
    int32_t committed;      /* postings valid for the current rows */
    int32_t reserved;
    int64_t device_bytes;   /* device memory held by this index */
} krag_stats_t;

/* --------------------------------------------------------------------- lifecycle */
int32_t krag_version(void);
const char* krag_last_error(void);
/* replaces: process-wide FAISS/BM25 imports of the RAGService (main.py:141-158) */
int32_t krag_init(const krag_config* cfg, krag_ctx** out);
int32_t krag_shutdown(krag_ctx* ctx);
/* number of kernels this library has launched since krag_init (bench.py gpu_launches) */
int64_t krag_launch_count(krag_ctx* ctx);
void* krag_ctx_stream(krag_ctx* ctx);  /* cudaStream_t of search slot 0 (for event timing) */

/* ------------------------------------------------------------------------- index */
/* replaces: faiss.IndexIDMap(faiss.IndexFlatL2(dim)) + FaissMapVectorStore,
 * vector_store/faiss_store.py:41-50 */
int32_t krag_index_create(krag_ctx* ctx, const char* name, int32_t dim, krag_index** out);
/* replaces: BaseVectorStore.delete_index (DELETE /indexes/{name}, main.py:774) */
int32_t krag_index_drop(krag_index* idx);
int32_t krag_index_reserve(krag_index* idx, int64_t rows, int64_t nnz);
/*
 * Append n nodes.  replaces: FaissMapVectorStore.add -> index.add_with_ids and the
 * docstore insert that BM25Retriever.from_defaults later tokenises
 * (vector_store/base.py:155-166, :499-511; hybrid_retriever.py:122-125).
 *   node_ids     [n]            caller-chosen unique u64 handles
 *   vecs         [n, dim]       fp32 row-major embeddings
 *   term_offsets [n+1]          CSR offsets into term_ids/term_tf (NULL: no sparse side)
 *   term_ids     [nnz]          unique term ids per node (host vocabulary)
 *   term_tf      [nnz]          term frequency within the node
 *   doc_len      [n]            token count of the node after stop-word removal
 */
int32_t krag_index_add(krag_index* idx, int64_t n, const uint64_t* node_ids, const float* vecs,
                       const int64_t* term_offsets, const uint32_t* term_ids, const uint16_t* term_tf,
                       const uint32_t* doc_len);
/* replaces: IndexIDMap.remove_ids via llama-index delete (vector_store/base.py:563-643) */
int32_t krag_index_remove(krag_index* idx, int64_t n, const uint64_t* node_ids, int64_t* n_removed);
/*
 * (Re)build BM25 postings for the rows added so far.  replaces the per-query
 * BM25Retriever.from_defaults rebuild (hybrid_retriever.py:104-130): same scores,
 * built once.  Single-shard form:
 */
int32_t krag_index_commit(krag_index* idx, int64_t vocab);
/* Multi-shard form: each rank reports local stats, the host all-reduces them (sum),
 * then every rank finishes with the global values (SURVEY.md section 8e). */
int32_t krag_index_commit_local(krag_index* idx, int64_t vocab, uint32_t* df_out /*[vocab] host*/,
                                int64_t* n_live_out, int64_t* total_len_out);
int32_t krag_index_commit_global(krag_index* idx, int64_t vocab, const uint32_t* df_global /*[vocab] host*/,
                                 int64_t n_docs_global, int64_t total_len_global, int64_t ordinal_base);
/* Global ordinal of local row r = ordinal_base + r * ordinal_stride (default base 0 / stride 1; krag_index_commit_global sets
 * the base of a contiguous shard).  The multi-GPU service deals nodes round-robin over G shards (node o -> shard o % G, row
 * o / G) and sets (base, stride) = (shard, G): ordinals -- and with them every tie-break -- equal the single-GPU insertion
 * order.  Call before krag_index_commit_global / searches; no counterpart in the reference (one replica, manifests.go:81). */
int32_t krag_index_set_ordinal_map(krag_index* idx, int64_t ordinal_base, int64_t ordinal_stride);
int32_t krag_index_stats(krag_index* idx, krag_stats_t* out);
/* ordinals (global) -> node ids for rows of THIS shard; KRAG_E_NOT_FOUND if out of range */
int32_t krag_index_node_ids(krag_index* idx, int64_t n, const int64_t* ordinals, uint64_t* node_ids_out);
/* replaces: StorageContext.persist / load_index_from_storage (vector_store/base.py:779-868) */
int32_t krag_index_persist(krag_index* idx, const char* dir);
int32_t krag_index_load(krag_ctx* ctx, const char* name, const char* dir, krag_index** out);

/* ------------------------------------------------- search, host buffers (1 shard) */
/*
 * replaces: IndexIDMap(IndexFlatL2).search(q, k) reached from
 * index.as_retriever(similarity_top_k=P).aretrieve (hybrid_retriever.py:209-213).
 *   q [batch, dim] fp32;  out_l2sq [batch, k] ascending (+inf pad);
 *   out_ordinals [batch, k] (-1 pad, like faiss' -1 labels).
 */
int32_t krag_search_dense(krag_index* idx, int32_t batch, const float* q, int32_t k,
                          float* out_l2sq, int64_t* out_ordinals);
/*
 * replaces: bm25_retriever.aretrieve(query) (hybrid_retriever.py:220) after host-side
 * tokenisation.  q_terms are term ids in query order, duplicates kept;
 * q_term_offsets [batch+1].  out_score [batch,k] descending; zero-score documents fill
 * short lists as bm25s' argpartition does; out_ordinals -1 past the live doc count.
 */
int32_t krag_search_bm25(krag_index* idx, int32_t batch, const uint32_t* q_terms, const int32_t* q_term_offsets,
                         int32_t k, float* out_score, int64_t* out_ordinals);
/*
 * The whole HybridRetriever._aretrieve (hybrid_retriever.py:205-237) for a batch:
 * dense top-P, BM25 top-P, keyword-side metadata post-filter (optional bitmap of
 * allowed LOCAL rows, 1 bit per row, at least (n_rows + 31) / 32 words -- fewer is KRAG_E_INVALID; NULL = no filter),
 * _fuse, top-k.
 *   P = int(k * max(1, cand_mult)).  q_terms == NULL or an uncommitted index selects
 *   the reference's vector-only fallback (:216-218): dense top-P cut to k.
 * Outputs are [batch, k]; out_count[batch] gives the valid prefix per query.
 *   out_final  fp64 fused score (dense-only fallback: the L2^2)
 *   out_dense  L2^2 or NaN;  out_sparse BM25 score or NaN;  out_rank BM25 rank or -1
 * fusion_mode | KRAG_FILTER_PUSHDOWN: the bitmap restricts both candidate scans instead (also in the vector-only case).
 */
int32_t krag_retrieve(krag_index* idx, int32_t batch, const float* q,
                      const uint32_t* q_terms, const int32_t* q_term_offsets,
                      int32_t k, double cand_mult, double vector_weight, double text_weight, int32_t fusion_mode,
                      const uint32_t* keyword_allow_bitmap, int64_t keyword_allow_words /* u32 words held by the bitmap */,
                      double* out_final, float* out_dense, float* out_sparse, int32_t* out_rank,
                      int64_t* out_ordinals, int32_t* out_count);

/* ------------------------------- stage API, DEVICE pointers (one process per GPU) */
/* All pointers are device pointers valid on ctx's device; `stream` is a cudaStream_t
 * (NULL = legacy default stream).  These let the host place one NCCL all-gather
 * between the local candidate stage and the merge/fuse stage (SURVEY.md section 8e). */
int32_t krag_dev_dense_candidates(krag_index* idx, int32_t batch, const float* d_q, int32_t P,
                                  uint64_t* d_keys_out /*[batch,P]*/, void* stream);
int32_t krag_dev_bm25_candidates(krag_index* idx, int32_t batch, const uint32_t* d_q_terms,
                                 const int32_t* d_q_term_offsets, const int32_t* h_q_term_offsets,
                                 int32_t P, uint64_t* d_keys_out /*[batch,P]*/, void* stream);
/* keys_in [n_lists, batch, P] -> keys_out [batch, P]: the P smallest keys per query */
int32_t krag_dev_merge(krag_ctx* ctx, int32_t n_lists, int32_t batch, int32_t P, const uint64_t* d_keys_in,
                       uint64_t* d_keys_out, void* stream);
/* HybridRetriever._fuse (hybrid_retriever.py:132-166) on merged candidate lists.
 * d_bm25_keys == NULL selects the vector-only fallback. d_allow: optional bitmap over
 * GLOBAL ordinals for the keyword-side post-filter (:227-235). */
int32_t krag_dev_fuse(krag_ctx* ctx, int32_t batch, int32_t P, int32_t k, const uint64_t* d_dense_keys,
                      const uint64_t* d_bm25_keys, double vector_weight, double text_weight, int32_t fusion_mode,
                      const uint32_t* d_allow, double* d_out_final, float* d_out_dense, float* d_out_sparse,
                      int32_t* d_out_rank, int64_t* d_out_ordinals, int32_t* d_out_count, void* stream);

/* ------------------------------------------------ synthetic corpora (bench / tests) */
/* Fill the index with n deterministic unit-norm rows generated ON THE DEVICE
 * (counter-based Philox4x32-10 keyed by seed and global row), plus, when vocab > 0,
 * Zipf(s=1.07) term lists with log-normal lengths (SURVEY.md section 8d).  Node id of a
 * synthetic row == its global ordinal.  Not on the product path. */
int32_t krag_synth_fill(krag_index* idx, int64_t n, int64_t row_base, uint64_t seed, int64_t vocab);
/* copy rows [row0,row0+n) back to host (parity spot checks at full size) */
int32_t krag_index_read_rows(krag_index* idx, int64_t row0, int64_t n, float* out /*[n,dim]*/);
/* copy the postings of one term back to host: returns count via *n_out (cap entries max) */
int32_t krag_index_read_postings(krag_index* idx, uint32_t term, int64_t cap, uint32_t* docs_out, float* scores_out,
                                 int64_t* n_out);
/* copy the rank-table row of one term back to host: out[i] = the 2^i-th best posting score of the term, i = 0..10
 * (0 where the term has fewer than 2^i postings) */
int32_t krag_index_read_rank_scores(krag_index* idx, uint32_t term, float* out /*[11]*/);

/* ----------------------------------------- peer-memory candidate exchange (one process per GPU, one box) */
/* The all-gather + merge of the per-shard candidate lists done by our own kernels over NVLink peer memory:
 * every rank creates a mailbox (cudaMalloc + CUDA IPC handle), the host exchanges the 64-byte handles (any
 * side channel; kaito_b200/sharded.py uses torch.distributed.all_gather_object), every rank connects, and
 * krag_dev_exchange_merge then (1) stores this rank's lists [n_lists, batch, P] into all mailboxes with P2P
 * writes + a system-scope release flag and (2) waits for all ranks' flags and merges G*P -> P locally.
 * No counterpart in the reference (single replica, SURVEY.md section 8e). */
typedef struct krag_p2p krag_p2p;
int32_t krag_p2p_create(krag_ctx* ctx, int32_t rank, int32_t world, int32_t max_batch, int32_t max_P, krag_p2p** out,
                        uint8_t* handle_out /*[64]*/);
int32_t krag_p2p_connect(krag_p2p* p, const uint8_t* handles /*[world][64], own entry ignored*/);
int32_t krag_dev_exchange_merge(krag_p2p* p, int32_t n_lists, int32_t batch, int32_t P, const uint64_t* d_local_keys,
                                uint64_t* d_merged_out /*[n_lists, batch, P]*/, void* stream);
int32_t krag_p2p_destroy(krag_p2p* p);

/* ------------------------------------------------------------- embedding forward (K5) */
/* replaces: LocalHuggingFaceEmbedding (embedding/huggingface_local_embedding.py:34-53) -> sentence-
 * transformers BertModel forward, CLS pooling, L2 normalisation.  Tokenisation (WordPiece) stays in
 * the host.  Weights are loaded by their Hugging Face BertModel names ("embeddings.word_embeddings.weight",
 * "encoder.layer.0.attention.self.query.weight", ...), fp32, row-major as torch stores them. */
typedef struct krag_embedder krag_embedder;
typedef struct krag_bert_config {
    int32_t layers, hidden, heads, intermediate, vocab, max_position, type_vocab;
    float ln_eps;
} krag_bert_config;
int32_t krag_embedder_create(krag_ctx* ctx, const krag_bert_config* cfg, krag_embedder** out);
int32_t krag_embedder_load_tensor(krag_embedder* e, const char* name, const float* data, int64_t n_elems);
int32_t krag_embedder_finalize(krag_embedder* e);
/* tok_ids: packed token ids of all sequences ([CLS] ... [SEP] each); tok_offsets [batch+1]; out [batch, hidden] */
int32_t krag_embed(krag_embedder* e, int32_t batch, const int32_t* tok_ids, const int32_t* tok_offsets, float* out);
/* same, result left on the device: rows of d_out with stride ld_out floats (>= hidden; the padded query layout
 * krag_dev_dense_candidates takes); `stream` (cudaStream_t) is made to wait for the embeddings. tok_* are HOST. */
int32_t krag_embed_dev(krag_embedder* e, int32_t batch, const int32_t* tok_ids, const int32_t* tok_offsets, float* d_out,
                       int32_t ld_out, void* stream);
int32_t krag_embedder_destroy(krag_embedder* e);

/* ------------------------------------------------- host-side text analysis (no GPU involved; ASCII input) */
/* The analysis chains the reference runs in native third-party code, for hosts that are not Python (a cgo host links the
 * same functions the Python host uses for ASCII text; kaito_b200/text.py is the Unicode-complete restatement and the spec).
 * krag_text_analyze: bm25s.tokenize(text, stopwords="english", stemmer=Snowball english) as used by
 *   BM25Retriever.from_defaults (hybrid_retriever.py:122-125): lower-case, \w\w+ tokens, 33 stop words dropped, Porter2 stems.
 *   Writes the stems separated by '\n' into out (if *out_len <= cap) and always reports the needed length and the token count.
 * krag_wordpiece_*: BertTokenizer (uncased) of the bge models (huggingface_local_embedding.py:34-53): BasicTokenizer +
 *   greedy longest-match WordPiece; vocab = the lines of vocab.txt joined by '\n'; encode_batch writes, per text,
 *   [CLS] ids[: max_len - 2] [SEP] into out_ids[i * max_len ...] and its length into out_n[i] (texts are threaded). */
typedef struct krag_wordpiece krag_wordpiece;
int32_t krag_text_analyze(const char* text, int64_t len, char* out, int64_t cap, int64_t* out_len, int32_t* n_terms);
int32_t krag_wordpiece_create(const char* vocab, int64_t len, int32_t lower_case, krag_wordpiece** out);
int32_t krag_wordpiece_encode_batch(const krag_wordpiece* w, int64_t n, const char* texts, const int64_t* offsets /*[n+1]*/,
                                    int32_t max_len, int32_t* out_ids /*[n * max_len]*/, int32_t* out_n /*[n]*/);
int32_t krag_wordpiece_destroy(krag_wordpiece* w);

/* ------------------------------------------------------------------- diagnostics */
/* C[M,N] = A[M,K] . B[N,K]^T + bias (+erf-GELU) (+residual) through K5's tcgen05 TF32 GEMM; host buffers.
 * N % 128 == 0, K % 32 == 0.  Test hook. */
int32_t krag_debug_gemm_tf32(krag_ctx* ctx, int32_t M, int32_t N, int32_t K, const float* A, const float* B,
                             const float* bias, const float* residual, int32_t gelu, float* C_out);
/* Y = LayerNorm(A . B^T + bias (+residual)) * gamma + beta through K5's linear-layer dispatcher (for a handful of rows:
 * 128 x 32 split-K tiles + the reduce/LayerNorm kernel).  Test hook. */
int32_t krag_debug_linear_ln(krag_ctx* ctx, int32_t M, int32_t N, int32_t K, const float* A, const float* B,
                             const float* bias, const float* residual, const float* ln_gamma, const float* ln_beta,
                             float eps, float* Y_out);
/* Switch the dense kernel policy (KRAG_DENSE_*) of the context this index lives in.  Switching to KRAG_DENSE_TC_BF16
 * builds the index's bf16 shadow if it does not exist yet (one conversion pass over the fp32 rows); switching away
 * keeps the shadow unless release_shadow != 0.  Results never change: every mode returns exact fp32 distances. */
int32_t krag_index_set_dense_mode(krag_index* idx, int32_t dense_mode, int32_t release_shadow);
/* queries whose tensor-core result failed the exactness certificate and were re-run on the
 * exact scan kernel (process-wide counter) */
int64_t krag_tc_fallback_queries(void);
/* CUDA-event duration of the dominant dense kernel of the last search on this process
 * (kernel_id 1 = K1 exact scan, 2 = K2 tcgen05 main pass), with the algorithmic bytes and
 * flops of that launch -- bench.py's roofline line is computed from it. */
int32_t krag_last_dense_kernel(float* ms, int32_t* kernel_id, int64_t* algorithmic_bytes, int64_t* flops);
/* raw K2 output a[j][r] = |x_r|^2 - 2 x_r.q_j (TF32) for every row, [nq_pad][S] row-major;
 * call with out == NULL to query S and nq_pad.  Test hook for the tcgen05 kernel. */
int32_t krag_debug_tc_dump(krag_index* idx, int32_t nq, const float* q, float* out, int64_t out_elems,
                           int64_t* S_out, int32_t* nq_pad_out);

#ifdef __cplusplus
}
#endif
#endif /* KAITO_RAG_H_ */
