// engine.h -- internal launcher interface between the kernel translation units and api.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <stdexcept>
namespace krag {

// device allocation failure with a message that says what was asked for and what was free (KRAG_E_OOM at the C ABI)
struct DevOom : std::runtime_error { using std::runtime_error::runtime_error; };

// global ordinal of a local row: base + row * stride.  Contiguous shards (bench, one GPU) use stride 1; the multi-GPU
// service deals nodes round-robin (node o -> shard o % G, row o / G), so base = shard, stride = G and ordinals -- hence
// every tie-break -- are exactly the single-GPU insertion order.
struct OrdMap {
    uint32_t base, stride;
    __host__ __device__ __forceinline__ uint32_t operator+(uint32_t row) const { return base + row * stride; }
};

struct DeviceInfo {
    int device = 0;
    int sm_count = 148;
    int cc_major = 0, cc_minor = 0;
    size_t smem_optin = 0;
};

// CUDA-event bracket around the dominant dense kernel of the last search (roofline evidence):
// recorded on the launching stream; read back after the stream is synchronised.
void dense_timer_begin(cudaStream_t st, int kernel_id, int64_t algorithmic_bytes, int64_t flops);
void dense_timer_end(cudaStream_t st);
bool dense_timer_read(float* ms, int* kernel_id, int64_t* bytes, int64_t* flops);

// launch counter (bench.py reports gpu_launches from it)
void count_launch(int n = 1);
int64_t launch_count();

// ---- K1: exact fp32 L2^2 scan + fused top-P (dense_scan.cu)
// q: device [batch, dpad] zero-padded.  part: workspace >= dense_scan_part_elems() u64.
// keys_out: device [batch, P], ascending, KEY_PAD padded, ordinals already global.
size_t dense_scan_part_elems(const DeviceInfo& di, int P);
void launch_dense_scan(const DeviceInfo& di, const float* X, int64_t n_rows, int dpad, const uint32_t* alive,
                       const float* q, int batch, int P, OrdMap ord_base, uint64_t* part, uint64_t* keys_out,
                       cudaStream_t st);

// ---- K2: tcgen05 TF32 candidate generation + exact fp32 rescoring (dense_tc.cu)
bool dense_tc_supported(const DeviceInfo& di, int dpad);
bool dense_tc_wants(int64_t n_rows, int batch);   // size heuristics: is K2 the better kernel for this call?
size_t dense_tc_workspace_bytes(const DeviceInfo& di, int64_t n_rows, int P);
// |x|^2 per row (+ running max) maintained at index time for K2's epilogue and certificate
void launch_row_norms(const float* X, int64_t row0, int64_t n, int dpad, float* xnorm, uint32_t* xn_max_bits,
                      cudaStream_t st);
// returns false when the tensor-core path cannot serve the request (caller falls back to K1 -- still GPU)
bool launch_dense_tc(const DeviceInfo& di, const float* X, int64_t n_rows, int dpad, const uint32_t* alive,
                     const float* xnorm, const uint32_t* xn_max_bits, const float* q, int batch, int P,
                     OrdMap ord_base, void* workspace, size_t workspace_bytes, uint64_t* part, uint64_t* keys_out,
                     cudaStream_t st, const uint16_t* Xh = nullptr /* optional bf16 shadow of X for the prune pass */,
                     bool allow_cvt = true /* fp32 rows rounded to bf16 on chip (kind::f16) instead of kind::tf32 */);
void launch_f32_to_bf16(const float* in, uint16_t* out, int64_t n_elems, cudaStream_t st);
int64_t dense_tc_fallback_queries();   // queries re-run on K1 because the exactness certificate failed
// diagnostics: a[j][r] = |x_r|^2 - 2 x_r.q_j for ALL rows through the tensor-core kernel (tests only)
bool dense_tc_debug_dump(const DeviceInfo& di, const float* X, int64_t n_rows, int dpad, const float* xnorm,
                         const float* q, int nq, float* dump_out /*[NQ_pad][S]*/, int64_t* S_out, int* nq_pad_out,
                         cudaStream_t st);

// ---- merge / fuse (merge_fuse.cu)
// per query: n_lists lists of list_len keys (element (l,i) at in[b*batch_stride + l*list_stride + i]) -> the P smallest
// only_flag != null: queries whose flag is 0 are left untouched
void launch_merge(const uint64_t* keys_in, int n_lists, int list_len, int batch, int P, int64_t list_stride,
                  int64_t batch_stride, uint64_t* keys_out, cudaStream_t st, const uint64_t* thr_hint = nullptr,
                  const uint32_t* only_flag = nullptr);
// peer-memory exchange: push local lists [nl, batch, P] into every rank's mailbox, then merge G*P -> P locally
size_t p2p_mailbox_words(int world, int nl, int max_batch, int max_P);
void launch_p2p_exchange_merge(uint64_t* const* d_mailboxes, uint64_t* own_mailbox, int rank, int world, int64_t slot_words,
                               unsigned long long seq, int nl, int batch, int P, const uint64_t* local, uint64_t* merged,
                               cudaStream_t st);
void launch_bitmap_and(uint32_t* dst, const uint32_t* other, int64_t words, cudaStream_t st);
// append zero-score fillers to short BM25 lists (bm25s argpartition semantics)
void launch_bm25_fill(uint64_t* keys /*[batch,P]*/, int batch, int P, const uint32_t* alive, int64_t n_rows,
                      OrdMap ord_base, cudaStream_t st);
void launch_fuse(int batch, int P, int k, const uint64_t* dense_keys, const uint64_t* bm25_keys, double w_v, double w_t,
                 int mode, const uint32_t* allow, double* out_final, float* out_dense, float* out_sparse,
                 int32_t* out_rank, int64_t* out_ord, int32_t* out_count, cudaStream_t st);

// ---- K3: BM25 (bm25.cu)
constexpr int BM25_SUB_DOCS = 2048;      // doc range of one tile-index column = one warp's shared-memory accumulator (K3)
constexpr int BM25_SUBS_PER_TILE = 8;
constexpr int BM25_TILE_DOCS = BM25_SUB_DOCS * BM25_SUBS_PER_TILE;   // doc range of one CTA in the legacy kernel (safety net)
struct Postings {
    int64_t* off = nullptr;    // [vocab+1]
    uint32_t* doc = nullptr;   // [nnz] local rows ascending inside a term
    float* score = nullptr;    // [nnz]
    int64_t vocab = 0, nnz = 0;
    // tile index: for terms with more than BM25_RARE_MAX postings, the offset (relative to off[t]) of the
    // first posting whose doc lies in each BM25_SUB_DOCS-sized doc range; removes per-query searches.  Terms below the
    // threshold get the same kind of row built per batch by bm25_resolve_kernel (a row costs 4 B per sub-tile, more than
    // the postings of a short list)
    int32_t* tile_slot = nullptr;   // [vocab]  slot of a frequent term, -1 for the others
    uint32_t* tile_off = nullptr;   // [n_slots][n_tiles + 1]
    int64_t n_slots = 0, n_tiles = 0;   // n_tiles = number of BM25_SUB_DOCS ranges
    // rank table: rank_score[t][i] = the 2^i-th best posting score of term t (the stored fp32 value), 0 when df(t) < 2^i.
    // Any query containing t has at least 2^i documents scoring >= that value: K3's admission threshold without a sample pass
    float* rank_score = nullptr;    // [vocab][BM25_RANKS]
};
constexpr int BM25_RARE_MAX = 2048;
constexpr int BM25_RANKS = 11;      // ranks 1, 2, 4, ..., 1024 = KRAG_MAX_POOL
void launch_df_histogram(const uint32_t* term_ids, const uint32_t* entry_doc, const uint32_t* alive, int64_t nnz,
                         uint32_t* df, cudaStream_t st);
void launch_expand_entry_doc(const int64_t* term_offsets, int64_t n_docs, uint32_t* entry_doc, cudaStream_t st);
// builds postings from CSR-by-doc arrays; idf is a device array [vocab] computed on the host (glibc log)
void build_postings(const uint32_t* term_ids, const uint16_t* term_tf, const uint32_t* entry_doc,
                    const uint32_t* doc_len, const uint32_t* alive, int64_t nnz, int64_t vocab, const float* idf,
                    double avgdl, int64_t n_docs_rows, Postings& out, cudaStream_t st);
size_t bm25_part_elems(int64_t n_rows, int batch, int P);
size_t bm25_resolve_bytes(int64_t n_rows, int n_terms_total);   // size of launch_bm25's resolve_ws
// alive_is_committed: `alive` admits exactly the documents the postings were built from (no delete since the commit, no
// filter), so the rank table bounds every query's P-th best score
void launch_bm25(const DeviceInfo& di, const Postings& post, int64_t n_rows, const uint32_t* alive, bool alive_is_committed,
                 const uint32_t* q_terms, const int32_t* q_term_offsets, int n_terms_total, void* resolve_ws, int batch, int P,
                 OrdMap ord_base, uint64_t* part, uint64_t* keys_out, cudaStream_t st);

// ---- K5: BERT encoder forward (embed.cu)
struct BertConfig;
struct Embedder;
Embedder* embedder_create(const DeviceInfo& di, const BertConfig& cfg);
void embedder_load(Embedder* e, const char* name, const float* data, int64_t n);
void embedder_finalize(Embedder* e);
void embedder_destroy(Embedder* e);
int embedder_hidden(const Embedder* e);
void embedder_forward(Embedder* e, int batch, const int32_t* tok_ids, const int32_t* tok_offsets, float* out_host,
                      float* out_dev = nullptr, int ld_out = 0, cudaStream_t consumer = nullptr);
// A fp32 matrix carried as two fp16 planes: v = hi + lo * 2^-11 (see embed.cu: split operands of the K5 GEMMs)
struct SplitMat { uint16_t* hi; uint16_t* lo; };
void launch_split_f16(const float* in, uint16_t* hi, uint16_t* lo, int64_t n /* % 8 == 0 */, cudaStream_t st);
// Linear layer on split operands: C = A . B^T + bias (+GELU) (+residual), fp32-accurate (three kind::f16 MMAs per step);
// outputs: fp32 C and / or the split planes of C; with ln_g the row LayerNorm of that goes to Y / Y planes (C is scratch).
// Picks CTA pairs / 128x128 tiles / 128xBN split-K tiles by problem size; ws = split-K workspace (may be null).
void launch_linear(const DeviceInfo& di, const SplitMat& A, const SplitMat& B, int M, int N, int K, const float* bias, const float* residual,
                   bool gelu, float* C, uint16_t* C_hi, uint16_t* C_lo, const float* ln_g, const float* ln_b, float eps, float* Y,
                   uint16_t* Y_hi, uint16_t* Y_lo, float* ws, size_t ws_floats, cudaStream_t st);
// test hook: fp32 device operands, split on the fly, then the path above
void launch_linear_f32(const DeviceInfo& di, const float* A, const float* B, int M, int N, int K, const float* bias, const float* residual,
                       bool gelu, float* C, const float* ln_g, const float* ln_b, float eps, float* Y, float* ws, size_t ws_floats,
                       cudaStream_t st);

// ---- synthetic data (synth.cu)
void launch_synth_dense(float* X, int64_t n, int d, int dpad, int64_t row_base, uint64_t seed, cudaStream_t st);
// two-pass: lengths -> offsets (host scan by caller via cub) -> fill
void synth_sparse(int64_t n, int64_t row_base, uint64_t seed, int64_t vocab, int64_t** term_offsets_out,
                  uint32_t** term_ids_out, uint16_t** term_tf_out, uint32_t** doc_len_out, int64_t* nnz_out,
                  cudaStream_t st);

}  // namespace krag
