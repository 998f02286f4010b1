// api.cu -- the C ABI of libkaito_rag.so (include/kaito_rag.h): context, index shards,
// host-buffer search entry points and the device-pointer stage API.
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <sys/stat.h>

#include <atomic>
#include <condition_variable>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/kaito_rag.h"
#include "common.cuh"
#include "embed_config.h"
#include "engine.h"

namespace krag {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
static std::atomic<int64_t> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int64_t launch_count() { return g_launches.load(std::memory_order_relaxed); }

// "last dense kernel" diagnostics (krag_last_dense_kernel, read by bench.py).  Process-wide and last-writer-wins: with
// concurrent searches the numbers describe one of them; the mutex only keeps the record itself consistent.
static std::mutex g_t_mu;
static cudaEvent_t g_t0 = nullptr, g_t1 = nullptr;
static int g_t_kernel = 0;
static int64_t g_t_bytes = 0, g_t_flops = 0;
static bool g_t_valid = false;
void dense_timer_begin(cudaStream_t st, int kernel_id, int64_t bytes, int64_t flops)
{
    std::lock_guard<std::mutex> lk(g_t_mu);
    if (!g_t0) { cudaEventCreate(&g_t0); cudaEventCreate(&g_t1); }
    g_t_kernel = kernel_id; g_t_bytes = bytes; g_t_flops = flops; g_t_valid = false;
    cudaEventRecord(g_t0, st);
}
void dense_timer_end(cudaStream_t st)
{
    std::lock_guard<std::mutex> lk(g_t_mu);
    cudaEventRecord(g_t1, st);
    g_t_valid = true;
}
bool dense_timer_read(float* ms, int* kernel_id, int64_t* bytes, int64_t* flops)
{
    std::lock_guard<std::mutex> lk(g_t_mu);
    if (!g_t_valid || cudaEventSynchronize(g_t1) != cudaSuccess || cudaEventElapsedTime(ms, g_t0, g_t1) != cudaSuccess) return false;
    *kernel_id = g_t_kernel; *bytes = g_t_bytes; *flops = g_t_flops;
    return true;
}

struct ApiError { int32_t code; std::string msg; };
#define KRAG_REQUIRE(cond, code, msg)                      \
    do {                                                   \
        if (!(cond)) throw ::krag::ApiError{(code), (msg)}; \
    } while (0)

template <class F>
static int32_t guarded(F&& f)
{
    try {
        f();
        return KRAG_OK;
    } catch (const ApiError& e) {
        set_error(e.msg);
        return e.code;
    } catch (const CudaError& e) {
        char buf[512];
        snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)e.e, cudaGetErrorString(e.e), e.file, e.line, e.what);
        set_error(buf);
        cudaGetLastError();
        return e.e == cudaErrorMemoryAllocation ? KRAG_E_OOM : KRAG_E_CUDA;
    } catch (const DevOom& e) {
        set_error(e.what());
        return KRAG_E_OOM;
    } catch (const std::bad_alloc&) {
        set_error("host allocation failed");
        return KRAG_E_OOM;
    } catch (const std::exception& e) {
        set_error(e.what());
        return KRAG_E_INVALID;
    }
}

// growable device array (copy-on-grow; krag_index_reserve avoids the copies for big corpora)
template <class T>
struct DevArray {
    T* p = nullptr;
    int64_t cap = 0;
    void reserve(int64_t n, int64_t used, cudaStream_t st)
    {
        if (n <= cap) return;
        int64_t ncap = cap + cap / 2;
        if (ncap < n) ncap = n;
        T* np = nullptr;
        KRAG_CUDA(cudaMalloc(&np, sizeof(T) * (size_t)ncap));
        if (p && used > 0) KRAG_CUDA(cudaMemcpyAsync(np, p, sizeof(T) * (size_t)used, cudaMemcpyDeviceToDevice, st));
        KRAG_CUDA(cudaStreamSynchronize(st));
        if (p) KRAG_CUDA(cudaFree(p));
        p = np;
        cap = ncap;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    int64_t bytes() const { return (int64_t)sizeof(T) * cap; }
};

// per-call search workspace
struct Slot {
    cudaStream_t st = nullptr;
    DevArray<float> q;
    DevArray<uint32_t> terms;
    DevArray<int32_t> toff;
    DevArray<uint64_t> dense_keys, bm25_keys, part;
    DevArray<unsigned char> tc_ws, bm25_res;
    DevArray<uint32_t> allow;
    DevArray<double> out_final;
    DevArray<float> out_dense, out_sparse;
    DevArray<int32_t> out_rank, out_count;
    DevArray<int64_t> out_ord;
    std::vector<float> hq;  // padded query staging
};

}  // namespace krag

using namespace krag;

struct krag_ctx {
    DeviceInfo di;
    krag_config cfg;
    std::mutex mu;
    std::condition_variable cv;
    std::vector<Slot*> all_slots, free_slots;
    cudaStream_t admin = nullptr;  // mutation / build stream
};

struct krag_index {
    krag_ctx* ctx = nullptr;
    std::string name;
    int dim = 0, dpad = 0;
    std::shared_mutex mu;
    // dense shard
    DevArray<float> X;
    DevArray<float> xnorm;          // |x|^2 per row (K2 epilogue)
    DevArray<uint16_t> Xh;          // optional bf16 shadow of X (KRAG_DENSE_TC_BF16): prune pass only
    DevArray<uint32_t> xn_max;      // [1] bits of max |x|^2 (K2 certificate)
    int64_t n_rows = 0, n_live = 0;
    std::vector<uint32_t> alive_h;
    DevArray<uint32_t> alive_d;
    bool has_dead = false;
    std::vector<uint64_t> node_ids;
    std::unordered_map<uint64_t, int64_t> id2row;
    // sparse raw (CSR by doc)
    bool has_sparse = false;
    DevArray<int64_t> toff;
    DevArray<uint32_t> tid;
    DevArray<uint16_t> ttf;
    DevArray<uint32_t> dlen;
    int64_t nnz = 0;
    uint32_t max_term_id = 0;       // largest term id ever added (commit requires vocab > max_term_id)
    // committed postings
    Postings post;
    DevArray<uint32_t> entry_doc;  // scratch kept between commit_local and commit_global
    bool committed = false;
    bool removed_since_commit = false;   // the alive bitmap admits fewer documents than the postings were built from
    int64_t committed_rows = 0;
    int64_t vocab = 0, n_docs_global = 0, total_len_global = 0;
    int64_t ord_base = 0, ord_stride = 1;   // global ordinal of local row r = ord_base + r * ord_stride
};

namespace {

struct SlotLease {
    krag_ctx* c;
    Slot* s;
    explicit SlotLease(krag_ctx* ctx) : c(ctx)
    {
        std::unique_lock<std::mutex> lk(c->mu);
        c->cv.wait(lk, [&] { return !c->free_slots.empty(); });
        s = c->free_slots.back();
        c->free_slots.pop_back();
    }
    ~SlotLease()
    {
        {
            std::lock_guard<std::mutex> lk(c->mu);
            c->free_slots.push_back(s);
        }
        c->cv.notify_one();
    }
};

const uint32_t* alive_ptr(const krag_index* ix) { return ix->has_dead ? ix->alive_d.p : nullptr; }
OrdMap ord_map(const krag_index* ix) { return OrdMap{(uint32_t)ix->ord_base, (uint32_t)ix->ord_stride}; }
int64_t ord_last(const krag_index* ix) { return ix->ord_base + (ix->n_rows > 0 ? (ix->n_rows - 1) * ix->ord_stride : 0); }

void check_P(int P) { KRAG_REQUIRE(P >= 1 && P <= KRAG_MAX_POOL, KRAG_E_INVALID, "candidate pool must be in [1, 1024]"); }

// dense candidates for device-resident padded queries
void dense_candidates_dev(krag_index* ix, Slot* s, const float* d_q, int batch, int P, uint64_t* d_keys, cudaStream_t st,
                          const uint32_t* eligible = nullptr)
{
    krag_ctx* c = ix->ctx;
    const uint32_t* alive = eligible ? eligible : alive_ptr(ix);     // rows the scan may return (tombstones [& filter])
    if (ix->n_rows == 0) {
        KRAG_CUDA(cudaMemsetAsync(d_keys, 0xFF, sizeof(uint64_t) * (size_t)batch * P, st));
        return;
    }
    KRAG_REQUIRE(ord_last(ix) < 0xFFFFFFFFll, KRAG_E_UNSUPPORTED, "global ordinal exceeds 32 bits");
    s->part.reserve((int64_t)dense_scan_part_elems(c->di, P), 0, st);
    int mode = c->cfg.dense_mode;
    bool use_tc = (mode == KRAG_DENSE_TC) || (mode == KRAG_DENSE_TC_TF32) || (mode == KRAG_DENSE_TC_BF16 && dense_tc_wants(ix->n_rows, batch)) ||
                  (mode == KRAG_DENSE_AUTO && dense_tc_wants(ix->n_rows, batch));
    if (use_tc && dense_tc_supported(c->di, ix->dpad)) {
        size_t ws = dense_tc_workspace_bytes(c->di, ix->n_rows, P);
        s->tc_ws.reserve((int64_t)ws, 0, st);
        if (launch_dense_tc(c->di, ix->X.p, ix->n_rows, ix->dpad, alive, ix->xnorm.p, ix->xn_max.p, d_q, batch, P,
                            ord_map(ix), s->tc_ws.p, ws, s->part.p, d_keys, st,
                            mode == KRAG_DENSE_TC_BF16 ? ix->Xh.p : nullptr, mode != KRAG_DENSE_TC_TF32))
            return;
    }
    KRAG_REQUIRE((mode != KRAG_DENSE_TC && mode != KRAG_DENSE_TC_TF32) || !dense_tc_wants(ix->n_rows, 16), KRAG_E_UNSUPPORTED, "tensor-core dense path unavailable for this index/device");
    launch_dense_scan(c->di, ix->X.p, ix->n_rows, ix->dpad, alive, d_q, batch, P, ord_map(ix),
                      s->part.p, d_keys, st);
}

void bm25_candidates_dev(krag_index* ix, Slot* s, const uint32_t* d_terms, const int32_t* d_toff, int n_terms_total, int batch,
                         int P, uint64_t* d_keys, cudaStream_t st, const uint32_t* eligible = nullptr)
{
    KRAG_REQUIRE(ix->committed, KRAG_E_STATE, "index has no committed postings (call krag_index_commit)");
    if (n_terms_total < 0) {   // caller did not provide the host copy of the offsets: read the total back (4 bytes)
        int32_t tot = 0;
        KRAG_CUDA(cudaMemcpyAsync(&tot, d_toff + batch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        KRAG_CUDA(cudaStreamSynchronize(st));
        n_terms_total = tot;
    }
    s->part.reserve((int64_t)bm25_part_elems(ix->committed_rows, batch, P), 0, st);
    s->bm25_res.reserve((int64_t)bm25_resolve_bytes(ix->committed_rows, n_terms_total), 0, st);
    launch_bm25(ix->ctx->di, ix->post, ix->committed_rows, eligible ? eligible : alive_ptr(ix), !eligible && !ix->removed_since_commit, d_terms, d_toff, n_terms_total, s->bm25_res.p, batch, P,
                ord_map(ix), s->part.p, d_keys, st);
}

// stage padded queries on the device
const float* upload_queries(krag_index* ix, Slot* s, const float* q, int batch)
{
    const int d = ix->dim, dp = ix->dpad;
    s->q.reserve((int64_t)batch * dp, 0, s->st);
    if (d == dp) {
        KRAG_CUDA(cudaMemcpyAsync(s->q.p, q, sizeof(float) * (size_t)batch * d, cudaMemcpyHostToDevice, s->st));
    } else {
        s->hq.assign((size_t)batch * dp, 0.f);
        for (int b = 0; b < batch; ++b) memcpy(&s->hq[(size_t)b * dp], q + (size_t)b * d, sizeof(float) * d);
        KRAG_CUDA(cudaMemcpyAsync(s->q.p, s->hq.data(), sizeof(float) * (size_t)batch * dp, cudaMemcpyHostToDevice, s->st));
    }
    return s->q.p;
}

void upload_terms(Slot* s, const uint32_t* q_terms, const int32_t* q_toff, int batch)
{
    const int nt = q_toff[batch];
    KRAG_REQUIRE(q_toff[0] == 0 && nt >= 0, KRAG_E_INVALID, "q_term_offsets must start at 0 and be non-decreasing");
    s->terms.reserve(nt > 0 ? nt : 1, 0, s->st);
    s->toff.reserve(batch + 1, 0, s->st);
    if (nt > 0) KRAG_CUDA(cudaMemcpyAsync(s->terms.p, q_terms, sizeof(uint32_t) * (size_t)nt, cudaMemcpyHostToDevice, s->st));
    KRAG_CUDA(cudaMemcpyAsync(s->toff.p, q_toff, sizeof(int32_t) * (size_t)(batch + 1), cudaMemcpyHostToDevice, s->st));
}

void mark_alive(krag_index* ix, int64_t row0, int64_t n, cudaStream_t st)
{
    int64_t words = (ix->n_rows + n + 31) / 32;
    if ((int64_t)ix->alive_h.size() < words) ix->alive_h.resize((size_t)words, 0u);
    for (int64_t r = row0; r < row0 + n; ++r) ix->alive_h[(size_t)(r >> 5)] |= 1u << (r & 31);
    ix->alive_d.reserve(words, (row0 + 31) / 32, st);
    int64_t w0 = row0 >> 5, w1 = (row0 + n + 31) >> 5;
    KRAG_CUDA(cudaMemcpyAsync(ix->alive_d.p + w0, ix->alive_h.data() + w0, sizeof(uint32_t) * (size_t)(w1 - w0),
                              cudaMemcpyHostToDevice, st));
}

void ensure_capacity(krag_index* ix, int64_t rows, int64_t nnz, cudaStream_t st)
{
    ix->X.reserve(rows * ix->dpad, ix->n_rows * ix->dpad, st);
    ix->xnorm.reserve(rows, ix->n_rows, st);
    if (ix->ctx->cfg.dense_mode == KRAG_DENSE_TC_BF16 || ix->Xh.p) ix->Xh.reserve(rows * ix->dpad, ix->n_rows * ix->dpad, st);
    if (ix->xn_max.p == nullptr) {
        ix->xn_max.reserve(1, 0, st);
        KRAG_CUDA(cudaMemsetAsync(ix->xn_max.p, 0, sizeof(uint32_t), st));
    }
    if (nnz >= 0) {
        ix->toff.reserve(rows + 1, ix->n_rows + 1, st);
        ix->dlen.reserve(rows, ix->n_rows, st);
        ix->tid.reserve(nnz > 0 ? nnz : 1, ix->nnz, st);
        ix->ttf.reserve(nnz > 0 ? nnz : 1, ix->nnz, st);
    }
}

void commit_local_impl(krag_index* ix, int64_t vocab, uint32_t* df_out, int64_t* n_live_out, int64_t* total_len_out)
{
    cudaStream_t st = ix->ctx->admin;
    KRAG_REQUIRE(ix->has_sparse || ix->n_rows == 0, KRAG_E_STATE, "index holds no term lists (dense-only)");
    KRAG_REQUIRE(vocab > 0 && vocab < 0x7fffffffll, KRAG_E_INVALID, "vocab out of range");
    ix->entry_doc.reserve(ix->nnz > 0 ? ix->nnz : 1, 0, st);
    if (ix->n_rows > 0) launch_expand_entry_doc(ix->toff.p, ix->n_rows, ix->entry_doc.p, st);
    uint32_t* df = nullptr;
    KRAG_CUDA(cudaMalloc(&df, sizeof(uint32_t) * (size_t)vocab));
    KRAG_CUDA(cudaMemsetAsync(df, 0, sizeof(uint32_t) * (size_t)vocab, st));
    // term ids >= vocab would make the df kernel write out of bounds: the largest id is tracked on the host at add time
    KRAG_REQUIRE(ix->nnz == 0 || vocab > (int64_t)ix->max_term_id, KRAG_E_INVALID,
                 "vocab must exceed the largest term id added to the index");
    if (ix->nnz > 0) {
        launch_df_histogram(ix->tid.p, ix->entry_doc.p, alive_ptr(ix), ix->nnz, df, st);
    }
    KRAG_CUDA(cudaMemcpyAsync(df_out, df, sizeof(uint32_t) * (size_t)vocab, cudaMemcpyDeviceToHost, st));
    // total length over live docs (host side: doc_len is small)
    std::vector<uint32_t> dl((size_t)ix->n_rows);
    if (ix->n_rows > 0)
        KRAG_CUDA(cudaMemcpyAsync(dl.data(), ix->dlen.p, sizeof(uint32_t) * (size_t)ix->n_rows, cudaMemcpyDeviceToHost, st));
    KRAG_CUDA(cudaStreamSynchronize(st));
    KRAG_CUDA(cudaFree(df));
    int64_t total = 0, live = 0;
    for (int64_t r = 0; r < ix->n_rows; ++r)
        if ((ix->alive_h[(size_t)(r >> 5)] >> (r & 31)) & 1u) { total += dl[(size_t)r]; ++live; }
    *n_live_out = live;
    *total_len_out = total;
}

void commit_global_impl(krag_index* ix, int64_t vocab, const uint32_t* df_global, int64_t n_docs_global,
                        int64_t total_len_global, int64_t ord_base)
{
    cudaStream_t st = ix->ctx->admin;
    KRAG_REQUIRE(ord_base >= 0 && ord_base + ix->n_rows * ix->ord_stride <= 0xFFFFFFFFll, KRAG_E_UNSUPPORTED, "global ordinal exceeds 32 bits");
    // n_docs_global == 0 is legal: every document deleted (the reference's docstore is then empty and its retriever
    // falls back to vector-only, hybrid_retriever.py:113-121); the postings come out empty and avgdl is irrelevant
    KRAG_REQUIRE(n_docs_global >= 0 && total_len_global >= 0, KRAG_E_INVALID, "n_docs_global / total_len_global must be >= 0");
    KRAG_REQUIRE(ix->nnz == 0 || vocab > (int64_t)ix->max_term_id, KRAG_E_INVALID,
                 "vocab must exceed the largest term id added to the index");
    // idf on the host with glibc log(): the same libm call chain as the reference's math.log
    std::vector<float> idf((size_t)vocab);
    for (int64_t t = 0; t < vocab; ++t) {
        double dfd = (double)df_global[t];
        idf[(size_t)t] = (float)log(1.0 + ((double)n_docs_global - dfd + 0.5) / (dfd + 0.5));
    }
    float* d_idf = nullptr;
    KRAG_CUDA(cudaMalloc(&d_idf, sizeof(float) * (size_t)vocab));
    KRAG_CUDA(cudaMemcpyAsync(d_idf, idf.data(), sizeof(float) * (size_t)vocab, cudaMemcpyHostToDevice, st));
    const double avgdl = n_docs_global > 0 ? (double)total_len_global / (double)n_docs_global : 1.0;
    if (ix->entry_doc.cap < (ix->nnz > 0 ? ix->nnz : 1)) {
        ix->entry_doc.reserve(ix->nnz > 0 ? ix->nnz : 1, 0, st);
        if (ix->n_rows > 0) launch_expand_entry_doc(ix->toff.p, ix->n_rows, ix->entry_doc.p, st);
    }
    build_postings(ix->tid.p, ix->ttf.p, ix->entry_doc.p, ix->dlen.p, alive_ptr(ix), ix->nnz, vocab, d_idf, avgdl,
                   ix->n_rows, ix->post, st);
    KRAG_CUDA(cudaStreamSynchronize(st));
    KRAG_CUDA(cudaFree(d_idf));
    ix->entry_doc.release();
    ix->vocab = vocab;
    ix->n_docs_global = n_docs_global;
    ix->total_len_global = total_len_global;
    ix->ord_base = ord_base;
    ix->committed = true;
    ix->removed_since_commit = false;
    ix->committed_rows = ix->n_rows;
}

}  // namespace

extern "C" {

int32_t krag_version(void) { return 100; }
const char* krag_last_error(void) { return g_err.c_str(); }

int32_t krag_init(const krag_config* cfg, krag_ctx** out)
{
    return guarded([&] {
        KRAG_REQUIRE(cfg && out, KRAG_E_INVALID, "null argument");
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        KRAG_REQUIRE(e == cudaSuccess && n > 0, KRAG_E_NO_DEVICE,
                     std::string("no CUDA device: ") + cudaGetErrorString(e) + " (libkaito_rag has no CPU fallback)");
        KRAG_REQUIRE(cfg->device_id >= 0 && cfg->device_id < n, KRAG_E_INVALID, "device_id out of range");
        KRAG_CUDA(cudaSetDevice(cfg->device_id));
        cudaDeviceProp p;
        KRAG_CUDA(cudaGetDeviceProperties(&p, cfg->device_id));
        KRAG_REQUIRE(p.major == 10, KRAG_E_NO_DEVICE,
                     std::string("device is sm_") + std::to_string(p.major) + std::to_string(p.minor) +
                         "; libkaito_rag is built for sm_100a only");
        krag_ctx* c = new krag_ctx();
        c->cfg = *cfg;
        if (c->cfg.world_size <= 0) c->cfg.world_size = 1;
        c->di.device = cfg->device_id;
        c->di.sm_count = p.multiProcessorCount;
        c->di.cc_major = p.major;
        c->di.cc_minor = p.minor;
        c->di.smem_optin = p.sharedMemPerBlockOptin;
        KRAG_CUDA(cudaStreamCreateWithFlags(&c->admin, cudaStreamNonBlocking));
        int ns = cfg->search_slots > 0 ? cfg->search_slots : 4;
        for (int i = 0; i < ns; ++i) {
            Slot* s = new Slot();
            KRAG_CUDA(cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking));
            c->all_slots.push_back(s);
            c->free_slots.push_back(s);
        }
        *out = c;
    });
}

int32_t krag_shutdown(krag_ctx* c)
{
    return guarded([&] {
        KRAG_REQUIRE(c, KRAG_E_INVALID, "null context");
        cudaSetDevice(c->di.device);
        cudaDeviceSynchronize();
        for (Slot* s : c->all_slots) {
            s->q.release(); s->terms.release(); s->toff.release(); s->dense_keys.release(); s->bm25_keys.release();
            s->part.release(); s->tc_ws.release(); s->bm25_res.release(); s->allow.release(); s->out_final.release(); s->out_dense.release();
            s->out_sparse.release(); s->out_rank.release(); s->out_count.release(); s->out_ord.release();
            cudaStreamDestroy(s->st);
            delete s;
        }
        cudaStreamDestroy(c->admin);
        delete c;
    });
}

int64_t krag_launch_count(krag_ctx*) { return launch_count(); }
void* krag_ctx_stream(krag_ctx* c) { return c ? (void*)c->all_slots[0]->st : nullptr; }

int32_t krag_index_create(krag_ctx* c, const char* name, int32_t dim, krag_index** out)
{
    return guarded([&] {
        KRAG_REQUIRE(c && name && out, KRAG_E_INVALID, "null argument");
        KRAG_REQUIRE(dim >= 1 && dim <= 16384, KRAG_E_INVALID, "dim must be in [1, 16384]");
        krag_index* ix = new krag_index();
        ix->ctx = c;
        ix->name = name;
        ix->dim = dim;
        ix->dpad = (dim + KRAG_LANES - 1) / KRAG_LANES * KRAG_LANES;
        ix->ord_base = 0;
        *out = ix;
    });
}

int32_t krag_index_drop(krag_index* ix)
{
    return guarded([&] {
        KRAG_REQUIRE(ix, KRAG_E_INVALID, "null index");
        {
            std::unique_lock<std::shared_mutex> lk(ix->mu);
            cudaSetDevice(ix->ctx->di.device);
            cudaDeviceSynchronize();
            ix->X.release(); ix->Xh.release(); ix->xnorm.release(); ix->xn_max.release(); ix->alive_d.release(); ix->toff.release(); ix->tid.release(); ix->ttf.release();
            ix->dlen.release(); ix->entry_doc.release();
            if (ix->post.off) cudaFree(ix->post.off);
            if (ix->post.doc) cudaFree(ix->post.doc);
            if (ix->post.score) cudaFree(ix->post.score);
            if (ix->post.rank_score) cudaFree(ix->post.rank_score);
            if (ix->post.tile_slot) cudaFree(ix->post.tile_slot);
            if (ix->post.tile_off) cudaFree(ix->post.tile_off);
        }
        delete ix;
    });
}

int32_t krag_index_reserve(krag_index* ix, int64_t rows, int64_t nnz)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && rows >= 0, KRAG_E_INVALID, "bad argument");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        ensure_capacity(ix, rows, nnz > 0 ? nnz : -1, ix->ctx->admin);
    });
}

int32_t krag_index_add(krag_index* ix, int64_t n, const uint64_t* node_ids, const float* vecs,
                       const int64_t* term_offsets, const uint32_t* term_ids, const uint16_t* term_tf,
                       const uint32_t* doc_len)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && n >= 0, KRAG_E_INVALID, "bad argument");
        if (n == 0) return;
        KRAG_REQUIRE(node_ids && vecs, KRAG_E_INVALID, "node_ids and vecs are required");
        const bool sparse = term_offsets != nullptr;
        KRAG_REQUIRE(!sparse || (term_ids && term_tf && doc_len), KRAG_E_INVALID, "term_ids/term_tf/doc_len required with term_offsets");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        cudaStream_t st = ix->ctx->admin;
        KRAG_REQUIRE(ix->n_rows == 0 || sparse == ix->has_sparse, KRAG_E_STATE,
                     "an index is either hybrid (term lists for every node) or dense-only");
        {
            std::unordered_map<uint64_t, int64_t> batch;   // ids must be new to the index AND unique inside the call
            batch.reserve((size_t)n);
            for (int64_t i = 0; i < n; ++i) {
                KRAG_REQUIRE(ix->id2row.find(node_ids[i]) == ix->id2row.end(), KRAG_E_INVALID, "duplicate node id");
                KRAG_REQUIRE(batch.emplace(node_ids[i], i).second, KRAG_E_INVALID, "duplicate node id inside the batch");
            }
        }
        const int64_t add_nnz = sparse ? term_offsets[n] - term_offsets[0] : 0;
        KRAG_REQUIRE(!sparse || (term_offsets[0] == 0 && add_nnz >= 0), KRAG_E_INVALID, "term_offsets must start at 0");
        ensure_capacity(ix, ix->n_rows + n, sparse ? ix->nnz + add_nnz : -1, st);
        float* dst = ix->X.p + ix->n_rows * ix->dpad;
        if (ix->dim == ix->dpad) {
            KRAG_CUDA(cudaMemcpyAsync(dst, vecs, sizeof(float) * (size_t)n * ix->dim, cudaMemcpyHostToDevice, st));
        } else {
            KRAG_CUDA(cudaMemsetAsync(dst, 0, sizeof(float) * (size_t)n * ix->dpad, st));
            KRAG_CUDA(cudaMemcpy2DAsync(dst, sizeof(float) * ix->dpad, vecs, sizeof(float) * ix->dim, sizeof(float) * ix->dim,
                                        (size_t)n, cudaMemcpyHostToDevice, st));
        }
        launch_row_norms(ix->X.p, ix->n_rows, n, ix->dpad, ix->xnorm.p, ix->xn_max.p, st);
        if (ix->Xh.p) launch_f32_to_bf16(dst, ix->Xh.p + ix->n_rows * ix->dpad, n * ix->dpad, st);
        std::vector<int64_t> shifted;
        if (sparse) {
            shifted.resize((size_t)n + 1);
            for (int64_t i = 0; i <= n; ++i) {
                KRAG_REQUIRE(i == 0 || term_offsets[i] >= term_offsets[i - 1], KRAG_E_INVALID, "term_offsets must be non-decreasing");
                shifted[(size_t)i] = ix->nnz + term_offsets[i];
            }
            KRAG_CUDA(cudaMemcpyAsync(ix->toff.p + ix->n_rows, shifted.data(), sizeof(int64_t) * (size_t)(n + 1),
                                      cudaMemcpyHostToDevice, st));
            KRAG_CUDA(cudaMemcpyAsync(ix->dlen.p + ix->n_rows, doc_len, sizeof(uint32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
            if (add_nnz > 0) {
                uint32_t mx = ix->max_term_id;
                for (int64_t i = 0; i < add_nnz; ++i) mx = term_ids[i] > mx ? term_ids[i] : mx;
                ix->max_term_id = mx;
                KRAG_CUDA(cudaMemcpyAsync(ix->tid.p + ix->nnz, term_ids, sizeof(uint32_t) * (size_t)add_nnz, cudaMemcpyHostToDevice, st));
                KRAG_CUDA(cudaMemcpyAsync(ix->ttf.p + ix->nnz, term_tf, sizeof(uint16_t) * (size_t)add_nnz, cudaMemcpyHostToDevice, st));
            }
        }
        mark_alive(ix, ix->n_rows, n, st);
        KRAG_CUDA(cudaStreamSynchronize(st));
        for (int64_t i = 0; i < n; ++i) {
            ix->id2row[node_ids[i]] = ix->n_rows + i;
            ix->node_ids.push_back(node_ids[i]);
        }
        ix->n_rows += n;
        ix->n_live += n;
        ix->nnz += add_nnz;
        ix->has_sparse = sparse;
        ix->committed = false;  // postings are stale until the next commit (reference rebuilds per query)
    });
}

int32_t krag_index_remove(krag_index* ix, int64_t n, const uint64_t* node_ids, int64_t* n_removed)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && (n == 0 || node_ids), KRAG_E_INVALID, "bad argument");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        int64_t removed = 0;
        for (int64_t i = 0; i < n; ++i) {
            auto it = ix->id2row.find(node_ids[i]);
            if (it == ix->id2row.end()) continue;
            int64_t r = it->second;
            ix->alive_h[(size_t)(r >> 5)] &= ~(1u << (r & 31));
            KRAG_CUDA(cudaMemcpyAsync(ix->alive_d.p + (r >> 5), &ix->alive_h[(size_t)(r >> 5)], sizeof(uint32_t),
                                      cudaMemcpyHostToDevice, ix->ctx->admin));
            ix->id2row.erase(it);
            ++removed;
        }
        KRAG_CUDA(cudaStreamSynchronize(ix->ctx->admin));
        if (removed) { ix->has_dead = true; ix->removed_since_commit = true; ix->n_live -= removed; }
        if (n_removed) *n_removed = removed;
    });
}

int32_t krag_index_commit_local(krag_index* ix, int64_t vocab, uint32_t* df_out, int64_t* n_live_out, int64_t* total_len_out)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && df_out && n_live_out && total_len_out, KRAG_E_INVALID, "null argument");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        commit_local_impl(ix, vocab, df_out, n_live_out, total_len_out);
    });
}

int32_t krag_index_commit_global(krag_index* ix, int64_t vocab, const uint32_t* df_global, int64_t n_docs_global,
                                 int64_t total_len_global, int64_t ordinal_base)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && df_global, KRAG_E_INVALID, "null argument");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        commit_global_impl(ix, vocab, df_global, n_docs_global, total_len_global, ordinal_base);
    });
}

int32_t krag_index_commit(krag_index* ix, int64_t vocab)
{
    return guarded([&] {
        KRAG_REQUIRE(ix, KRAG_E_INVALID, "null index");
        KRAG_REQUIRE(vocab >= 1 && vocab <= (int64_t)1 << 31, KRAG_E_INVALID, "vocab must be in [1, 2^31]");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        std::vector<uint32_t> df((size_t)vocab);
        int64_t live = 0, total = 0;
        commit_local_impl(ix, vocab, df.data(), &live, &total);
        commit_global_impl(ix, vocab, df.data(), live, total, ix->ord_base);
    });
}

int32_t krag_index_set_ordinal_map(krag_index* ix, int64_t ordinal_base, int64_t ordinal_stride)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && ordinal_base >= 0 && ordinal_stride >= 1 && ordinal_stride <= 64, KRAG_E_INVALID, "bad argument");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_REQUIRE(ordinal_base + ix->n_rows * ordinal_stride <= 0xFFFFFFFFll, KRAG_E_UNSUPPORTED, "global ordinal exceeds 32 bits");
        ix->ord_base = ordinal_base; ix->ord_stride = ordinal_stride;
    });
}

int32_t krag_index_stats(krag_index* ix, krag_stats_t* out)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && out, KRAG_E_INVALID, "null argument");
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        memset(out, 0, sizeof *out);
        out->n_rows = ix->n_rows; out->n_live = ix->n_live; out->nnz = ix->committed ? ix->post.nnz : ix->nnz;
        out->n_docs_global = ix->n_docs_global; out->total_len_global = ix->total_len_global; out->vocab = ix->vocab;
        out->ordinal_base = ix->ord_base; out->dim = ix->dim; out->dim_padded = ix->dpad;
        out->committed = ix->committed && ix->committed_rows == ix->n_rows;
        out->device_bytes = ix->X.bytes() + ix->Xh.bytes() + ix->xnorm.bytes() + ix->alive_d.bytes() + ix->toff.bytes() + ix->tid.bytes() + ix->ttf.bytes() +
                            ix->dlen.bytes() + (ix->committed ? (int64_t)(ix->post.nnz * 8 + (ix->post.vocab + 1) * 8) : 0);
    });
}

int32_t krag_index_node_ids(krag_index* ix, int64_t n, const int64_t* ordinals, uint64_t* out)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && (n == 0 || (ordinals && out)), KRAG_E_INVALID, "null argument");
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        for (int64_t i = 0; i < n; ++i) {
            const int64_t off = ordinals[i] - ix->ord_base;
            KRAG_REQUIRE(off >= 0 && off % ix->ord_stride == 0, KRAG_E_NOT_FOUND, "ordinal is not held by this shard");
            const int64_t r = off / ix->ord_stride;
            KRAG_REQUIRE(r < ix->n_rows, KRAG_E_NOT_FOUND, "ordinal is not held by this shard");
            out[i] = ix->node_ids[(size_t)r];
        }
    });
}

// ------------------------------------------------------------------ host-buffer search
int32_t krag_search_dense(krag_index* ix, int32_t batch, const float* q, int32_t k, float* out_l2sq, int64_t* out_ord)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && q && out_l2sq && out_ord && batch >= 1, KRAG_E_INVALID, "bad argument");
        check_P(k);
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        SlotLease lease(ix->ctx);
        Slot* s = lease.s;
        const float* dq = upload_queries(ix, s, q, batch);
        s->dense_keys.reserve((int64_t)batch * k, 0, s->st);
        dense_candidates_dev(ix, s, dq, batch, k, s->dense_keys.p, s->st);
        std::vector<uint64_t> keys((size_t)batch * k);
        KRAG_CUDA(cudaMemcpyAsync(keys.data(), s->dense_keys.p, sizeof(uint64_t) * keys.size(), cudaMemcpyDeviceToHost, s->st));
        KRAG_CUDA(cudaStreamSynchronize(s->st));
        for (size_t i = 0; i < keys.size(); ++i) {
            if (keys[i] == KEY_PAD) { out_l2sq[i] = INFINITY; out_ord[i] = -1; }
            else { out_l2sq[i] = key_value_asc(keys[i]); out_ord[i] = (int64_t)key_ordinal(keys[i]); }
        }
    });
}

int32_t krag_search_bm25(krag_index* ix, int32_t batch, const uint32_t* q_terms, const int32_t* q_toff, int32_t k,
                         float* out_score, int64_t* out_ord)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && q_toff && out_score && out_ord && batch >= 1, KRAG_E_INVALID, "bad argument");
        check_P(k);
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        SlotLease lease(ix->ctx);
        Slot* s = lease.s;
        upload_terms(s, q_terms, q_toff, batch);
        s->bm25_keys.reserve((int64_t)batch * k, 0, s->st);
        bm25_candidates_dev(ix, s, s->terms.p, s->toff.p, q_toff[batch], batch, k, s->bm25_keys.p, s->st);
        std::vector<uint64_t> keys((size_t)batch * k);
        KRAG_CUDA(cudaMemcpyAsync(keys.data(), s->bm25_keys.p, sizeof(uint64_t) * keys.size(), cudaMemcpyDeviceToHost, s->st));
        KRAG_CUDA(cudaStreamSynchronize(s->st));
        for (size_t i = 0; i < keys.size(); ++i) {
            if (keys[i] == KEY_PAD) { out_score[i] = 0.f; out_ord[i] = -1; }
            else { out_score[i] = key_value_desc(keys[i]); out_ord[i] = (int64_t)key_ordinal(keys[i]); }
        }
    });
}

int32_t krag_retrieve(krag_index* ix, int32_t batch, const float* q, const uint32_t* q_terms, const int32_t* q_toff,
                      int32_t k, double cand_mult, double vector_weight, double text_weight, int32_t fusion_mode,
                      const uint32_t* keyword_allow_bitmap, int64_t keyword_allow_words, double* out_final, float* out_dense,
                      float* out_sparse, int32_t* out_rank, int64_t* out_ord, int32_t* out_count)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && q && out_final && out_dense && out_sparse && out_rank && out_ord && out_count && batch >= 1,
                     KRAG_E_INVALID, "bad argument");
        KRAG_REQUIRE(k >= 1 && k <= KRAG_MAX_TOP_K, KRAG_E_INVALID, "k must be in [1, 300]");
        KRAG_REQUIRE(vector_weight + text_weight > 0, KRAG_E_INVALID, "weights must sum to a positive value");
        // HybridRetriever.__init__ (hybrid_retriever.py:91-98)
        const double total = vector_weight + text_weight;
        const double w_v = vector_weight / total, w_t = text_weight / total;
        const double mult = cand_mult > 1.0 ? cand_mult : 1.0;
        const int P = (int)((double)k * mult);
        check_P(P);
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        // the bitmap is read (n_rows + 31) / 32 words deep: the caller states how many it holds, so a bitmap built
        // before a concurrent krag_index_add is refused instead of over-read
        KRAG_REQUIRE(keyword_allow_bitmap == nullptr || keyword_allow_words >= (ix->n_rows + 31) / 32, KRAG_E_INVALID,
                     "keyword_allow_bitmap holds fewer words than the index has rows / 32");
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        SlotLease lease(ix->ctx);
        Slot* s = lease.s;
        cudaStream_t st = s->st;
        const bool hybrid = q_terms != nullptr && q_toff != nullptr && ix->committed;
        const bool pushdown = (fusion_mode & KRAG_FILTER_PUSHDOWN) != 0 && keyword_allow_bitmap != nullptr;
        fusion_mode &= 0xFF;
        const uint32_t* eligible = nullptr;
        if (pushdown) {   // eligible = allow & alive, consumed by K1/K2/K3 in place of the tombstone bitmap
            const int64_t words = (ix->n_rows + 31) / 32;
            s->allow.reserve(words > 0 ? words : 1, 0, st);
            KRAG_CUDA(cudaMemcpyAsync(s->allow.p, keyword_allow_bitmap, sizeof(uint32_t) * (size_t)words, cudaMemcpyHostToDevice, st));
            if (ix->has_dead && words > 0) launch_bitmap_and(s->allow.p, ix->alive_d.p, words, st);
            eligible = s->allow.p;
        }
        const float* dq = upload_queries(ix, s, q, batch);
        s->dense_keys.reserve((int64_t)batch * P, 0, st);
        dense_candidates_dev(ix, s, dq, batch, P, s->dense_keys.p, st, eligible);
        const uint32_t* d_allow = nullptr;
        if (hybrid) {
            upload_terms(s, q_terms, q_toff, batch);
            s->bm25_keys.reserve((int64_t)batch * P, 0, st);
            bm25_candidates_dev(ix, s, s->terms.p, s->toff.p, q_toff[batch], batch, P, s->bm25_keys.p, st, eligible);
            if (keyword_allow_bitmap && !pushdown) {
                // bitmap is over local rows; fuse tests global ordinals -> shift by ord_base words is only
                // valid when ord_base % 32 == 0; the host path is single-shard (ord_base == 0)
                KRAG_REQUIRE(ix->ord_base == 0 && ix->ord_stride == 1, KRAG_E_UNSUPPORTED, "keyword filter on host path requires ordinal_base 0, stride 1");
                int64_t words = (ix->n_rows + 31) / 32;
                s->allow.reserve(words, 0, st);
                KRAG_CUDA(cudaMemcpyAsync(s->allow.p, keyword_allow_bitmap, sizeof(uint32_t) * (size_t)words, cudaMemcpyHostToDevice, st));
                d_allow = s->allow.p;
            }
        }
        const int64_t nk = (int64_t)batch * k;
        s->out_final.reserve(nk, 0, st); s->out_dense.reserve(nk, 0, st); s->out_sparse.reserve(nk, 0, st);
        s->out_rank.reserve(nk, 0, st); s->out_ord.reserve(nk, 0, st); s->out_count.reserve(batch, 0, st);
        launch_fuse(batch, P, k, s->dense_keys.p, hybrid ? s->bm25_keys.p : nullptr, w_v, w_t, fusion_mode, d_allow,
                    s->out_final.p, s->out_dense.p, s->out_sparse.p, s->out_rank.p, s->out_ord.p, s->out_count.p, st);
        KRAG_CUDA(cudaMemcpyAsync(out_final, s->out_final.p, sizeof(double) * (size_t)nk, cudaMemcpyDeviceToHost, st));
        KRAG_CUDA(cudaMemcpyAsync(out_dense, s->out_dense.p, sizeof(float) * (size_t)nk, cudaMemcpyDeviceToHost, st));
        KRAG_CUDA(cudaMemcpyAsync(out_sparse, s->out_sparse.p, sizeof(float) * (size_t)nk, cudaMemcpyDeviceToHost, st));
        KRAG_CUDA(cudaMemcpyAsync(out_rank, s->out_rank.p, sizeof(int32_t) * (size_t)nk, cudaMemcpyDeviceToHost, st));
        KRAG_CUDA(cudaMemcpyAsync(out_ord, s->out_ord.p, sizeof(int64_t) * (size_t)nk, cudaMemcpyDeviceToHost, st));
        KRAG_CUDA(cudaMemcpyAsync(out_count, s->out_count.p, sizeof(int32_t) * (size_t)batch, cudaMemcpyDeviceToHost, st));
        KRAG_CUDA(cudaStreamSynchronize(st));
    });
}

// ---------------------------------------------------------------- device stage API
int32_t krag_dev_dense_candidates(krag_index* ix, int32_t batch, const float* d_q, int32_t P, uint64_t* d_keys, void* stream)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && d_q && d_keys && batch >= 1, KRAG_E_INVALID, "bad argument");
        check_P(P);
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        SlotLease lease(ix->ctx);
        dense_candidates_dev(ix, lease.s, d_q, batch, P, d_keys, (cudaStream_t)stream);
    });
}

int32_t krag_dev_bm25_candidates(krag_index* ix, int32_t batch, const uint32_t* d_terms, const int32_t* d_toff,
                                 const int32_t* h_toff, int32_t P, uint64_t* d_keys, void* stream)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && d_toff && d_keys && batch >= 1, KRAG_E_INVALID, "bad argument");
        check_P(P);
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        SlotLease lease(ix->ctx);
        bm25_candidates_dev(ix, lease.s, d_terms, d_toff, h_toff ? h_toff[batch] : -1, batch, P, d_keys, (cudaStream_t)stream);
    });
}

int32_t krag_dev_merge(krag_ctx* c, int32_t n_lists, int32_t batch, int32_t P, const uint64_t* d_in, uint64_t* d_out, void* stream)
{
    return guarded([&] {
        KRAG_REQUIRE(c && d_in && d_out && n_lists >= 1 && batch >= 1, KRAG_E_INVALID, "bad argument");
        check_P(P);
        KRAG_CUDA(cudaSetDevice(c->di.device));
        launch_merge(d_in, n_lists, P, batch, P, (int64_t)batch * P, P, d_out, (cudaStream_t)stream);
    });
}

int32_t krag_dev_fuse(krag_ctx* c, int32_t batch, int32_t P, int32_t k, const uint64_t* d_dense, const uint64_t* d_bm25,
                      double vector_weight, double text_weight, int32_t fusion_mode, const uint32_t* d_allow,
                      double* d_final, float* d_dense_out, float* d_sparse_out, int32_t* d_rank, int64_t* d_ord,
                      int32_t* d_count, void* stream)
{
    return guarded([&] {
        KRAG_REQUIRE(c && d_dense && d_final && d_dense_out && d_sparse_out && d_rank && d_ord && d_count && batch >= 1,
                     KRAG_E_INVALID, "bad argument");
        KRAG_REQUIRE(k >= 1 && k <= KRAG_MAX_POOL, KRAG_E_INVALID, "k out of range");
        check_P(P);
        const double total = vector_weight + text_weight;
        KRAG_REQUIRE(total > 0, KRAG_E_INVALID, "weights must sum to a positive value");
        KRAG_CUDA(cudaSetDevice(c->di.device));
        launch_fuse(batch, P, k, d_dense, d_bm25, vector_weight / total, text_weight / total, fusion_mode, d_allow, d_final,
                    d_dense_out, d_sparse_out, d_rank, d_ord, d_count, (cudaStream_t)stream);
    });
}

// -------------------------------------------------------------------- synthetic / io
int32_t krag_synth_fill(krag_index* ix, int64_t n, int64_t row_base, uint64_t seed, int64_t vocab)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && n >= 0, KRAG_E_INVALID, "bad argument");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        cudaStream_t st = ix->ctx->admin;
        KRAG_REQUIRE(ix->n_rows == 0, KRAG_E_STATE, "synthetic fill needs an empty index");
        ensure_capacity(ix, n, -1, st);
        launch_synth_dense(ix->X.p, n, ix->dim, ix->dpad, row_base, seed, st);
        launch_row_norms(ix->X.p, 0, n, ix->dpad, ix->xnorm.p, ix->xn_max.p, st);
        if (ix->Xh.p) launch_f32_to_bf16(ix->X.p, ix->Xh.p, n * ix->dpad, st);
        if (vocab > 0) {
            int64_t* off = nullptr; uint32_t* ids = nullptr; uint16_t* tf = nullptr; uint32_t* dl = nullptr; int64_t nnz = 0;
            synth_sparse(n, row_base, seed, vocab, &off, &ids, &tf, &dl, &nnz, st);
            ix->toff.release(); ix->tid.release(); ix->ttf.release(); ix->dlen.release();
            ix->toff.p = off; ix->toff.cap = n + 1;
            ix->tid.p = ids; ix->tid.cap = nnz > 0 ? nnz : 1;
            ix->ttf.p = tf; ix->ttf.cap = nnz > 0 ? nnz : 1;
            ix->dlen.p = dl; ix->dlen.cap = n > 0 ? n : 1;
            ix->nnz = nnz;
            ix->max_term_id = (uint32_t)(vocab - 1);     // the generator draws ids in [0, vocab)
            ix->has_sparse = true;
        }
        mark_alive(ix, 0, n, st);
        KRAG_CUDA(cudaStreamSynchronize(st));
        ix->node_ids.resize((size_t)n);
        for (int64_t i = 0; i < n; ++i) { ix->node_ids[(size_t)i] = (uint64_t)(row_base + i); ix->id2row[(uint64_t)(row_base + i)] = i; }
        ix->n_rows = n; ix->n_live = n; ix->ord_base = row_base; ix->ord_stride = 1; ix->committed = false;
    });
}

int32_t krag_index_read_rows(krag_index* ix, int64_t row0, int64_t n, float* out)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && out && row0 >= 0 && n >= 0 && row0 + n <= ix->n_rows, KRAG_E_INVALID, "row range out of bounds");
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        if (n == 0) return;
        KRAG_CUDA(cudaMemcpy2D(out, sizeof(float) * ix->dim, ix->X.p + row0 * ix->dpad, sizeof(float) * ix->dpad,
                               sizeof(float) * ix->dim, (size_t)n, cudaMemcpyDeviceToHost));
    });
}

int32_t krag_index_read_postings(krag_index* ix, uint32_t term, int64_t cap, uint32_t* docs_out, float* scores_out, int64_t* n_out)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && n_out, KRAG_E_INVALID, "null argument");
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_REQUIRE(ix->committed, KRAG_E_STATE, "index not committed");
        KRAG_REQUIRE((int64_t)term < ix->post.vocab, KRAG_E_INVALID, "term id out of range");
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        int64_t be[2];
        KRAG_CUDA(cudaMemcpy(be, ix->post.off + term, sizeof be, cudaMemcpyDeviceToHost));
        int64_t cnt = be[1] - be[0];
        *n_out = cnt;
        int64_t m = cnt < cap ? cnt : cap;
        if (m > 0 && docs_out) KRAG_CUDA(cudaMemcpy(docs_out, ix->post.doc + be[0], sizeof(uint32_t) * (size_t)m, cudaMemcpyDeviceToHost));
        if (m > 0 && scores_out) KRAG_CUDA(cudaMemcpy(scores_out, ix->post.score + be[0], sizeof(float) * (size_t)m, cudaMemcpyDeviceToHost));
    });
}

int32_t krag_index_read_rank_scores(krag_index* ix, uint32_t term, float* out)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && out, KRAG_E_INVALID, "null argument");
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_REQUIRE(ix->committed, KRAG_E_STATE, "index not committed");
        KRAG_REQUIRE((int64_t)term < ix->post.vocab, KRAG_E_INVALID, "term id out of range");
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        KRAG_CUDA(cudaMemcpy(out, ix->post.rank_score + (size_t)term * BM25_RANKS, sizeof(float) * BM25_RANKS, cudaMemcpyDeviceToHost));
    });
}

int32_t krag_index_set_dense_mode(krag_index* ix, int32_t dense_mode, int32_t release_shadow)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && dense_mode >= KRAG_DENSE_AUTO && dense_mode <= KRAG_DENSE_TC_TF32, KRAG_E_INVALID, "bad argument");
        std::unique_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        cudaStream_t st = ix->ctx->admin;
        if (dense_mode == KRAG_DENSE_TC_BF16 && ix->Xh.p == nullptr && ix->X.p != nullptr) {
            ix->Xh.reserve(ix->X.cap, 0, st);                     // same capacity as the fp32 rows: later appends convert in place
            launch_f32_to_bf16(ix->X.p, ix->Xh.p, ix->n_rows * ix->dpad, st);
        }
        if (dense_mode != KRAG_DENSE_TC_BF16 && release_shadow) ix->Xh.release();
        KRAG_CUDA(cudaStreamSynchronize(st));
        ix->ctx->cfg.dense_mode = dense_mode;
    });
}

int64_t krag_tc_fallback_queries(void) { return dense_tc_fallback_queries(); }

int32_t krag_last_dense_kernel(float* ms, int32_t* kernel_id, int64_t* algorithmic_bytes, int64_t* flops)
{
    return guarded([&] {
        KRAG_REQUIRE(ms && kernel_id && algorithmic_bytes && flops, KRAG_E_INVALID, "null argument");
        int kid = 0;
        KRAG_REQUIRE(dense_timer_read(ms, &kid, algorithmic_bytes, flops), KRAG_E_STATE, "no dense kernel timed yet");
        *kernel_id = kid;
    });
}

int32_t krag_debug_tc_dump(krag_index* ix, int32_t nq, const float* q, float* out, int64_t out_elems, int64_t* S_out, int32_t* nq_pad_out)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && q && S_out && nq_pad_out && nq >= 1 && nq <= 256, KRAG_E_INVALID, "bad argument");
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        SlotLease lease(ix->ctx);
        Slot* s = lease.s;
        int64_t S = 0; int nqp = 0;
        KRAG_REQUIRE(dense_tc_debug_dump(ix->ctx->di, ix->X.p, ix->n_rows, ix->dpad, ix->xnorm.p, nullptr, nq, nullptr, &S, &nqp, s->st),
                     KRAG_E_UNSUPPORTED, "tensor-core path unavailable");
        *S_out = S; *nq_pad_out = nqp;
        if (!out) return;
        KRAG_REQUIRE(out_elems >= S * nqp, KRAG_E_INVALID, "output buffer too small");
        const float* dq = upload_queries(ix, s, q, nq);
        s->tc_ws.reserve(S * nqp * 4, 0, s->st);
        KRAG_REQUIRE(dense_tc_debug_dump(ix->ctx->di, ix->X.p, ix->n_rows, ix->dpad, ix->xnorm.p, dq, nq, (float*)s->tc_ws.p, &S, &nqp, s->st),
                     KRAG_E_UNSUPPORTED, "tensor-core dump failed");
        KRAG_CUDA(cudaMemcpyAsync(out, s->tc_ws.p, sizeof(float) * (size_t)(S * nqp), cudaMemcpyDeviceToHost, s->st));
        KRAG_CUDA(cudaStreamSynchronize(s->st));
    });
}

// ------------------------------------------------------------- peer-memory exchange (one process per GPU)
struct krag_p2p {
    krag_ctx* ctx; int rank, world, nl, max_batch, max_P; int64_t slot_words;
    uint64_t* own = nullptr;                 // this rank's mailbox (cudaMalloc, IPC-exported)
    std::vector<uint64_t*> peers;            // [world] device pointers: own + IPC-opened peers
    uint64_t** d_peers = nullptr;            // device copy of the pointer table
    unsigned long long seq = 0;
};

int32_t krag_p2p_create(krag_ctx* c, int32_t rank, int32_t world, int32_t max_batch, int32_t max_P, krag_p2p** out, uint8_t* handle_out /*[64]*/)
{
    return guarded([&] {
        KRAG_REQUIRE(c && out && handle_out && world >= 1 && world <= 64 && rank >= 0 && rank < world, KRAG_E_INVALID, "bad argument");
        KRAG_CUDA(cudaSetDevice(c->di.device));
        krag_p2p* p = new krag_p2p();
        p->ctx = c; p->rank = rank; p->world = world; p->nl = 2; p->max_batch = max_batch; p->max_P = max_P;
        p->slot_words = (int64_t)2 * max_batch * max_P;
        const size_t words = p2p_mailbox_words(world, 2, max_batch, max_P);
        KRAG_CUDA(cudaMalloc(&p->own, words * 8));
        KRAG_CUDA(cudaMemset(p->own, 0, words * 8));
        cudaIpcMemHandle_t h;
        KRAG_CUDA(cudaIpcGetMemHandle(&h, p->own));
        static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
        memcpy(handle_out, &h, 64);
        p->peers.assign((size_t)world, nullptr);
        p->peers[(size_t)rank] = p->own;
        *out = p;
    });
}

int32_t krag_p2p_connect(krag_p2p* p, const uint8_t* handles /*[world][64]*/)
{
    return guarded([&] {
        KRAG_REQUIRE(p && handles, KRAG_E_INVALID, "null argument");
        KRAG_CUDA(cudaSetDevice(p->ctx->di.device));
        for (int r = 0; r < p->world; ++r) {
            if (r == p->rank) continue;
            cudaIpcMemHandle_t h;
            memcpy(&h, handles + (size_t)r * 64, 64);
            void* ptr = nullptr;
            KRAG_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
            p->peers[(size_t)r] = (uint64_t*)ptr;
        }
        KRAG_CUDA(cudaMalloc(&p->d_peers, sizeof(uint64_t*) * (size_t)p->world));
        KRAG_CUDA(cudaMemcpy(p->d_peers, p->peers.data(), sizeof(uint64_t*) * (size_t)p->world, cudaMemcpyHostToDevice));
    });
}

int32_t krag_dev_exchange_merge(krag_p2p* p, int32_t n_lists, int32_t batch, int32_t P, const uint64_t* d_local, uint64_t* d_merged, void* stream)
{
    return guarded([&] {
        KRAG_REQUIRE(p && p->d_peers && d_local && d_merged, KRAG_E_INVALID, "bad argument / not connected");
        KRAG_REQUIRE(n_lists >= 1 && n_lists <= 2 && batch >= 1 && (int64_t)n_lists * batch * P <= p->slot_words, KRAG_E_INVALID,
                     "exchange exceeds the mailbox the ranks agreed on");
        check_P(P);
        KRAG_CUDA(cudaSetDevice(p->ctx->di.device));
        ++p->seq;
        launch_p2p_exchange_merge(p->d_peers, p->own, p->rank, p->world, p->slot_words, p->seq, n_lists, batch, P, d_local, d_merged,
                                  (cudaStream_t)stream);
    });
}

int32_t krag_p2p_destroy(krag_p2p* p)
{
    return guarded([&] {
        KRAG_REQUIRE(p, KRAG_E_INVALID, "null argument");
        cudaSetDevice(p->ctx->di.device);
        cudaDeviceSynchronize();
        for (int r = 0; r < p->world; ++r) if (r != p->rank && p->peers[(size_t)r]) cudaIpcCloseMemHandle(p->peers[(size_t)r]);
        if (p->d_peers) cudaFree(p->d_peers);
        if (p->own) cudaFree(p->own);
        delete p;
    });
}

// ---------------------------------------------------------------------- K5 embedder
struct krag_embedder { krag_ctx* ctx; Embedder* e; };

int32_t krag_embedder_create(krag_ctx* c, const krag_bert_config* cfg, krag_embedder** out)
{
    return guarded([&] {
        KRAG_REQUIRE(c && cfg && out, KRAG_E_INVALID, "null argument");
        KRAG_CUDA(cudaSetDevice(c->di.device));
        BertConfig bc{cfg->layers, cfg->hidden, cfg->heads, cfg->intermediate, cfg->vocab, cfg->max_position, cfg->type_vocab, cfg->ln_eps};
        krag_embedder* h = new krag_embedder{c, embedder_create(c->di, bc)};
        *out = h;
    });
}
int32_t krag_embedder_load_tensor(krag_embedder* h, const char* name, const float* data, int64_t n)
{
    return guarded([&] {
        KRAG_REQUIRE(h && name && data && n > 0, KRAG_E_INVALID, "bad argument");
        KRAG_CUDA(cudaSetDevice(h->ctx->di.device));
        embedder_load(h->e, name, data, n);
    });
}
int32_t krag_embedder_finalize(krag_embedder* h)
{
    return guarded([&] {
        KRAG_REQUIRE(h, KRAG_E_INVALID, "null embedder");
        KRAG_CUDA(cudaSetDevice(h->ctx->di.device));
        embedder_finalize(h->e);
    });
}
int32_t krag_embed(krag_embedder* h, int32_t batch, const int32_t* tok_ids, const int32_t* tok_offsets, float* out)
{
    return guarded([&] {
        KRAG_REQUIRE(h && tok_ids && tok_offsets && out && batch >= 1, KRAG_E_INVALID, "bad argument");
        KRAG_REQUIRE(tok_offsets[0] == 0, KRAG_E_INVALID, "tok_offsets must start at 0");
        KRAG_CUDA(cudaSetDevice(h->ctx->di.device));
        embedder_forward(h->e, batch, tok_ids, tok_offsets, out);
    });
}
int32_t krag_embed_dev(krag_embedder* h, int32_t batch, const int32_t* tok_ids, const int32_t* tok_offsets, float* d_out,
                       int32_t ld_out, void* stream)
{
    return guarded([&] {
        KRAG_REQUIRE(h && tok_ids && tok_offsets && d_out && batch >= 1 && ld_out >= embedder_hidden(h->e), KRAG_E_INVALID, "bad argument");
        KRAG_REQUIRE(tok_offsets[0] == 0, KRAG_E_INVALID, "tok_offsets must start at 0");
        KRAG_CUDA(cudaSetDevice(h->ctx->di.device));
        embedder_forward(h->e, batch, tok_ids, tok_offsets, nullptr, d_out, ld_out, (cudaStream_t)stream);
    });
}
int32_t krag_embedder_destroy(krag_embedder* h)
{
    return guarded([&] {
        KRAG_REQUIRE(h, KRAG_E_INVALID, "null embedder");
        cudaSetDevice(h->ctx->di.device);
        embedder_destroy(h->e);
        delete h;
    });
}
static void debug_linear(krag_ctx* c, int32_t M, int32_t N, int32_t K, const float* A, const float* B, const float* bias,
                         const float* residual, int32_t gelu, const float* ln_g, const float* ln_b, float eps, float* out)
{
    KRAG_REQUIRE(c && A && B && bias && out && M >= 1 && N % 128 == 0 && K % 64 == 0, KRAG_E_INVALID, "bad argument (N % 128, K % 64)");
    KRAG_CUDA(cudaSetDevice(c->di.device));
    float *dA, *dB, *db, *dr = nullptr, *dC, *dY = nullptr, *dg = nullptr, *dlb = nullptr, *ws;
    const size_t ws_floats = (size_t)4 << 20;
    KRAG_CUDA(cudaMalloc(&dA, 4 * (size_t)M * K)); KRAG_CUDA(cudaMalloc(&dB, 4 * (size_t)N * K)); KRAG_CUDA(cudaMalloc(&db, 4 * (size_t)N));
    KRAG_CUDA(cudaMalloc(&dC, 4 * (size_t)M * N)); KRAG_CUDA(cudaMalloc(&ws, 4 * ws_floats));
    KRAG_CUDA(cudaMemcpy(dA, A, 4 * (size_t)M * K, cudaMemcpyHostToDevice)); KRAG_CUDA(cudaMemcpy(dB, B, 4 * (size_t)N * K, cudaMemcpyHostToDevice));
    KRAG_CUDA(cudaMemcpy(db, bias, 4 * (size_t)N, cudaMemcpyHostToDevice));
    if (residual) { KRAG_CUDA(cudaMalloc(&dr, 4 * (size_t)M * N)); KRAG_CUDA(cudaMemcpy(dr, residual, 4 * (size_t)M * N, cudaMemcpyHostToDevice)); }
    if (ln_g) {
        KRAG_CUDA(cudaMalloc(&dg, 4 * (size_t)N)); KRAG_CUDA(cudaMalloc(&dlb, 4 * (size_t)N)); KRAG_CUDA(cudaMalloc(&dY, 4 * (size_t)M * N));
        KRAG_CUDA(cudaMemcpy(dg, ln_g, 4 * (size_t)N, cudaMemcpyHostToDevice)); KRAG_CUDA(cudaMemcpy(dlb, ln_b, 4 * (size_t)N, cudaMemcpyHostToDevice));
    }
    launch_linear_f32(c->di, dA, dB, M, N, K, db, dr, gelu != 0, dC, dg, dlb, eps, dY, ws, ws_floats, c->admin);
    KRAG_CUDA(cudaStreamSynchronize(c->admin));
    KRAG_CUDA(cudaMemcpy(out, ln_g ? dY : dC, 4 * (size_t)M * N, cudaMemcpyDeviceToHost));
    cudaFree(dA); cudaFree(dB); cudaFree(db); cudaFree(dC); cudaFree(ws);
    if (dr) cudaFree(dr);
    if (dg) { cudaFree(dg); cudaFree(dlb); cudaFree(dY); }
}

int32_t krag_debug_gemm_tf32(krag_ctx* c, int32_t M, int32_t N, int32_t K, const float* A, const float* B, const float* bias,
                             const float* residual, int32_t gelu, float* C_out)
{
    return guarded([&] { debug_linear(c, M, N, K, A, B, bias, residual, gelu, nullptr, nullptr, 0.f, C_out); });
}

int32_t krag_debug_linear_ln(krag_ctx* c, int32_t M, int32_t N, int32_t K, const float* A, const float* B, const float* bias,
                             const float* residual, const float* ln_gamma, const float* ln_beta, float eps, float* Y_out)
{
    return guarded([&] {
        KRAG_REQUIRE(ln_gamma && ln_beta, KRAG_E_INVALID, "null LayerNorm parameters");
        debug_linear(c, M, N, K, A, B, bias, residual, 0, ln_gamma, ln_beta, eps, Y_out);
    });
}

// Own on-disk format (SURVEY.md section 5: the snapshot only needs to round-trip itself).
static const char kMagic[8] = {'K', 'R', 'A', 'G', 'I', 'D', 'X', '1'};

int32_t krag_index_persist(krag_index* ix, const char* dir)
{
    return guarded([&] {
        KRAG_REQUIRE(ix && dir, KRAG_E_INVALID, "null argument");
        std::shared_lock<std::shared_mutex> lk(ix->mu);
        KRAG_CUDA(cudaSetDevice(ix->ctx->di.device));
        mkdir(dir, 0755);
        std::string path = std::string(dir) + "/krag_index.bin";
        FILE* f = fopen((path + ".tmp").c_str(), "wb");
        KRAG_REQUIRE(f, KRAG_E_IO, "cannot open " + path + ".tmp for writing");
        auto W = [&](const void* p, size_t n) { if (n && fwrite(p, 1, n, f) != n) { fclose(f); throw ApiError{KRAG_E_IO, "short write to " + path}; } };
        int64_t hdr[8] = {ix->dim, ix->n_rows, ix->nnz, ix->has_sparse ? 1 : 0, ix->committed ? ix->vocab : 0, 0, 0, 0};
        W(kMagic, 8); W(hdr, sizeof hdr);
        W(ix->node_ids.data(), sizeof(uint64_t) * (size_t)ix->n_rows);
        W(ix->alive_h.data(), sizeof(uint32_t) * (size_t)((ix->n_rows + 31) / 32));
        const int64_t chunk = 1 << 16;
        std::vector<float> rows((size_t)chunk * ix->dim);
        for (int64_t r = 0; r < ix->n_rows; r += chunk) {
            int64_t m = ix->n_rows - r < chunk ? ix->n_rows - r : chunk;
            KRAG_CUDA(cudaMemcpy2D(rows.data(), sizeof(float) * ix->dim, ix->X.p + r * ix->dpad, sizeof(float) * ix->dpad,
                                   sizeof(float) * ix->dim, (size_t)m, cudaMemcpyDeviceToHost));
            W(rows.data(), sizeof(float) * (size_t)m * ix->dim);
        }
        if (ix->has_sparse) {
            std::vector<int64_t> off((size_t)ix->n_rows + 1);
            std::vector<uint32_t> dl((size_t)ix->n_rows), ids((size_t)ix->nnz);
            std::vector<uint16_t> tf((size_t)ix->nnz);
            KRAG_CUDA(cudaMemcpy(off.data(), ix->toff.p, sizeof(int64_t) * off.size(), cudaMemcpyDeviceToHost));
            if (ix->n_rows) KRAG_CUDA(cudaMemcpy(dl.data(), ix->dlen.p, sizeof(uint32_t) * dl.size(), cudaMemcpyDeviceToHost));
            if (ix->nnz) {
                KRAG_CUDA(cudaMemcpy(ids.data(), ix->tid.p, sizeof(uint32_t) * ids.size(), cudaMemcpyDeviceToHost));
                KRAG_CUDA(cudaMemcpy(tf.data(), ix->ttf.p, sizeof(uint16_t) * tf.size(), cudaMemcpyDeviceToHost));
            }
            W(off.data(), sizeof(int64_t) * off.size()); W(dl.data(), sizeof(uint32_t) * dl.size());
            W(ids.data(), sizeof(uint32_t) * ids.size()); W(tf.data(), sizeof(uint16_t) * tf.size());
        }
        KRAG_REQUIRE(fclose(f) == 0, KRAG_E_IO, "close failed for " + path);
        KRAG_REQUIRE(rename((path + ".tmp").c_str(), path.c_str()) == 0, KRAG_E_IO, "rename failed for " + path);
    });
}

int32_t krag_index_load(krag_ctx* c, const char* name, const char* dir, krag_index** out)
{
    krag_index* ix = nullptr;
    int32_t rc = guarded([&] {
        KRAG_REQUIRE(c && name && dir && out, KRAG_E_INVALID, "null argument");
        std::string path = std::string(dir) + "/krag_index.bin";
        FILE* f = fopen(path.c_str(), "rb");
        KRAG_REQUIRE(f, KRAG_E_IO, "cannot open " + path);
        auto R = [&](void* p, size_t n) { if (n && fread(p, 1, n, f) != n) { fclose(f); throw ApiError{KRAG_E_IO, "short read from " + path}; } };
        char magic[8]; int64_t hdr[8];
        R(magic, 8); R(hdr, sizeof hdr);
        if (memcmp(magic, kMagic, 8) != 0) { fclose(f); throw ApiError{KRAG_E_IO, path + " is not a krag index snapshot"}; }
        const int64_t dim = hdr[0], n = hdr[1], nnz = hdr[2], sparse = hdr[3], vocab = hdr[4];
        int32_t rc2 = krag_index_create(c, name, (int32_t)dim, &ix);
        if (rc2 != KRAG_OK) { fclose(f); throw ApiError{rc2, g_err}; }
        std::vector<uint64_t> ids((size_t)n);
        std::vector<uint32_t> alive((size_t)((n + 31) / 32));
        R(ids.data(), sizeof(uint64_t) * ids.size()); R(alive.data(), sizeof(uint32_t) * alive.size());
        std::vector<float> rows((size_t)n * dim);
        R(rows.data(), sizeof(float) * rows.size());
        std::vector<int64_t> off; std::vector<uint32_t> dl, tids; std::vector<uint16_t> tf;
        if (sparse) {
            off.resize((size_t)n + 1); dl.resize((size_t)n); tids.resize((size_t)nnz); tf.resize((size_t)nnz);
            R(off.data(), sizeof(int64_t) * off.size()); R(dl.data(), sizeof(uint32_t) * dl.size());
            R(tids.data(), sizeof(uint32_t) * tids.size()); R(tf.data(), sizeof(uint16_t) * tf.size());
        }
        fclose(f);
        if (n > 0) {
            rc2 = krag_index_add(ix, n, ids.data(), rows.data(), sparse ? off.data() : nullptr, sparse ? tids.data() : nullptr,
                                 sparse ? tf.data() : nullptr, sparse ? dl.data() : nullptr);
            if (rc2 != KRAG_OK) throw ApiError{rc2, g_err};
            std::vector<uint64_t> dead;
            for (int64_t r = 0; r < n; ++r) if (!((alive[(size_t)(r >> 5)] >> (r & 31)) & 1u)) dead.push_back(ids[(size_t)r]);
            if (!dead.empty()) { rc2 = krag_index_remove(ix, (int64_t)dead.size(), dead.data(), nullptr); if (rc2 != KRAG_OK) throw ApiError{rc2, g_err}; }
        }
        if (sparse && vocab > 0) { rc2 = krag_index_commit(ix, vocab); if (rc2 != KRAG_OK) throw ApiError{rc2, g_err}; }
        *out = ix;
    });
    if (rc != KRAG_OK && ix) { std::string keep = g_err; krag_index_drop(ix); set_error(keep); }
    return rc;
}

}  // extern "C"
