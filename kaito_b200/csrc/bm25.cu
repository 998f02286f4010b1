// bm25.cu -- K3: BM25 postings build (index time) and score/accumulate/select (query time).
//
// Replaces, with identical arithmetic, what the reference does on EVERY query at
// presets/ragengine/vector_store/retriever/hybrid_retriever.py:104-130 (BM25Retriever.
// from_defaults -> bm25s "lucene" score matrix) and :220 (bm25_retriever.aretrieve):
//   score(t,d) = (f32)( (f64) idf32[t] * tf / (k1*((1-b) + b*dl/avgdl) + tf) ),  k1=1.5, b=0.75
//   acc[d]    += score(t,d)  for the query's term ids in query order (fp32, duplicates kept)
//   result     = top-P by (score desc, ordinal asc)
// idf32 is computed on the host with glibc log() (the library the reference's math.log
// uses); every other operation is a correctly rounded IEEE op issued without contraction.
//
// Query kernel: one CTA per (doc-range tile, query).  The tile's fp32 accumulators live in
// shared memory, postings are read exactly once with coalesced loads (8 bytes per posting
// = the algorithmic traffic), terms are applied one after another (doc ids are unique
// inside a term, so no atomics and a fixed fp32 summation order), and the top-P select
// runs over shared memory.
#include <math_constants.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>

#include <stdlib.h>
#include <algorithm>
#include <stdexcept>
#include <vector>

#include "engine.h"
#include "select.cuh"

namespace krag {

// -------------------------------------------------------------------------- index time
__global__ void expand_entry_doc_kernel(const int64_t* __restrict__ off, int64_t n_docs, uint32_t* __restrict__ entry_doc)
{
    // one warp per document
    int64_t d = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (d >= n_docs) return;
    for (int64_t i = off[d] + lane; i < off[d + 1]; i += 32) entry_doc[i] = (uint32_t)d;
}
void launch_expand_entry_doc(const int64_t* term_offsets, int64_t n_docs, uint32_t* entry_doc, cudaStream_t st)
{
    if (n_docs == 0) return;
    int64_t threads = n_docs * 32;
    expand_entry_doc_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(term_offsets, n_docs, entry_doc);
    KRAG_CUDA(cudaGetLastError());
    count_launch();
}

__global__ void df_hist_kernel(const uint32_t* __restrict__ term_ids, const uint32_t* __restrict__ entry_doc,
                               const uint32_t* __restrict__ alive, int64_t nnz, uint32_t* __restrict__ df)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x)
        if (alive == nullptr || bit_test(alive, entry_doc[i])) atomicAdd(&df[term_ids[i]], 1u);
}
void launch_df_histogram(const uint32_t* term_ids, const uint32_t* entry_doc, const uint32_t* alive, int64_t nnz,
                         uint32_t* df, cudaStream_t st)
{
    if (nnz == 0) return;
    df_hist_kernel<<<148 * 8, 256, 0, st>>>(term_ids, entry_doc, alive, nnz, df);
    KRAG_CUDA(cudaGetLastError());
    count_launch();
}

// Stable compaction of the index entries that belong to one TERM RANGE [t_lo, t_hi) of live documents: the postings are built
// range by range (radix sort of one range at a time), so the sort's four key/value buffers hold one range, not the whole index.
// Two passes over the raw entries: per-block counts, (exclusive scan,) ordered scatter.
constexpr int CC_THREADS = 256;
constexpr int CC_ITEMS = 8;                       // consecutive entries per thread: 2048 per block
__device__ __forceinline__ bool chunk_member(const uint32_t* __restrict__ term_ids, const uint32_t* __restrict__ entry_doc,
                                             const uint32_t* __restrict__ alive, int64_t i, uint32_t t_lo, uint32_t t_hi)
{
    const uint32_t t = term_ids[i];
    return t >= t_lo && t < t_hi && (alive == nullptr || bit_test(alive, entry_doc[i]));
}
__global__ void __launch_bounds__(CC_THREADS)
chunk_count_kernel(const uint32_t* __restrict__ term_ids, const uint32_t* __restrict__ entry_doc,
                   const uint32_t* __restrict__ alive, int64_t nnz, uint32_t t_lo, uint32_t t_hi, uint32_t* __restrict__ block_cnt)
{
    __shared__ uint32_t s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const int64_t base = ((int64_t)blockIdx.x * CC_THREADS + threadIdx.x) * CC_ITEMS;
    uint32_t c = 0;
#pragma unroll
    for (int k = 0; k < CC_ITEMS; ++k)
        if (base + k < nnz && chunk_member(term_ids, entry_doc, alive, base + k, t_lo, t_hi)) ++c;
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) block_cnt[blockIdx.x] = s_cnt;
}
__global__ void __launch_bounds__(CC_THREADS)
chunk_scatter_kernel(const uint32_t* __restrict__ term_ids, const uint16_t* __restrict__ term_tf,
                     const uint32_t* __restrict__ entry_doc, const uint32_t* __restrict__ alive, int64_t nnz, uint32_t t_lo,
                     uint32_t t_hi, const uint32_t* __restrict__ block_off, uint32_t* __restrict__ keys,
                     uint64_t* __restrict__ vals)
{
    typedef cub::BlockScan<uint32_t, CC_THREADS> Scan;
    __shared__ typename Scan::TempStorage tmp;
    const int64_t base = ((int64_t)blockIdx.x * CC_THREADS + threadIdx.x) * CC_ITEMS;
    bool ok[CC_ITEMS];
    uint32_t c = 0;
#pragma unroll
    for (int k = 0; k < CC_ITEMS; ++k) {
        ok[k] = base + k < nnz && chunk_member(term_ids, entry_doc, alive, base + k, t_lo, t_hi);
        c += ok[k] ? 1u : 0u;
    }
    uint32_t excl;
    Scan(tmp).ExclusiveSum(c, excl);
    uint32_t at = block_off[blockIdx.x] + excl;          // entry order = document order: the stable sort keeps it inside a term
#pragma unroll
    for (int k = 0; k < CC_ITEMS; ++k)
        if (ok[k]) {
            keys[at] = term_ids[base + k];
            vals[at] = ((uint64_t)entry_doc[base + k] << 16) | term_tf[base + k];
            ++at;
        }
}

__global__ void score_postings_kernel(const uint32_t* __restrict__ sorted_terms, const uint64_t* __restrict__ sorted_vals,
                                      const uint32_t* __restrict__ doc_len, const float* __restrict__ idf, double avgdl,
                                      int64_t nnz_live, uint32_t* __restrict__ post_doc, float* __restrict__ post_score)
{
    const double k1 = 1.5, b = 0.75;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz_live; i += (int64_t)gridDim.x * blockDim.x) {
        uint64_t v = sorted_vals[i];
        uint32_t d = (uint32_t)(v >> 16);
        double tf = (double)(uint32_t)(v & 0xffffu);
        // tf / (k1 * ((1 - b) + b * dl / avgdl) + tf), left-to-right as Python evaluates it
        double t1 = __dmul_rn(b, (double)doc_len[d]);
        double t2 = __ddiv_rn(t1, avgdl);
        double t3 = __dadd_rn(__dsub_rn(1.0, b), t2);
        double t4 = __dmul_rn(k1, t3);
        double t5 = __dadd_rn(t4, tf);
        double tfc = __ddiv_rn(tf, t5);
        post_doc[i] = d;
        post_score[i] = __double2float_rn(__dmul_rn((double)idf[sorted_terms[i]], tfc));
    }
}

__global__ void df_to_i64_kernel(const uint32_t* __restrict__ df_local, int64_t vocab, int64_t* __restrict__ out)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= vocab; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = i < vocab ? (int64_t)df_local[i] : 0;
}

// ---- tile index (frequent terms only)
__global__ void tile_flag_kernel(const int64_t* __restrict__ off, int64_t vocab, int32_t* __restrict__ flag)
{
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t <= vocab; t += (int64_t)gridDim.x * blockDim.x)
        flag[t] = (t < vocab && off[t + 1] - off[t] > BM25_RARE_MAX) ? 1 : 0;
}
__global__ void tile_slot_kernel(const int32_t* __restrict__ flag, const int32_t* __restrict__ scan, int64_t vocab,
                                 int32_t* __restrict__ slot)
{
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < vocab; t += (int64_t)gridDim.x * blockDim.x)
        slot[t] = flag[t] ? scan[t] : -1;
}
__global__ void tile_index_kernel(const uint32_t* __restrict__ sorted_terms, const uint32_t* __restrict__ post_doc,
                                  const int64_t* __restrict__ off, const int32_t* __restrict__ slot, int64_t p_base,
                                  int64_t p_count, int64_t n_tiles, uint32_t* __restrict__ tile_off)
{
    // sorted_terms: the term ids of postings [p_base, p_base + p_count) (one term range of the build); post_doc: all postings
    for (int64_t pl = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pl < p_count; pl += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = p_base + pl;
        const uint32_t t = sorted_terms[pl];
        const int32_t sl = slot[t];
        if (sl < 0) continue;
        const int64_t b = off[t], e = off[t + 1];
        const int64_t i = p - b;
        const int64_t tile_d = post_doc[p] / BM25_SUB_DOCS;
        const int64_t prev = (i == 0) ? -1 : (int64_t)(post_doc[p - 1] / BM25_SUB_DOCS);
        uint32_t* row = tile_off + (int64_t)sl * (n_tiles + 1);
        for (int64_t tl = prev + 1; tl <= tile_d; ++tl) row[tl] = (uint32_t)i;
        if (p == e - 1) for (int64_t tl = tile_d + 1; tl <= n_tiles; ++tl) row[tl] = (uint32_t)(e - b);
    }
}

// ---- rank table (Postings::rank_score), built per term range right after its scores.  Scores are compared as
// f32_ordered_bits keys and written back from the same bits: the table holds stored posting scores bit for bit.
constexpr int RK_TOP = 1 << (BM25_RANKS - 1);     // 1024: deepest rank of the table
constexpr int RS_WARPS = 8;
// terms with 1 <= df <= RK_TOP: one warp per term, bitonic sort (descending) of the term's keys in shared memory
__global__ void __launch_bounds__(RS_WARPS * 32)
rank_small_kernel(const int64_t* __restrict__ off, const float* __restrict__ score, int64_t t_lo, int64_t t_hi,
                  float* __restrict__ rank)
{
    __shared__ uint32_t s_key[RS_WARPS][RK_TOP];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* key = s_key[warp];
    for (int64_t t = t_lo + (int64_t)blockIdx.x * RS_WARPS + warp; t < t_hi; t += (int64_t)gridDim.x * RS_WARPS) {
        const int64_t b = off[t], df = off[t + 1] - b;
        if (df == 0 || df > RK_TOP) continue;
        const int n = (int)df, n2 = next_pow2(max(n, 2));
        for (int i = lane; i < n2; i += 32) key[i] = i < n ? f32_ordered_bits(score[b + i]) : 0u;   // 0: below every score
        __syncwarp();
        for (int k = 2; k <= n2; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int p = lane; p < (n2 >> 1); p += 32) {
                    const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1)), q = i | j;
                    const uint32_t a = key[i], c = key[q];
                    if ((a < c) == ((i & k) == 0)) { key[i] = c; key[q] = a; }
                }
                __syncwarp();
            }
        }
        if (lane < BM25_RANKS) rank[t * BM25_RANKS + lane] = (1 << lane) <= n ? f32_from_ordered_bits(key[(1 << lane) - 1]) : 0.f;
        __syncwarp();
    }
}
// terms with df > RK_TOP: one CTA per term.  Radix select (digits of 11, 11 and 10 bits from the top) of T = the RK_TOP-th
// best key; then the < RK_TOP keys above T are collected and sorted, and ranks past them are T itself (ties)
constexpr int RL_THREADS = 512;
template <typename F>
__device__ __forceinline__ void rank_for_each_key(const float* __restrict__ s, int64_t n, F f)
{
    const int64_t head = min(n, (int64_t)((16 - ((uintptr_t)s & 15)) & 15) / 4);      // scalars up to 16-byte alignment
    if ((int64_t)threadIdx.x < head) f(f32_ordered_bits(s[threadIdx.x]));
    const float4* s4 = reinterpret_cast<const float4*>(s + head);
    const int64_t n4 = (n - head) / 4;
    int64_t i = threadIdx.x;
    for (; i + 3 * RL_THREADS < n4; i += 4 * RL_THREADS) {          // four independent 16-byte loads per thread in flight
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldg(s4 + i + u * RL_THREADS);
#pragma unroll
        for (int u = 0; u < 4; ++u) { f(f32_ordered_bits(v[u].x)); f(f32_ordered_bits(v[u].y)); f(f32_ordered_bits(v[u].z)); f(f32_ordered_bits(v[u].w)); }
    }
    for (; i < n4; i += RL_THREADS) {
        const float4 v = __ldg(s4 + i);
        f(f32_ordered_bits(v.x)); f(f32_ordered_bits(v.y)); f(f32_ordered_bits(v.z)); f(f32_ordered_bits(v.w));
    }
    for (int64_t k = head + n4 * 4 + threadIdx.x; k < n; k += RL_THREADS) f(f32_ordered_bits(s[k]));
}
__global__ void __launch_bounds__(RL_THREADS)
rank_large_kernel(const int64_t* __restrict__ off, const float* __restrict__ score, const uint32_t* __restrict__ terms,
                  float* __restrict__ rank)
{
    typedef cub::BlockScan<uint32_t, RL_THREADS> Scan;
    __shared__ typename Scan::TempStorage s_scan;
    __shared__ uint32_t s_hist[2048];
    __shared__ uint32_t s_top[RK_TOP];
    __shared__ uint32_t s_prefix, s_need, s_cnt;
    const int tid = threadIdx.x;
    const uint32_t t = terms[blockIdx.x];
    const int64_t b = off[t], df = off[t + 1] - b;
    const float* s = score + b;
    uint32_t prefix = 0, mask = 0, need = RK_TOP;                   // need: rank of T among the keys that match prefix
    for (int pass = 0; pass < 3; ++pass) {
        const int shift = pass == 0 ? 21 : (pass == 1 ? 10 : 0);
        const uint32_t dmask = pass == 2 ? 0x3FFu : 0x7FFu;
        for (int i = tid; i < 2048; i += RL_THREADS) s_hist[i] = 0;
        __syncthreads();
        rank_for_each_key(s, df, [&](uint32_t k) { if ((k & mask) == prefix) atomicAdd(&s_hist[(k >> shift) & dmask], 1u); });
        __syncthreads();
        // bins from the top: thread tid holds bins 2047 - 4 tid ... 2044 - 4 tid; the bin where the running count reaches
        // `need` holds T
        uint32_t c[4], sum = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) { c[e] = s_hist[2047 - 4 * tid - e]; sum += c[e]; }
        uint32_t above;
        Scan(s_scan).ExclusiveSum(sum, above);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (above < need && above + c[e] >= need) { s_prefix = prefix | ((uint32_t)(2047 - 4 * tid - e) << shift); s_need = need - above; }
            above += c[e];
        }
        __syncthreads();
        prefix = s_prefix; need = s_need; mask |= dmask << shift;
    }
    // prefix == T; RK_TOP - need keys are above it
    if (tid == 0) s_cnt = 0;
    for (int i = tid; i < RK_TOP; i += RL_THREADS) s_top[i] = 0;
    __syncthreads();
    rank_for_each_key(s, df, [&](uint32_t k) { if (k > prefix) s_top[atomicAdd(&s_cnt, 1u)] = k; });
    __syncthreads();
    for (int k = 2; k <= RK_TOP; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int p = tid; p < RK_TOP / 2; p += RL_THREADS) {
                const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1)), q = i | j;
                const uint32_t x = s_top[i], y = s_top[q];
                if ((x < y) == ((i & k) == 0)) { s_top[i] = y; s_top[q] = x; }
            }
            __syncthreads();
        }
    }
    const uint32_t n_above = RK_TOP - need;
    if (tid < BM25_RANKS) rank[(int64_t)t * BM25_RANKS + tid] = f32_from_ordered_bits((1u << tid) <= n_above ? s_top[(1 << tid) - 1] : prefix);
}
// device scratch of the index build: everything allocated through it is freed on scope exit (also when a CUDA call
// throws half-way), except what keep() hands over to the Postings
struct DevScratch {
    std::vector<void*> ptrs;
    template <typename T> T* alloc(size_t n)
    {
        void* p = nullptr;
        const size_t bytes = sizeof(T) * (n ? n : 1);
        const cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaErrorMemoryAllocation) {          // say how much was asked for and what was left: the build is the memory peak
            cudaGetLastError();
            size_t free_b = 0, total_b = 0;
            cudaMemGetInfo(&free_b, &total_b);
            char msg[256];
            snprintf(msg, sizeof msg, "bm25 index build: out of device memory (wanted %.2f GB, %.2f of %.2f GB free)", bytes / 1e9, free_b / 1e9,
                     total_b / 1e9);
            throw DevOom{msg};
        }
        KRAG_CUDA(e);
        ptrs.push_back(p);
        return static_cast<T*>(p);
    }
    void free_now(void* p)
    {
        for (auto& q : ptrs) if (q == p && q) { cudaFree(q); q = nullptr; }
    }
    template <typename T> T* keep(T* p)
    {
        for (auto& q : ptrs) if (q == static_cast<void*>(p)) q = nullptr;
        return p;
    }
    ~DevScratch() { for (void* p : ptrs) if (p) cudaFree(p); }
};

// slots of the frequent terms (df > BM25_RARE_MAX) and the (still empty) boundary table; filled range by range below
static void prepare_tile_index(const int64_t* off, int64_t vocab, int64_t n_rows, Postings& out, cudaStream_t st)
{
    DevScratch sc;
    int32_t* flag = sc.alloc<int32_t>((size_t)(vocab + 1));
    int32_t* scan = sc.alloc<int32_t>((size_t)(vocab + 1));
    int32_t* slot = sc.alloc<int32_t>((size_t)vocab);
    tile_flag_kernel<<<256, 256, 0, st>>>(off, vocab, flag);
    count_launch();
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, flag, scan, (int)(vocab + 1), st);
    void* tmp = sc.alloc<unsigned char>(bytes);
    cub::DeviceScan::ExclusiveSum(tmp, bytes, flag, scan, (int)(vocab + 1), st);
    count_launch();
    tile_slot_kernel<<<256, 256, 0, st>>>(flag, scan, vocab, slot);
    count_launch();
    int32_t n_slots = 0;
    KRAG_CUDA(cudaMemcpyAsync(&n_slots, scan + vocab, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    KRAG_CUDA(cudaStreamSynchronize(st));
    sc.free_now(tmp); sc.free_now(flag); sc.free_now(scan);
    int64_t n_tiles = (n_rows + BM25_SUB_DOCS - 1) / BM25_SUB_DOCS;
    if (n_tiles < 1) n_tiles = 1;
    uint32_t* tile_off = sc.alloc<uint32_t>((size_t)((int64_t)(n_slots > 0 ? n_slots : 1) * (n_tiles + 1)));
    if (out.tile_slot) cudaFree(out.tile_slot);
    if (out.tile_off) cudaFree(out.tile_off);
    sc.keep(slot); sc.keep(tile_off);
    out.tile_slot = slot; out.tile_off = tile_off; out.n_slots = n_slots; out.n_tiles = n_tiles;
}

// postings per term range of the build: KRAG_BM25_BUILD_CHUNK, else what fits in 70 % of the free device memory at 24 bytes
// of sort buffers per posting + 12 for the alternate key/value buffers the radix sort keeps in its temporary storage
static int64_t build_chunk_cap(int64_t nnz_live)
{
    int64_t cap = 0;
    if (const char* e = getenv("KRAG_BM25_BUILD_CHUNK")) cap = atoll(e);
    if (cap <= 0) {
        size_t free_b = 0, total_b = 0;
        KRAG_CUDA(cudaMemGetInfo(&free_b, &total_b));
        cap = (int64_t)((double)free_b * 0.7 / 37.0);
        if (cap < ((int64_t)1 << 20)) cap = (int64_t)1 << 20;
    }
    const int64_t hard = ((int64_t)1 << 31) - 4096;              // 32-bit block offsets / cub item counts
    if (cap > hard) cap = hard;
    return cap < nnz_live ? cap : nnz_live;
}

void build_postings(const uint32_t* term_ids, const uint16_t* term_tf, const uint32_t* entry_doc,
                    const uint32_t* doc_len, const uint32_t* alive, int64_t nnz, int64_t vocab, const float* idf,
                    double avgdl, int64_t n_docs_rows, Postings& out, cudaStream_t st)
{
    // local df (live docs only) -> exclusive scan -> offsets
    DevScratch sc;
    uint32_t* df_local = sc.alloc<uint32_t>((size_t)(vocab + 1));
    KRAG_CUDA(cudaMemsetAsync(df_local, 0, sizeof(uint32_t) * (size_t)(vocab + 1), st));
    launch_df_histogram(term_ids, entry_doc, alive, nnz, df_local, st);
    int64_t* off = sc.alloc<int64_t>((size_t)(vocab + 1));
    int64_t* tmp64 = sc.alloc<int64_t>((size_t)(vocab + 1));
    df_to_i64_kernel<<<256, 256, 0, st>>>(df_local, vocab, tmp64);
    count_launch();
    size_t scan_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, tmp64, off, (int)(vocab + 1), st);
    void* scan_tmp = sc.alloc<unsigned char>(scan_bytes);
    cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, tmp64, off, (int)(vocab + 1), st);
    count_launch();
    std::vector<int64_t> h_off((size_t)(vocab + 1));
    KRAG_CUDA(cudaMemcpyAsync(h_off.data(), off, sizeof(int64_t) * (size_t)(vocab + 1), cudaMemcpyDeviceToHost, st));
    KRAG_CUDA(cudaStreamSynchronize(st));
    const int64_t nnz_live = h_off[(size_t)vocab];
    sc.free_now(scan_tmp); sc.free_now(tmp64); sc.free_now(df_local);

    uint32_t* post_doc = sc.alloc<uint32_t>((size_t)(nnz_live > 0 ? nnz_live : 1));
    float* post_score = sc.alloc<float>((size_t)(nnz_live > 0 ? nnz_live : 1));
    float* rank_score = sc.alloc<float>((size_t)vocab * BM25_RANKS);
    KRAG_CUDA(cudaMemsetAsync(rank_score, 0, sizeof(float) * (size_t)vocab * BM25_RANKS, st));

    if (nnz > 0 && nnz_live > 0) {
        prepare_tile_index(off, vocab, n_docs_rows, out, st);
        // terms too long for a warp sort (df > RK_TOP), ascending: the ones of a term range are a contiguous run
        std::vector<uint32_t> h_big;
        for (int64_t t = 0; t < vocab; ++t)
            if (h_off[(size_t)t + 1] - h_off[(size_t)t] > RK_TOP) h_big.push_back((uint32_t)t);
        uint32_t* big = sc.alloc<uint32_t>(h_big.size());
        if (!h_big.empty())
            KRAG_CUDA(cudaMemcpyAsync(big, h_big.data(), sizeof(uint32_t) * h_big.size(), cudaMemcpyHostToDevice, st));
        // term ranges [t_lo, t_hi) of at most `cap` postings each (a single term longer than that is a range of its own).  The
        // sort buffers are sized for the widest range; if they do not fit after all (fragmentation, another context on the
        // device), the ranges are halved until they do
        int64_t cap = build_chunk_cap(nnz_live);
        const int64_t n_blocks = (nnz + (int64_t)CC_THREADS * CC_ITEMS - 1) / ((int64_t)CC_THREADS * CC_ITEMS);
        if (n_blocks >= ((int64_t)1 << 31)) throw std::runtime_error("bm25 build: too many index entries on one shard");
        uint32_t* block_cnt = sc.alloc<uint32_t>((size_t)n_blocks);
        uint32_t* block_off = sc.alloc<uint32_t>((size_t)n_blocks);
        size_t bscan_bytes = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, bscan_bytes, block_cnt, block_off, (int)n_blocks, st);
        void* bscan_tmp = sc.alloc<unsigned char>(bscan_bytes);
        int end_bit = 1;
        while (((int64_t)1 << end_bit) < vocab) ++end_bit;  // keys range over [0, vocab)
        std::vector<int64_t> cuts;
        uint32_t *k_in = nullptr, *k_out = nullptr;
        uint64_t *v_in = nullptr, *v_out = nullptr;
        void* sort_tmp = nullptr;
        size_t sort_bytes = 0;
        for (;;) {
            cuts.assign(1, 0);
            int64_t widest = 0;
            while (cuts.back() < vocab) {
                const int64_t t_lo = cuts.back();
                int64_t t_hi = (int64_t)(std::upper_bound(h_off.begin() + t_lo, h_off.end(), h_off[(size_t)t_lo] + cap) - h_off.begin()) - 1;
                if (t_hi <= t_lo) t_hi = t_lo + 1;
                if (t_hi > vocab) t_hi = vocab;
                cuts.push_back(t_hi);
                widest = std::max(widest, h_off[(size_t)t_hi] - h_off[(size_t)t_lo]);
            }
            if (widest >= ((int64_t)1 << 31)) throw std::runtime_error("bm25 build: a single term has too many postings for one build range");
            try {
                // stable LSD radix sort by term id keeps documents ascending inside every term
                k_in = sc.alloc<uint32_t>((size_t)widest);
                k_out = sc.alloc<uint32_t>((size_t)widest);
                v_in = sc.alloc<uint64_t>((size_t)widest);
                v_out = sc.alloc<uint64_t>((size_t)widest);
                sort_bytes = 0;
                cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, k_in, k_out, v_in, v_out, widest, 0, end_bit, st);
                sort_tmp = sc.alloc<unsigned char>(sort_bytes);
                break;
            } catch (const DevOom&) {
                sc.free_now(k_in); sc.free_now(k_out); sc.free_now(v_in); sc.free_now(v_out);
                k_in = k_out = nullptr; v_in = v_out = nullptr;
                if (cap <= ((int64_t)1 << 22) || widest > cap) throw;      // cannot get smaller: the widest range is one term
                cap /= 2;
            }
        }
        for (size_t c = 0; c + 1 < cuts.size(); ++c) {
            const int64_t t_lo = cuts[c], t_hi = cuts[c + 1];
            const int64_t p_base = h_off[(size_t)t_lo], m = h_off[(size_t)t_hi] - p_base;
            if (m == 0) continue;
            chunk_count_kernel<<<(unsigned)n_blocks, CC_THREADS, 0, st>>>(term_ids, entry_doc, alive, nnz, (uint32_t)t_lo, (uint32_t)t_hi,
                                                                         block_cnt);
            KRAG_CUDA(cudaGetLastError());
            count_launch();
            cub::DeviceScan::ExclusiveSum(bscan_tmp, bscan_bytes, block_cnt, block_off, (int)n_blocks, st);
            count_launch();
            chunk_scatter_kernel<<<(unsigned)n_blocks, CC_THREADS, 0, st>>>(term_ids, term_tf, entry_doc, alive, nnz, (uint32_t)t_lo,
                                                                           (uint32_t)t_hi, block_off, k_in, v_in);
            KRAG_CUDA(cudaGetLastError());
            count_launch();
            size_t sb = sort_bytes;
            cub::DeviceRadixSort::SortPairs(sort_tmp, sb, k_in, k_out, v_in, v_out, m, 0, end_bit, st);
            count_launch();
            score_postings_kernel<<<148 * 8, 256, 0, st>>>(k_out, v_out, doc_len, idf, avgdl, m, post_doc + p_base, post_score + p_base);
            count_launch();
            const int64_t small_grid = std::min<int64_t>((t_hi - t_lo + RS_WARPS - 1) / RS_WARPS, 148 * 16);
            rank_small_kernel<<<(unsigned)small_grid, RS_WARPS * 32, 0, st>>>(off, post_score, t_lo, t_hi, rank_score);
            KRAG_CUDA(cudaGetLastError());
            count_launch();
            const size_t b0 = std::lower_bound(h_big.begin(), h_big.end(), (uint32_t)t_lo) - h_big.begin();
            const size_t b1 = std::lower_bound(h_big.begin(), h_big.end(), (uint32_t)t_hi) - h_big.begin();
            if (b1 > b0) {
                rank_large_kernel<<<(unsigned)(b1 - b0), RL_THREADS, 0, st>>>(off, post_score, big + b0, rank_score);
                KRAG_CUDA(cudaGetLastError());
                count_launch();
            }
            if (out.n_slots > 0) {
                tile_index_kernel<<<148 * 8, 256, 0, st>>>(k_out, post_doc, off, out.tile_slot, p_base, m, out.n_tiles, out.tile_off);
                KRAG_CUDA(cudaGetLastError());
                count_launch();
            }
        }
        KRAG_CUDA(cudaStreamSynchronize(st));
    }
    if (nnz_live == 0 || nnz == 0) {   // no postings: every term is "rare" with an empty list
        int32_t* slot = sc.alloc<int32_t>((size_t)vocab);
        KRAG_CUDA(cudaMemset(slot, 0xFF, sizeof(int32_t) * (size_t)vocab));
        uint32_t* toff = sc.alloc<uint32_t>(4);
        if (out.tile_slot) cudaFree(out.tile_slot);
        if (out.tile_off) cudaFree(out.tile_off);
        out.tile_slot = sc.keep(slot); out.tile_off = sc.keep(toff); out.n_slots = 0;
        out.n_tiles = (n_docs_rows + BM25_SUB_DOCS - 1) / BM25_SUB_DOCS < 1 ? 1 : (n_docs_rows + BM25_SUB_DOCS - 1) / BM25_SUB_DOCS;
    }
    if (out.off) cudaFree(out.off);
    if (out.doc) cudaFree(out.doc);
    if (out.score) cudaFree(out.score);
    if (out.rank_score) cudaFree(out.rank_score);
    sc.keep(off); sc.keep(post_doc); sc.keep(post_score); sc.keep(rank_score);
    out.off = off; out.doc = post_doc; out.score = post_score; out.rank_score = rank_score; out.vocab = vocab; out.nnz = nnz_live;
}

// -------------------------------------------------------------------------- query time
// Two kernels.  bm25_warp_kernel (further down) is the one that runs: warp-autonomous sub-tiles, a sampled per-query
// admission threshold, global candidate lists.  bm25_tile_kernel below is the first-generation CTA-per-tile kernel, kept as
// the exact SAFETY NET for queries whose candidate list overflows (launched after every batch, it skips every query whose
// overflow flag is 0) and selectable as a whole with KRAG_BM25_LEGACY=1.
constexpr int BQ_THREADS = 256;   // a term contributes ~200 postings to a 16384-doc tile: 256-wide slabs keep the lanes busy
constexpr int BQ_MAX_TERMS = 32;    // query terms resolved per pass; longer queries loop
constexpr int BQ_MAX_SLABS = 96;    // 512-posting slabs per pass
constexpr int BQ_PREFETCH = 8;      // slabs held in registers at a time
constexpr int BQ_GROUP_MAX = 32;    // upper bound of the group size (shared-memory table)
// consecutive doc tiles handled by one work item (same query): one resolve, one select, one store.  Runtime value
// (KRAG_BM25_GROUP, default 8): larger groups mean fewer per-item sorts/stores and tighter own thresholds, smaller
// ones more items to balance over the 444 resident CTAs
static int bq_group()
{
    static int v = -1;
    if (v < 0) { const char* e = getenv("KRAG_BM25_GROUP"); int g = e ? atoi(e) : 8; v = g < 1 ? 1 : (g > BQ_GROUP_MAX ? BQ_GROUP_MAX : g); }
    return v;
}

// A "slab" is up to 512 consecutive postings of one query term that fall into this CTA's doc
// range (frequent terms: looked up in the tile index; rare terms: the whole <= 256-entry list,
// filtered by doc).  Slabs are applied in query-term order with a barrier in between, which
// fixes the per-document fp32 summation order to the oracle's.
__global__ void __launch_bounds__(BQ_THREADS)
bm25_tile_kernel(const int64_t* __restrict__ post_off, const uint32_t* __restrict__ post_doc,
                 const float* __restrict__ post_score, const int32_t* __restrict__ tile_slot,
                 const uint32_t* __restrict__ tile_off, int64_t n_tiles_idx, int64_t vocab,
                 const uint32_t* __restrict__ q_terms, const int32_t* __restrict__ q_term_offsets,
                 const int32_t* __restrict__ q_slot, const int64_t* __restrict__ q_base, const int32_t* __restrict__ q_rare_len,
                 int64_t n_rows, const uint32_t* __restrict__ alive, int P, int cap, OrdMap ord_base, int batch, int n_tiles, int group,
                 uint64_t* __restrict__ part /*[batch][n_groups][P]*/, unsigned long long* __restrict__ g_thr /*[batch]*/,
                 const uint32_t* __restrict__ only_flag /* != null: only queries whose flag is set */)
{
    // the tile index has one column per BM25_SUB_DOCS docs; this kernel's tiles are BM25_SUBS_PER_TILE of them
    auto idx_col = [&](int tile) -> int64_t {
        const int64_t c = (int64_t)tile * BM25_SUBS_PER_TILE;
        return c < n_tiles_idx ? c : n_tiles_idx;
    };
    extern __shared__ __align__(16) unsigned char bsm[];
    float* acc = reinterpret_cast<float*>(bsm);                                          // [BM25_TILE_DOCS]
    uint64_t* sbuf = reinterpret_cast<uint64_t*>(bsm + (size_t)BM25_TILE_DOCS * 4);      // [cap]
    __shared__ int s_count;
    __shared__ uint64_t s_thr;
    __shared__ int64_t s_lo[BQ_MAX_TERMS];
    __shared__ int s_len[BQ_MAX_TERMS];
    __shared__ int64_t s_slab_lo[BQ_MAX_SLABS];
    __shared__ int s_slab_n[BQ_MAX_SLABS];
    __shared__ int s_nslab, s_next_term, s_next_off;
    __shared__ int32_t s_slot[BQ_MAX_TERMS], s_rare[BQ_MAX_TERMS];
    __shared__ int64_t s_base[BQ_MAX_TERMS];
    __shared__ uint32_t s_toff[BQ_MAX_TERMS][BQ_GROUP_MAX + 1];

    const int tid = threadIdx.x;
    // the accumulators are zeroed once: every touched entry is reset by the claim step
    for (int i = tid; i < BM25_TILE_DOCS / 4; i += BQ_THREADS) reinterpret_cast<float4*>(acc)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    SelectBuf sel{sbuf, &s_count, &s_thr, cap};

    // persistent loop over (tile group, query) work items, query fastest.  A work item covers BQ_GROUP consecutive
    // doc tiles of one query: the term -> posting-range lookups are fetched once for the whole group, the select
    // buffer (and its threshold) carries over from tile to tile, and one top-P list is stored per item.
    // g_thr[q] (min over finished items of their P-th best key -- an upper bound of the global P-th best) prunes
    // almost every candidate of later items before it reaches the select buffer.
    const int n_groups = (n_tiles + group - 1) / group;
    const int64_t n_items = (int64_t)n_groups * batch;
    for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int tg = (int)(item / batch), qi = (int)(item - (int64_t)tg * batch);
    if (only_flag != nullptr && only_flag[qi] == 0) continue;      // uniform over the CTA, before any barrier of the item
    const int tile0 = tg * group, gcount = min(group, n_tiles - tile0);
    const int tb = q_term_offsets[qi], te = q_term_offsets[qi + 1];
    const bool single_chunk = (te - tb <= BQ_MAX_TERMS);
    __syncthreads();   // previous item fully stored
    if (tid == 0) {
        const unsigned long long h = __ldcg(&g_thr[qi]);
        s_count = 0;
        s_thr = (h == KEY_PAD) ? KEY_PAD : h + 1;   // admit keys <= hint
    }
    if (single_chunk && tid < te - tb) {
        // one fetch per item: slot/base of the term and its posting offsets at the group's tile boundaries
        const int32_t sl = q_slot[tb + tid];
        s_slot[tid] = sl; s_base[tid] = q_base[tb + tid]; s_rare[tid] = q_rare_len[tb + tid];
        if (sl >= 0) {
            const uint32_t* row = tile_off + (int64_t)sl * (n_tiles_idx + 1);
            for (int g = 0; g <= gcount; ++g) s_toff[tid][g] = row[idx_col(tile0 + g)];
        }
    }
    __syncthreads();
    uint64_t thr = s_thr;

    for (int gi = 0; gi < gcount; ++gi) {
    const int tile = tile0 + gi;
    const int64_t t0 = (int64_t)tile * BM25_TILE_DOCS;
    const int tile_n = (int)min((int64_t)BM25_TILE_DOCS, n_rows - t0);

    // posting range of each term of the chunk [c0, c0+nt) inside this tile
    auto resolve = [&](int c0, int nt) {
        __syncthreads();
        if (tid < nt) {
            // (slot, base, rare length) of every query term were resolved once per batch by bm25_resolve_kernel
            const int32_t sl = q_slot[c0 + tid];
            int64_t lo = 0; int len = 0;
            if (sl >= 0) {
                const uint32_t* row = tile_off + (int64_t)sl * (n_tiles_idx + 1);
                const uint32_t o0 = row[idx_col(tile)], o1 = row[idx_col(tile + 1)];
                lo = q_base[c0 + tid] + o0; len = (int)(o1 - o0);
            } else if (sl == -1) {
                lo = q_base[c0 + tid]; len = q_rare_len[c0 + tid];   // rare: whole list, filtered by doc range below
            }
            s_lo[tid] = lo; s_len[tid] = len;
        }
        if (tid == 0) { s_next_term = 0; s_next_off = 0; }
        __syncthreads();
    };
    // next pass of at most BQ_MAX_SLABS slabs of the resolved chunk; returns the slab count
    auto next_pass = [&](int nt) -> int {
        if (tid == 0) {
            int ns = 0, j = s_next_term, o = s_next_off;
            while (j < nt && ns < BQ_MAX_SLABS) {
                const int rem = s_len[j] - o;
                if (rem <= 0) { ++j; o = 0; continue; }
                s_slab_lo[ns] = s_lo[j] + o; s_slab_n[ns] = rem < BQ_THREADS ? rem : BQ_THREADS; ++ns;
                o += BQ_THREADS;
            }
            s_nslab = ns; s_next_term = j; s_next_off = o;
        }
        __syncthreads();
        return s_nslab;
    };
    // acc[doc] += score, slab after slab (query-term order), BQ_PREFETCH slabs in registers at a time
    auto accumulate = [&](int ns) {
        for (int s0 = 0; s0 < ns; s0 += BQ_PREFETCH) {
            uint32_t d[BQ_PREFETCH]; float sc[BQ_PREFETCH];
#pragma unroll
            for (int u = 0; u < BQ_PREFETCH; ++u) {
                d[u] = 0xFFFFFFFFu; sc[u] = 0.f;
                if (s0 + u < ns && tid < s_slab_n[s0 + u]) {
                    const int64_t p = s_slab_lo[s0 + u] + tid;
                    d[u] = post_doc[p]; sc[u] = post_score[p];
                }
            }
#pragma unroll
            for (int u = 0; u < BQ_PREFETCH; ++u) {
                if (s0 + u < ns) {
                    const uint32_t rel = d[u] - (uint32_t)t0;     // wraps to a huge value for docs below t0
                    if (d[u] != 0xFFFFFFFFu && rel < (uint32_t)tile_n) acc[rel] += sc[u];
                    __syncthreads();
                }
            }
        }
    };
    // every touched document is pushed exactly once with its final score (first claimer takes it)
    auto claim = [&](int ns) {
        for (int s0 = 0; s0 < ns; s0 += BQ_PREFETCH) {
            uint32_t d[BQ_PREFETCH];
#pragma unroll
            for (int u = 0; u < BQ_PREFETCH; ++u) {
                d[u] = 0xFFFFFFFFu;
                if (s0 + u < ns && tid < s_slab_n[s0 + u]) d[u] = post_doc[s_slab_lo[s0 + u] + tid];
            }
#pragma unroll
            for (int u = 0; u < BQ_PREFETCH; ++u) {
                if (s0 + u < ns) {
                    const uint32_t rel = d[u] - (uint32_t)t0;
                    if (d[u] != 0xFFFFFFFFu && rel < (uint32_t)tile_n) {
                        const float sum = atomicExch(&acc[rel], 0.f);
                        if (sum > 0.f && (alive == nullptr || bit_test(alive, d[u])))
                            select_push(sel, make_key_desc(sum, ord_base + d[u]), thr);
                    }
                    __syncthreads();
                    if (s_count + BQ_THREADS > cap) select_prune<BQ_THREADS>(sel, P, tid, 0);
                    thr = s_thr;
                }
            }
        }
    };

    bool done = false;
    if (single_chunk) {
        // common case: the whole query resolves in one chunk (ranges come from the per-item shared-memory copy);
        // if it also fits one pass, accumulate and claim without resolving twice
        __syncthreads();
        if (tid < te - tb) {
            const int32_t sl = s_slot[tid];
            int64_t lo = 0; int len = 0;
            if (sl >= 0) { lo = s_base[tid] + s_toff[tid][gi]; len = (int)(s_toff[tid][gi + 1] - s_toff[tid][gi]); }
            else if (sl == -1) { lo = s_base[tid]; len = s_rare[tid]; }
            s_lo[tid] = lo; s_len[tid] = len;
        }
        if (tid == 0) { s_next_term = 0; s_next_off = 0; }
        __syncthreads();
        const int ns = next_pass(te - tb);
        const bool more = (s_next_term < te - tb);   // uniform: written before the barrier inside next_pass
        if (!more && ns <= BQ_PREFETCH) {
            // all slabs of the item fit the register window: accumulate and claim from the same registers
            uint32_t d[BQ_PREFETCH]; float sc[BQ_PREFETCH];
#pragma unroll
            for (int u = 0; u < BQ_PREFETCH; ++u) {
                d[u] = 0xFFFFFFFFu; sc[u] = 0.f;
                if (u < ns && tid < s_slab_n[u]) {
                    const int64_t p = s_slab_lo[u] + tid;
                    d[u] = post_doc[p]; sc[u] = post_score[p];
                }
            }
#pragma unroll
            for (int u = 0; u < BQ_PREFETCH; ++u) {
                if (u < ns) {
                    const uint32_t rel = d[u] - (uint32_t)t0;
                    if (d[u] != 0xFFFFFFFFu && rel < (uint32_t)tile_n) acc[rel] += sc[u];
                    __syncthreads();
                }
            }
#pragma unroll
            for (int u = 0; u < BQ_PREFETCH; ++u) {
                if (u < ns) {
                    const uint32_t rel = d[u] - (uint32_t)t0;
                    if (d[u] != 0xFFFFFFFFu && rel < (uint32_t)tile_n) {
                        const float sum = atomicExch(&acc[rel], 0.f);
                        if (sum > 0.f && (alive == nullptr || bit_test(alive, d[u])))
                            select_push(sel, make_key_desc(sum, ord_base + d[u]), thr);
                    }
                    __syncthreads();
                    if (s_count + BQ_THREADS > cap) select_prune<BQ_THREADS>(sel, P, tid, 0);
                    thr = s_thr;
                }
            }
            done = true;
        } else if (!more) {
            accumulate(ns);
            claim(ns);
            done = true;
        }
    }
    if (!done) {
        // general case: ALL terms are accumulated before any document is claimed
        for (int sweep = 0; sweep < 2; ++sweep) {
            for (int c0 = tb; c0 < te; c0 += BQ_MAX_TERMS) {
                const int nt = min(BQ_MAX_TERMS, te - c0);
                resolve(c0, nt);
                for (int ns = next_pass(nt); ns > 0; ns = next_pass(nt)) {
                    if (sweep == 0) accumulate(ns); else claim(ns);
                    __syncthreads();
                }
            }
        }
    }
    }   // tiles of the group
    select_prune<BQ_THREADS>(sel, P, tid, 0);
    select_store<BQ_THREADS>(sel, P, part + ((size_t)qi * n_groups + tg) * P, tid);
    if (tid == 0 && s_count == P) atomicMin(&g_thr[qi], (unsigned long long)sbuf[P - 1]);
    }   // work items
}

// ---------------------------------------------------------------------------------------------------------------------
// K3, second generation: bm25_warp_kernel.
//
// The legacy kernel spends its time on per-(tile, query) bookkeeping -- ~17 CTA barriers, slab tables and a bitonic sort
// per work item -- not on postings (ncu: DRAM 4.6 % busy, ~195 thread instructions per posting).  Here a WARP owns a
// BM25_SUB_DOCS-document range ("sub-tile") with its fp32 accumulators in shared memory and walks the query's terms on its
// own: no CTA barrier anywhere.  Documents are unique inside a term, so the lanes of a 32-posting round never collide;
// rounds are issued in query-term order with a __syncwarp() in between, which fixes every document's fp32 summation
// order to the oracle's (bit-exact).  All postings of a sub-tile (up to BW_ROUNDS rounds) are loaded into registers up
// front -- the loads of all terms are in flight together -- then accumulated, then every touched document is claimed
// once (atomicExch resets the accumulator) and, if it passes the query's admission threshold, appended to the query's
// candidate list in global memory (one warp-aggregated atomic per round).  No per-item sort, no per-item list.
//
// Threshold: scores are positive and fp32 round-to-nearest addition is monotone, so a document's sum is >= the score of
// any one query term it contains.  Term t has at least 2^i postings scoring >= rank_score[t][i] (the rank table, built at
// commit), hence for 2^i >= P the largest such entry over the query's terms bounds the query's P-th best score from below
// (bm25_rank_threshold_kernel).  The pass over all sub-tiles admits only documents at or above it, and bm25_select_kernel
// takes the exact top-P of them.  The table counts the documents that were alive at commit: when the bitmap of the call
// admits fewer (a delete since, a pushdown filter), a first pass over every `stride`-th sub-tile (no threshold) fills the
// lists with a sample instead, and its P-th best key is the bound (P real documents are at least that good).
// A list that overflows (adversarial score layouts) raises the query's flag and the legacy kernel recomputes that query.
//
// Term -> posting range lookups: one u32 row of sub-tile boundaries per query term.  Frequent terms (> BM25_RARE_MAX
// postings) have theirs in the persistent tile index; for the others bm25_resolve_kernel builds the row per batch from
// the term's <= 2048 document ids (binary searches out of shared memory).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int BW_WARPS = 8;                 // warps per CTA: 8 x (8 KB accumulators + 6 KB staging), 2 CTAs per SM = 16 warps
constexpr int BW_THREADS = BW_WARPS * 32;
constexpr int BW_CHUNK = 8;                 // consecutive (sampled) sub-tiles of one query per work unit
constexpr int BW_STAGE_ROUNDS = 12;         // 32-posting rounds per staging buffer: a whole sub-tile in the common case
constexpr int BW_STAGE_WORDS = BW_STAGE_ROUNDS * 32 * 2;           // docs[12][32] | scores[12][32]
constexpr int BW_WARP_WORDS = BM25_SUB_DOCS + 2 * BW_STAGE_WORDS;  // per-warp shared memory, 4-byte words (14 KB)

// once per batch and query-term position: posting base, boundary row, and the legacy kernel's (slot, rare length)
__global__ void __launch_bounds__(256)
bm25_resolve_kernel(const uint32_t* __restrict__ q_terms, int n_terms, const int64_t* __restrict__ post_off,
                    const uint32_t* __restrict__ post_doc, const int32_t* __restrict__ tile_slot,
                    const uint32_t* __restrict__ tile_off, int64_t vocab, int64_t n_sub, uint32_t* __restrict__ scratch_rows,
                    const uint32_t** __restrict__ q_row, int64_t* __restrict__ q_base, int32_t* __restrict__ q_slot,
                    int32_t* __restrict__ q_rare_len)
{
    __shared__ uint32_t s_doc[BM25_RARE_MAX];
    const int i = blockIdx.x, tid = threadIdx.x;
    if (i >= n_terms) return;
    const uint32_t t = q_terms[i];
    if ((int64_t)t >= vocab) {                                   // out-of-vocabulary id: contributes nothing
        if (tid == 0) { q_row[i] = nullptr; q_base[i] = 0; q_slot[i] = -2; q_rare_len[i] = 0; }
        return;
    }
    const int64_t b = post_off[t];
    const int df = (int)min((int64_t)0x7fffffff, post_off[t + 1] - b);
    const int32_t sl = tile_slot[t];
    if (sl >= 0) {
        if (tid == 0) { q_row[i] = tile_off + (int64_t)sl * (n_sub + 1); q_base[i] = b; q_slot[i] = sl; q_rare_len[i] = 0; }
        return;
    }
    // short list (df <= BM25_RARE_MAX): boundary row built here
    for (int k = tid; k < df; k += 256) s_doc[k] = post_doc[b + k];
    __syncthreads();
    uint32_t* row = scratch_rows + (int64_t)i * (n_sub + 1);
    for (int64_t sidx = tid; sidx <= n_sub; sidx += 256) {
        const uint64_t target = (uint64_t)sidx * BM25_SUB_DOCS;  // first posting with doc >= target
        int lo = 0, hi = df;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if ((uint64_t)s_doc[mid] < target) lo = mid + 1; else hi = mid; }
        row[sidx] = (uint32_t)lo;
    }
    if (tid == 0) { q_row[i] = row; q_base[i] = b; q_slot[i] = -1; q_rare_len[i] = df; }
}

// per query: thr_q = the weakest key whose score is the largest rank-table entry of rank 2^lg >= P over its terms (every
// tie at that score is admitted), or KEY_PAD (admit everything) when that is 0: out-of-vocabulary terms and terms with
// fewer than 2^lg postings contribute nothing
__global__ void bm25_rank_threshold_kernel(const uint32_t* __restrict__ q_terms, const int32_t* __restrict__ q_term_offsets,
                                           int batch, const float* __restrict__ rank_score, int64_t vocab, int lg,
                                           unsigned long long* __restrict__ thr_q)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= batch) return;
    float s = 0.f;
    for (int i = q_term_offsets[q]; i < q_term_offsets[q + 1]; ++i) {
        const uint32_t t = q_terms[i];
        if ((int64_t)t < vocab) s = fmaxf(s, rank_score[(int64_t)t * BM25_RANKS + lg]);
    }
    thr_q[q] = s > 0.f ? (make_key_desc(s, 0u) | 0xFFFFFFFFull) : KEY_PAD;
}

struct BwCtx {
    const uint32_t* post_doc; const float* post_score; float* acc; const uint32_t* alive;
    unsigned long long* cand_q; uint32_t* cnt_q; unsigned long long thr; float thr_score;
    uint32_t t0; OrdMap ord_base; int64_t n_rows; int capq, lane;
};
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// cursor over the (term, 32-posting round) sequence of one sub-tile; lane j < nt holds term j's posting range
struct BwCursor {
    int64_t my_start; int my_len; int nt;
    int j, r;                 // next round to issue: term j, round r of that term
    int R, issued;            // rounds of the sub-tile / rounds staged so far
    uint32_t t0;
};
__device__ __forceinline__ void bw_cursor_reset(BwCursor& cur, int64_t my_start, int my_len, int nt, uint32_t t0)
{
    cur.my_start = my_start; cur.my_len = my_len; cur.nt = nt; cur.j = 0; cur.r = 0; cur.issued = 0; cur.t0 = t0;
    cur.R = (int)__reduce_add_sync(0xffffffffu, (unsigned)((my_len + 31) >> 5));     // one REDUX
}
// Stage (cp.async: the loads of all rounds are in flight together and nobody waits for them here) up to BW_STAGE_ROUNDS
// rounds at the cursor: docs[round][lane] | scores[round][lane]; lanes past the end of a term's list get doc = ~0.
// Outer loop over the terms (one pair of shuffles per term), inner loop over the 32-posting rounds of the term.
__device__ __forceinline__ int bw_issue(const BwCtx& c, BwCursor& cur, uint32_t* buf)
{
    int n = 0;
    uint32_t* dd = buf + c.lane;
    bool full = false;
#pragma unroll 1
    while (cur.j < cur.nt && !full) {
        const int len = __shfl_sync(0xffffffffu, cur.my_len, cur.j);
        int base = cur.r * 32;
        if (base < len) {
            const int64_t st = __shfl_sync(0xffffffffu, cur.my_start, cur.j);
            const uint32_t* pd = c.post_doc + st + c.lane;
            const float* ps = c.post_score + st + c.lane;
#pragma unroll 1
            for (; base < len; base += 32) {
                if (n == BW_STAGE_ROUNDS) { full = true; break; }
                if (base + c.lane < len) {
                    cp_async4(dd, pd + base);
                    cp_async4(dd + BW_STAGE_ROUNDS * 32, ps + base);
                } else {
                    *dd = 0xFFFFFFFFu;
                }
                dd += 32; ++n; ++cur.r;
            }
            if (full) break;
        }
        ++cur.j; cur.r = 0;
    }
    cur.issued += n;
    cp_async_commit();
    return n;
}
// acc[doc] += score for the staged rounds, one round after the other: rounds follow the query-term order, documents are
// unique inside a term (no two lanes of a round collide) and a __syncwarp() separates the rounds, so every document's
// fp32 sum is built in the oracle's order
__device__ __forceinline__ void bw_accumulate(const BwCtx& c, const uint32_t* buf, int n)
{
    const uint32_t* pd = buf + c.lane;
    const uint32_t* ps = buf + BW_STAGE_ROUNDS * 32 + c.lane;
    int u = 0;
#pragma unroll 1
    for (; u + 1 < n; u += 2) {            // two rounds per iteration: the staged loads of the second overlap the first's RMW
        const uint32_t d0 = pd[u * 32], d1 = pd[u * 32 + 32];
        const float s0 = __uint_as_float(ps[u * 32]), s1 = __uint_as_float(ps[u * 32 + 32]);
        const uint32_t r0 = d0 - c.t0, r1 = d1 - c.t0;
        if (d0 != 0xFFFFFFFFu && r0 < (uint32_t)BM25_SUB_DOCS) c.acc[r0] += s0;
        __syncwarp();
        if (d1 != 0xFFFFFFFFu && r1 < (uint32_t)BM25_SUB_DOCS) c.acc[r1] += s1;
        __syncwarp();
    }
    if (u < n) {
        const uint32_t d0 = pd[u * 32];
        const uint32_t r0 = d0 - c.t0;
        if (d0 != 0xFFFFFFFFu && r0 < (uint32_t)BM25_SUB_DOCS) c.acc[r0] += __uint_as_float(ps[u * 32]);
        __syncwarp();
    }
}
__device__ __forceinline__ void bw_push(const BwCtx& c, bool hit, unsigned long long key)
{
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (m) {                                                               // one atomic per hit group and warp
        const int leader = __ffs(m) - 1;
        uint32_t base_slot = 0;
        if (c.lane == leader) base_slot = atomicAdd(c.cnt_q, (uint32_t)__popc(m));
        base_slot = __shfl_sync(0xffffffffu, base_slot, leader);
        if (hit) {
            const uint32_t at = base_slot + (uint32_t)__popc(m & ((1u << c.lane) - 1u));
            if (at < (uint32_t)c.capq) c.cand_q[at] = key;                 // past capq: counted, dropped -> overflow flag
        }
    }
}
// All terms of the sub-tile are accumulated and its postings are still staged: every touched document is claimed once
// (atomicExch resets the accumulator; later occurrences of the same document read 0) and appended to the query's
// candidate list if it passes the admission threshold.
__device__ __forceinline__ void bw_claim_one(const BwCtx& c, uint32_t d, float sum)
{
    bool hit = false;
    unsigned long long key = 0;
    if (sum > 0.f && sum >= c.thr_score && (c.alive == nullptr || bit_test(c.alive, d))) {
        key = make_key_desc(sum, c.ord_base + d);
        hit = key <= c.thr;
    }
    bw_push(c, hit, key);
}
__device__ __forceinline__ void bw_claim_staged(const BwCtx& c, const uint32_t* buf, int n)
{
    const uint32_t* pd = buf + c.lane;
#pragma unroll 1
    for (int u = 0; u < n; u += 2) {       // two rounds per iteration: both exchanges are in flight together
        const uint32_t d0 = pd[u * 32], d1 = (u + 1 < n) ? pd[u * 32 + 32] : 0xFFFFFFFFu;
        const uint32_t r0 = d0 - c.t0, r1 = d1 - c.t0;
        float sum0 = 0.f, sum1 = 0.f;
        if (d0 != 0xFFFFFFFFu && r0 < (uint32_t)BM25_SUB_DOCS) sum0 = atomicExch(&c.acc[r0], 0.f);
        if (d1 != 0xFFFFFFFFu && r1 < (uint32_t)BM25_SUB_DOCS) sum1 = atomicExch(&c.acc[r1], 0.f);   // same document again: reads 0
        const bool maybe = (sum0 > 0.f && sum0 >= c.thr_score) || (sum1 > 0.f && sum1 >= c.thr_score);
        if (!__any_sync(0xffffffffu, maybe)) continue;
        bw_claim_one(c, d0, sum0);
        bw_claim_one(c, d1, sum1);
    }
    __syncwarp();
}
// sub-tiles with more rounds than a staging buffer holds: accumulated block by block, then claimed by a sweep over the
// accumulators (vectorised, conflict-free)
__device__ __forceinline__ void bw_claim_sweep(const BwCtx& c)
{
    float4* acc4 = reinterpret_cast<float4*>(c.acc);
#pragma unroll 1
    for (int k = 0; k < BM25_SUB_DOCS / 128; ++k) {
        const int slot = k * 32 + c.lane;
        const float4 v = acc4[slot];
        const bool nz = (v.x != 0.f) | (v.y != 0.f) | (v.z != 0.f) | (v.w != 0.f);     // scores are positive: touched <=> nonzero
        if (nz) acc4[slot] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!__any_sync(0xffffffffu, nz)) continue;
        const float comp[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            bool hit = false;
            unsigned long long key = 0;
            if (comp[e] > 0.f && comp[e] >= c.thr_score) {
                const uint32_t row = c.t0 + (uint32_t)(slot * 4 + e);
                if ((int64_t)row < c.n_rows && (c.alive == nullptr || bit_test(c.alive, row))) {
                    key = make_key_desc(comp[e], c.ord_base + row);
                    hit = key <= c.thr;
                }
            }
            bw_push(c, hit, key);
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(BW_THREADS, 2)
bm25_warp_kernel(const uint32_t* __restrict__ post_doc, const float* __restrict__ post_score,
                 const int32_t* __restrict__ q_term_offsets, const uint32_t* const* __restrict__ q_row,
                 const int64_t* __restrict__ q_base, int64_t n_rows, const uint32_t* __restrict__ alive, OrdMap ord_base,
                 int batch, int n_s /* sub-tiles visited */, int stride /* every stride-th sub-tile */,
                 const unsigned long long* __restrict__ thr_q /* null: admit everything */, unsigned long long* __restrict__ cand,
                 uint32_t* __restrict__ cand_cnt, int capq, unsigned long long* __restrict__ unit_counter)
{
    extern __shared__ __align__(16) uint32_t bw_smem[];                    // [BW_WARPS][accumulators | staging x 2]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* wbase = bw_smem + (size_t)warp * BW_WARP_WORDS;
    float* acc = reinterpret_cast<float*>(wbase);
    uint32_t* stage = wbase + BM25_SUB_DOCS;
    for (int i = lane; i < BM25_SUB_DOCS / 4; i += 32) reinterpret_cast<float4*>(acc)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();                                                          // zeroed once: the claim step resets what was touched

    const int n_chunks = (n_s + BW_CHUNK - 1) / BW_CHUNK;
    const long long n_units = (long long)n_chunks * batch;
    BwCtx c;
    c.post_doc = post_doc; c.post_score = post_score; c.acc = acc; c.alive = alive; c.ord_base = ord_base; c.capq = capq; c.lane = lane;
    c.n_rows = n_rows;
    for (;;) {
        unsigned long long unit = 0;
        if (lane == 0) unit = atomicAdd(unit_counter, 1ull);               // dynamic: units differ a lot in postings
        unit = __shfl_sync(0xffffffffu, unit, 0);
        if ((long long)unit >= n_units) break;
        const int q = (int)(unit % (unsigned long long)batch), ch = (int)(unit / (unsigned long long)batch);
        const int tb = q_term_offsets[q], te = q_term_offsets[q + 1];
        if (te <= tb) continue;
        c.thr = thr_q ? thr_q[q] : KEY_PAD;
        c.thr_score = (c.thr == KEY_PAD) ? -CUDART_INF_F : key_value_desc(c.thr);
        c.cand_q = cand + (size_t)q * capq; c.cnt_q = cand_cnt + q;
        const int s0 = ch * BW_CHUNK, ns = min(BW_CHUNK, n_s - s0);
        if (te - tb <= 32) {
            // common case: every term of the query lives in one lane; the boundary offsets of the whole chunk are fetched
            // at once (independent loads).  Then a two-deep pipeline runs across the chunk's sub-tiles: while sub-tile i is
            // accumulated and claimed out of one staging buffer, the postings of sub-tile i + 1 are in flight to the other.
            const int nt = te - tb;
            const uint32_t* row = nullptr; int64_t base = 0;
            if (lane < nt) { row = q_row[tb + lane]; base = q_base[tb + lane]; }
            // boundary offsets of the sub-tile AFTER the one being staged are fetched one step ahead (two independent loads
            // whose latency hides under a whole sub-tile of work)
            uint32_t nlo = 0, nhi = 0;
            if (row != nullptr) { const int64_t sub = (int64_t)s0 * stride; nlo = row[sub]; nhi = row[sub + 1]; }
            BwCursor cur;
            int ii = -1, buf = 0;
            int nb_n = 0, nb_R = 0; uint32_t nb_t0 = 0;                    // sub-tile in flight: rounds staged, rounds total
            // stage the first (up to BW_STAGE_ROUNDS) rounds of the next non-empty sub-tile; false at the end of the unit
            auto next_subtile = [&](uint32_t* dst) -> bool {
                for (;;) {
                    if (++ii >= ns) return false;
                    const uint32_t lo = nlo, hi = nhi;
                    if (row != nullptr && ii + 1 < ns) { const int64_t sub = (int64_t)(s0 + ii + 1) * stride; nlo = row[sub]; nhi = row[sub + 1]; }
                    bw_cursor_reset(cur, base + lo, (int)(hi - lo), nt, (uint32_t)((int64_t)(s0 + ii) * stride * BM25_SUB_DOCS));
                    if (cur.R == 0) continue;
                    nb_n = bw_issue(c, cur, dst);
                    nb_R = cur.R; nb_t0 = cur.t0;
                    return true;
                }
            };
            bool have = next_subtile(stage);
            while (have) {
                const int cb_n = nb_n, cb_R = nb_R;
                uint32_t* cbuf = stage + buf * BW_STAGE_WORDS;
                c.t0 = nb_t0;
                if (cb_R <= BW_STAGE_ROUNDS) {
                    buf ^= 1;
                    have = next_subtile(stage + buf * BW_STAGE_WORDS);     // next sub-tile's loads fly while this one is processed
                    if (have) cp_async_wait<1>(); else cp_async_wait<0>();
                    __syncwarp();
                    bw_accumulate(c, cbuf, cb_n);
                    bw_claim_staged(c, cbuf, cb_n);
                } else {
                    // rare: more rounds than a buffer holds -> block by block out of this buffer, then the sweep
                    int n = cb_n;
                    for (;;) {
                        cp_async_wait<0>();
                        __syncwarp();
                        bw_accumulate(c, cbuf, n);
                        if (cur.issued >= cur.R) break;
                        n = bw_issue(c, cur, cbuf);
                    }
                    bw_claim_sweep(c);
                    buf ^= 1;
                    have = next_subtile(stage + buf * BW_STAGE_WORDS);
                }
            }
        } else {
            // long queries: term chunks of 32; ALL chunks are accumulated (in query order) before the claim sweep
            for (int i = 0; i < ns; ++i) {
                const int64_t sub = (int64_t)(s0 + i) * stride;
                c.t0 = (uint32_t)(sub * BM25_SUB_DOCS);
                bool touched = false;
                for (int c0 = tb; c0 < te; c0 += 32) {
                    int64_t my_start = 0; int my_len = 0;
                    if (lane < te - c0) {
                        const uint32_t* row = q_row[c0 + lane];
                        if (row != nullptr) { const uint32_t lo = row[sub], hi = row[sub + 1]; my_start = q_base[c0 + lane] + lo; my_len = (int)(hi - lo); }
                    }
                    BwCursor cur;
                    bw_cursor_reset(cur, my_start, my_len, min(32, te - c0), c.t0);
                    while (cur.issued < cur.R) {
                        const int n = bw_issue(c, cur, stage);
                        cp_async_wait<0>();
                        __syncwarp();
                        bw_accumulate(c, stage, n);
                        touched = true;
                    }
                }
                if (touched) bw_claim_sweep(c);
            }
        }
    }
}

// per query: top-P of the candidate list.  mode 0 (after the sample pass): thr[q] = P-th best key (KEY_PAD when the sample
// holds fewer than P documents), list emptied.  mode 1 (after the main pass): the sorted top-P to keys_out, or flag[q] = 1
// when the list overflowed (the legacy kernel then recomputes the query; keys_out is left alone).
constexpr int BS_THREADS = 512;
constexpr int BS_CAP = 2048;   // >= KRAG_MAX_POOL + 2 * BS_THREADS
__global__ void __launch_bounds__(BS_THREADS)
bm25_select_kernel(const unsigned long long* __restrict__ cand, uint32_t* __restrict__ cand_cnt, int capq, int P, int mode,
                   unsigned long long* __restrict__ thr_q, uint64_t* __restrict__ keys_out, uint32_t* __restrict__ flags)
{
    __shared__ uint64_t s_buf[BS_CAP];
    __shared__ int s_count;
    __shared__ uint64_t s_thr;
    const int tid = threadIdx.x, q = blockIdx.x;
    const uint32_t n_raw = cand_cnt[q];
    if (mode == 1) {
        if (tid == 0) flags[q] = n_raw > (uint32_t)capq ? 1u : 0u;
        if (n_raw > (uint32_t)capq) return;                                // uniform
    }
    const int n = (int)min(n_raw, (uint32_t)capq);
    SelectBuf sel{s_buf, &s_count, &s_thr, BS_CAP};
    select_init(sel, tid);
    __syncthreads();
    const unsigned long long* src = cand + (size_t)q * capq;
    const int epoch = (BS_CAP - P) / BS_THREADS;                           // >= 2 for P <= 1024
    uint64_t thr = KEY_PAD;
    int it = 0;
    for (int i0 = 0; i0 < n; i0 += BS_THREADS, ++it) {
        const int i = i0 + tid;
        if (i < n) select_push(sel, src[i], thr);
        if ((it + 1) % epoch == 0) {
            __syncthreads();
            if (s_count + epoch * BS_THREADS > BS_CAP) select_prune<BS_THREADS>(sel, P, tid, 0);
            thr = s_thr;
        }
    }
    select_prune<BS_THREADS>(sel, P, tid, 0);
    if (mode == 0) {
        if (tid == 0) { thr_q[q] = (s_count == P) ? s_buf[P - 1] : KEY_PAD; cand_cnt[q] = 0; }
    } else {
        select_store<BS_THREADS>(sel, P, keys_out + (size_t)q * P, tid);
    }
}

static int bq_cap(int P) { return P <= 256 ? 512 : (P <= 512 ? 1024 : 2048); }   // cap - P >= BQ_THREADS; small caps keep 3 CTAs per SM

static int env_int(const char* name, int dflt)
{
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}
// candidate-list capacity per query: the main pass admits ~stride * P documents with stride = capq / (4 P)
static int bw_capq(int P)
{
    const int forced = env_int("KRAG_BM25_CAPQ", -1);     // read per call: the tests force overflows with it
    if (forced > 0) return forced < P ? P : forced;
    int c = 32768;
    while (c < 256 * P && c < 262144) c <<= 1;
    return c;
}
// which query kernel serves a shard: KRAG_BM25_KERNEL = auto (default) | warp | legacy; KRAG_BM25_LEGACY=1 == legacy.
// auto: with the rank-table threshold the warp kernel's fixed passes are a resolve, the threshold and one select; measured
// per 256-query batch of the bench's queries (scripts/k3_cutover.py, B200 at 1000 W) warp vs first generation: 0.17 vs
// 0.085 ms at 40k rows, 0.128 vs 0.110 at 80k, 0.128 vs 0.169 at 160k, 0.15 vs 0.24 at 320k, 0.27 vs 0.54 at 1.25M, 0.73 vs
// 1.67 at 5M: the curves cross between 80k and 160k rows
constexpr int64_t BW_AUTO_MIN_ROWS = 160000;
static bool bw_legacy(int64_t n_rows)
{
    if (env_int("KRAG_BM25_LEGACY", 0) != 0) return true;
    const char* k = getenv("KRAG_BM25_KERNEL");
    if (k && k[0] == 'w') return false;
    if (k && k[0] == 'l') return true;
    return n_rows < BW_AUTO_MIN_ROWS;
}

struct BmLayout {   // carve-up of the caller's u64 workspace (`part`)
    size_t legacy_part, g_thr, cand, thr, cnt_flags, counters, total;
    int64_t n_tiles, n_groups;
    int capq;
};
static BmLayout bm_layout(int64_t n_rows, int batch, int P)
{
    BmLayout L;
    L.n_tiles = (n_rows + BM25_TILE_DOCS - 1) / BM25_TILE_DOCS;
    if (L.n_tiles < 1) L.n_tiles = 1;
    L.n_groups = (L.n_tiles + bq_group() - 1) / bq_group();
    L.capq = bw_capq(P);
    size_t o = 0;
    L.legacy_part = o; o += (size_t)L.n_groups * batch * P;
    L.g_thr = o; o += (size_t)batch;
    L.cand = o; o += (size_t)batch * L.capq;
    L.thr = o; o += (size_t)batch;
    L.cnt_flags = o; o += (size_t)batch;          // u32 cnt[batch] then u32 flags[batch]
    L.counters = o; o += 4;                       // work-unit counters of the two passes
    L.total = o;
    return L;
}

size_t bm25_part_elems(int64_t n_rows, int batch, int P) { return bm_layout(n_rows, batch, P).total; }

size_t bm25_resolve_bytes(int64_t n_rows, int n_terms_total)
{
    const size_t n = (size_t)(n_terms_total > 0 ? n_terms_total : 1);
    int64_t n_sub = (n_rows + BM25_SUB_DOCS - 1) / BM25_SUB_DOCS;
    if (n_sub < 1) n_sub = 1;
    return n * (8 + 8 + 4 + 4) + n * (size_t)(n_sub + 1) * 4 + 64;
}

void launch_bm25(const DeviceInfo& di, const Postings& post, int64_t n_rows, const uint32_t* alive, bool alive_is_committed,
                 const uint32_t* q_terms, const int32_t* q_term_offsets, int n_terms_total, void* resolve_ws, int batch, int P,
                 OrdMap ord_base, uint64_t* part, uint64_t* keys_out, cudaStream_t st)
{
    const size_t nt = (size_t)(n_terms_total > 0 ? n_terms_total : 1);
    const int64_t n_sub = post.n_tiles;
    // resolve_ws: bm25_resolve_bytes(n_rows, n_terms_total)
    int64_t* q_base = reinterpret_cast<int64_t*>(resolve_ws);
    const uint32_t** q_row = reinterpret_cast<const uint32_t**>(q_base + nt);
    int32_t* q_slot = reinterpret_cast<int32_t*>(q_row + nt);
    int32_t* q_rare = q_slot + nt;
    uint32_t* scratch_rows = reinterpret_cast<uint32_t*>(q_rare + nt);
    if (n_terms_total > 0) {
        bm25_resolve_kernel<<<n_terms_total, 256, 0, st>>>(q_terms, n_terms_total, post.off, post.doc, post.tile_slot, post.tile_off,
                                                           post.vocab, n_sub, scratch_rows, q_row, q_base, q_slot, q_rare);
        KRAG_CUDA(cudaGetLastError());
        count_launch();
    }
    const BmLayout L = bm_layout(n_rows, batch, P);
    unsigned long long* g_thr = reinterpret_cast<unsigned long long*>(part + L.g_thr);
    unsigned long long* cand = reinterpret_cast<unsigned long long*>(part + L.cand);
    unsigned long long* thr_q = reinterpret_cast<unsigned long long*>(part + L.thr);
    uint32_t* cand_cnt = reinterpret_cast<uint32_t*>(part + L.cnt_flags);
    uint32_t* flags = cand_cnt + batch;
    unsigned long long* counters = reinterpret_cast<unsigned long long*>(part + L.counters);
    const bool legacy_only = bw_legacy(n_rows);
    const bool complete = n_rows <= (int64_t)L.capq;     // one pass without threshold cannot overflow the lists
    bool need_safety_net = legacy_only;

    if (!legacy_only) {
        static bool attr_set = false;
        const size_t smem = (size_t)BW_WARPS * BW_WARP_WORDS * 4;
        if (!attr_set) {
            KRAG_CUDA(cudaFuncSetAttribute(bm25_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_set = true;
        }
        // cnt[batch] + flags[batch] (u32) and the counters are contiguous: one memset
        KRAG_CUDA(cudaMemsetAsync(part + L.cnt_flags, 0, sizeof(uint64_t) * ((size_t)batch + 4), st));
        auto pass = [&](int stride, const unsigned long long* thr, unsigned long long* counter) {
            const int n_s = (int)((n_sub + stride - 1) / stride);
            const long long units = (long long)((n_s + BW_CHUNK - 1) / BW_CHUNK) * batch;
            const long long want = (units + BW_WARPS - 1) / BW_WARPS;
            const long long max_grid = 2LL * di.sm_count;
            const int grid = (int)(want < max_grid ? (want > 0 ? want : 1) : max_grid);
            bm25_warp_kernel<<<grid, BW_THREADS, smem, st>>>(post.doc, post.score, q_term_offsets, q_row, q_base, n_rows, alive, ord_base,
                                                             batch, n_s, stride, thr, cand, cand_cnt, L.capq, counter);
            KRAG_CUDA(cudaGetLastError());
            count_launch();
        };
        if (!complete && alive_is_committed) {
            // the rank table was built over exactly the documents `alive` admits: its bound holds, no sample pass
            int lg = 0;
            while ((1 << lg) < P) ++lg;
            bm25_rank_threshold_kernel<<<(batch + 127) / 128, 128, 0, st>>>(q_terms, q_term_offsets, batch, post.rank_score, post.vocab,
                                                                         lg, thr_q);
            KRAG_CUDA(cudaGetLastError());
            count_launch();
            pass(1, thr_q, counters);
            need_safety_net = true;
        } else if (!complete) {
            // deletes since the commit or a pushdown filter: documents the rank table counted may be excluded, so its bound
            // may not hold.  Sample every stride-th sub-tile instead: the main pass then admits ~stride * P documents per
            // query.  Small strides cost a larger sample pass (1 / stride of the main pass) but tighten the threshold
            int stride = L.capq / (4 * P);
            if (stride > 64) stride = 64;
            if (stride < 1) stride = 1;
            if ((int64_t)stride > n_sub) stride = (int)n_sub;
            pass(stride, nullptr, counters);                               // sample: every stride-th sub-tile, everything admitted
            bm25_select_kernel<<<batch, BS_THREADS, 0, st>>>(cand, cand_cnt, L.capq, P, 0, thr_q, keys_out, flags);
            KRAG_CUDA(cudaGetLastError());
            count_launch();
            pass(1, thr_q, counters + 1);                                  // main: all sub-tiles, key <= thr[q]
            need_safety_net = true;
        } else {
            pass(1, nullptr, counters);
        }
        bm25_select_kernel<<<batch, BS_THREADS, 0, st>>>(cand, cand_cnt, L.capq, P, 1, thr_q, keys_out, flags);
        KRAG_CUDA(cudaGetLastError());
        count_launch();
    }
    if (need_safety_net) {
        // legacy kernel: every query (KRAG_BM25_LEGACY=1) or only the queries whose list overflowed (normally none: its
        // CTAs read one flag per work item and leave)
        const int cap = bq_cap(P);
        const size_t smem = (size_t)BM25_TILE_DOCS * 4 + (size_t)cap * 8;
        static bool attr_set = false;
        if (!attr_set) {
            KRAG_CUDA(cudaFuncSetAttribute(bm25_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
            attr_set = true;
        }
        KRAG_CUDA(cudaMemsetAsync(g_thr, 0xFF, sizeof(unsigned long long) * (size_t)batch, st));
        const int64_t n_items = L.n_groups * batch;
        const int per_sm = (smem <= 74 * 1024) ? 3 : 2;
        const int64_t max_grid = (int64_t)per_sm * di.sm_count;
        const int grid = (int)(n_items < max_grid ? n_items : max_grid);
        const uint32_t* only = legacy_only ? nullptr : flags;
        bm25_tile_kernel<<<grid, BQ_THREADS, smem, st>>>(post.off, post.doc, post.score, post.tile_slot, post.tile_off,
                                                         post.n_tiles, post.vocab, q_terms, q_term_offsets, q_slot, q_base, q_rare, n_rows,
                                                         alive, P, cap, ord_base, batch, (int)L.n_tiles, bq_group(), part + L.legacy_part, g_thr, only);
        KRAG_CUDA(cudaGetLastError());
        count_launch();
        launch_merge(part + L.legacy_part, (int)L.n_groups, P, batch, P, /*list_stride=*/P, /*batch_stride=*/L.n_groups * P, keys_out, st,
                     reinterpret_cast<const uint64_t*>(g_thr), only);
    }
    launch_bm25_fill(keys_out, batch, P, alive, n_rows, ord_base, st);
}

}  // namespace krag
