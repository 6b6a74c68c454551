// kb_common.cuh -- shared declarations for libkarma_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <nvtx3/nvToolsExt.h>          // header-only (NVTX v3): ranges are no-ops unless a profiler is attached
#include "../../include/karma_b200.h"

#define KB_N_TIMERS 17
#define KB_EV_RING 128

struct kb_ctx {
    int device;
    int sm_count;
    cudaStream_t stream;
    int timing;
    // per-stage ring of CUDA-event pairs recorded on the launching stream; read (and
    // reset) by kb_stage_ms without synchronising inside the timed region
    cudaEvent_t (*ev0)[KB_EV_RING];
    cudaEvent_t (*ev1)[KB_EV_RING];
    int ev_n[KB_N_TIMERS];          // launches recorded since the last reset
    int64_t launches;
    // K1 scratch: work counter + long-contig list
    int32_t* d_k1_scratch;          // [0] contig counter, [1] n_long, [2..] long ids
    int64_t k1_scratch_cap;         // capacity in int32 entries
    // exotic side path (owned)
    uint64_t* d_ex_keys;            // unique keys (sorted k-mer path: the low 8 characters)
    uint64_t* d_ex_keys_hi;         // sorted k-mer path (k >= 8): the first 8 characters of every unique key
    int32_t* d_ex_row; int32_t* d_ex_keyidx; uint32_t* d_ex_cnt;
    int64_t ex_n_keys, ex_n_entries;
    // read-graph edges of the last kb_readgraph_build (owned)
    int32_t* d_rg_a; int32_t* d_rg_b; double* d_rg_w; uint64_t* d_rg_shared; int64_t rg_edges;
    // group-pair connection weights of the last kb_links_build: one grow-only scratch block (owned), results point into it
    void* d_lk_scratch; int64_t lk_scratch_bytes;
    int32_t* d_lk_a; int32_t* d_lk_b; double* d_lk_w; int64_t* d_lk_edges; int64_t* d_lk_over; int64_t lk_pairs;
    // fuzzy simplicial set (CSR) of the last kb_fuzzy_graph_build, in pool memory (owned)
    int64_t* d_fg_indptr; int32_t* d_fg_indices; double* d_fg_data; int64_t fg_n, fg_nnz;
    // stream-ordered pool for the temporaries of the read-graph build (created lazily, keeps its memory)
    cudaMemPool_t pool;
    // tensor-map encoder (driver entry point, resolved lazily)
    void* encode_tiled;
    // kNN plans and uploaded piece tables (kb_knn.cu)
    void* knn_cache;
    // the spectral initialisation of the last kb_spectral_build (kb_spectral.cu, owned)
    void* spectral;
    // the MCL result of the last kb_mcl_build (kb_mcl.cu, owned)
    void* mcl;
};

void kb_set_error(const char* fmt, ...);
int kb_cuda_fail(cudaError_t e, const char* what);

#define KB_CUDA(call)                                                   \
    do {                                                                \
        cudaError_t _e = (call);                                        \
        if (_e != cudaSuccess) return kb_cuda_fail(_e, #call);          \
    } while (0)

#define KB_CHECK_ARG(cond, msg)                                         \
    do {                                                                \
        if (!(cond)) { kb_set_error("invalid argument: %s", msg); return KB_EINVAL; } \
    } while (0)

// One stage of the path on the host timeline: an NVTX range (SURVEY 5: per-stage ranges for nsys / ncu --nvtx) and,
// with timing enabled, a CUDA-event pair on the launching stream.
static const char* const kb_stage_names[KB_N_TIMERS] = {
    "kb:K1 count", "kb:K1 count (split contigs)", "kb:K2 compact", "kb:K3 normalise", "kb:K4 distance GEMM + top-k",
    "kb:K5 merge + exact rerank", "kb:K4x/K6 exact distances", "kb:read graph", "kb:group links",
    "kb:K9 core distances", "kb:K9 Boruvka round", "kb:K9 edge sort", "kb:K10 components", "kb:K10 eigensolve",
    "kb:K10 meta-embedding", "kb:K11 set-up", "kb:K11 iteration"};
struct KbTimer {
    kb_ctx* c; int which; int slot;
    KbTimer(kb_ctx* ctx, int w) : c(ctx), which(w), slot(0) {
        nvtxRangePushA(kb_stage_names[which]);
        if (c->timing) { slot = c->ev_n[which] % KB_EV_RING; cudaEventRecord(c->ev0[which][slot], c->stream); }
    }
    ~KbTimer() {
        if (c->timing) { cudaEventRecord(c->ev1[which][slot], c->stream); c->ev_n[which]++; }
        nvtxRangePop();
    }
};

// mode description shared by host and device
struct KbMode {
    int ka;        // first component k (0 = none)
    int kb;        // second component k (0 = none)
    int pal_b;     // second component: string-palindromic windows only, binned by rank
    int bins_a;    // 4^ka
    int bins_b;    // 4^kb, or 4^(kb/2) when pal_b
    int permute;   // columns are a permutation of [A bins | B bins] (5p6 sorted order)
    int cols;      // bins_a + bins_b
};
int kb_mode_describe(int mode, KbMode* out);

// internal launchers (defined in the per-kernel .cu files)
int kb_launch_count_kernels(kb_ctx* ctx, const KbMode& m, const uint8_t* d_bases,
                            const int64_t* d_offsets, int64_t n, uint32_t* d_counts,
                            int64_t ld, uint32_t* d_exotic, uint32_t* d_presence, int track_columns);

void kb_links_free(kb_ctx* c);
void kb_fuzzy_free(kb_ctx* c);
void kb_knn_cache_free(kb_ctx* c);
void kb_spectral_free(kb_ctx* c);
void kb_mcl_free(kb_ctx* c);
// host-side file input shared by the FASTA and eq_classes parsers (kb_fasta.cu)
int64_t kb_host_threads();
int kb_host_read_file(const char* path, uint8_t** img, int64_t* size);
int kb_pool_get(kb_ctx* c, cudaMemPool_t* out);

// temporary from the context's stream-ordered pool, returned to it (not to the driver) when it goes out of scope
struct PoolBuf {
    cudaMemPool_t pool = nullptr;
    cudaStream_t stream = 0;
    void* p = nullptr;
    PoolBuf(cudaMemPool_t pl, cudaStream_t st) : pool(pl), stream(st) {}
    ~PoolBuf() { if (p) cudaFreeAsync(p, stream); }
    cudaError_t alloc(size_t bytes) { return cudaMallocFromPoolAsync(&p, bytes ? bytes : 1, pool, stream); }
    template <class T> T* as() { return reinterpret_cast<T*>(p); }
};

static inline int64_t kb_round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// ---- a fuzzy graph's CSR rows, checked as K8 and K10 check them ----
constexpr unsigned KB_CSR_BAD_INDPTR = 1u, KB_CSR_BAD_INDEX = 2u, KB_CSR_BAD_DATA = 4u;

__device__ __forceinline__ bool kb_csr_row(const int64_t* __restrict__ indptr, int64_t r, int64_t nnz, int64_t* lo, int64_t* hi) {
    *lo = indptr[r];
    *hi = indptr[r + 1];
    return *lo >= 0 && *lo <= *hi && *hi <= nnz;
}

__device__ __forceinline__ bool kb_weight_ok(double w) { return w > 0.0 && w <= 1.7976931348623157e308; }

// thread per row: indptr monotone from 0 to nnz, indices in [0, n), data finite and > 0 (KB_CSR_BAD_* into *flags); the
// largest weight into *wmax_bits (atomicMax on the bits of a positive double, order-free).  No read beyond nnz entries.
static __global__ void kb_csr_check(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                    const double* __restrict__ data, int64_t n, int64_t nnz,
                                    unsigned long long* __restrict__ flags, unsigned long long* __restrict__ wmax_bits) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    unsigned f = 0;
    if (r == 0 && (indptr[0] != 0 || indptr[n] != nnz)) f |= KB_CSR_BAD_INDPTR;
    int64_t lo, hi;
    double mx = 0.0;
    if (!kb_csr_row(indptr, r, nnz, &lo, &hi)) {
        f |= KB_CSR_BAD_INDPTR;
    } else {
        for (int64_t e = lo; e < hi; ++e) {
            const int32_t c = indices[e];
            if (c < 0 || (int64_t)c >= n) f |= KB_CSR_BAD_INDEX;
            const double w = data[e];
            if (!kb_weight_ok(w)) f |= KB_CSR_BAD_DATA;
            else if (w > mx) mx = w;
        }
    }
    if (f) atomicOr(flags, (unsigned long long)f);
    if (mx > 0.0) atomicMax(wmax_bits, (unsigned long long)__double_as_longlong(mx));
}

// ---- hooking union-find over components (K9's Boruvka rounds, K10's connected components) ----
// comp[i] is i's component, named by its root vertex (comp[c] == c); comp_key[c] is the edge (min << 32 | max) along which
// component c hooks, ~0 for none.  With every component hooking along its minimum edge under one strict total order, the
// successor graph is a forest whose only cycles are pairs that chose the same edge.
__device__ __forceinline__ unsigned long long hd_key(int64_t a, int64_t b) {
    return a < b ? ((unsigned long long)a << 32) | (unsigned long long)b : ((unsigned long long)b << 32) | (unsigned long long)a;
}

// each component's successor: the component at the other end of its edge (itself when it has none)
static __global__ void hd_hook(const int32_t* __restrict__ comp, const unsigned long long* __restrict__ comp_key,
                               int32_t* __restrict__ succ, int64_t n) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n || comp[c] != c) return;
    const unsigned long long key = comp_key[c];
    if (key == ~0ull) { succ[c] = (int32_t)c; return; }
    const int32_t ca = comp[key >> 32], cb = comp[key & 0xffffffffull];
    succ[c] = ca == c ? cb : ca;
}

// one pointer-jumping step over the components' parents; every value written is an ancestor, so concurrent reads are safe
static __global__ void hd_jump(const int32_t* __restrict__ comp, int32_t* par, int64_t n) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n || comp[c] != c) return;
    par[c] = par[par[c]];
}

// comp[i] <- its root; *n_comp counts the roots
static __global__ void hd_relabel(int32_t* __restrict__ comp, const int32_t* __restrict__ par, int64_t n,
                                  unsigned long long* __restrict__ n_comp) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t c = comp[i];
    const int32_t r = par[c];
    comp[i] = r;
    if (c == i && r == i) atomicAdd(n_comp, 1ull);
}

static __global__ void hd_iota(int32_t* __restrict__ comp, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) comp[i] = (int32_t)i;
}
