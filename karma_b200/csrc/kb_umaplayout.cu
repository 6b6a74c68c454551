// kb_umaplayout.cu -- K8: UMAP's layout optimisation over the fuzzy graph (the stage after K7).
//
// Replaces the tail of umap.umap_.simplicial_set_embedding of umap-learn 0.3.9 (pruning, make_epochs_per_sample,
// optimize_layout), which karma reaches through UMAP.fit at kmer.py:285-290.  umap's loop is sequential: every
// sample moves the embedding in place and the next sample sees the move.  The device runs ONE deterministic
// algorithm instead, epoch-synchronous with exact fixed-point accumulation (rules frozen in
// oracle/umap_layout_oracle.py, optimize_layout_sync):
//   * the schedule is umap's, in fp64: an edge fires in epoch n when epoch_of_next_sample <= n,
//     n_neg = int((n - epoch_of_next_negative_sample) / epochs_per_negative_sample), both counters advance as in umap;
//   * every sample of epoch n reads the positions Y as they were at the start of the epoch;
//   * the negative sample p of kept edge e in epoch n is vertex H(seed, e, n, p): splitmix64 finalisers chained over
//     (seed, e, n, p), multiply-shift of the high 32 bits onto [0, N) -- no state, so no dependence on order;
//   * every gradient coordinate (fp64, umap's formulas; no FMA contraction) is rounded to an int64 at 2^-32 and added
//     to a per-vertex, per-coordinate int64 accumulator: integer addition is associative, so the sum does not depend
//     on the order the atomics land in; then Y <- fp32(fp64(Y) + acc * 2^-32) and acc <- 0.
// GPU formulation:
//   0. before the one host synchronisation (thread per row; no read beyond the caller's nnz entries):
//      kb_csr_check   indptr monotone from 0 to nnz, indices in [0, N), data finite and > 0, row max -> fp64 max (atomicMax
//                     on the bits of a positive double, order-free);  ul_check_init: init finite
//      ul_rows_keep   kept edges per row (w >= max / n_epochs, umap's pruning), total degree of every vertex
//      ul_max_degree  the largest total degree, for the fixed-point range check
//   1. after it: scan of the kept counts, ul_compact writes head / tail / epochs_per_sample / both counters in CSR order
//   2. per epoch, enqueued back to back with no host synchronisation: ul_epoch<DMAX> (a thread owns UL_CHUNK
//      consecutive kept edges; CSR rows are grouped by head, so it sums its head's moves in registers and adds them
//      once per head it meets; only tails need an atomic per sample), then ul_apply
#include "kb_common.cuh"
#include <cub/cub.cuh>
#include <cmath>

namespace {

constexpr int UL_THREADS = 128;
constexpr int UL_CHUNK = 16;
constexpr unsigned UL_BAD_INIT = 8u;     // above kb_csr_check's KB_CSR_BAD_* bits

struct UlStatus {                 // device word block read back by the one host synchronisation
    unsigned long long flags;
    unsigned long long wmax_bits; // fp64 bits of the largest weight (positive doubles order like their bits)
    unsigned long long kept;
    unsigned long long max_degree;
};

struct UlParams {
    double a, b, bm1, c_att, c_rep, rate;
    uint64_t seed_mixed;          // mix64(seed)
    int64_t n_vertices;
    int dim;
    int has_neg;
};

__host__ __device__ __forceinline__ uint64_t ul_mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

__global__ void ul_check_init(const float* __restrict__ y, int64_t total, UlStatus* __restrict__ st) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x)
        if (!isfinite(y[t])) { atomicOr(&st->flags, (unsigned long long)UL_BAD_INIT); return; }
}

// umap's pruning: data < max / n_epochs is dropped
__device__ __forceinline__ double ul_threshold(const UlStatus* st, int n_epochs) {
    return __ddiv_rn(__longlong_as_double((long long)st->wmax_bits), (double)n_epochs);
}

__global__ void __launch_bounds__(UL_THREADS) ul_rows_keep(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                           const double* __restrict__ data, int64_t n, int64_t nnz,
                                                           int n_epochs, UlStatus* __restrict__ st, int64_t* __restrict__ row_kept,
                                                           int* __restrict__ degree) {
    typedef cub::BlockReduce<unsigned long long, UL_THREADS> Red;
    __shared__ typename Red::TempStorage tmp;
    const int64_t r = (int64_t)blockIdx.x * UL_THREADS + threadIdx.x;
    unsigned long long kept = 0;
    if (r < n) {
        const double thr = ul_threshold(st, n_epochs);
        int64_t lo, hi;
        if (kb_csr_row(indptr, r, nnz, &lo, &hi)) {
            for (int64_t e = lo; e < hi; ++e) {
                const int32_t c = indices[e];
                const double w = data[e];
                if (c < 0 || (int64_t)c >= n || !kb_weight_ok(w) || w < thr) continue;
                ++kept;
                atomicAdd(&degree[c], 1);
            }
            if (kept) atomicAdd(&degree[r], (int)kept);
        }
        row_kept[r] = (int64_t)kept;
    }
    const unsigned long long total = Red(tmp).Sum(kept);
    if (threadIdx.x == 0 && total) atomicAdd(&st->kept, total);
}

__global__ void __launch_bounds__(256) ul_max_degree(const int* __restrict__ degree, int64_t n, UlStatus* __restrict__ st) {
    typedef cub::BlockReduce<int, 256> Red;
    __shared__ typename Red::TempStorage tmp;
    int mx = 0;
    for (int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x; t < n; t += (int64_t)gridDim.x * 256) mx = max(mx, degree[t]);
    const int m = Red(tmp).Reduce(mx, cub::Max());
    if (threadIdx.x == 0 && m) atomicMax(&st->max_degree, (unsigned long long)m);
}

// kept edges in CSR order: head, tail, epochs_per_sample = n_epochs / (n_epochs * (w / max)) and the two counters
__global__ void __launch_bounds__(UL_THREADS) ul_compact(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                         const double* __restrict__ data, int64_t n, int n_epochs, double rate,
                                                         const UlStatus* __restrict__ st, const int64_t* __restrict__ row_off,
                                                         int32_t* __restrict__ head, int32_t* __restrict__ tail,
                                                         double* __restrict__ eps, double* __restrict__ next_pos,
                                                         double* __restrict__ next_neg) {
    const int64_t r = (int64_t)blockIdx.x * UL_THREADS + threadIdx.x;
    if (r >= n) return;
    const double wmax = __longlong_as_double((long long)st->wmax_bits);
    const double thr = ul_threshold(st, n_epochs);
    const double fn = (double)n_epochs;
    int64_t o = row_off[r];
    for (int64_t e = indptr[r]; e < indptr[r + 1]; ++e) {
        const double w = data[e];
        if (w < thr) continue;
        const double s = __ddiv_rn(fn, __dmul_rn(fn, __ddiv_rn(w, wmax)));
        head[o] = (int32_t)r;
        tail[o] = indices[e];
        eps[o] = s;
        next_pos[o] = s;
        next_neg[o] = rate > 0.0 ? __ddiv_rn(s, rate) : 0.0;
        ++o;
    }
}

// umap's clip; NaN passes through
__device__ __forceinline__ double ul_clip(double v) { return v > 4.0 ? 4.0 : (v < -4.0 ? -4.0 : v); }

__device__ __forceinline__ long long ul_fixed(double g) { return __double2ll_rn(__dmul_rn(g, 4294967296.0)); }

// umap's rdist, summed in coordinate order (yj stays in registers: the loop is unrolled over DMAX)
template <int DMAX>
__device__ __forceinline__ double ul_rdist(const float (&yj)[DMAX], const float* __restrict__ yo, int dim) {
    double d2 = 0.0;
#pragma unroll
    for (int d = 0; d < DMAX; ++d) {
        if (d >= dim) break;
        const double df = __dsub_rn((double)yj[d], (double)__ldg(yo + d));
        d2 = __dadd_rn(d2, __dmul_rn(df, df));
    }
    return d2;
}

template <int DMAX>
__device__ __forceinline__ void ul_flush(unsigned long long* __restrict__ acc, int64_t row, int dim, long long* hs) {
#pragma unroll
    for (int d = 0; d < DMAX; ++d)
        if (d < dim && hs[d]) atomicAdd(&acc[row * dim + d], (unsigned long long)hs[d]);
}

template <int DMAX>
__global__ void __launch_bounds__(UL_THREADS) ul_epoch(const int32_t* __restrict__ head, const int32_t* __restrict__ tail,
                                                       const double* __restrict__ eps, double* __restrict__ next_pos,
                                                       double* __restrict__ next_neg, int64_t m, const float* __restrict__ y,
                                                       unsigned long long* __restrict__ acc, UlParams P, int epoch,
                                                       double alpha, long long* __restrict__ samples) {
    int64_t e = ((int64_t)blockIdx.x * UL_THREADS + threadIdx.x) * UL_CHUNK;
    if (e >= m) return;
    const int64_t e_end = min(e + (int64_t)UL_CHUNK, m);
    const int dim = P.dim;
    const double fe = (double)epoch;
    const double g4 = __dmul_rn(4.0, alpha);
    long long hs[DMAX];
    float yj[DMAX];
    int64_t cur = -1;
    for (; e < e_end; ++e) {
        const double np = next_pos[e];
        if (np > fe) continue;
        const int64_t j = head[e];
        if (j != cur) {
            if (cur >= 0) ul_flush<DMAX>(acc, cur, dim, hs);
            cur = j;
#pragma unroll
            for (int d = 0; d < DMAX; ++d) {
                hs[d] = 0;
                yj[d] = d < dim ? y[j * dim + d] : 0.f;
            }
        }
        // attraction: head and tail are the same array (umap's move_other)
        const int64_t k = tail[e];
        const float* yk = y + k * dim;
        double d2 = ul_rdist<DMAX>(yj, yk, dim);
        double coef = 0.0;
        if (d2 > 0.0)
            coef = __ddiv_rn(__dmul_rn(P.c_att, pow(d2, P.bm1)), __dadd_rn(__dmul_rn(P.a, pow(d2, P.b)), 1.0));
#pragma unroll
        for (int d = 0; d < DMAX; ++d) {
            if (d >= dim) break;
            const double df = __dsub_rn((double)yj[d], (double)__ldg(yk + d));
            const long long q = ul_fixed(__dmul_rn(ul_clip(__dmul_rn(coef, df)), alpha));
            hs[d] += q;
            if (q) atomicAdd(&acc[k * dim + d], (unsigned long long)(-q));
        }
        const double s = eps[e];
        next_pos[e] = __dadd_rn(np, s);
        long long n_neg = 0;
        if (P.has_neg) {
            // repulsion: the head alone moves
            const double epn = __ddiv_rn(s, P.rate);
            const double nn = next_neg[e];
            n_neg = __double2ll_rz(__ddiv_rn(__dsub_rn(fe, nn), epn));
            const uint64_t hee = ul_mix64(ul_mix64(P.seed_mixed ^ (uint64_t)e) ^ (uint64_t)epoch);
            for (long long p = 0; p < n_neg; ++p) {
                const uint64_t h = ul_mix64(hee ^ (uint64_t)p);
                const int64_t v = (int64_t)(((h >> 32) * (uint64_t)P.n_vertices) >> 32);
                const float* yv = y + v * dim;
                d2 = ul_rdist<DMAX>(yj, yv, dim);
                if (d2 > 0.0)
                    coef = __ddiv_rn(P.c_rep, __dmul_rn(__dadd_rn(0.001, d2), __dadd_rn(__dmul_rn(P.a, pow(d2, P.b)), 1.0)));
                else if (v == j)
                    continue;
                else
                    coef = 0.0;
#pragma unroll
                for (int d = 0; d < DMAX; ++d) {
                    if (d >= dim) break;
                    const double df = __dsub_rn((double)yj[d], (double)__ldg(yv + d));
                    const double g = coef > 0.0 ? __dmul_rn(ul_clip(__dmul_rn(coef, df)), alpha) : g4;   // umap 0.3.9: 4
                    hs[d] += ul_fixed(g);
                }
            }
            next_neg[e] = __dadd_rn(nn, __dmul_rn((double)n_neg, epn));
        }
        if (samples) {
            samples[2 * e] += 1;
            samples[2 * e + 1] += n_neg > 0 ? n_neg : 0;
        }
    }
    if (cur >= 0) ul_flush<DMAX>(acc, cur, dim, hs);
}

__global__ void ul_apply(float* __restrict__ y, unsigned long long* __restrict__ acc, int64_t total) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const long long a = (long long)acc[t];
        y[t] = __double2float_rn(__dadd_rn((double)y[t], __dmul_rn(__ll2double_rn(a), 0x1p-32)));
        acc[t] = 0;
    }
}

template <int DMAX>
void ul_launch_epoch(unsigned blocks, cudaStream_t st, const int32_t* head, const int32_t* tail, const double* eps,
                     double* next_pos, double* next_neg, int64_t m, const float* y, unsigned long long* acc,
                     const UlParams& P, int epoch, double alpha, long long* samples) {
    ul_epoch<DMAX><<<blocks, UL_THREADS, 0, st>>>(head, tail, eps, next_pos, next_neg, m, y, acc, P, epoch, alpha, samples);
}

}  // namespace

extern "C" int kb_umap_layout(kb_ctx* ctx, int64_t n, int64_t nnz, const int64_t* d_indptr, const int32_t* d_indices, const double* d_data,
                              int32_t dim, int32_t n_epochs, double a, double b, double gamma, double initial_alpha,
                              double negative_sample_rate, uint64_t seed, float* d_embedding, int64_t* d_samples,
                              int64_t* nnz_kept) {
    KB_CHECK_ARG(ctx && nnz_kept && (n == 0 || (d_indptr && d_embedding)) && (nnz == 0 || (d_indices && d_data)),
                 "null pointer");
    KB_CHECK_ARG(n >= 0 && n <= INT32_MAX, "n (0 <= n < 2^31)");
    KB_CHECK_ARG(nnz >= 0 && (n > 0 || nnz == 0), "nnz (>= 0, 0 when n is 0)");
    KB_CHECK_ARG(dim >= 1, "dim must be >= 1");
    KB_CHECK_ARG(n_epochs >= 1, "n_epochs must be >= 1");
    KB_CHECK_ARG(std::isfinite(a) && std::isfinite(b) && std::isfinite(gamma), "a, b and gamma must be finite");
    KB_CHECK_ARG(std::isfinite(initial_alpha) && initial_alpha >= 0.0, "initial_alpha must be finite and >= 0");
    KB_CHECK_ARG(std::isfinite(negative_sample_rate) && negative_sample_rate >= 0.0, "negative_sample_rate must be finite and >= 0");
    if (dim > 64) { kb_set_error("umap layout: n_components = %d, this build serves 1..64", dim); return KB_EUNSUPPORTED; }
    *nnz_kept = 0;
    if (n == 0) return KB_OK;
    KB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    cudaMemPool_t pool;
    { int rc = kb_pool_get(ctx, &pool); if (rc) return rc; }
    // 0. validation, max, pruning counts and degrees; then the one host synchronisation
    PoolBuf status(pool, st), row_kept(pool, st), degree(pool, st);
    KB_CUDA(status.alloc(sizeof(UlStatus)));
    KB_CUDA(row_kept.alloc((size_t)(n + 1) * 8));
    KB_CUDA(degree.alloc((size_t)n * 4));
    KB_CUDA(cudaMemsetAsync(status.p, 0, sizeof(UlStatus), st));
    KB_CUDA(cudaMemsetAsync(degree.p, 0, (size_t)n * 4, st));
    UlStatus* d_st = status.as<UlStatus>();
    const unsigned row_blocks = (unsigned)((n + UL_THREADS - 1) / UL_THREADS);
    const int64_t total = n * dim;
    const unsigned flat_blocks = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 16);
    kb_csr_check<<<row_blocks, UL_THREADS, 0, st>>>(d_indptr, d_indices, d_data, n, nnz, &d_st->flags, &d_st->wmax_bits);
    ul_check_init<<<flat_blocks, 256, 0, st>>>(d_embedding, total, d_st);
    ul_rows_keep<<<row_blocks, UL_THREADS, 0, st>>>(d_indptr, d_indices, d_data, n, nnz, n_epochs, d_st, row_kept.as<int64_t>(),
                                                     degree.as<int>());
    ul_max_degree<<<(unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8), 256, 0, st>>>(degree.as<int>(), n, d_st);
    ctx->launches += 4;
    KB_CUDA(cudaGetLastError());
    UlStatus h;
    KB_CUDA(cudaMemcpyAsync(&h, d_st, sizeof(UlStatus), cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    if (h.flags & KB_CSR_BAD_INDPTR) { kb_set_error("umap layout: indptr must run from 0 to nnz and never decrease"); return KB_EINVAL; }
    if (h.flags & KB_CSR_BAD_INDEX) { kb_set_error("umap layout: a column index is outside [0, n)"); return KB_EINVAL; }
    if (h.flags & KB_CSR_BAD_DATA) { kb_set_error("umap layout: every weight must be finite and > 0"); return KB_EINVAL; }
    if (h.flags & UL_BAD_INIT) { kb_set_error("umap layout: the initial embedding holds a value that is not finite"); return KB_EINVAL; }
    const int64_t m = (int64_t)h.kept;
    *nnz_kept = m;
    if (m == 0) return KB_OK;
    // A vertex collects per epoch one attraction per incident kept edge and, as a head, n_neg repulsions per out-edge
    // (an edge fires at most once per epoch), every coordinate at most 4 * alpha.  One firing draws fewer than
    // 2 * rate + 1 negative samples (DESIGN §3 K8), so at most ceil(2 * rate); one more absorbs fp64 rounding.
    const double neg_max = negative_sample_rate > 0.0 ? std::ceil(2.0 * negative_sample_rate) + 1.0 : 0.0;
    const double bound = (double)h.max_degree * (1.0 + neg_max) * 4.0 * initial_alpha * 4294967296.0;
    if (!(bound < 4611686018427387904.0)) {
        kb_set_error("umap layout: max degree %llu x (2 + ceil(2 * rate)) x 4 x initial_alpha may leave the int64 fixed-point "
                     "range at 2^-32", h.max_degree);
        return KB_EUNSUPPORTED;
    }
    // 1. kept edges in CSR order
    PoolBuf row_off(pool, st), scan_tmp(pool, st), head(pool, st), tail(pool, st), eps(pool, st), next_pos(pool, st),
        next_neg(pool, st), acc(pool, st);
    KB_CUDA(row_off.alloc((size_t)(n + 1) * 8));
    size_t tb = 0;
    KB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, row_kept.as<int64_t>(), row_off.as<int64_t>(), n, st));
    KB_CUDA(scan_tmp.alloc(tb));
    KB_CUDA(cub::DeviceScan::ExclusiveSum(scan_tmp.p, tb, row_kept.as<int64_t>(), row_off.as<int64_t>(), n, st));
    KB_CUDA(head.alloc((size_t)m * 4)); KB_CUDA(tail.alloc((size_t)m * 4));
    KB_CUDA(eps.alloc((size_t)m * 8)); KB_CUDA(next_pos.alloc((size_t)m * 8)); KB_CUDA(next_neg.alloc((size_t)m * 8));
    KB_CUDA(acc.alloc((size_t)total * 8));
    KB_CUDA(cudaMemsetAsync(acc.p, 0, (size_t)total * 8, st));
    if (d_samples) KB_CUDA(cudaMemsetAsync(d_samples, 0, (size_t)m * 16, st));
    ul_compact<<<row_blocks, UL_THREADS, 0, st>>>(d_indptr, d_indices, d_data, n, n_epochs, negative_sample_rate, d_st,
                                                   row_off.as<int64_t>(), head.as<int32_t>(), tail.as<int32_t>(), eps.as<double>(),
                                                   next_pos.as<double>(), next_neg.as<double>());
    ctx->launches += 2;
    // 2. the epochs, enqueued back to back
    UlParams P;
    P.a = a; P.b = b; P.bm1 = b - 1.0;
    P.c_att = (-2.0 * a) * b;
    P.c_rep = (2.0 * gamma) * b;
    P.rate = negative_sample_rate;
    P.has_neg = negative_sample_rate > 0.0;
    P.seed_mixed = ul_mix64(seed);
    P.n_vertices = n;
    P.dim = dim;
    const unsigned epoch_blocks = (unsigned)(((m + UL_CHUNK - 1) / UL_CHUNK + UL_THREADS - 1) / UL_THREADS);
    const unsigned apply_blocks = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 32);
    auto launch = dim <= 2 ? ul_launch_epoch<2> : dim <= 4 ? ul_launch_epoch<4> : dim <= 8 ? ul_launch_epoch<8>
                : dim <= 16 ? ul_launch_epoch<16> : dim <= 32 ? ul_launch_epoch<32> : ul_launch_epoch<64>;
    double alpha = initial_alpha;
    for (int ep = 0; ep < n_epochs; ++ep) {
        launch(epoch_blocks, st, head.as<int32_t>(), tail.as<int32_t>(), eps.as<double>(), next_pos.as<double>(),
               next_neg.as<double>(), m, d_embedding, acc.as<unsigned long long>(), P, ep, alpha, (long long*)d_samples);
        ul_apply<<<apply_blocks, 256, 0, st>>>(d_embedding, acc.as<unsigned long long>(), total);
        alpha = initial_alpha * (1.0 - ((double)ep / (double)n_epochs));     // umap: set after epoch ep, used in ep + 1
    }
    ctx->launches += 2 * (int64_t)n_epochs;
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}
