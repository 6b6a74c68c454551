// kb_hdbscan.cu -- K9: HDBSCAN's mutual-reachability minimum spanning tree (device) and its clusters (host).
//
// Replaces hdbscan.HDBSCAN(min_cluster_size=m).fit(embedding) of hdbscan 0.8.22 (kmer.py:296-301); the reference of
// record is scikit-learn 1.9.0's port of its tree code (sklearn/cluster/_hdbscan/_linkage.pyx, _tree.pyx).  Rules
// frozen in oracle/hdbscan_oracle.py:
//   * d(i, j) = RN(sqrt(sum_c (x_ic - x_jc)^2)) in fp64 from the float32 coordinates, in coordinate order, no FMA
//     contraction (sklearn's EuclideanDistance64.rdist, then sqrt);
//   * core_i = the core_k-th smallest of {d(i, j) : all j}, d(i, i) = 0 and duplicates counted (kneighbors);
//   * w(i, j) = max(core_i, core_j, d(i, j)) (mst_from_data_matrix, alpha 1);
//   * edges are totally ordered by (w, min(i, j), max(i, j)): the MST is unique, and it is returned oriented
//     (min, max) and sorted in that order, which is the order make_single_linkage consumes.
// GPU formulation:
//   hd_check   non-finite coordinates -> one flag word
//   hd_core    all-pairs tile sweep: a thread owns a row (coordinates widened to fp64 in registers), column tiles are
//              staged in shared memory as fp64; the row keeps its core_k smallest d^2 (sorted, local memory) and takes
//              one sqrt at the end (sqrt is monotone and correctly rounded, so this is the core_k-th smallest d)
//   Boruvka rounds over the implicit complete graph, until one component is left (at most ceil(log2 N) rounds; the
//   host reads the component count once per round):
//   hd_round   the same sweep: row i's minimum (w, j) over comp[j] != comp[i].  Columns run in ascending j, so a tie never
//              replaces, and for a fixed i the (w, j) order is the (w, min, max) order.  A pair is skipped before its
//              distance when max(core_i, core_j) >= best, and before its sqrt when d^2 >= RU(best^2) (then
//              RN(sqrt(d^2)) >= best): both skips provably leave the fp64 w of every kept candidate unchanged.
//              atomicMin of the weight bits per component (non-negative doubles order like their bits)
//   hd_comp_key  rows whose weight is their component's minimum: atomicMin of the key (min << 32 | max)
//   hd_hook    (kb_common.cuh) each component's successor: the component at the other end of its minimum edge
//   hd_link    the only cycles are pairs choosing the same edge: the smaller id becomes a root, the other appends it
//   hd_jump    pointer jumping to the roots, hd_relabel: comp[i] <- root, count the components
//   edge sort  two stable CUB radix sorts: by (min << 32 | max), then by the weight bits -> (w, min, max)
#include "kb_common.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <cmath>
#include <vector>

namespace {

constexpr int HD_THREADS = 128;
constexpr int HD_TJ = 64;             // columns per shared-memory tile
constexpr int HD_KMAX = 128;
constexpr int HD_DIM_MAX = 64;
constexpr unsigned HD_BAD_X = 1u;

struct HdStatus {                     // device words read back once per round
    unsigned long long flags;
    unsigned long long n_comp;
    unsigned long long n_edges;
};

__global__ void hd_check(const float* __restrict__ x, int64_t total, HdStatus* __restrict__ st) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x)
        if (!isfinite(x[t])) { atomicOr(&st->flags, (unsigned long long)HD_BAD_X); return; }
}

// columns [j0, j0 + HD_TJ) of x, widened to fp64, at a row stride of DMAX
template <int DMAX>
__device__ __forceinline__ void hd_load_tile(double* xs, const float* __restrict__ x, int64_t n, int dim, int64_t j0) {
    const int64_t jn = min((int64_t)HD_TJ, n - j0);
    const float* src = x + j0 * dim;
    for (int t = threadIdx.x; t < jn * dim; t += HD_THREADS) {
        const int jj = t / dim, c = t - jj * dim;
        xs[jj * DMAX + c] = (double)src[t];
    }
}

template <int DMAX>
__device__ __forceinline__ void hd_load_row(double (&xi)[DMAX], const float* __restrict__ x, int64_t i, int dim) {
#pragma unroll
    for (int c = 0; c < DMAX; ++c) xi[c] = c < dim ? (double)x[i * dim + c] : 0.0;
}

// sklearn's rdist: the squares summed in coordinate order, no contraction
template <int DMAX>
__device__ __forceinline__ double hd_d2(const double (&xi)[DMAX], const double* xj, int dim) {
    double d2 = 0.0;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) {
        if (c >= dim) break;
        const double df = __dsub_rn(xi[c], xj[c]);
        d2 = __dadd_rn(d2, __dmul_rn(df, df));
    }
    return d2;
}

template <int DMAX>
__global__ void __launch_bounds__(HD_THREADS) hd_core(const float* __restrict__ x, int64_t n, int dim, int k,
                                                      double* __restrict__ core) {
    __shared__ double xs[HD_TJ * DMAX];
    const int64_t i = (int64_t)blockIdx.x * HD_THREADS + threadIdx.x;
    const bool live = i < n;
    double xi[DMAX];
    hd_load_row<DMAX>(xi, x, live ? i : 0, dim);
    double lst[HD_KMAX];              // the k smallest d^2 so far, ascending
    int cnt = 0;
    double thr = INFINITY;            // lst[k - 1] once full: d^2 is finite for finite float32 input
    for (int64_t j0 = 0; j0 < n; j0 += HD_TJ) {
        __syncthreads();
        hd_load_tile<DMAX>(xs, x, n, dim, j0);
        __syncthreads();
        if (!live) continue;
        const int jn = (int)min((int64_t)HD_TJ, n - j0);
        for (int jj = 0; jj < jn; ++jj) {
            const double d2 = hd_d2<DMAX>(xi, xs + jj * DMAX, dim);
            if (!(d2 < thr)) continue;
            int p = cnt < k ? cnt++ : k - 1;
            while (p > 0 && lst[p - 1] > d2) { lst[p] = lst[p - 1]; --p; }
            lst[p] = d2;
            if (cnt == k) thr = lst[k - 1];
        }
    }
    if (live) core[i] = __dsqrt_rn(lst[k - 1]);
}

template <int DMAX>
__global__ void __launch_bounds__(HD_THREADS) hd_round(const float* __restrict__ x, int64_t n, int dim,
                                                       const double* __restrict__ core, const int32_t* __restrict__ comp,
                                                       double* __restrict__ row_w, int32_t* __restrict__ row_j,
                                                       unsigned long long* __restrict__ comp_w) {
    __shared__ double xs[HD_TJ * DMAX];
    __shared__ double cs[HD_TJ];
    __shared__ int32_t ms[HD_TJ];
    const int64_t i = (int64_t)blockIdx.x * HD_THREADS + threadIdx.x;
    const bool live = i < n;
    double xi[DMAX];
    hd_load_row<DMAX>(xi, x, live ? i : 0, dim);
    const double ci = live ? core[i] : 0.0;
    const int32_t mi = live ? comp[i] : -1;
    double bw = INFINITY, thr = INFINITY;
    int32_t bj = -1;
    for (int64_t j0 = 0; j0 < n; j0 += HD_TJ) {
        __syncthreads();
        hd_load_tile<DMAX>(xs, x, n, dim, j0);
        const int jn = (int)min((int64_t)HD_TJ, n - j0);
        if (threadIdx.x < jn) {
            cs[threadIdx.x] = core[j0 + threadIdx.x];
            ms[threadIdx.x] = comp[j0 + threadIdx.x];
        }
        __syncthreads();
        if (!live) continue;
        for (int jj = 0; jj < jn; ++jj) {
            if (ms[jj] == mi) continue;
            const double cj = cs[jj];
            const double m = cj > ci ? cj : ci;
            if (!(m < bw)) continue;                  // w >= m: cannot beat the best, and a tie never replaces
            const double d2 = hd_d2<DMAX>(xi, xs + jj * DMAX, dim);
            if (d2 >= thr) continue;                  // d^2 >= RU(bw^2) >= bw^2, so RN(sqrt(d^2)) >= bw
            const double s = __dsqrt_rn(d2);
            const double w = s > m ? s : m;
            if (w < bw) {
                bw = w;
                bj = (int32_t)(j0 + jj);
                thr = __dmul_ru(bw, bw);
            }
        }
    }
    if (!live) return;
    row_w[i] = bw;
    row_j[i] = bj;
    atomicMin(&comp_w[mi], (unsigned long long)__double_as_longlong(bw));
}

__global__ void hd_comp_key(const double* __restrict__ row_w, const int32_t* __restrict__ row_j, const int32_t* __restrict__ comp,
                            const unsigned long long* __restrict__ comp_w, unsigned long long* __restrict__ comp_key, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t c = comp[i];
    if ((unsigned long long)__double_as_longlong(row_w[i]) == comp_w[c]) atomicMin(&comp_key[c], hd_key(i, row_j[i]));
}

__global__ void hd_link(const int32_t* __restrict__ comp, const int32_t* __restrict__ succ, int32_t* __restrict__ par,
                        const unsigned long long* __restrict__ comp_w, const unsigned long long* __restrict__ comp_key,
                        unsigned long long* __restrict__ edge_key, unsigned long long* __restrict__ edge_w, int64_t n,
                        HdStatus* __restrict__ st) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n || comp[c] != c) return;
    const int32_t o = succ[c];
    if (succ[o] == c && c < o) {
        par[c] = (int32_t)c;
        return;
    }
    par[c] = o;
    const unsigned long long pos = atomicAdd(&st->n_edges, 1ull);
    edge_key[pos] = comp_key[c];
    edge_w[pos] = comp_w[c];
}

__global__ void hd_unpack(const unsigned long long* __restrict__ key, const unsigned long long* __restrict__ wbits, int64_t m,
                          int32_t* __restrict__ edges, double* __restrict__ weights) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    edges[2 * e] = (int32_t)(key[e] >> 32);
    edges[2 * e + 1] = (int32_t)(key[e] & 0xffffffffull);
    weights[e] = __longlong_as_double((long long)wbits[e]);
}

template <int DMAX>
void hd_launch_core(unsigned blocks, cudaStream_t st, const float* x, int64_t n, int dim, int k, double* core) {
    hd_core<DMAX><<<blocks, HD_THREADS, 0, st>>>(x, n, dim, k, core);
}

template <int DMAX>
void hd_launch_round(unsigned blocks, cudaStream_t st, const float* x, int64_t n, int dim, const double* core,
                     const int32_t* comp, double* row_w, int32_t* row_j, unsigned long long* comp_w) {
    hd_round<DMAX><<<blocks, HD_THREADS, 0, st>>>(x, n, dim, core, comp, row_w, row_j, comp_w);
}

}  // namespace

extern "C" int kb_hdbscan_mst(kb_ctx* ctx, int64_t n, int32_t dim, const float* d_x, int32_t core_k, double* d_core,
                              int32_t* d_edges, double* d_weights) {
    KB_CHECK_ARG(ctx && d_x && d_core && d_edges && d_weights, "null pointer");
    KB_CHECK_ARG(n >= 2 && n <= INT32_MAX, "n (2 <= n < 2^31)");
    KB_CHECK_ARG(dim >= 1, "dim must be >= 1");
    KB_CHECK_ARG(core_k >= 1 && core_k <= n, "core_k (1 <= core_k <= n)");
    if (dim > HD_DIM_MAX) { kb_set_error("hdbscan mst: dim = %d, this build serves 1..%d", dim, HD_DIM_MAX); return KB_EUNSUPPORTED; }
    if (core_k > HD_KMAX) { kb_set_error("hdbscan mst: core_k = %d, this build serves 1..%d", core_k, HD_KMAX); return KB_EUNSUPPORTED; }
    KB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    cudaMemPool_t pool;
    { int rc = kb_pool_get(ctx, &pool); if (rc) return rc; }
    PoolBuf status(pool, st), comp(pool, st), succ(pool, st), par(pool, st), row_w(pool, st), row_j(pool, st),
        comp_w(pool, st), comp_key(pool, st), ek(pool, st), ew(pool, st), ek2(pool, st), ew2(pool, st), sort_tmp(pool, st);
    KB_CUDA(status.alloc(sizeof(HdStatus)));
    KB_CUDA(cudaMemsetAsync(status.p, 0, sizeof(HdStatus), st));
    HdStatus* d_st = status.as<HdStatus>();
    const int64_t total = n * dim;
    const unsigned row_blocks = (unsigned)((n + HD_THREADS - 1) / HD_THREADS);
    const unsigned flat_blocks = (unsigned)((n + 255) / 256);
    const int dmax = dim <= 2 ? 2 : dim <= 4 ? 4 : dim <= 8 ? 8 : dim <= 16 ? 16 : dim <= 32 ? 32 : 64;
    // 0. input check and core distances, then the first host synchronisation
    hd_check<<<(unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 16), 256, 0, st>>>(d_x, total, d_st);
    ctx->launches += 1;
    {
        KbTimer t(ctx, 9);
        auto core = dmax == 2 ? hd_launch_core<2> : dmax == 4 ? hd_launch_core<4> : dmax == 8 ? hd_launch_core<8>
                  : dmax == 16 ? hd_launch_core<16> : dmax == 32 ? hd_launch_core<32> : hd_launch_core<64>;
        core(row_blocks, st, d_x, n, dim, core_k, d_core);
        ctx->launches += 1;
    }
    KB_CUDA(cudaGetLastError());
    HdStatus h;
    KB_CUDA(cudaMemcpyAsync(&h, d_st, sizeof(HdStatus), cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    if (h.flags & HD_BAD_X) { kb_set_error("hdbscan mst: a coordinate is not finite"); return KB_EINVAL; }
    // 1. Boruvka rounds
    KB_CUDA(comp.alloc((size_t)n * 4)); KB_CUDA(succ.alloc((size_t)n * 4)); KB_CUDA(par.alloc((size_t)n * 4));
    KB_CUDA(row_w.alloc((size_t)n * 8)); KB_CUDA(row_j.alloc((size_t)n * 4));
    KB_CUDA(comp_w.alloc((size_t)n * 8)); KB_CUDA(comp_key.alloc((size_t)n * 8));
    KB_CUDA(ek.alloc((size_t)(n - 1) * 8)); KB_CUDA(ew.alloc((size_t)(n - 1) * 8));
    hd_iota<<<flat_blocks, 256, 0, st>>>(comp.as<int32_t>(), n);
    ctx->launches += 1;
    auto round = dmax == 2 ? hd_launch_round<2> : dmax == 4 ? hd_launch_round<4> : dmax == 8 ? hd_launch_round<8>
               : dmax == 16 ? hd_launch_round<16> : dmax == 32 ? hd_launch_round<32> : hd_launch_round<64>;
    int64_t n_comp = n;
    int rounds = 0;
    while (n_comp > 1) {
        if (++rounds > 64) { kb_set_error("hdbscan mst: Boruvka did not converge"); return KB_EINVAL; }
        int jumps = 0;                 // a chain of n_comp components is at most n_comp - 1 long: ceil(log2(n_comp))
        while ((int64_t)1 << jumps < n_comp) ++jumps;                   // jumps reach every root
        {
            KbTimer t(ctx, 10);
            KB_CUDA(cudaMemsetAsync(comp_w.p, 0xff, (size_t)n * 8, st));
            KB_CUDA(cudaMemsetAsync(comp_key.p, 0xff, (size_t)n * 8, st));
            KB_CUDA(cudaMemsetAsync(&d_st->n_comp, 0, 8, st));
            round(row_blocks, st, d_x, n, dim, d_core, comp.as<int32_t>(), row_w.as<double>(), row_j.as<int32_t>(),
                  comp_w.as<unsigned long long>());
            hd_comp_key<<<flat_blocks, 256, 0, st>>>(row_w.as<double>(), row_j.as<int32_t>(), comp.as<int32_t>(),
                                                     comp_w.as<unsigned long long>(), comp_key.as<unsigned long long>(), n);
            hd_hook<<<flat_blocks, 256, 0, st>>>(comp.as<int32_t>(), comp_key.as<unsigned long long>(), succ.as<int32_t>(), n);
            hd_link<<<flat_blocks, 256, 0, st>>>(comp.as<int32_t>(), succ.as<int32_t>(), par.as<int32_t>(),
                                                 comp_w.as<unsigned long long>(), comp_key.as<unsigned long long>(),
                                                 ek.as<unsigned long long>(), ew.as<unsigned long long>(), n, d_st);
            for (int s = 0; s < jumps; ++s) hd_jump<<<flat_blocks, 256, 0, st>>>(comp.as<int32_t>(), par.as<int32_t>(), n);
            hd_relabel<<<flat_blocks, 256, 0, st>>>(comp.as<int32_t>(), par.as<int32_t>(), n, &d_st->n_comp);
            ctx->launches += 5 + jumps;
        }
        KB_CUDA(cudaGetLastError());
        KB_CUDA(cudaMemcpyAsync(&h, d_st, sizeof(HdStatus), cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        if (h.n_comp == 0 || (int64_t)h.n_comp >= n_comp || h.n_edges != (unsigned long long)(n - (int64_t)h.n_comp)) {
            kb_set_error("hdbscan mst: round %d left %llu components and %llu edges", rounds, h.n_comp, h.n_edges);
            return KB_EINVAL;
        }
        n_comp = (int64_t)h.n_comp;
    }
    // 2. the canonical order: by (min, max), then stably by the weight bits
    {
        KbTimer t(ctx, 11);
        const int64_t m = n - 1;
        KB_CUDA(ek2.alloc((size_t)m * 8)); KB_CUDA(ew2.alloc((size_t)m * 8));
        unsigned long long *k0 = ek.as<unsigned long long>(), *w0 = ew.as<unsigned long long>();
        unsigned long long *k1 = ek2.as<unsigned long long>(), *w1 = ew2.as<unsigned long long>();
        size_t tb0 = 0, tb1 = 0;
        KB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb0, k0, k1, w0, w1, m, 0, 64, st));
        KB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb1, w1, w0, k1, k0, m, 0, 64, st));
        KB_CUDA(sort_tmp.alloc(std::max(tb0, tb1)));
        KB_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp.p, tb0, k0, k1, w0, w1, m, 0, 64, st));
        KB_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp.p, tb1, w1, w0, k1, k0, m, 0, 64, st));
        hd_unpack<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(k0, w0, m, d_edges, d_weights);
        ctx->launches += 3;
        KB_CUDA(cudaGetLastError());
    }
    return KB_OK;
}

// ---------------------------------------------------------------------------------------------
// host: scikit-learn 1.9.0's make_single_linkage (_linkage.pyx) and, from _tree.pyx, _condense_tree,
// _compute_stability, _get_clusters (eom), _do_labelling and get_probabilities, with their fp64 operation and
// summation order.  No FMA: x86-64's baseline has none, and the build does not enable it.
// ---------------------------------------------------------------------------------------------
namespace {

struct Cond { int64_t parent, child; double value; int64_t size; };

// bfs_from_hierarchy: level by level from root; an internal node x (>= n) has children hier[x - n]
void hd_bfs(const std::vector<int64_t>& left, const std::vector<int64_t>& right, int64_t n, int64_t root,
            std::vector<int64_t>& out) {
    out.clear();
    std::vector<int64_t> q{root}, next;
    while (!q.empty()) {
        out.insert(out.end(), q.begin(), q.end());
        next.clear();
        for (int64_t x : q)
            if (x >= n) { next.push_back(left[x - n]); next.push_back(right[x - n]); }
        q.swap(next);
    }
}

// sklearn's TreeUnionFind (union by rank, find with path compression)
struct TreeUF {
    std::vector<int64_t> parent, rank;
    explicit TreeUF(int64_t size) : parent(size), rank(size, 0) { for (int64_t i = 0; i < size; ++i) parent[i] = i; }
    int64_t find(int64_t x) {
        int64_t r = x;
        while (parent[r] != r) r = parent[r];
        while (parent[x] != r) { int64_t nx = parent[x]; parent[x] = r; x = nx; }
        return r;
    }
    void unite(int64_t x, int64_t y) {
        const int64_t xr = find(x), yr = find(y);
        if (rank[xr] < rank[yr]) parent[xr] = yr;
        else if (rank[xr] > rank[yr]) parent[yr] = xr;
        else { parent[yr] = xr; rank[xr] += 1; }
    }
};

}  // namespace

extern "C" int kb_hdbscan_labels(int64_t n, const int32_t* edges, const double* weights, int32_t min_cluster_size,
                                 int32_t allow_single_cluster, int32_t* labels, double* probabilities, int64_t* n_clusters) {
    KB_CHECK_ARG(edges && weights && labels && probabilities && n_clusters, "null pointer");
    KB_CHECK_ARG(n >= 2 && n <= INT32_MAX, "n (2 <= n < 2^31)");
    KB_CHECK_ARG(min_cluster_size >= 2, "min_cluster_size must be >= 2");
    const int64_t m = n - 1;
    for (int64_t e = 0; e < m; ++e) {
        const int64_t a = edges[2 * e], b = edges[2 * e + 1];
        const double w = weights[e];
        if (a < 0 || b >= n || !(a < b)) { kb_set_error("hdbscan labels: edge %lld is not (min, max) within [0, n)", (long long)e); return KB_EINVAL; }
        if (!std::isfinite(w) || w < 0.0) { kb_set_error("hdbscan labels: weight %lld is negative or not finite", (long long)e); return KB_EINVAL; }
        if (e > 0) {
            const double pw = weights[e - 1];
            const int64_t pa = edges[2 * e - 2], pb = edges[2 * e - 1];
            if (w < pw || (w == pw && (a < pa || (a == pa && b <= pb)))) {
                kb_set_error("hdbscan labels: edges %lld and %lld are not in (w, min, max) order", (long long)e - 1, (long long)e);
                return KB_EINVAL;
            }
        }
    }
    // make_single_linkage (UnionFind of _hierarchical_fast: parent -1, labels n.., fast_find with path shortcut)
    std::vector<int64_t> uf_parent(2 * n - 1, -1), uf_size(2 * n - 1, 0);
    std::fill(uf_size.begin(), uf_size.begin() + n, 1);
    std::vector<int64_t> left(m), right(m), hsize(m);
    std::vector<double> hval(m);
    auto fast_find = [&](int64_t x) {
        int64_t p = x;
        while (uf_parent[x] != -1) x = uf_parent[x];
        // sklearn's loop, entered at a root, also writes parent[-1] (wraparound: label 2n - 2, which no find reaches
        // before the last union creates it); stopping at the root leaves every result the same
        while (p != x && uf_parent[p] != x) { const int64_t np = uf_parent[p]; uf_parent[p] = x; p = np; }
        return x;
    };
    int64_t next_label = n;
    for (int64_t e = 0; e < m; ++e) {
        const int64_t ca = fast_find(edges[2 * e]), cb = fast_find(edges[2 * e + 1]);
        if (ca == cb) { kb_set_error("hdbscan labels: edge %lld closes a cycle", (long long)e); return KB_EINVAL; }
        left[e] = ca; right[e] = cb; hval[e] = weights[e];
        hsize[e] = uf_size[ca] + uf_size[cb];
        uf_parent[ca] = next_label; uf_parent[cb] = next_label;
        uf_size[next_label] = hsize[e];
        ++next_label;
    }
    // _condense_tree
    const int64_t root = 2 * m, mcs = min_cluster_size;
    std::vector<int64_t> node_list, sub;
    hd_bfs(left, right, n, root, node_list);
    std::vector<int64_t> relabel(root + 1, 0);
    std::vector<uint8_t> ignore(node_list.size(), 0);
    relabel[root] = n;
    int64_t nlabel = n + 1;
    std::vector<Cond> ct;
    ct.reserve((size_t)(2 * n));
    auto shed = [&](int64_t parent, int64_t from, double lam) {
        hd_bfs(left, right, n, from, sub);
        for (int64_t s : sub) {
            if (s < n) ct.push_back({parent, s, lam, 1});
            ignore[s] = 1;
        }
    };
    for (int64_t node : node_list) {
        if (ignore[node] || node < n) continue;
        const int64_t h = node - n, l = left[h], r = right[h];
        const double dist = hval[h];
        const double lam = dist > 0.0 ? 1.0 / dist : INFINITY;
        const int64_t lc = l >= n ? hsize[l - n] : 1, rc = r >= n ? hsize[r - n] : 1;
        if (lc >= mcs && rc >= mcs) {
            relabel[l] = nlabel++;
            ct.push_back({relabel[node], relabel[l], lam, lc});
            relabel[r] = nlabel++;
            ct.push_back({relabel[node], relabel[r], lam, rc});
        } else if (lc < mcs && rc < mcs) {
            shed(relabel[node], l, lam);
            shed(relabel[node], r, lam);
        } else if (lc < mcs) {
            relabel[r] = relabel[node];
            shed(relabel[node], l, lam);
        } else {
            relabel[l] = relabel[node];
            shed(relabel[node], r, lam);
        }
    }
    // _compute_stability
    int64_t largest_child = 0, smallest = INT64_MAX, largest_parent = 0;
    for (const Cond& c : ct) {
        largest_child = std::max(largest_child, c.child);
        smallest = std::min(smallest, c.parent);
        largest_parent = std::max(largest_parent, c.parent);
    }
    largest_child = std::max(largest_child, smallest);
    const int64_t n_ids = largest_parent - smallest + 1;
    std::vector<double> births(largest_child + 1, NAN), stability(n_ids, 0.0);
    for (const Cond& c : ct) births[c.child] = c.value;
    births[smallest] = 0.0;
    for (const Cond& c : ct) stability[c.parent - smallest] += (c.value - births[c.parent]) * (double)c.size;
    // _get_clusters, eom: ids descending (children before parents); a node either gives way to its children's summed
    // stability or is kept, and a kept node deselects everything below it.  is_cluster[x] ends true iff x was kept and
    // no ancestor was.
    std::vector<int64_t> kid0(n_ids, -1), kid1(n_ids, -1), up(n_ids, -1);
    for (const Cond& c : ct)
        if (c.size > 1) {
            const int64_t p = c.parent - smallest;
            (kid0[p] < 0 ? kid0[p] : kid1[p]) = c.child;
            up[c.child - smallest] = p;
        }
    std::vector<uint8_t> kept(n_ids, 0);
    const int64_t lowest = allow_single_cluster ? 0 : 1;      // the root is excluded unless allow_single_cluster
    for (int64_t id = n_ids - 1; id >= lowest; --id) {
        double sub_stab = 0.0;
        if (kid0[id] >= 0) sub_stab = stability[kid0[id] - smallest];
        if (kid1[id] >= 0) sub_stab = sub_stab + stability[kid1[id] - smallest];
        if (sub_stab > stability[id]) stability[id] = sub_stab;
        else kept[id] = 1;
    }
    std::vector<uint8_t> selected(n_ids, 0);
    std::vector<uint8_t> under(n_ids, 0);                       // a kept ancestor exists
    std::vector<int64_t> cluster_label(n_ids, -1);
    int64_t n_sel = 0;
    for (int64_t id = 0; id < n_ids; ++id) {                    // parents before children
        if (up[id] >= 0) under[id] = under[up[id]] || selected[up[id]];
        if (id >= lowest && kept[id] && !under[id]) { selected[id] = 1; cluster_label[id] = n_sel++; }
    }
    // _do_labelling
    TreeUF uf(largest_parent + 1);
    for (const Cond& c : ct)
        if (!(c.child >= smallest && c.child <= largest_parent && selected[c.child - smallest])) uf.unite(c.parent, c.child);
    double root_threshold = -INFINITY;
    std::vector<double> point_lambda;
    if (n_sel == 1 && allow_single_cluster) {
        point_lambda.assign(n, 0.0);
        bool first = true;
        for (const Cond& c : ct) {
            if (c.child < n) point_lambda[c.child] = c.value;
            if (c.parent == smallest) {
                if (first || c.value > root_threshold) root_threshold = c.value;      // numpy's max
                first = false;
            }
        }
    }
    for (int64_t p = 0; p < n; ++p) {
        const int64_t c = uf.find(p);
        int64_t label = -1;
        if (c != smallest) {
            label = cluster_label[c - smallest];
        } else if (n_sel == 1 && allow_single_cluster) {
            if (point_lambda[p] >= root_threshold) {
                // Only the root can be the one selected cluster here: a root that gives way has two cluster children,
                // and EOM keeps at least one cluster below each.  sklearn would raise a KeyError otherwise.
                if (!selected[0]) {
                    kb_set_error("hdbscan labels: internal inconsistency: point %lld joins the root, which is not the "
                                 "selected cluster", (long long)p);
                    return KB_EINVAL;
                }
                label = cluster_label[0];
            }
        }
        labels[p] = (int32_t)label;
    }
    // get_probabilities: max_lambdas keeps, per parent, the maximum of its LAST run of consecutive rows
    std::vector<double> deaths(largest_parent + 1, 0.0);
    int64_t cur = ct[0].parent;
    double mx = ct[0].value;
    for (size_t r = 1; r < ct.size(); ++r) {
        if (ct[r].parent == cur) { if (ct[r].value > mx) mx = ct[r].value; }
        else { deaths[cur] = mx; cur = ct[r].parent; mx = ct[r].value; }
    }
    deaths[cur] = mx;
    std::vector<int64_t> label_cluster(n_sel);
    for (int64_t id = 0; id < n_ids; ++id) if (selected[id]) label_cluster[cluster_label[id]] = id + smallest;
    std::fill(probabilities, probabilities + n, 0.0);
    for (const Cond& c : ct) {
        if (c.child >= smallest) continue;
        const int32_t lab = labels[c.child];
        if (lab == -1) continue;
        const double max_lambda = deaths[label_cluster[lab]];
        if (max_lambda == 0.0 || std::isinf(c.value)) probabilities[c.child] = 1.0;
        else probabilities[c.child] = (max_lambda < c.value ? max_lambda : c.value) / max_lambda;
    }
    *n_clusters = n_sel;
    return KB_OK;
}
