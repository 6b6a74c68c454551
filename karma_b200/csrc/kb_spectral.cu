// kb_spectral.cu -- K10: UMAP's spectral initialisation over the pruned fuzzy graph (the stage between K7 and K8).
//
// Replaces umap.spectral.spectral_layout of umap-learn 0.3.9 (UMAP.fit's init="spectral"), disconnected graphs
// included.  Rules frozen in oracle/umap_spectral_oracle.py:
//   * the graph is pruned with K8's rule (w >= max / n_epochs); its weakly connected components are numbered in the
//     order of their smallest vertex (scipy.sparse.csgraph.connected_components);
//   * a connected graph, and every component of at least 2 * dim vertices of a disconnected one, gets the unit
//     eigenvectors of the dim smallest non-trivial eigenvalues of L = I - D^-1/2 W D^-1/2 (D: degrees), each with its
//     largest-|.| entry positive (scikit-learn's _deterministic_vector_sign_flip);
//   * a disconnected graph places its components around meta points: with more than 2 * dim components, the spectral
//     embedding of the components' float32 centroids under exp(-d^2) (scikit-learn 1.9.0's spectral_embedding: the
//     diagonal ignored, eigenvectors divided by sqrt(degree), sign flipped, the first dropped), over its global max;
//     otherwise the rows of [eye(k), 0; -eye(k), 0], k = ceil(n_comp / 2);
//   * data_range of a component is half the smallest positive euclidean distance from its meta point to the others,
//     in fp64, coordinate order, no FMA (0.3.9 takes it from pairwise_distances, whose self-distance is often not 0:
//     DESIGN §3 K10); a solved component is scaled to data_range / max|v| and offset by its meta point, every other one
//     is data_range * uniform(-1, 1) + meta, with the uniform draws taken on the host from umap's random_state.
// GPU formulation:
//   kb_csr_check, sp_keep   validation; kept edges per row and the fp64 degree (CSR order)
//   components   hooking rounds (kb_common.cuh's union-find): every component hooks along its minimum kept edge
//                (min << 32 | max), one host read per round; labels from the smallest vertex and a scan
//   sp_perm_*    vertices sorted by (label, vertex) with CUB: every component is a contiguous block of a permuted CSR
//                of M = D^-1/2 W D^-1/2
//   eigensolve   one fp64 Lanczos driver (full reorthogonalisation, twice; thick restart) for the largest eigenvalues of
//                M on the complement of the trivial vector D^1/2 1, serving the component SpMV and the dense meta
//                matvec; dot products are fixed-order two-stage reductions; the Ritz problems are solved on the host
//                by cyclic Jacobi, so the same inputs give the same bits
//   meta         sp_centroid (float32 sums in row order), sp_affinity (16 x 16 tiles), sp_meta_deg, the dense solve;
//                sp_range: every component against every meta point (shared-memory tiles, dim <= 64)
//   sp_assemble  the float32 [N, dim] layout, after the host has drawn its uniforms
#include "kb_common.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <cmath>
#include <vector>

namespace {

constexpr int SP_THREADS = 256;
constexpr int SP_DIM_MAX = 64;
constexpr int64_t SP_META_MAX = 65536;     // n_comp^2 fp64 of dense affinity: 34 GB at the limit
constexpr int SP_RESTART_CAP = 500;        // thick restarts per solve before a component counts as not converged
constexpr double SP_TOL = 1e-9;            // Ritz residual bound ||M v - theta v|| of every returned vector
constexpr double SP_BREAK = 1e-10;         // a Lanczos step whose new direction is shorter spans an invariant subspace
constexpr int64_t SP_DOT_CHUNK = 8192;
constexpr unsigned SP_BAD_X = 8u, SP_ZERO_AFFINITY = 16u;   // above kb_csr_check's KB_CSR_BAD_* bits
enum { SP_DRAW = 0, SP_SOLVED = 1, SP_NOT_CONVERGED = 2 };

struct SpStatus {
    unsigned long long flags;
    unsigned long long wmax_bits;
    unsigned long long hooks;
    unsigned long long n_comp;
};

__host__ __device__ __forceinline__ uint64_t sp_mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

__device__ __forceinline__ double sp_threshold(const SpStatus* st, int n_epochs) {
    return n_epochs > 0 ? __ddiv_rn(__longlong_as_double((long long)st->wmax_bits), (double)n_epochs) : 0.0;
}

__global__ void sp_check_x(const void* __restrict__ x, int f64, int64_t total, SpStatus* __restrict__ st) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const float v = f64 ? (float)((const double*)x)[t] : ((const float*)x)[t];
        if (!isfinite(v)) { atomicOr(&st->flags, (unsigned long long)SP_BAD_X); return; }
    }
}

// kept edges per row and the degree (kept weights summed in CSR order)
__global__ void sp_keep(const int64_t* __restrict__ indptr, const double* __restrict__ data, int64_t n, int n_epochs,
                        const SpStatus* __restrict__ st, int64_t* __restrict__ row_kept, double* __restrict__ deg) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const double thr = sp_threshold(st, n_epochs);
    int64_t k = 0;
    double s = 0.0;
    for (int64_t e = indptr[r]; e < indptr[r + 1]; ++e)
        if (data[e] >= thr) { ++k; s = __dadd_rn(s, data[e]); }
    row_kept[r] = k;
    deg[r] = s;
}

// every component's minimum kept edge to another component (both ends: weak connectivity)
__global__ void sp_edge_min(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                            const double* __restrict__ data, int64_t n, int n_epochs, const SpStatus* __restrict__ st,
                            const int32_t* __restrict__ comp, unsigned long long* __restrict__ comp_key) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const double thr = sp_threshold(st, n_epochs);
    const int32_t cr = comp[r];
    unsigned long long best = ~0ull;
    for (int64_t e = indptr[r]; e < indptr[r + 1]; ++e) {
        if (data[e] < thr) continue;
        const int32_t c = indices[e];
        const int32_t cc = comp[c];
        if (cc == cr) continue;
        const unsigned long long key = hd_key(r, c);
        atomicMin(&comp_key[cc], key);
        best = key < best ? key : best;
    }
    if (best != ~0ull) atomicMin(&comp_key[cr], best);
}

// a pair that chose the same edge: the smaller id becomes the root; a component without an edge stays a root
__global__ void sp_link(const int32_t* __restrict__ comp, const int32_t* __restrict__ succ, int32_t* __restrict__ par,
                        int64_t n, SpStatus* __restrict__ st) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n || comp[c] != c) return;
    const int32_t o = succ[c];
    if (o == c) { par[c] = (int32_t)c; return; }
    atomicAdd(&st->hooks, 1ull);
    par[c] = succ[o] == c && c < o ? (int32_t)c : o;
}

__global__ void sp_min_vertex(const int32_t* __restrict__ comp, int64_t n, int32_t* __restrict__ minv) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicMin(&minv[comp[i]], (int32_t)i);
}

__global__ void sp_first(const int32_t* __restrict__ comp, const int32_t* __restrict__ minv, int64_t n, int32_t* __restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = minv[comp[i]] == i ? 1 : 0;
}

__global__ void sp_label(const int32_t* __restrict__ comp, const int32_t* __restrict__ minv, const int32_t* __restrict__ rank,
                         int64_t n, int32_t* __restrict__ label, int32_t* __restrict__ size) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t l = rank[minv[comp[i]]];
    label[i] = l;
    atomicAdd(&size[l], 1);
}

__global__ void sp_perm_count(const int32_t* __restrict__ perm, const int64_t* __restrict__ row_kept, int64_t n,
                              int32_t* __restrict__ pos, int64_t* __restrict__ cnt) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int32_t r = perm[t];
    pos[r] = (int32_t)t;
    cnt[t] = row_kept[r];
}

// the permuted CSR of M: row t is vertex perm[t], columns are permuted positions, values (w / sqrt(d_r)) / sqrt(d_c)
__global__ void sp_perm_fill(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                             const double* __restrict__ data, int64_t n, int n_epochs, const SpStatus* __restrict__ st,
                             const int32_t* __restrict__ perm, const int32_t* __restrict__ pos, const double* __restrict__ deg,
                             const int64_t* __restrict__ pindptr, int32_t* __restrict__ pidx, double* __restrict__ pval) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const double thr = sp_threshold(st, n_epochs);
    const int32_t r = perm[t];
    const double sr = __dsqrt_rn(deg[r]);
    int64_t o = pindptr[t];
    for (int64_t e = indptr[r]; e < indptr[r + 1]; ++e) {
        const double w = data[e];
        if (w < thr) continue;
        const int32_t c = indices[e];
        pidx[o] = pos[c];
        pval[o] = __ddiv_rn(__ddiv_rn(w, sr), __dsqrt_rn(deg[c]));
        ++o;
    }
}

// ---- the Lanczos driver's kernels ----
// y = M x over the rows [row0, row0 + n) of the permuted CSR (one component's block)
__global__ void sp_spmv(const int64_t* __restrict__ pindptr, const int32_t* __restrict__ pidx, const double* __restrict__ pval,
                        int64_t row0, int64_t n, const double* __restrict__ x, double* __restrict__ y) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    double s = 0.0;
    for (int64_t e = pindptr[row0 + t]; e < pindptr[row0 + t + 1]; ++e) s += pval[e] * x[pidx[e] - row0];
    y[t] = s;
}

// y = A x for a dense row-major n x n matrix: a warp per row, lanes strided, a fixed butterfly
__global__ void sp_densemv(const double* __restrict__ a, int64_t n, const double* __restrict__ x, double* __restrict__ y) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const double* ar = a + row * n;
    double s = 0.0;
    for (int64_t b = lane; b < n; b += 32) s += ar[b] * x[b];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) y[row] = s;
}

// part[b * ncols + j] = sum over the rows of chunk b of V[j * n + r] * w[r]
__global__ void __launch_bounds__(SP_THREADS) sp_dots_part(const double* __restrict__ v, int64_t n, int ncols,
                                                           const double* __restrict__ w, double* __restrict__ part) {
    typedef cub::BlockReduce<double, SP_THREADS> Red;
    __shared__ typename Red::TempStorage tmp;
    const int64_t r0 = (int64_t)blockIdx.x * SP_DOT_CHUNK, r1 = min(n, r0 + SP_DOT_CHUNK);
    const double* vj = v + (int64_t)blockIdx.y * n;
    double s = 0.0;
    for (int64_t r = r0 + threadIdx.x; r < r1; r += SP_THREADS) s += vj[r] * w[r];
    s = Red(tmp).Sum(s);
    if (threadIdx.x == 0) part[(int64_t)blockIdx.x * ncols + blockIdx.y] = s;
}

__global__ void sp_dots_sum(const double* __restrict__ part, int nb, int ncols, double* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ncols) return;
    double s = 0.0;
    for (int b = 0; b < nb; ++b) s += part[(int64_t)b * ncols + j];
    out[j] = s;
}

// w -= V h over the first ncols columns
__global__ void sp_sub(const double* __restrict__ v, int64_t n, int ncols, const double* __restrict__ h, double* __restrict__ w) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double s = 0.0;
    for (int j = 0; j < ncols; ++j) s += v[(int64_t)j * n + r] * h[j];
    w[r] -= s;
}

__global__ void sp_scale(const double* __restrict__ x, int64_t n, double d, double* __restrict__ y) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) y[t] = x[t] / d;
}

__global__ void sp_random(double* __restrict__ x, int64_t n, uint64_t seed) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) x[t] = (double)(sp_mix64(seed ^ sp_mix64((uint64_t)t)) >> 11) * 0x1p-52 - 1.0;
}

// out[c * n + r] = sum_j V[(j + 1) * n + r] * Y[j * k + c], j < m: Ritz vectors from the basis
__global__ void sp_combine(const double* __restrict__ v, int64_t n, int m, const double* __restrict__ y, int k, double* __restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (r >= n) return;
    double s = 0.0;
    for (int j = 0; j < m; ++j) s += v[(int64_t)(j + 1) * n + r] * y[j * k + c];
    out[(int64_t)c * n + r] = s;
}

// per column of x (n x k, column-major): squared norm
__global__ void __launch_bounds__(SP_THREADS) sp_colnorm2(const double* __restrict__ x, int64_t n, double* __restrict__ out) {
    typedef cub::BlockReduce<double, SP_THREADS> Red;
    __shared__ typename Red::TempStorage tmp;
    const double* xc = x + (int64_t)blockIdx.x * n;
    double s = 0.0;
    for (int64_t r = threadIdx.x; r < n; r += SP_THREADS) s += xc[r] * xc[r];
    s = Red(tmp).Sum(s);
    if (threadIdx.x == 0) out[blockIdx.x] = s;
}

__global__ void sp_colscale(double* __restrict__ x, int64_t n, int k, const double* __restrict__ norm2) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * k) return;
    x[t] = x[t] / __dsqrt_rn(norm2[t / n]);
}

struct SpArg { double a; double v; int64_t i; };
struct SpArgMax {                          // the largest |v|, the first such index on ties (numpy's argmax)
    __device__ __forceinline__ SpArg operator()(const SpArg& x, const SpArg& y) const {
        return (x.a > y.a || (x.a == y.a && x.i < y.i)) ? x : y;
    }
};

__global__ void __launch_bounds__(SP_THREADS) sp_colargmax(const double* __restrict__ x, int64_t n, double* __restrict__ val) {
    typedef cub::BlockReduce<SpArg, SP_THREADS> Red;
    __shared__ typename Red::TempStorage tmp;
    const double* xc = x + (int64_t)blockIdx.x * n;
    SpArg b{-1.0, 0.0, INT64_MAX};
    for (int64_t r = threadIdx.x; r < n; r += SP_THREADS) {
        const double a = fabs(xc[r]);
        if (a > b.a) b = SpArg{a, xc[r], r};
    }
    b = Red(tmp).Reduce(b, SpArgMax());
    if (threadIdx.x == 0) { val[2 * blockIdx.x] = b.v; val[2 * blockIdx.x + 1] = b.a; }
}

// a component's vectors, signs fixed, into vertex order: vec[perm[row0 + t] * dim + c]
__global__ void sp_vec_out(const double* __restrict__ x, int64_t n, int k, const double* __restrict__ sgn,
                           const int32_t* __restrict__ perm, int64_t row0, double* __restrict__ vec) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * k) return;
    const int64_t r = t % n;
    const int c = (int)(t / n);
    vec[(int64_t)perm[row0 + r] * k + c] = x[t] * sgn[c];
}

__global__ void sp_sqrt_deg(const double* __restrict__ deg, const int32_t* __restrict__ perm, int64_t row0, int64_t n,
                            double* __restrict__ q) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) q[t] = __dsqrt_rn(deg[perm ? perm[row0 + t] : t]);
}

// ---- meta-embedding ----
// numpy's float32 mean(axis=0) of a component's rows: float32 sum in row order, then the division
__global__ void sp_centroid(const void* __restrict__ x, int f64, int64_t cols, const int32_t* __restrict__ perm,
                            const int64_t* __restrict__ off, const int32_t* __restrict__ size, int64_t n_comp,
                            double* __restrict__ cent) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_comp * cols) return;
    const int64_t c = t / cols, d = t - c * cols;
    float s = 0.f;
    for (int64_t p = off[c]; p < off[c] + size[c]; ++p) {
        const int64_t at = (int64_t)perm[p] * cols + d;
        s = __fadd_rn(s, f64 ? (float)((const double*)x)[at] : ((const float*)x)[at]);
    }
    cent[t] = (double)__double2float_rn(__ddiv_rn((double)s, (double)size[c]));
}

// a[i][j] = exp(-d^2(i, j)), 0 on the diagonal; d^2 in fp64, coordinate order, no FMA
constexpr int SP_TILE = 16;
__global__ void __launch_bounds__(SP_TILE * SP_TILE) sp_affinity(const double* __restrict__ cent, int64_t n, int64_t cols,
                                                                 double* __restrict__ a, SpStatus* __restrict__ st) {
    __shared__ double si[SP_TILE][SP_TILE + 1], sj[SP_TILE][SP_TILE + 1];
    const int tx = threadIdx.x % SP_TILE, ty = threadIdx.x / SP_TILE;
    const int64_t i = (int64_t)blockIdx.y * SP_TILE + ty, j = (int64_t)blockIdx.x * SP_TILE + tx;
    double d2 = 0.0;
    for (int64_t d0 = 0; d0 < cols; d0 += SP_TILE) {
        const int64_t li = (int64_t)blockIdx.y * SP_TILE + ty, lj = (int64_t)blockIdx.x * SP_TILE + ty;
        si[ty][tx] = li < n && d0 + tx < cols ? cent[li * cols + d0 + tx] : 0.0;
        sj[ty][tx] = lj < n && d0 + tx < cols ? cent[lj * cols + d0 + tx] : 0.0;
        __syncthreads();
        const int dn = (int)min((int64_t)SP_TILE, cols - d0);
        for (int k = 0; k < dn; ++k) {
            const double df = __dsub_rn(si[ty][k], sj[tx][k]);
            d2 = __dadd_rn(d2, __dmul_rn(df, df));
        }
        __syncthreads();
    }
    if (i >= n || j >= n) return;
    const double v = i == j ? 0.0 : exp(-d2);
    if (i != j && !(v > 0.0)) atomicOr(&st->flags, (unsigned long long)SP_ZERO_AFFINITY);
    a[i * n + j] = v;
}

// degree of every meta point (its row summed in a fixed order), then a[i][j] <- (a[i][j] / sqrt(d_j)) / sqrt(d_i)
__global__ void __launch_bounds__(SP_THREADS) sp_rowsum(const double* __restrict__ a, int64_t n, double* __restrict__ deg) {
    typedef cub::BlockReduce<double, SP_THREADS> Red;
    __shared__ typename Red::TempStorage tmp;
    const double* ar = a + (int64_t)blockIdx.x * n;
    double s = 0.0;
    for (int64_t j = threadIdx.x; j < n; j += SP_THREADS) s += ar[j];
    s = Red(tmp).Sum(s);
    if (threadIdx.x == 0) deg[blockIdx.x] = s;
}

__global__ void sp_normalise(double* __restrict__ a, int64_t n, const double* __restrict__ deg) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * n) return;
    const int64_t i = t / n, j = t - i * n;
    a[t] = __ddiv_rn(__ddiv_rn(a[t], __dsqrt_rn(deg[j])), __dsqrt_rn(deg[i]));
}

// half the smallest positive euclidean distance from meta point c to the others (NaN when there is none)
constexpr int SP_RJ = 64;
template <int DMAX>
__global__ void __launch_bounds__(SP_THREADS) sp_range(const double* __restrict__ meta, int64_t n, int dim, double* __restrict__ range) {
    __shared__ double ms[SP_RJ * DMAX];
    const int64_t c = (int64_t)blockIdx.x * SP_THREADS + threadIdx.x;
    const bool live = c < n;
    double mc[DMAX];
#pragma unroll
    for (int d = 0; d < DMAX; ++d) mc[d] = live && d < dim ? meta[c * dim + d] : 0.0;
    double best = INFINITY;
    for (int64_t j0 = 0; j0 < n; j0 += SP_RJ) {
        const int jn = (int)min((int64_t)SP_RJ, n - j0);
        __syncthreads();
        for (int t = threadIdx.x; t < jn * dim; t += SP_THREADS) ms[(t / dim) * DMAX + t % dim] = meta[j0 * dim + t];
        __syncthreads();
        if (!live) continue;
        for (int jj = 0; jj < jn; ++jj) {
            double d2 = 0.0;
#pragma unroll
            for (int d = 0; d < DMAX; ++d) {
                if (d >= dim) break;
                const double df = __dsub_rn(mc[d], ms[jj * DMAX + d]);
                d2 = __dadd_rn(d2, __dmul_rn(df, df));
            }
            if (d2 > 0.0 && d2 < best) best = d2;
        }
    }
    if (live) range[c] = best < INFINITY ? __dsqrt_rn(best) * 0.5 : NAN;
}

template <int DMAX>
void sp_launch_range(unsigned blocks, cudaStream_t st, const double* meta, int64_t n, int dim, double* range) {
    sp_range<DMAX><<<blocks, SP_THREADS, 0, st>>>(meta, n, dim, range);
}

// umap's arithmetic after each draw: fp32((low + (high - low) * u) + meta), or fp32(v * (range / max|v|) + meta)
__global__ void sp_assemble(const int32_t* __restrict__ label, const int32_t* __restrict__ status, const double* __restrict__ range,
                            const double* __restrict__ expansion, const double* __restrict__ meta, const double* __restrict__ vec,
                            const double* __restrict__ u, int64_t n, int dim, float* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * dim) return;
    const int32_t c = label[t / dim];
    const int d = (int)(t % dim);
    const bool solved = status[c] == SP_SOLVED;
    const double r = range[c];
    double v = solved ? vec[t] : __dadd_rn(-r, __dmul_rn(__dsub_rn(r, -r), u[t]));
    if (meta) v = __dadd_rn(solved ? __dmul_rn(v, expansion[c]) : v, meta[(int64_t)c * dim + d]);
    out[t] = __double2float_rn(v);
}

inline unsigned sp_blocks(int64_t n, int threads = SP_THREADS) { return (unsigned)((n + threads - 1) / threads); }

// ---- host: the Ritz problem ----
// eigenpairs of the symmetric m x m matrix a (row-major, destroyed) by cyclic Jacobi; theta descending, the vector of
// theta[i] in column i of z (row-major)
void sp_jacobi(int m, std::vector<double>& a, std::vector<double>& theta, std::vector<double>& z) {
    std::vector<double> v((size_t)m * m, 0.0);
    for (int i = 0; i < m; ++i) v[(size_t)i * m + i] = 1.0;
    for (int sweep = 0; sweep < 100; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int p = 0; p < m; ++p) {
            diag += a[(size_t)p * m + p] * a[(size_t)p * m + p];
            for (int q = p + 1; q < m; ++q) off += a[(size_t)p * m + q] * a[(size_t)p * m + q];
        }
        if (off == 0.0 || off < 1e-34 * diag) break;
        for (int p = 0; p < m - 1; ++p)
            for (int q = p + 1; q < m; ++q) {
                const double apq = a[(size_t)p * m + q];
                const double app = a[(size_t)p * m + p], aqq = a[(size_t)q * m + q];
                const double g = 100.0 * std::fabs(apq);
                if (sweep > 4 && std::fabs(app) + g == std::fabs(app) && std::fabs(aqq) + g == std::fabs(aqq)) {
                    a[(size_t)p * m + q] = a[(size_t)q * m + p] = 0.0;
                    continue;
                }
                if (apq == 0.0) continue;
                const double th = (aqq - app) / (2.0 * apq);
                double t = 1.0 / (std::fabs(th) + std::sqrt(th * th + 1.0));
                if (th < 0.0) t = -t;
                const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int r = 0; r < m; ++r) {
                    if (r == p || r == q) continue;
                    const double arp = a[(size_t)r * m + p], arq = a[(size_t)r * m + q];
                    a[(size_t)r * m + p] = a[(size_t)p * m + r] = c * arp - s * arq;
                    a[(size_t)r * m + q] = a[(size_t)q * m + r] = s * arp + c * arq;
                }
                a[(size_t)p * m + p] = app - t * apq;
                a[(size_t)q * m + q] = aqq + t * apq;
                a[(size_t)p * m + q] = a[(size_t)q * m + p] = 0.0;
                for (int r = 0; r < m; ++r) {
                    const double vrp = v[(size_t)r * m + p], vrq = v[(size_t)r * m + q];
                    v[(size_t)r * m + p] = c * vrp - s * vrq;
                    v[(size_t)r * m + q] = s * vrp + c * vrq;
                }
            }
    }
    std::vector<int> order(m);
    for (int i = 0; i < m; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return a[(size_t)x * m + x] > a[(size_t)y * m + y]; });
    theta.resize(m);
    z.assign((size_t)m * m, 0.0);
    for (int i = 0; i < m; ++i) {
        theta[i] = a[(size_t)order[i] * m + order[i]];
        for (int r = 0; r < m; ++r) z[(size_t)r * m + i] = v[(size_t)r * m + order[i]];
    }
}

// the operator: rows [row0, row0 + n) of the permuted CSR, or a dense n x n matrix
struct SpOp {
    const int64_t* pindptr; const int32_t* pidx; const double* pval; int64_t row0;
    const double* dense;
    int64_t n;
};

struct SpSolve { int64_t steps = 0, restarts = 0; bool converged = false; };

void sp_apply(const SpOp& op, cudaStream_t st, const double* x, double* y) {
    if (op.dense) sp_densemv<<<sp_blocks(op.n * 32), SP_THREADS, 0, st>>>(op.dense, op.n, x, y);
    else sp_spmv<<<sp_blocks(op.n), SP_THREADS, 0, st>>>(op.pindptr, op.pidx, op.pval, op.row0, op.n, x, y);
}

// out[0 .. ncols) = V[:, j]^T w for the first ncols columns of V (n rows), in a fixed order
void sp_dots(cudaStream_t st, const double* v, int64_t n, int ncols, const double* w, double* part, double* out) {
    const int nb = (int)((n + SP_DOT_CHUNK - 1) / SP_DOT_CHUNK);
    sp_dots_part<<<dim3(nb, ncols), SP_THREADS, 0, st>>>(v, n, ncols, w, part);
    sp_dots_sum<<<sp_blocks(ncols), SP_THREADS, 0, st>>>(part, nb, ncols, out);
}

// Lanczos with full reorthogonalisation (two Gram-Schmidt passes per step) and thick restart: the nev largest
// eigenvalues of op on the complement of q0 (unit, an eigenvector of op).  Writes the Ritz vectors, unnormalised, to
// out (n x nev, column-major), largest first.  A step whose new direction is shorter than SP_BREAK continues from a
// fresh deterministic random direction orthogonal to the basis (the Krylov space was invariant).
int sp_lanczos(kb_ctx* ctx, cudaMemPool_t pool, const SpOp& op, int nev, uint64_t seed, const double* d_q0, double* d_out,
               SpSolve* res) {
    cudaStream_t st = ctx->stream;
    const int64_t n = op.n;
    const int m = (int)std::min<int64_t>(n - 1, std::max(2 * nev + 32, 64));
    const int kk = std::max(nev, std::min(m - 1, nev + (m - nev) / 2));
    const int cols = m + 2;                                       // q0, v_0 .. v_m
    const bool complete = m == n - 1;                             // the basis can span q0's whole complement
    const int nb = (int)((n + SP_DOT_CHUNK - 1) / SP_DOT_CHUNK);
    PoolBuf V(pool, st), w(pool, st), part(pool, st), hb(pool, st), yd(pool, st), tmp(pool, st);
    KB_CUDA(V.alloc((size_t)n * cols * 8)); KB_CUDA(w.alloc((size_t)n * 8));
    KB_CUDA(part.alloc((size_t)nb * cols * 8)); KB_CUDA(hb.alloc((size_t)(2 * cols + 1) * 8));
    KB_CUDA(yd.alloc((size_t)m * m * 8)); KB_CUDA(tmp.alloc((size_t)n * kk * 8));
    double *Vp = V.as<double>(), *wp = w.as<double>(), *hp = hb.as<double>();
    KB_CUDA(cudaMemcpyAsync(Vp, d_q0, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
    std::vector<double> hh(2 * cols + 1), H((size_t)m * m, 0.0), theta, Y, ysub;
    // w <- w minus its projection on the first ncol columns, twice; returns the coefficients of both passes and |w|^2
    auto orth = [&](int ncol) -> int {
        sp_dots(st, Vp, n, ncol, wp, part.as<double>(), hp);
        sp_sub<<<sp_blocks(n), SP_THREADS, 0, st>>>(Vp, n, ncol, hp, wp);
        sp_dots(st, Vp, n, ncol, wp, part.as<double>(), hp + cols);
        sp_sub<<<sp_blocks(n), SP_THREADS, 0, st>>>(Vp, n, ncol, hp + cols, wp);
        sp_dots(st, wp, n, 1, wp, part.as<double>(), hp + 2 * cols);
        ctx->launches += 8;
        KB_CUDA(cudaGetLastError());
        KB_CUDA(cudaMemcpyAsync(hh.data(), hp, hh.size() * 8, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        return KB_OK;
    };
    uint64_t draws = 0;
    auto fresh = [&](int ncol, double* dst) -> int {               // a random unit direction orthogonal to ncol columns
        sp_random<<<sp_blocks(n), SP_THREADS, 0, st>>>(wp, n, sp_mix64(seed + draws++));
        ctx->launches += 1;
        int rc = orth(ncol);
        if (rc) return rc;
        const double nrm2 = hh[2 * cols];
        if (!(nrm2 > 0.0)) { kb_set_error("spectral: no direction is left orthogonal to the Lanczos basis"); return KB_EINVAL; }
        sp_scale<<<sp_blocks(n), SP_THREADS, 0, st>>>(wp, n, std::sqrt(nrm2), dst);
        ctx->launches += 1;
        return KB_OK;
    };
    { int rc = fresh(1, Vp + n); if (rc) return rc; }
    int j = 0;
    double beta = 0.0;
    for (;;) {
        for (; j < m; ++j) {
            sp_apply(op, st, Vp + (int64_t)(j + 1) * n, wp);
            ctx->launches += 1;
            ++res->steps;
            int rc = orth(j + 2);
            if (rc) return rc;
            for (int i = 0; i <= j; ++i) H[(size_t)i * m + j] = H[(size_t)j * m + i] = hh[i + 1] + hh[cols + i + 1];
            beta = std::sqrt(hh[2 * cols]);
            if (complete && j == m - 1) { beta = 0.0; break; }
            if (beta > SP_BREAK) {
                sp_scale<<<sp_blocks(n), SP_THREADS, 0, st>>>(wp, n, beta, Vp + (int64_t)(j + 2) * n);
                ctx->launches += 1;
            } else {
                beta = 0.0;
                rc = fresh(j + 2, Vp + (int64_t)(j + 2) * n);
                if (rc) return rc;
            }
        }
        std::vector<double> a = H;
        sp_jacobi(m, a, theta, Y);
        bool conv = true;
        for (int i = 0; i < nev; ++i) conv = conv && std::fabs(beta * Y[(size_t)(m - 1) * m + i]) <= SP_TOL;
        const bool done = conv || res->restarts >= SP_RESTART_CAP;
        const int keep = done ? nev : kk;
        ysub.resize((size_t)m * keep);
        for (int r = 0; r < m; ++r)
            for (int c = 0; c < keep; ++c) ysub[(size_t)r * keep + c] = Y[(size_t)r * m + c];
        KB_CUDA(cudaMemcpyAsync(yd.p, ysub.data(), ysub.size() * 8, cudaMemcpyHostToDevice, st));
        sp_combine<<<dim3(sp_blocks(n), keep), SP_THREADS, 0, st>>>(Vp, n, m, yd.as<double>(), keep, done ? d_out : tmp.as<double>());
        ctx->launches += 1;
        KB_CUDA(cudaGetLastError());
        if (done) {
            KB_CUDA(cudaStreamSynchronize(st));                    // ysub is read by the copy above
            res->converged = conv;
            return KB_OK;
        }
        // thick restart: [Ritz vectors 0 .. kk-1, v_m]; the kept block of H is diagonal
        KB_CUDA(cudaMemcpyAsync(Vp + n, tmp.p, (size_t)n * kk * 8, cudaMemcpyDeviceToDevice, st));
        KB_CUDA(cudaMemcpyAsync(Vp + (int64_t)(kk + 1) * n, Vp + (int64_t)(m + 1) * n, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
        KB_CUDA(cudaStreamSynchronize(st));
        std::fill(H.begin(), H.end(), 0.0);
        for (int i = 0; i < kk; ++i) H[(size_t)i * m + i] = theta[i];
        j = kk;
        ++res->restarts;
    }
}

// unit vectors with their largest-|.| entry positive (in place, n x k column-major); sgn / amax: device k doubles each
int sp_finish_vectors(kb_ctx* ctx, cudaMemPool_t pool, double* x, int64_t n, int k, std::vector<double>& amax) {
    cudaStream_t st = ctx->stream;
    PoolBuf nrm(pool, st), arg(pool, st);
    KB_CUDA(nrm.alloc((size_t)k * 8)); KB_CUDA(arg.alloc((size_t)2 * k * 8));
    sp_colnorm2<<<k, SP_THREADS, 0, st>>>(x, n, nrm.as<double>());
    sp_colscale<<<sp_blocks(n * k), SP_THREADS, 0, st>>>(x, n, k, nrm.as<double>());
    sp_colargmax<<<k, SP_THREADS, 0, st>>>(x, n, arg.as<double>());
    ctx->launches += 3;
    KB_CUDA(cudaGetLastError());
    std::vector<double> h(2 * k);
    KB_CUDA(cudaMemcpyAsync(h.data(), arg.p, h.size() * 8, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    amax.resize(2 * k);
    for (int c = 0; c < k; ++c) { amax[2 * c] = h[2 * c] < 0.0 ? -1.0 : 1.0; amax[2 * c + 1] = h[2 * c + 1]; }
    return KB_OK;
}

// the result of the last build, kept in the context for fetch and assemble
struct SpState {
    int64_t n = 0, n_comp = 0, cols = 0;
    int dim = 0;
    std::vector<int32_t> size, status;
    std::vector<double> range, expansion;
    int64_t stats[6] = {0, 0, 0, 0, 0, 0};
    int32_t *d_label = nullptr, *d_status = nullptr;
    double *d_range = nullptr, *d_expansion = nullptr, *d_meta = nullptr, *d_vec = nullptr, *d_cent = nullptr;
    ~SpState() {
        for (void* p : {(void*)d_label, (void*)d_status, (void*)d_range, (void*)d_expansion, (void*)d_meta, (void*)d_vec, (void*)d_cent})
            if (p) cudaFree(p);
    }
};

}  // namespace

void kb_spectral_free(kb_ctx* c) {
    delete (SpState*)c->spectral;
    c->spectral = nullptr;
}

extern "C" int kb_spectral_build(kb_ctx* ctx, int64_t n, int64_t nnz, const int64_t* d_indptr, const int32_t* d_indices,
                                 const double* d_data, int32_t n_epochs, int32_t dim, const void* d_x, int32_t x_dtype,
                                 int64_t x_cols, int64_t* n_comp_out) {
    KB_CHECK_ARG(ctx && n_comp_out && d_indptr && (nnz == 0 || (d_indices && d_data)), "null pointer");
    KB_CHECK_ARG(n >= 2 && n <= INT32_MAX, "n (2 <= n < 2^31)");
    KB_CHECK_ARG(nnz >= 0, "nnz must be >= 0");
    KB_CHECK_ARG(n_epochs >= 0, "n_epochs must be >= 0 (0: no pruning)");
    KB_CHECK_ARG(dim >= 1, "dim must be >= 1");
    KB_CHECK_ARG(x_dtype == 0 || (d_x && (x_dtype == 1 || x_dtype == 2) && x_cols >= 1),
                 "data: x_dtype 0 (none), 1 (float32) or 2 (float64) with x_cols >= 1");
    if (dim > SP_DIM_MAX) { kb_set_error("spectral: dim = %d, this build serves 1..%d", dim, SP_DIM_MAX); return KB_EUNSUPPORTED; }
    *n_comp_out = 0;
    kb_spectral_free(ctx);
    KB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    cudaMemPool_t pool;
    { int rc = kb_pool_get(ctx, &pool); if (rc) return rc; }
    SpState* S = new SpState();
    ctx->spectral = S;
    S->n = n; S->dim = dim;
    PoolBuf status(pool, st), row_kept(pool, st), deg(pool, st), comp(pool, st), succ(pool, st), par(pool, st),
        comp_key(pool, st), minv(pool, st), flag(pool, st), rank(pool, st), size(pool, st), off(pool, st), keys(pool, st),
        iota(pool, st), perm(pool, st), pos(pool, st), cnt(pool, st), pindptr(pool, st), pidx(pool, st), pval(pool, st),
        szpad(pool, st), tmp(pool, st);
    KB_CUDA(status.alloc(sizeof(SpStatus)));
    KB_CUDA(cudaMemsetAsync(status.p, 0, sizeof(SpStatus), st));
    SpStatus* d_st = status.as<SpStatus>();
    SpStatus h;
    const unsigned nbk = sp_blocks(n);
    int64_t n_comp = n;
    // 1. validation, pruning, degrees, components, labels, the permuted CSR
    {
        KbTimer t(ctx, 12);
        kb_csr_check<<<nbk, SP_THREADS, 0, st>>>(d_indptr, d_indices, d_data, n, nnz, &d_st->flags, &d_st->wmax_bits);
        if (x_dtype) {
            const int64_t total = n * x_cols;
            sp_check_x<<<(unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 16), 256, 0, st>>>(
                d_x, x_dtype == 2, total, d_st);
        }
        ctx->launches += x_dtype ? 2 : 1;
        KB_CUDA(cudaGetLastError());
        KB_CUDA(cudaMemcpyAsync(&h, d_st, sizeof(h), cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        if (h.flags & KB_CSR_BAD_INDPTR) { kb_set_error("spectral: indptr must run from 0 to nnz and never decrease"); return KB_EINVAL; }
        if (h.flags & KB_CSR_BAD_INDEX) { kb_set_error("spectral: a column index is outside [0, n)"); return KB_EINVAL; }
        if (h.flags & KB_CSR_BAD_DATA) { kb_set_error("spectral: every weight must be finite and > 0"); return KB_EINVAL; }
        if (h.flags & SP_BAD_X) { kb_set_error("spectral: the data hold a value that is not finite as float32"); return KB_EINVAL; }
        KB_CUDA(row_kept.alloc((size_t)n * 8)); KB_CUDA(deg.alloc((size_t)n * 8));
        sp_keep<<<nbk, SP_THREADS, 0, st>>>(d_indptr, d_data, n, n_epochs, d_st, row_kept.as<int64_t>(), deg.as<double>());
        KB_CUDA(comp.alloc((size_t)n * 4)); KB_CUDA(succ.alloc((size_t)n * 4)); KB_CUDA(par.alloc((size_t)n * 4));
        KB_CUDA(comp_key.alloc((size_t)n * 8));
        hd_iota<<<nbk, SP_THREADS, 0, st>>>(comp.as<int32_t>(), n);
        ctx->launches += 2;
        int rounds = 0;
        for (;;) {
            if (++rounds > 64) { kb_set_error("spectral: the component rounds did not converge"); return KB_EINVAL; }
            int jumps = 0;
            while ((int64_t)1 << jumps < n_comp) ++jumps;
            KB_CUDA(cudaMemsetAsync(comp_key.p, 0xff, (size_t)n * 8, st));
            KB_CUDA(cudaMemsetAsync(&d_st->hooks, 0, 16, st));
            sp_edge_min<<<nbk, SP_THREADS, 0, st>>>(d_indptr, d_indices, d_data, n, n_epochs, d_st, comp.as<int32_t>(),
                                                    comp_key.as<unsigned long long>());
            hd_hook<<<nbk, SP_THREADS, 0, st>>>(comp.as<int32_t>(), comp_key.as<unsigned long long>(), succ.as<int32_t>(), n);
            sp_link<<<nbk, SP_THREADS, 0, st>>>(comp.as<int32_t>(), succ.as<int32_t>(), par.as<int32_t>(), n, d_st);
            for (int s = 0; s < jumps; ++s) hd_jump<<<nbk, SP_THREADS, 0, st>>>(comp.as<int32_t>(), par.as<int32_t>(), n);
            hd_relabel<<<nbk, SP_THREADS, 0, st>>>(comp.as<int32_t>(), par.as<int32_t>(), n, &d_st->n_comp);
            ctx->launches += 4 + jumps;
            KB_CUDA(cudaGetLastError());
            KB_CUDA(cudaMemcpyAsync(&h, d_st, sizeof(h), cudaMemcpyDeviceToHost, st));
            KB_CUDA(cudaStreamSynchronize(st));
            n_comp = (int64_t)h.n_comp;
            if (h.hooks == 0) break;
        }
        S->stats[4] = rounds;
        KB_CUDA(minv.alloc((size_t)n * 4)); KB_CUDA(flag.alloc((size_t)n * 4)); KB_CUDA(rank.alloc((size_t)n * 4));
        KB_CUDA(size.alloc((size_t)n_comp * 4)); KB_CUDA(off.alloc((size_t)(n_comp + 1) * 8));
        KB_CUDA(cudaMalloc(&S->d_label, (size_t)n * 4));
        KB_CUDA(cudaMemsetAsync(minv.p, 0x7f, (size_t)n * 4, st));
        KB_CUDA(cudaMemsetAsync(size.p, 0, (size_t)n_comp * 4, st));
        sp_min_vertex<<<nbk, SP_THREADS, 0, st>>>(comp.as<int32_t>(), n, minv.as<int32_t>());
        sp_first<<<nbk, SP_THREADS, 0, st>>>(comp.as<int32_t>(), minv.as<int32_t>(), n, flag.as<int32_t>());
        size_t tb = 0, tb2 = 0, tb3 = 0, tb4 = 0;
        KB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, flag.as<int32_t>(), rank.as<int32_t>(), n, st));
        KB_CUDA(keys.alloc((size_t)n * 4)); KB_CUDA(iota.alloc((size_t)n * 4)); KB_CUDA(perm.alloc((size_t)n * 4));
        KB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb2, S->d_label, keys.as<int32_t>(), iota.as<int32_t>(),
                                                perm.as<int32_t>(), n, 0, 32, st));
        KB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb3, size.as<int32_t>(), off.as<int64_t>(), n_comp + 1, st));   // sizes only
        KB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb4, row_kept.as<int64_t>(), row_kept.as<int64_t>(), n + 1, st));
        KB_CUDA(tmp.alloc(std::max(std::max(tb, tb2), std::max(tb3, tb4))));
        KB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, flag.as<int32_t>(), rank.as<int32_t>(), n, st));
        sp_label<<<nbk, SP_THREADS, 0, st>>>(comp.as<int32_t>(), minv.as<int32_t>(), rank.as<int32_t>(), n, S->d_label,
                                             size.as<int32_t>());
        hd_iota<<<nbk, SP_THREADS, 0, st>>>(iota.as<int32_t>(), n);
        KB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tb2, S->d_label, keys.as<int32_t>(), iota.as<int32_t>(),
                                                perm.as<int32_t>(), n, 0, 32, st));
        // offsets: the exclusive scan of the sizes, zero-padded to n_comp + 1 entries
        KB_CUDA(szpad.alloc((size_t)(n_comp + 1) * 4));
        KB_CUDA(cudaMemsetAsync(szpad.p, 0, (size_t)(n_comp + 1) * 4, st));
        KB_CUDA(cudaMemcpyAsync(szpad.p, size.p, (size_t)n_comp * 4, cudaMemcpyDeviceToDevice, st));
        KB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb3, szpad.as<int32_t>(), off.as<int64_t>(), n_comp + 1, st));
        KB_CUDA(pos.alloc((size_t)n * 4)); KB_CUDA(cnt.alloc((size_t)(n + 1) * 8)); KB_CUDA(pindptr.alloc((size_t)(n + 1) * 8));
        KB_CUDA(cudaMemsetAsync(cnt.as<int64_t>() + n, 0, 8, st));
        sp_perm_count<<<nbk, SP_THREADS, 0, st>>>(perm.as<int32_t>(), row_kept.as<int64_t>(), n, pos.as<int32_t>(), cnt.as<int64_t>());
        KB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb4, cnt.as<int64_t>(), pindptr.as<int64_t>(), n + 1, st));
        ctx->launches += 10;
        KB_CUDA(cudaGetLastError());
        int64_t kept = 0;
        KB_CUDA(cudaMemcpyAsync(&kept, pindptr.as<int64_t>() + n, 8, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        KB_CUDA(pidx.alloc((size_t)kept * 4)); KB_CUDA(pval.alloc((size_t)kept * 8));
        sp_perm_fill<<<nbk, SP_THREADS, 0, st>>>(d_indptr, d_indices, d_data, n, n_epochs, d_st, perm.as<int32_t>(),
                                                 pos.as<int32_t>(), deg.as<double>(), pindptr.as<int64_t>(), pidx.as<int32_t>(),
                                                 pval.as<double>());
        ctx->launches += 1;
        KB_CUDA(cudaGetLastError());
    }
    S->n_comp = n_comp;
    S->size.resize(n_comp);
    S->status.assign(n_comp, SP_DRAW);
    S->range.assign(n_comp, 10.0);
    S->expansion.assign(n_comp, 1.0);
    KB_CUDA(cudaMemcpyAsync(S->size.data(), size.p, (size_t)n_comp * 4, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    if (n_comp == 1 && n <= (int64_t)dim + 1) {
        kb_set_error("spectral: a connected graph of %lld vertices has fewer than dim = %d non-trivial eigenvectors",
                     (long long)n, dim);
        return KB_EINVAL;
    }
    const bool want_meta = n_comp > 2 * (int64_t)dim;
    if (want_meta && n_comp > SP_META_MAX) {
        kb_set_error("spectral: %lld components; the dense meta-embedding serves at most %lld", (long long)n_comp,
                     (long long)SP_META_MAX);
        return KB_EUNSUPPORTED;
    }
    if (want_meta && !x_dtype) {
        kb_set_error("spectral: %lld components > 2 * dim need the data for their centroids", (long long)n_comp);
        return KB_EINVAL;
    }
    std::vector<int64_t> offs(n_comp + 1, 0);
    for (int64_t c = 0; c < n_comp; ++c) offs[c + 1] = offs[c] + S->size[c];
    // 2. every component's eigenvectors
    KB_CUDA(cudaMalloc(&S->d_vec, (size_t)n * dim * 8));
    KB_CUDA(cudaMemsetAsync(S->d_vec, 0, (size_t)n * dim * 8, st));
    {
        KbTimer t(ctx, 13);
        PoolBuf q0(pool, st), out(pool, st), sgn(pool, st), nrm(pool, st);
        KB_CUDA(sgn.alloc((size_t)dim * 8)); KB_CUDA(nrm.alloc(8));
        for (int64_t c = 0; c < n_comp; ++c) {
            const int64_t sc = S->size[c];
            if (n_comp > 1 && sc < 2 * (int64_t)dim) continue;
            if (!q0.p) { KB_CUDA(q0.alloc((size_t)n * 8)); KB_CUDA(out.alloc((size_t)n * dim * 8)); }
            // q0 = D^1/2 1, normalised
            sp_sqrt_deg<<<sp_blocks(sc), SP_THREADS, 0, st>>>(deg.as<double>(), perm.as<int32_t>(), offs[c], sc, q0.as<double>());
            sp_colnorm2<<<1, SP_THREADS, 0, st>>>(q0.as<double>(), sc, nrm.as<double>());
            sp_colscale<<<sp_blocks(sc), SP_THREADS, 0, st>>>(q0.as<double>(), sc, 1, nrm.as<double>());
            ctx->launches += 3;
            SpOp op{pindptr.as<int64_t>(), pidx.as<int32_t>(), pval.as<double>(), offs[c], nullptr, sc};
            SpSolve res;
            int rc = sp_lanczos(ctx, pool, op, dim, sp_mix64(0x5eed0000ull + (uint64_t)c), q0.as<double>(), out.as<double>(), &res);
            if (rc) return rc;
            S->stats[0] += res.steps;
            S->stats[1] += res.restarts;
            if (!res.converged) { S->status[c] = SP_NOT_CONVERGED; continue; }
            std::vector<double> am;
            rc = sp_finish_vectors(ctx, pool, out.as<double>(), sc, dim, am);
            if (rc) return rc;
            std::vector<double> sg(dim);
            double mx = 0.0;
            for (int k = 0; k < dim; ++k) { sg[k] = am[2 * k]; mx = std::max(mx, am[2 * k + 1]); }
            KB_CUDA(cudaMemcpyAsync(sgn.p, sg.data(), (size_t)dim * 8, cudaMemcpyHostToDevice, st));
            sp_vec_out<<<sp_blocks(sc * dim), SP_THREADS, 0, st>>>(out.as<double>(), sc, dim, sgn.as<double>(),
                                                                   perm.as<int32_t>(), offs[c], S->d_vec);
            ctx->launches += 1;
            KB_CUDA(cudaGetLastError());
            KB_CUDA(cudaStreamSynchronize(st));                    // sg is read by the copy above
            S->status[c] = SP_SOLVED;
            S->expansion[c] = mx;                                  // max|v| until the range is known
        }
    }
    // 3. meta points and data ranges
    if (n_comp > 1) {
        KbTimer t(ctx, 14);
        KB_CUDA(cudaMalloc(&S->d_meta, (size_t)n_comp * dim * 8));
        std::vector<double> meta((size_t)n_comp * dim, 0.0);
        if (want_meta) {
            S->cols = x_cols;
            KB_CUDA(cudaMalloc(&S->d_cent, (size_t)n_comp * x_cols * 8));
            PoolBuf aff(pool, st), mdeg(pool, st), q0(pool, st), out(pool, st), nrm(pool, st);
            sp_centroid<<<sp_blocks(n_comp * x_cols), SP_THREADS, 0, st>>>(d_x, x_dtype == 2, x_cols, perm.as<int32_t>(),
                                                                          off.as<int64_t>(), size.as<int32_t>(), n_comp, S->d_cent);
            KB_CUDA(aff.alloc((size_t)n_comp * n_comp * 8));
            const unsigned tiles = (unsigned)((n_comp + SP_TILE - 1) / SP_TILE);
            sp_affinity<<<dim3(tiles, tiles), SP_TILE * SP_TILE, 0, st>>>(S->d_cent, n_comp, x_cols, aff.as<double>(), d_st);
            KB_CUDA(mdeg.alloc((size_t)n_comp * 8));
            sp_rowsum<<<(unsigned)n_comp, SP_THREADS, 0, st>>>(aff.as<double>(), n_comp, mdeg.as<double>());
            sp_normalise<<<sp_blocks(n_comp * n_comp), SP_THREADS, 0, st>>>(aff.as<double>(), n_comp, mdeg.as<double>());
            ctx->launches += 4;
            KB_CUDA(cudaGetLastError());
            KB_CUDA(cudaMemcpyAsync(&h, d_st, sizeof(h), cudaMemcpyDeviceToHost, st));
            KB_CUDA(cudaStreamSynchronize(st));
            if (h.flags & SP_ZERO_AFFINITY) {
                kb_set_error("spectral: exp(-d^2) between two centroids underflows to 0; the meta graph may be disconnected");
                return KB_EUNSUPPORTED;
            }
            KB_CUDA(q0.alloc((size_t)n_comp * 8)); KB_CUDA(out.alloc((size_t)n_comp * dim * 8)); KB_CUDA(nrm.alloc(8));
            sp_sqrt_deg<<<sp_blocks(n_comp), SP_THREADS, 0, st>>>(mdeg.as<double>(), nullptr, 0, n_comp, q0.as<double>());
            sp_colnorm2<<<1, SP_THREADS, 0, st>>>(q0.as<double>(), n_comp, nrm.as<double>());
            sp_colscale<<<sp_blocks(n_comp), SP_THREADS, 0, st>>>(q0.as<double>(), n_comp, 1, nrm.as<double>());
            ctx->launches += 3;
            SpOp op{nullptr, nullptr, nullptr, 0, aff.as<double>(), n_comp};
            SpSolve res;
            int rc = sp_lanczos(ctx, pool, op, dim, sp_mix64(0x3e7a0000ull), q0.as<double>(), out.as<double>(), &res);
            if (rc) return rc;
            S->stats[2] = res.steps;
            S->stats[3] = res.restarts;
            if (!res.converged) {
                kb_set_error("spectral: the meta-embedding did not converge in %d restarts", SP_RESTART_CAP);
                return KB_EINVAL;
            }
            sp_colnorm2<<<dim, SP_THREADS, 0, st>>>(out.as<double>(), n_comp, aff.as<double>());
            sp_colscale<<<sp_blocks(n_comp * dim), SP_THREADS, 0, st>>>(out.as<double>(), n_comp, dim, aff.as<double>());
            ctx->launches += 2;
            std::vector<double> u((size_t)n_comp * dim), dd(n_comp);
            KB_CUDA(cudaMemcpyAsync(u.data(), out.p, u.size() * 8, cudaMemcpyDeviceToHost, st));
            KB_CUDA(cudaMemcpyAsync(dd.data(), mdeg.p, dd.size() * 8, cudaMemcpyDeviceToHost, st));
            KB_CUDA(cudaStreamSynchronize(st));
            // scikit-learn: divided by sqrt(degree), the sign flipped, then 0.3.9 divides by the global max
            for (int64_t a = 0; a < n_comp; ++a) dd[a] = std::sqrt(dd[a]);
            double gmax = -INFINITY;
            for (int k = 0; k < dim; ++k) {
                int64_t arg = 0;
                for (int64_t a = 0; a < n_comp; ++a) {
                    double& e = u[(size_t)k * n_comp + a];
                    e = e / dd[a];
                    if (std::fabs(e) > std::fabs(u[(size_t)k * n_comp + arg])) arg = a;
                }
                const double s = u[(size_t)k * n_comp + arg] < 0.0 ? -1.0 : 1.0;
                for (int64_t a = 0; a < n_comp; ++a) {
                    const double e = u[(size_t)k * n_comp + a] * s;
                    meta[(size_t)a * dim + k] = e;
                    gmax = std::max(gmax, e);
                }
            }
            for (double& e : meta) e = e / gmax;
        } else {
            const int64_t k = (n_comp + 1) / 2;
            for (int64_t c = 0; c < n_comp; ++c) meta[(size_t)c * dim + (c < k ? c : c - k)] = c < k ? 1.0 : -1.0;
        }
        KB_CUDA(cudaMemcpyAsync(S->d_meta, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, st));
        PoolBuf rng(pool, st);
        KB_CUDA(rng.alloc((size_t)n_comp * 8));
        auto launch = dim <= 2 ? sp_launch_range<2> : dim <= 4 ? sp_launch_range<4> : dim <= 8 ? sp_launch_range<8>
                    : dim <= 16 ? sp_launch_range<16> : dim <= 32 ? sp_launch_range<32> : sp_launch_range<64>;
        launch(sp_blocks(n_comp), st, S->d_meta, n_comp, dim, rng.as<double>());
        ctx->launches += 1;
        KB_CUDA(cudaGetLastError());
        KB_CUDA(cudaMemcpyAsync(S->range.data(), rng.p, (size_t)n_comp * 8, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        for (int64_t c = 0; c < n_comp; ++c)
            if (!(S->range[c] > 0.0)) {
                kb_set_error("spectral: meta point %lld coincides with every other one", (long long)c);
                return KB_EINVAL;
            }
    }
    for (int64_t c = 0; c < n_comp; ++c)
        S->expansion[c] = S->status[c] == SP_SOLVED && n_comp > 1 ? S->range[c] / S->expansion[c] : 1.0;
    KB_CUDA(cudaMalloc(&S->d_status, (size_t)n_comp * 4));
    KB_CUDA(cudaMalloc(&S->d_range, (size_t)n_comp * 8));
    KB_CUDA(cudaMalloc(&S->d_expansion, (size_t)n_comp * 8));
    KB_CUDA(cudaMemcpyAsync(S->d_status, S->status.data(), (size_t)n_comp * 4, cudaMemcpyHostToDevice, st));
    KB_CUDA(cudaMemcpyAsync(S->d_range, S->range.data(), (size_t)n_comp * 8, cudaMemcpyHostToDevice, st));
    KB_CUDA(cudaMemcpyAsync(S->d_expansion, S->expansion.data(), (size_t)n_comp * 8, cudaMemcpyHostToDevice, st));
    KB_CUDA(cudaStreamSynchronize(st));
    *n_comp_out = n_comp;
    return KB_OK;
}

extern "C" int kb_spectral_fetch(kb_ctx* ctx, int32_t* h_size, int32_t* h_status, double* h_range, int64_t* h_stats,
                                 int32_t* d_labels, double* d_meta, double* d_vectors, double* d_centroids) {
    KB_CHECK_ARG(ctx, "null pointer");
    const SpState* S = (const SpState*)ctx->spectral;
    if (!S || !S->d_status) { kb_set_error("spectral fetch: no successful kb_spectral_build on this context"); return KB_EINVAL; }
    KB_CHECK_ARG(!d_meta || S->d_meta, "d_meta: a connected graph has no meta points");
    KB_CHECK_ARG(!d_centroids || S->d_cent, "d_centroids: no centroids were computed (n_comp <= 2 * dim)");
    const int64_t nc = S->n_comp;
    if (h_size) std::copy(S->size.begin(), S->size.end(), h_size);
    if (h_status) std::copy(S->status.begin(), S->status.end(), h_status);
    if (h_range) std::copy(S->range.begin(), S->range.end(), h_range);
    if (h_stats) std::copy(S->stats, S->stats + 6, h_stats);
    KB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (d_labels) KB_CUDA(cudaMemcpyAsync(d_labels, S->d_label, (size_t)S->n * 4, cudaMemcpyDeviceToDevice, st));
    if (d_meta) KB_CUDA(cudaMemcpyAsync(d_meta, S->d_meta, (size_t)nc * S->dim * 8, cudaMemcpyDeviceToDevice, st));
    if (d_vectors) KB_CUDA(cudaMemcpyAsync(d_vectors, S->d_vec, (size_t)S->n * S->dim * 8, cudaMemcpyDeviceToDevice, st));
    if (d_centroids) KB_CUDA(cudaMemcpyAsync(d_centroids, S->d_cent, (size_t)nc * S->cols * 8, cudaMemcpyDeviceToDevice, st));
    return KB_OK;
}

extern "C" int kb_spectral_assemble(kb_ctx* ctx, const double* d_u, float* d_out) {
    KB_CHECK_ARG(ctx && d_out, "null pointer");
    const SpState* S = (const SpState*)ctx->spectral;
    if (!S || !S->d_status) { kb_set_error("spectral assemble: no successful kb_spectral_build on this context"); return KB_EINVAL; }
    const bool draws = std::any_of(S->status.begin(), S->status.end(), [](int32_t s) { return s != SP_SOLVED; });
    KB_CHECK_ARG(d_u || !draws, "d_u: a component takes uniform draws");
    KB_CUDA(cudaSetDevice(ctx->device));
    const int64_t total = S->n * S->dim;
    sp_assemble<<<sp_blocks(total), SP_THREADS, 0, ctx->stream>>>(S->d_label, S->d_status, S->d_range, S->d_expansion,
                                                                  S->d_meta, S->d_vec, d_u, S->n, S->dim, d_out);
    ctx->launches += 1;
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}
