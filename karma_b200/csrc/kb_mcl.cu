// kb_mcl.cu -- K11: MCL (Markov clustering) of many groups of a read graph in one call.
//
// karma runs `mcl - --abc -o -` once per k-mer cluster (Mcl.run_pipe).  Here every group's abc stream becomes one
// diagonal block of a single column-stochastic matrix, and all blocks iterate together; a group whose chaos falls
// below the threshold leaves the active set, so its columns are exactly what a run of that group alone gives.
// The arithmetic is frozen in oracle/mcl_oracle.py: fp64, every product and sum rounded separately (no FMA), every
// sum a left fold from 0.0 in ascending rows, expansion terms added in ascending k.
//
//   set-up (stage 15): validate, label each group's nodes by first appearance (atomicMin of 2*edge + side, then a
//     radix sort by (group, key)), build the block-diagonal CSC with loops (a radix sort of (column, row) keys) into
//     a fixed-capacity layout: column j keeps room for min(n_g, max(S, R)) entries (and its initial length), which
//     pruning never exceeds, so the loop allocates nothing.
//   one iteration (stage 16, one record per iteration): per active column a team (a warp for groups of <= 256
//     nodes, a CTA above) expands into a dense fp64 accumulator indexed by the group's local row (shared memory up to
//     16 384 rows, a per-CTA global slice above), compacts it in row order, prunes, inflates, renormalises, writes
//     the column once into the other buffer and raises its group's chaos (atomicMax on the bits of a non-negative
//     double); then groups below the threshold are frozen and the active lists compacted.  The host reads the three
//     list lengths once per iteration.
//   interpretation: the final columns are gathered on the device and read back; attractor systems, membership and
//     the output order are O(nnz) host work in this library (kb_mcl_build), over a matrix that has about one entry
//     per column once converged.
#include "kb_common.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <cmath>
#include <vector>

namespace {

// mcl 14-137's default resource scheme and convergence threshold as remembered (unpinned; DESIGN §3 K11); the oracle
// holds the same values
constexpr int MC_P = 7000, MC_S = 900, MC_R = 1000, MC_PCT = 90;
constexpr int MC_CAP = MC_S > MC_R ? MC_S : MC_R;
constexpr double MC_CHAOS_EPS = 1e-4;
constexpr int MC_MAX_ITER = 1000;
constexpr int MC_WARP_ROWS = 256;        // groups up to this size: one warp per column
constexpr int MC_SMEM_ROWS = 16384;      // up to this size: one CTA per column, accumulator in shared memory
constexpr int MC_BLOCK = 256;
constexpr unsigned MC_BAD_INDEX = 1u, MC_BAD_GROUP = 2u, MC_BAD_SELF = 4u, MC_BAD_WEIGHT = 8u, MC_BAD_DUP = 16u;

struct McState {
    std::vector<void*> bufs;             // device allocations of the last build
    int64_t n_nodes = 0, n_groups = 0, n_cols = 0, nnz = 0;
    std::vector<int32_t> local, cluster;
    std::vector<int64_t> n_clusters, iterations, overlap, colptr;
    std::vector<int32_t> rows;
    std::vector<double> vals;
    void release() {
        for (void* p : bufs) cudaFree(p);
        bufs.clear();
    }
};

// ---- teams: a warp or a whole CTA works on one column ----
template <int TEAM> struct Team;
template <> struct Team<32> {
    struct Scratch {};
    __device__ static int lane() { return threadIdx.x & 31; }
    __device__ static void sync() { __syncwarp(); }
    __device__ static int scan(bool p, int* total, Scratch&) {
        const unsigned b = __ballot_sync(0xffffffffu, p);
        *total = __popc(b);
        return __popc(b & ((1u << lane()) - 1));
    }
    __device__ static int sum(int x, Scratch&) {
        for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        return x;
    }
    __device__ static double max(double x, Scratch&) {
        for (int o = 16; o; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
        return x;
    }
    __device__ static double bcast(double x, Scratch&) { return __shfl_sync(0xffffffffu, x, 0); }
    __device__ static int bcast(int x, Scratch&) { return __shfl_sync(0xffffffffu, x, 0); }
};
template <> struct Team<MC_BLOCK> {
    struct Scratch { int i[MC_BLOCK / 32]; double d[MC_BLOCK / 32]; };
    __device__ static int lane() { return threadIdx.x; }
    __device__ static void sync() { __syncthreads(); }
    __device__ static int scan(bool p, int* total, Scratch& s) {
        const unsigned b = __ballot_sync(0xffffffffu, p);
        const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
        if (l == 0) s.i[w] = __popc(b);
        __syncthreads();
        int before = 0, all = 0;
        for (int k = 0; k < MC_BLOCK / 32; ++k) { before += k < w ? s.i[k] : 0; all += s.i[k]; }
        __syncthreads();
        *total = all;
        return before + __popc(b & ((1u << l) - 1));
    }
    __device__ static int sum(int x, Scratch& s) {
        for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if ((threadIdx.x & 31) == 0) s.i[threadIdx.x >> 5] = x;
        __syncthreads();
        int all = 0;
        for (int k = 0; k < MC_BLOCK / 32; ++k) all += s.i[k];
        __syncthreads();
        return all;
    }
    __device__ static double max(double x, Scratch& s) {
        for (int o = 16; o; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
        if ((threadIdx.x & 31) == 0) s.d[threadIdx.x >> 5] = x;
        __syncthreads();
        double all = 0.0;
        for (int k = 0; k < MC_BLOCK / 32; ++k) all = fmax(all, s.d[k]);
        __syncthreads();
        return all;
    }
    __device__ static double bcast(double x, Scratch& s) {
        if (threadIdx.x == 0) s.d[0] = x;
        __syncthreads();
        x = s.d[0];
        __syncthreads();
        return x;
    }
    __device__ static int bcast(int x, Scratch& s) {
        if (threadIdx.x == 0) s.i[0] = x;
        __syncthreads();
        x = s.i[0];
        __syncthreads();
        return x;
    }
};

// entry i of the compacted column is kept when it is not after entry b in the order (value desc, row asc)
__device__ __forceinline__ bool mc_kept_by(const double* v, int i, int b) { return v[i] > v[b] || (v[i] == v[b] && i <= b); }

// One iteration of the columns in `list`.  Per team: acc[rows_cap] fp64 (zero on entry and on exit), lrow[rows_cap],
// sidx[min(rows_cap, CAP)]; in shared memory, or (GLOB) in the CTA's slice of the global scratch.
template <int TEAM, bool GLOB>
__global__ void __launch_bounds__(MC_BLOCK) mc_column(
        const int32_t* __restrict__ list, int n_list, const int32_t* __restrict__ col_group, const int64_t* __restrict__ goff,
        const int64_t* __restrict__ ptr, const int32_t* __restrict__ ln_cur, const int32_t* __restrict__ rows_cur,
        const double* __restrict__ vals_cur, int32_t* __restrict__ ln_nxt, int32_t* __restrict__ rows_nxt,
        double* __restrict__ vals_nxt, double inflation, unsigned long long* __restrict__ chaos_bits, int rows_cap,
        double* __restrict__ g_acc, int32_t* __restrict__ g_idx) {
    using T = Team<TEAM>;
    __shared__ typename T::Scratch tsc[MC_BLOCK / TEAM];
    extern __shared__ double smem[];
    constexpr int TPB = MC_BLOCK / TEAM;
    const int team = threadIdx.x / TEAM, lane = T::lane();
    typename T::Scratch& sc = tsc[team];
    const int sidx_cap = rows_cap < MC_CAP ? rows_cap : MC_CAP;
    double* acc;
    int32_t* lrow;
    int32_t* sidx;
    if (GLOB) {
        acc = g_acc + (size_t)blockIdx.x * rows_cap;
        lrow = g_idx + (size_t)blockIdx.x * (rows_cap + sidx_cap);
        sidx = lrow + rows_cap;
    } else {
        acc = smem + (size_t)team * rows_cap;
        int32_t* ibase = reinterpret_cast<int32_t*>(smem + (size_t)TPB * rows_cap);
        lrow = ibase + (size_t)team * (rows_cap + sidx_cap);
        sidx = lrow + rows_cap;
        for (int r = lane; r < rows_cap; r += TEAM) acc[r] = 0.0;
        T::sync();
    }
    const double cut = 1.0 / MC_P, recover = MC_PCT / 100.0;
    for (int w = blockIdx.x * TPB + team; w < n_list; w += gridDim.x * TPB) {
        const int32_t j = list[w];
        const int32_t g = col_group[j];
        const int64_t base = goff[g];
        const int ng = (int)(goff[g + 1] - base);
        const int64_t p0 = ptr[j];
        const int lj = ln_cur[j];
        // expansion: acc[i] += M[i,k] * M[k,j], k ascending; the rows of one column k are distinct
        for (int t = 0; t < lj; ++t) {
            const int32_t k = rows_cur[p0 + t];
            const double mkj = vals_cur[p0 + t];
            const int64_t q0 = ptr[k];
            const int lk = ln_cur[k];
            for (int u = lane; u < lk; u += TEAM) {
                const int i = (int)(rows_cur[q0 + u] - base);
                acc[i] = __dadd_rn(acc[i], __dmul_rn(vals_cur[q0 + u], mkj));
            }
            T::sync();
        }
        // the present rows (sum != 0), compacted in place in row order: values in acc[0, m), rows in lrow
        int m = 0;
        for (int r0 = 0; r0 < ng; r0 += TEAM) {
            const int r = r0 + lane;
            double v = 0.0;
            if (r < ng) { v = acc[r]; if (v != 0.0) acc[r] = 0.0; }
            int tot;
            const int pos = m + T::scan(v != 0.0, &tot, sc);
            T::sync();
            if (v != 0.0) { acc[pos] = v; lrow[pos] = r; }
            m += tot;
            T::sync();
        }
        // pruning: the mass and the cutoff count
        int c = 0;
        for (int i = lane; i < m; i += TEAM) c += acc[i] >= cut;
        c = T::sum(c, sc);
        const bool select = c > MC_S;
        double total = 0.0, mass = 0.0;
        int k = select ? MC_S : c, b = -1;
        bool sorted = false;
        auto rank_sort = [&]() {   // sidx[r] = the entry of rank r in (value desc, row asc), r < min(m, CAP)
            const int lim = m < MC_CAP ? m : MC_CAP;
            for (int i = lane; i < m; i += TEAM) {
                const double vi = acc[i];
                int rank = 0;
                for (int q = 0; q < m && rank < lim; ++q) rank += acc[q] > vi || (acc[q] == vi && q < i);
                if (rank < lim) sidx[rank] = i;
            }
            T::sync();
            sorted = true;
        };
        if (select) { rank_sort(); b = sidx[MC_S - 1]; }
        if (lane == 0) {
            for (int i = 0; i < m; ++i) {
                const double v = acc[i];
                total = __dadd_rn(total, v);
                if (select ? mc_kept_by(acc, i, b) : v >= cut) mass = __dadd_rn(mass, v);
            }
        }
        total = T::bcast(total, sc);
        mass = T::bcast(mass, sc);
        const double lim_mass = __dmul_rn(recover, total);
        double s = mass;
        if (k < MC_R && k < m && mass < lim_mass) {
            if (!sorted) rank_sort();
            if (lane == 0) {
                while (k < MC_R && k < m && mass < lim_mass) { mass = __dadd_rn(mass, acc[sidx[k]]); ++k; }
                b = sidx[k - 1];
                s = 0.0;
                for (int i = 0; i < m; ++i) if (mc_kept_by(acc, i, b)) s = __dadd_rn(s, acc[i]);
            }
            s = T::bcast(s, sc);
            b = T::bcast(b, sc);
        }
        const bool by_rank = b >= 0;
        const double vb = by_rank ? acc[b] : 0.0;
        T::sync();
        // normalise and inflate the kept entries; the dropped ones become 0
        for (int i = lane; i < m; i += TEAM) {
            const double v = acc[i];
            double y = 0.0;
            if (by_rank ? (v > vb || (v == vb && i <= b)) : v >= cut) {
                const double x = __ddiv_rn(v, s);
                y = inflation == 2.0 ? __dmul_rn(x, x) : pow(x, inflation);
            }
            acc[i] = y;
        }
        T::sync();
        double sy = 0.0;
        if (lane == 0) for (int i = 0; i < m; ++i) sy = __dadd_rn(sy, acc[i]);
        sy = T::bcast(sy, sc);
        double mx = 0.0;
        for (int i = lane; i < m; i += TEAM) {
            const double z = acc[i] == 0.0 ? 0.0 : __ddiv_rn(acc[i], sy);
            acc[i] = z;
            mx = fmax(mx, z);
        }
        mx = T::max(mx, sc);
        T::sync();
        double sq = 0.0;
        if (lane == 0) for (int i = 0; i < m; ++i) sq = __dadd_rn(sq, __dmul_rn(acc[i], acc[i]));
        sq = T::bcast(sq, sc);
        // write the column once: its entries > 0 in row order
        int n_out = 0;
        for (int i0 = 0; i0 < m; i0 += TEAM) {
            const int i = i0 + lane;
            const bool keep = i < m && acc[i] > 0.0;
            int tot;
            const int pos = n_out + T::scan(keep, &tot, sc);
            if (keep) {
                rows_nxt[p0 + pos] = (int32_t)(base + lrow[i]);
                vals_nxt[p0 + pos] = acc[i];
            }
            n_out += tot;
        }
        T::sync();
        for (int i = lane; i < m; i += TEAM) acc[i] = 0.0;
        if (lane == 0) {
            ln_nxt[j] = n_out;
            const double ch = fmax(0.0, __dsub_rn(__ddiv_rn(mx, sq), 1.0));
            atomicMax(chaos_bits + g, (unsigned long long)__double_as_longlong(ch));
        }
        T::sync();
    }
}

// ---- set-up ----
__global__ void mc_check_nodes(const int32_t* __restrict__ group, int64_t n, int64_t n_groups, unsigned* __restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && (group[i] < -1 || group[i] >= n_groups)) atomicOr(flags, MC_BAD_GROUP);
}

// the stream edges: first appearance, degree, largest weight; pair keys for the duplicate check
__global__ void mc_edges(const int32_t* __restrict__ a, const int32_t* __restrict__ b, const double* __restrict__ w,
                         int64_t n_edges, int64_t n, int64_t n_groups, const int32_t* __restrict__ group,
                         unsigned* __restrict__ first, int32_t* __restrict__ deg, unsigned long long* __restrict__ wmax,
                         uint64_t* __restrict__ pair, unsigned* __restrict__ flags) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_edges) return;
    const int32_t u = a[e], v = b[e];
    pair[e] = ~0ull;
    if (u < 0 || v < 0 || u >= n || v >= n) { atomicOr(flags, MC_BAD_INDEX); return; }
    const int32_t g = group[u];
    if (g < 0 || g >= n_groups || g != group[v]) return;
    const double x = w[e];
    if (u == v) { atomicOr(flags, MC_BAD_SELF); return; }
    if (!kb_weight_ok(x)) { atomicOr(flags, MC_BAD_WEIGHT); return; }
    pair[e] = u < v ? ((uint64_t)u << 32) | (uint32_t)v : ((uint64_t)v << 32) | (uint32_t)u;
    atomicMin(first + u, (unsigned)(2 * e));
    atomicMin(first + v, (unsigned)(2 * e + 1));
    atomicAdd(deg + u, 1);
    atomicAdd(deg + v, 1);
    atomicMax(wmax + u, (unsigned long long)__double_as_longlong(x));
    atomicMax(wmax + v, (unsigned long long)__double_as_longlong(x));
}

__global__ void mc_dups(const uint64_t* __restrict__ sorted, int64_t n, unsigned* __restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i + 1 < n && sorted[i] != ~0ull && sorted[i] == sorted[i + 1]) atomicOr(flags, MC_BAD_DUP);
}

__global__ void mc_node_keys(const int32_t* __restrict__ group, const unsigned* __restrict__ first, int64_t n,
                             uint64_t* __restrict__ key, int32_t* __restrict__ node, int64_t* __restrict__ size,
                             unsigned long long* __restrict__ n_cols) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    node[i] = (int32_t)i;
    if (first[i] == 0xffffffffu) { key[i] = ~0ull; return; }
    const int32_t g = group[i];
    key[i] = ((uint64_t)(uint32_t)g << 32) | first[i];
    atomicAdd((unsigned long long*)(size + g), 1ull);
    atomicAdd(n_cols, 1ull);
}

__global__ void mc_place(const uint64_t* __restrict__ key, const int32_t* __restrict__ node, int64_t n_cols,
                         const int64_t* __restrict__ size, const int32_t* __restrict__ deg, int32_t* __restrict__ col_node,
                         int32_t* __restrict__ col_group, int32_t* __restrict__ node_col, int64_t* __restrict__ len,
                         int64_t* __restrict__ cap) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_cols) return;
    const int32_t v = node[p];
    const int32_t g = (int32_t)(key[p] >> 32);
    col_node[p] = v;
    col_group[p] = g;
    node_col[v] = (int32_t)p;
    const int64_t l = (int64_t)deg[v] + 1;
    const int64_t room = size[g] < MC_CAP ? size[g] : MC_CAP;
    len[p] = l;
    cap[p] = l > room ? l : room;
}

// entries (column << 32 | row, value): both directions of every stream edge, and the loops
__global__ void mc_emit(const int32_t* __restrict__ a, const int32_t* __restrict__ b, const double* __restrict__ w,
                        const uint64_t* __restrict__ pair, int64_t n_edges, const int32_t* __restrict__ node_col,
                        const int32_t* __restrict__ col_node, int64_t n_cols, const unsigned long long* __restrict__ wmax,
                        unsigned long long* __restrict__ counter, uint64_t* __restrict__ key, double* __restrict__ val) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n_edges && pair[e] != ~0ull) {
        const uint64_t cu = (uint32_t)node_col[a[e]], cv = (uint32_t)node_col[b[e]];
        const unsigned long long at = atomicAdd(counter, 2ull);
        key[at] = (cv << 32) | cu; val[at] = w[e];
        key[at + 1] = (cu << 32) | cv; val[at + 1] = w[e];
    }
    if (e < n_cols) {
        const unsigned long long at = atomicAdd(counter, 1ull);
        key[at] = ((uint64_t)e << 32) | (uint64_t)e;
        val[at] = __longlong_as_double((long long)wmax[col_node[e]]);
    }
}

__global__ void mc_fill(const uint64_t* __restrict__ key, const double* __restrict__ val, int64_t n_ent,
                        const int64_t* __restrict__ lptr, const int64_t* __restrict__ ptr, int32_t* __restrict__ rows,
                        double* __restrict__ vals) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_ent) return;
    const int64_t c = (int64_t)(key[t] >> 32);
    const int64_t at = ptr[c] + (t - lptr[c]);
    rows[at] = (int32_t)(key[t] & 0xffffffffull);
    vals[at] = val[t];
}

// M = A / column sum (ascending rows)
__global__ void mc_normalise(const int64_t* __restrict__ ptr, const int64_t* __restrict__ len, int64_t n_cols,
                             double* __restrict__ vals, int32_t* __restrict__ ln) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cols) return;
    const int64_t p = ptr[c], l = len[c];
    double s = 0.0;
    for (int64_t t = 0; t < l; ++t) s = __dadd_rn(s, vals[p + t]);
    for (int64_t t = 0; t < l; ++t) vals[p + t] = __ddiv_rn(vals[p + t], s);
    ln[c] = (int32_t)l;
}

// initial active lists by path
__global__ void mc_lists(const int32_t* __restrict__ col_group, const int64_t* __restrict__ size, int64_t n_cols,
                         int32_t* __restrict__ l0, int32_t* __restrict__ l1, int32_t* __restrict__ l2,
                         int* __restrict__ counts) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cols) return;
    const int64_t ng = size[col_group[c]];
    if (ng <= MC_WARP_ROWS) l0[atomicAdd(counts + 0, 1)] = (int32_t)c;
    else if (ng <= MC_SMEM_ROWS) l1[atomicAdd(counts + 1, 1)] = (int32_t)c;
    else l2[atomicAdd(counts + 2, 1)] = (int32_t)c;
}

// after an iteration: groups below the threshold stop; the chaos words are cleared for the next one
__global__ void mc_freeze(unsigned long long* __restrict__ chaos_bits, uint8_t* __restrict__ active,
                          int64_t* __restrict__ iters, int64_t n_groups, int t) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    if (active[g]) {
        iters[g] = t;
        if (__longlong_as_double((long long)chaos_bits[g]) < MC_CHAOS_EPS) active[g] = 0;
    }
    chaos_bits[g] = 0ull;
}

__global__ void mc_compact(const int32_t* __restrict__ in, int n, const int32_t* __restrict__ col_group,
                           const uint8_t* __restrict__ active, int32_t* __restrict__ out, int* __restrict__ count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && active[col_group[in[i]]]) out[atomicAdd(count, 1)] = in[i];
}

__global__ void mc_final_len(const int32_t* __restrict__ col_group, const int64_t* __restrict__ iters,
                             const int32_t* __restrict__ ln0, const int32_t* __restrict__ ln1, int64_t n_cols,
                             int64_t* __restrict__ flen) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_cols) flen[c] = (iters[col_group[c]] & 1) ? ln1[c] : ln0[c];
}

__global__ void mc_gather(const int32_t* __restrict__ col_group, const int64_t* __restrict__ iters,
                          const int64_t* __restrict__ goff, const int64_t* __restrict__ ptr, const int64_t* __restrict__ fptr,
                          int64_t n_cols, const int32_t* __restrict__ r0, const double* __restrict__ v0,
                          const int32_t* __restrict__ r1, const double* __restrict__ v1, int32_t* __restrict__ frow,
                          double* __restrict__ fval) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cols) return;
    const int32_t g = col_group[c];
    const bool odd = iters[g] & 1;
    const int32_t* r = odd ? r1 : r0;
    const double* v = odd ? v1 : v0;
    const int64_t p = ptr[c], base = goff[g];
    for (int64_t t = fptr[c]; t < fptr[c + 1]; ++t) {
        frow[t] = (int32_t)(r[p + t - fptr[c]] - base);
        fval[t] = v[p + t - fptr[c]];
    }
}

inline unsigned grid_for(int64_t n, int bs = 256) { return (unsigned)((n + bs - 1) / bs); }

// attractor systems, membership and output order of one group (local indices 0..n-1, columns c0..c0+n-1)
void interpret(int64_t n, const int64_t* cp, const int32_t* rows, const double* vals, int32_t* cluster_of_col,
               int64_t* n_clusters, int64_t* overlap) {
    std::vector<char> attractor(n, 0);
    for (int64_t j = 0; j < n; ++j)
        for (int64_t t = cp[j]; t < cp[j + 1]; ++t)
            if (rows[t] == j && vals[t] > 0) attractor[j] = 1;
    std::vector<int64_t> parent(n);
    for (int64_t i = 0; i < n; ++i) parent[i] = i;
    auto find = [&](int64_t x) {
        while (parent[x] != x) { parent[x] = parent[parent[x]]; x = parent[x]; }
        return x;
    };
    for (int64_t bb = 0; bb < n; ++bb) {
        if (!attractor[bb]) continue;
        for (int64_t t = cp[bb]; t < cp[bb + 1]; ++t) {
            const int64_t aa = rows[t];
            if (vals[t] > 0 && attractor[aa]) {
                const int64_t ra = find(aa), rb = find(bb);
                if (ra != rb) parent[std::max(ra, rb)] = std::min(ra, rb);
            }
        }
    }
    // key per node: its system (the smallest attractor of it), or n + j alone
    std::vector<int64_t> key(n), first(n), count(n, 0);
    int64_t over = 0;
    for (int64_t j = 0; j < n; ++j) {
        int64_t best = -1;
        bool several = false;
        for (int64_t t = cp[j]; t < cp[j + 1]; ++t) {
            const int64_t aa = rows[t];
            if (vals[t] > 0 && attractor[aa]) {
                const int64_t s = find(aa);
                if (best < 0) best = s;
                else if (s != best) { several = true; best = std::min(best, s); }
            }
        }
        over += several;
        key[j] = best >= 0 ? best : n + j;
    }
    // clusters: size desc, then smallest member asc; numbered in that order
    std::vector<int64_t> members_min(2 * n, -1), size(2 * n, 0);
    for (int64_t j = 0; j < n; ++j) {
        ++size[key[j]];
        if (members_min[key[j]] < 0) members_min[key[j]] = j;
    }
    std::vector<int64_t> keys;
    for (int64_t k = 0; k < 2 * n; ++k) if (size[k]) keys.push_back(k);
    std::sort(keys.begin(), keys.end(), [&](int64_t x, int64_t y) {
        return size[x] != size[y] ? size[x] > size[y] : members_min[x] < members_min[y];
    });
    std::vector<int32_t> number(2 * n, -1);
    for (size_t r = 0; r < keys.size(); ++r) number[keys[r]] = (int32_t)r;
    for (int64_t j = 0; j < n; ++j) cluster_of_col[j] = number[key[j]];
    *n_clusters = (int64_t)keys.size();
    *overlap = over;
}

}  // namespace

void kb_mcl_free(kb_ctx* c) {
    if (!c->mcl) return;
    auto* st = reinterpret_cast<McState*>(c->mcl);
    st->release();
    delete st;
    c->mcl = nullptr;
}

extern "C" int kb_mcl_build(kb_ctx* ctx, int64_t n_nodes, int64_t n_edges, const int32_t* d_a, const int32_t* d_b,
                            const double* d_w, const int32_t* d_group, int64_t n_groups, double inflation,
                            int64_t* n_cols_out, int64_t* nnz_out) {
    KB_CHECK_ARG(ctx, "ctx");
    KB_CHECK_ARG(n_nodes >= 0 && n_nodes < (1LL << 31) - 1, "node count (below 2^31 - 1)");
    KB_CHECK_ARG(n_edges >= 0 && n_edges < (1LL << 30), "edge count (below 2^30)");
    KB_CHECK_ARG(n_groups >= 0 && n_groups < (1LL << 31) - 1, "group count");
    KB_CHECK_ARG(n_edges == 0 || (d_a && d_b && d_w), "edge arrays");
    KB_CHECK_ARG(n_nodes == 0 || d_group, "group array");
    KB_CHECK_ARG(std::isfinite(inflation) && inflation > 1.0, "inflation must be finite and > 1");
    KB_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->mcl) ctx->mcl = new McState();
    McState& S = *reinterpret_cast<McState*>(ctx->mcl);
    S.release();
    S.n_nodes = n_nodes; S.n_groups = n_groups; S.n_cols = 0; S.nnz = 0;
    S.local.assign(n_nodes, -1); S.cluster.assign(n_nodes, -1);
    S.n_clusters.assign(n_groups, 0); S.iterations.assign(n_groups, 0); S.overlap.assign(n_groups, 0);
    S.colptr.assign(1, 0); S.rows.clear(); S.vals.clear();
    if (n_cols_out) *n_cols_out = 0;
    if (nnz_out) *nnz_out = 0;
    cudaStream_t st = ctx->stream;
    auto alloc = [&S](void** p, size_t bytes) -> cudaError_t {
        cudaError_t e = cudaMalloc(p, bytes ? bytes : 8);
        if (e == cudaSuccess) S.bufs.push_back(*p);
        return e;
    };
#define MC_ALLOC(ptr, type, count) KB_CUDA(alloc((void**)&(ptr), (size_t)(count) * sizeof(type)))
    const int64_t n1 = n_nodes > 0 ? n_nodes : 1, e1 = n_edges > 0 ? n_edges : 1, g1 = n_groups + 1;

    // ---- set-up ----
    unsigned* flags; unsigned* first; int32_t* deg; unsigned long long* wmax; uint64_t* pair; uint64_t* pair_s;
    uint64_t* nkey; uint64_t* nkey_s; int32_t* nnode; int32_t* nnode_s; int64_t* size; int64_t* goff;
    unsigned long long* counters;
    MC_ALLOC(flags, unsigned, 1); MC_ALLOC(first, unsigned, n1); MC_ALLOC(deg, int32_t, n1);
    MC_ALLOC(wmax, unsigned long long, n1); MC_ALLOC(pair, uint64_t, e1); MC_ALLOC(pair_s, uint64_t, e1);
    MC_ALLOC(nkey, uint64_t, n1); MC_ALLOC(nkey_s, uint64_t, n1); MC_ALLOC(nnode, int32_t, n1); MC_ALLOC(nnode_s, int32_t, n1);
    MC_ALLOC(size, int64_t, g1); MC_ALLOC(goff, int64_t, g1); MC_ALLOC(counters, unsigned long long, 2);
    int64_t n_cols = 0;
    {
        KbTimer timer(ctx, 15);
        KB_CUDA(cudaMemsetAsync(flags, 0, 4, st));
        KB_CUDA(cudaMemsetAsync(first, 0xff, (size_t)n1 * 4, st));
        KB_CUDA(cudaMemsetAsync(deg, 0, (size_t)n1 * 4, st));
        KB_CUDA(cudaMemsetAsync(wmax, 0, (size_t)n1 * 8, st));
        KB_CUDA(cudaMemsetAsync(size, 0, (size_t)g1 * 8, st));
        KB_CUDA(cudaMemsetAsync(counters, 0, 16, st));
        if (n_nodes) mc_check_nodes<<<grid_for(n_nodes), 256, 0, st>>>(d_group, n_nodes, n_groups, flags);
        if (n_edges) mc_edges<<<grid_for(n_edges), 256, 0, st>>>(d_a, d_b, d_w, n_edges, n_nodes, n_groups, d_group, first, deg,
                                                                 wmax, pair, flags);
        ctx->launches += 2;
        KB_CUDA(cudaGetLastError());
        size_t tb = 0, t1 = 0;
        KB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, t1, pair, pair_s, (int)e1, 0, 64, st)); tb = std::max(tb, t1);
        KB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, t1, nkey, nkey_s, nnode, nnode_s, (int)n1, 0, 64, st)); tb = std::max(tb, t1);
        KB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, t1, size, goff, (int)g1, st)); tb = std::max(tb, t1);
        void* tmp; MC_ALLOC(tmp, uint8_t, tb);
        if (n_edges) {
            KB_CUDA(cub::DeviceRadixSort::SortKeys(tmp, tb, pair, pair_s, (int)n_edges, 0, 64, st));
            mc_dups<<<grid_for(n_edges), 256, 0, st>>>(pair_s, n_edges, flags);
            ctx->launches += 2;
        }
        unsigned h_flags = 0;
        KB_CUDA(cudaMemcpyAsync(&h_flags, flags, 4, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        if (h_flags & MC_BAD_INDEX) { kb_set_error("invalid argument: mcl: an edge end is outside [0, %lld)", (long long)n_nodes); return KB_EINVAL; }
        if (h_flags & MC_BAD_GROUP) { kb_set_error("invalid argument: mcl: a group id is outside [-1, %lld)", (long long)n_groups); return KB_EINVAL; }
        if (h_flags & MC_BAD_SELF) { kb_set_error("invalid argument: mcl: a self-edge inside a group"); return KB_EINVAL; }
        if (h_flags & MC_BAD_WEIGHT) { kb_set_error("invalid argument: mcl: an edge weight inside a group is not finite and > 0"); return KB_EINVAL; }
        if (h_flags & MC_BAD_DUP) { kb_set_error("invalid argument: mcl: the same pair of nodes is listed twice"); return KB_EINVAL; }
        if (n_nodes) {
            mc_node_keys<<<grid_for(n_nodes), 256, 0, st>>>(d_group, first, n_nodes, nkey, nnode, size, counters);
            KB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, nkey, nkey_s, nnode, nnode_s, (int)n_nodes, 0, 64, st));
            ctx->launches += 2;
        }
        KB_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, size, goff, (int)g1, st));
        ctx->launches += 1;
        unsigned long long h_cols = 0;
        KB_CUDA(cudaMemcpyAsync(&h_cols, counters, 8, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        n_cols = (int64_t)h_cols;
    }
    std::vector<int64_t> h_size(n_groups), h_off(n_groups + 1);
    if (n_groups) {
        KB_CUDA(cudaMemcpyAsync(h_size.data(), size, (size_t)n_groups * 8, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaMemcpyAsync(h_off.data(), goff, (size_t)(n_groups + 1) * 8, cudaMemcpyDeviceToHost, st));
    }
    KB_CUDA(cudaStreamSynchronize(st));
    if (n_cols == 0) return KB_OK;
    const int64_t c1 = n_cols + 1;
    int32_t *col_node, *col_group, *node_col, *ln0, *ln1, *r0, *r1, *lists[2][3], *frow;
    int64_t *len, *cap, *lptr, *ptr, *flen, *fptr, *iters;
    double *v0, *v1, *fval;
    uint64_t *ekey, *ekey_s; double *eval, *eval_s;
    unsigned long long* chaos; uint8_t* active; int* counts;
    MC_ALLOC(col_node, int32_t, n_cols); MC_ALLOC(col_group, int32_t, n_cols); MC_ALLOC(node_col, int32_t, n1);
    MC_ALLOC(len, int64_t, c1); MC_ALLOC(cap, int64_t, c1); MC_ALLOC(lptr, int64_t, c1); MC_ALLOC(ptr, int64_t, c1);
    int64_t total_cap = 0, n_entries = 0;
    {
        KbTimer timer(ctx, 15);
        KB_CUDA(cudaMemsetAsync(len + n_cols, 0, 8, st));
        KB_CUDA(cudaMemsetAsync(cap + n_cols, 0, 8, st));
        mc_place<<<grid_for(n_cols), 256, 0, st>>>(nkey_s, nnode_s, n_cols, size, deg, col_node, col_group, node_col, len, cap);
        size_t tb = 0, t1 = 0;
        KB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, t1, len, lptr, (int)c1, st)); tb = std::max(tb, t1);
        void* tmp; MC_ALLOC(tmp, uint8_t, tb);
        KB_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, len, lptr, (int)c1, st));
        KB_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, cap, ptr, (int)c1, st));
        ctx->launches += 3;
        KB_CUDA(cudaGetLastError());
        KB_CUDA(cudaMemcpyAsync(&n_entries, lptr + n_cols, 8, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaMemcpyAsync(&total_cap, ptr + n_cols, 8, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
    }
    if (n_entries >= (1LL << 31)) { kb_set_error("mcl: %lld matrix entries (at most 2^31 - 1)", (long long)n_entries); return KB_EUNSUPPORTED; }
    MC_ALLOC(ekey, uint64_t, n_entries); MC_ALLOC(ekey_s, uint64_t, n_entries);
    MC_ALLOC(eval, double, n_entries); MC_ALLOC(eval_s, double, n_entries);
    MC_ALLOC(r0, int32_t, total_cap); MC_ALLOC(r1, int32_t, total_cap);
    MC_ALLOC(v0, double, total_cap); MC_ALLOC(v1, double, total_cap);
    MC_ALLOC(ln0, int32_t, n_cols); MC_ALLOC(ln1, int32_t, n_cols);
    for (int b = 0; b < 2; ++b) for (int p = 0; p < 3; ++p) MC_ALLOC(lists[b][p], int32_t, n_cols);
    MC_ALLOC(chaos, unsigned long long, n_groups); MC_ALLOC(active, uint8_t, n_groups); MC_ALLOC(iters, int64_t, n_groups);
    MC_ALLOC(counts, int, 3);
    // the largest group of each CTA path sizes its accumulator
    int64_t max1 = 0, max2 = 0;
    std::vector<uint8_t> h_active(n_groups);
    for (int64_t g = 0; g < n_groups; ++g) {
        h_active[g] = h_size[g] > 0;
        if (h_size[g] > MC_WARP_ROWS && h_size[g] <= MC_SMEM_ROWS) max1 = std::max(max1, h_size[g]);
        if (h_size[g] > MC_SMEM_ROWS) max2 = std::max(max2, h_size[g]);
    }
    const int sidx0 = std::min(MC_WARP_ROWS, MC_CAP);
    const size_t smem0 = (size_t)(MC_BLOCK / 32) * (MC_WARP_ROWS * 12 + sidx0 * 4);
    const int sidx1 = (int)std::min<int64_t>(max1, MC_CAP);
    const size_t smem1 = (size_t)max1 * 12 + (size_t)sidx1 * 4;
    KB_CUDA(cudaFuncSetAttribute(mc_column<32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0));
    if (max1) KB_CUDA(cudaFuncSetAttribute(mc_column<MC_BLOCK, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
    int occ0 = 0, occ1 = 0;
    KB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ0, mc_column<32, false>, MC_BLOCK, smem0));
    if (max1) KB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ1, mc_column<MC_BLOCK, false>, MC_BLOCK, smem1));
    const int64_t grid0_max = (int64_t)std::max(occ0, 1) * ctx->sm_count, grid1_max = (int64_t)std::max(occ1, 1) * ctx->sm_count;
    const int64_t grid2 = 2LL * ctx->sm_count;
    const int sidx2 = (int)std::min<int64_t>(max2, MC_CAP);
    double* g_acc = nullptr; int32_t* g_idx = nullptr;
    if (max2) {
        MC_ALLOC(g_acc, double, grid2 * max2);
        MC_ALLOC(g_idx, int32_t, grid2 * (max2 + sidx2));
        KB_CUDA(cudaMemsetAsync(g_acc, 0, (size_t)grid2 * max2 * 8, st));
    }
    {
        KbTimer timer(ctx, 15);
        KB_CUDA(cudaMemsetAsync(counters, 0, 8, st));
        const int64_t ge = std::max(n_edges, n_cols);
        mc_emit<<<grid_for(ge), 256, 0, st>>>(d_a, d_b, d_w, pair, n_edges, node_col, col_node, n_cols, wmax, counters, ekey, eval);
        size_t tb = 0;
        KB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, ekey, ekey_s, eval, eval_s, (int)n_entries, 0, 64, st));
        void* tmp; MC_ALLOC(tmp, uint8_t, tb);
        KB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, ekey, ekey_s, eval, eval_s, (int)n_entries, 0, 64, st));
        mc_fill<<<grid_for(n_entries), 256, 0, st>>>(ekey_s, eval_s, n_entries, lptr, ptr, r0, v0);
        mc_normalise<<<grid_for(n_cols), 256, 0, st>>>(ptr, len, n_cols, v0, ln0);
        KB_CUDA(cudaMemsetAsync(counts, 0, 12, st));
        mc_lists<<<grid_for(n_cols), 256, 0, st>>>(col_group, size, n_cols, lists[0][0], lists[0][1], lists[0][2], counts);
        KB_CUDA(cudaMemsetAsync(chaos, 0, (size_t)std::max<int64_t>(n_groups, 1) * 8, st));
        KB_CUDA(cudaMemsetAsync(iters, 0, (size_t)std::max<int64_t>(n_groups, 1) * 8, st));
        KB_CUDA(cudaMemcpyAsync(active, h_active.data(), (size_t)n_groups, cudaMemcpyHostToDevice, st));
        ctx->launches += 5;
        KB_CUDA(cudaGetLastError());
    }
    int h_counts[3] = {0, 0, 0};
    KB_CUDA(cudaMemcpyAsync(h_counts, counts, 12, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));

    // ---- iterations ----
    int cur = 0;
    for (int t = 1; h_counts[0] + h_counts[1] + h_counts[2] > 0; ++t) {
        if (t > MC_MAX_ITER) {
            KB_CUDA(cudaMemcpy(h_active.data(), active, (size_t)n_groups, cudaMemcpyDeviceToHost));
            int64_t bad = 0;
            while (bad < n_groups && !h_active[bad]) ++bad;
            kb_set_error("invalid argument: mcl: group %lld did not converge in %d iterations", (long long)bad, MC_MAX_ITER);
            return KB_EINVAL;
        }
        KbTimer timer(ctx, 16);
        const int rd = (t - 1) & 1;           // buffer 0 holds M0; iteration t reads (t-1)&1 and writes t&1
        const int32_t* rc = rd ? r1 : r0; const double* vc = rd ? v1 : v0; const int32_t* lc = rd ? ln1 : ln0;
        int32_t* rn = rd ? r0 : r1; double* vn = rd ? v0 : v1; int32_t* ln_n = rd ? ln0 : ln1;
        if (h_counts[0]) {
            const unsigned grid = (unsigned)std::min<int64_t>((h_counts[0] + MC_BLOCK / 32 - 1) / (MC_BLOCK / 32), grid0_max);
            mc_column<32, false><<<grid, MC_BLOCK, smem0, st>>>(lists[cur][0], h_counts[0], col_group, goff, ptr, lc, rc, vc,
                                                                ln_n, rn, vn, inflation, chaos, MC_WARP_ROWS, nullptr, nullptr);
            ctx->launches++;
        }
        if (h_counts[1]) {
            const unsigned grid = (unsigned)std::min<int64_t>(h_counts[1], grid1_max);
            mc_column<MC_BLOCK, false><<<grid, MC_BLOCK, smem1, st>>>(lists[cur][1], h_counts[1], col_group, goff, ptr, lc, rc, vc,
                                                                      ln_n, rn, vn, inflation, chaos, (int)max1, nullptr, nullptr);
            ctx->launches++;
        }
        if (h_counts[2]) {
            const unsigned grid = (unsigned)std::min<int64_t>(h_counts[2], grid2);
            mc_column<MC_BLOCK, true><<<grid, MC_BLOCK, 0, st>>>(lists[cur][2], h_counts[2], col_group, goff, ptr, lc, rc, vc,
                                                                 ln_n, rn, vn, inflation, chaos, (int)max2, g_acc, g_idx);
            ctx->launches++;
        }
        mc_freeze<<<grid_for(n_groups), 256, 0, st>>>(chaos, active, iters, n_groups, t);
        KB_CUDA(cudaMemsetAsync(counts, 0, 12, st));
        for (int p = 0; p < 3; ++p)
            if (h_counts[p]) {
                mc_compact<<<grid_for(h_counts[p]), 256, 0, st>>>(lists[cur][p], h_counts[p], col_group, active, lists[cur ^ 1][p], counts + p);
                ctx->launches++;
            }
        ctx->launches++;
        KB_CUDA(cudaGetLastError());
        KB_CUDA(cudaMemcpyAsync(h_counts, counts, 12, cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        cur ^= 1;
    }

    // ---- the final columns, and their interpretation on the host ----
    MC_ALLOC(flen, int64_t, c1); MC_ALLOC(fptr, int64_t, c1);
    KB_CUDA(cudaMemsetAsync(flen + n_cols, 0, 8, st));
    mc_final_len<<<grid_for(n_cols), 256, 0, st>>>(col_group, iters, ln0, ln1, n_cols, flen);
    {
        size_t tb = 0;
        KB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, flen, fptr, (int)c1, st));
        void* tmp; MC_ALLOC(tmp, uint8_t, tb);
        KB_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, flen, fptr, (int)c1, st));
    }
    int64_t nnz = 0;
    KB_CUDA(cudaMemcpyAsync(&nnz, fptr + n_cols, 8, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    MC_ALLOC(frow, int32_t, nnz); MC_ALLOC(fval, double, nnz);
    mc_gather<<<grid_for(n_cols), 256, 0, st>>>(col_group, iters, goff, ptr, fptr, n_cols, r0, v0, r1, v1, frow, fval);
    ctx->launches += 3;
    KB_CUDA(cudaGetLastError());
    S.colptr.resize(c1); S.rows.resize(nnz); S.vals.resize(nnz);
    std::vector<int32_t> h_col_node(n_cols), h_col_group(n_cols);
    KB_CUDA(cudaMemcpyAsync(S.colptr.data(), fptr, (size_t)c1 * 8, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaMemcpyAsync(S.rows.data(), frow, (size_t)nnz * 4, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaMemcpyAsync(S.vals.data(), fval, (size_t)nnz * 8, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaMemcpyAsync(h_col_node.data(), col_node, (size_t)n_cols * 4, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaMemcpyAsync(S.iterations.data(), iters, (size_t)n_groups * 8, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> cl(n_cols);
    for (int64_t g = 0; g < n_groups; ++g) {
        const int64_t c0 = h_off[g], ng = h_size[g];
        if (!ng) continue;
        std::vector<int64_t> cp(ng + 1);
        for (int64_t j = 0; j <= ng; ++j) cp[j] = S.colptr[c0 + j] - S.colptr[c0];
        interpret(ng, cp.data(), S.rows.data() + S.colptr[c0], S.vals.data() + S.colptr[c0], cl.data() + c0,
                  &S.n_clusters[g], &S.overlap[g]);
        for (int64_t j = 0; j < ng; ++j) {
            S.local[h_col_node[c0 + j]] = (int32_t)j;
            S.cluster[h_col_node[c0 + j]] = cl[c0 + j];
        }
    }
    S.n_cols = n_cols; S.nnz = nnz;
    S.release();                                      // the device copies are no longer needed
    if (n_cols_out) *n_cols_out = n_cols;
    if (nnz_out) *nnz_out = nnz;
#undef MC_ALLOC
    return KB_OK;
}

extern "C" int kb_mcl_fetch(kb_ctx* ctx, int32_t* h_local, int32_t* h_cluster, int64_t* h_n_clusters, int64_t* h_iterations,
                            int64_t* h_overlap, int64_t* h_colptr, int32_t* h_rows, double* h_vals) {
    KB_CHECK_ARG(ctx, "ctx");
    KB_CHECK_ARG(ctx->mcl, "no kb_mcl_build result in this context");
    const McState& S = *reinterpret_cast<const McState*>(ctx->mcl);
    auto put = [](auto* dst, const auto& src) { if (dst && !src.empty()) std::copy(src.begin(), src.end(), dst); };
    put(h_local, S.local); put(h_cluster, S.cluster); put(h_n_clusters, S.n_clusters); put(h_iterations, S.iterations);
    put(h_overlap, S.overlap); put(h_colptr, S.colptr); put(h_rows, S.rows); put(h_vals, S.vals);
    return KB_OK;
}
