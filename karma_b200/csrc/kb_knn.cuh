// kb_knn.cuh -- shared between the SIMT and tcgen05 candidate kernels and the rerank.
#pragma once
#include "kb_common.cuh"

#define KB_KNN_KP_MAX 64          // widest candidate list (tensor and SIMT kernels)
#define KB_KNN_K_MAX 60           // largest k served by the candidate kernels; beyond: exact pass over all keys
#define KB_KNN_MAX_CAND 512       // K5 merges at most this many candidates per row (slots * KP)

// One piece of work of the tensor kernel: query-block group `group` (2 adjacent 128-row blocks, one
// per CTA of the pair) against the key tiles tile(i), i in [i_lo, i_lo + i_cnt), of the sweep
//     tile(i) = (t_lo + ((i + shift) mod cnt)) mod n_tiles
// (a band of `cnt` key tiles starting at t_lo -- for a query shard it may wrap round the end of the key set --
// rotated so that the band holding the group's diagonal starts AT the diagonal).  The running top-KP list of
// every row is written to candidate slot `slot`.
struct KbPiece {
    int32_t group, slot, t_lo, cnt, shift, i_lo, i_cnt, pad;
};

// Candidate-search plan.
//  SIMT kernel: grid (m_blocks, slots); slot s covers key tiles [n_tiles*s/slots, n_tiles*(s+1)/slots).
//  Tensor kernel: a table of pieces per worker (= CTA pair), built on the host so that every worker
//  gets the same number of tile visits and all workers sweep the same band of key tiles at the same time.
struct KbKnnPlan {
    int impl;            // KB_KNN_SIMT / KB_KNN_TC, or 0: no candidate kernel (k > KB_KNN_K_MAX: exact pass only)
    int kp;              // candidates kept per (row, slot): 8 ... 64
    int bm, bn;          // tile shape
    int64_t m_blocks;    // ceil(nq / bm)
    int64_t n_tiles;     // ceil(nk / bn)
    int64_t nq;          // query rows
    int shard;           // the queries are a row shard of the keys (the other shards arrive over NVLink)
    int cl;              // query blocks per group: 2 on the tensor path (one per CTA of a pair), 1 on SIMT
    int64_t groups;      // ceil(m_blocks / cl)
    int workers;         // tensor path: CTA pairs launched
    int slots;           // candidate lists per query row (upper bound; per group see slot_count)
    int bands;           // tensor path: S
    int sched_kind;      // 0: whole units dealt round-robin, 1: every band cut into equal ranges
    int64_t n_pieces;
    double piece_cost;   // what a piece costs on top of its tile visits, in tile visits (model)
    double makespan;     // tile visits (+ piece_cost per piece) of the busiest worker
    // workspace offsets (bytes)
    int64_t off_score, off_idx, off_rowthr, off_xidx, off_xd2, off_uncert, total;
};

int kb_knn_plan(int sm_count, int impl, int64_t nq, int64_t nk, int64_t q_row0, int32_t dp, int32_t k, int64_t n_flag, KbKnnPlan* p);
// tensor path: fills `pieces` (ordered by worker), `piece_start` (workers + 1) and `slot_count` (groups)
void kb_knn_plan_pieces(const KbKnnPlan& p, int64_t q_row0, KbPiece* pieces, int32_t* piece_start, int32_t* slot_count);

// score of key j for query i, up to a per-row constant and positive factor:
//   l_i * d2_ij - n_i/l_i = l_i * n_j/l_j^2 - 2 g_ij / l_j  =  fma(g, cm_x, l_i * cm_y)
// kb_rowmeta carries { cm_x = -2/l_j , cm_y = n_j/l_j^2 }  (+inf in cm_y masks a key)
__device__ __forceinline__ float kb_score(float g, float2 cm, float li) {
    return fmaf(g, cm.x, li * cm.y);
}
__device__ __forceinline__ float2 kb_load_cm(const kb_rowmeta* __restrict__ rowmeta, int64_t j, int64_t nk) {
    float2 cm = make_float2(0.f, __int_as_float(0x7f800000));
    if (j < nk) cm = *reinterpret_cast<const float2*>(reinterpret_cast<const char*>(rowmeta + j) + 16);
    return cm;
}

// Per-row running top-KP list in shared memory, entry e of row r at [e*ROWS + r]
// (bank = r % 32: conflict-free for one thread per row).  The list is unsorted and
// organised as KP/8 groups of 8 slots; the worst entry of every group (value + slot) is
// cached in registers, so replacing the overall worst entry costs one 8-slot rescan
// whatever KP is.  `bound` = the KP-th best score seen so far (+inf until the list is full).
template <int KP, int ROWS>
struct KbRowList {
    static constexpr int NG = KP / 8;
    static_assert(KP % 8 == 0 && NG >= 1 && NG <= 8, "KP must be a multiple of 8, at most 64");
    float* s; int32_t* i;
    float gmax[NG]; int gpos[NG];
    float bound;
    __device__ __forceinline__ KbRowList(float* s_, int32_t* i_) : s(s_), i(i_), bound(0.f) {}
    __device__ __forceinline__ void init(int r) {
        const float inf = __int_as_float(0x7f800000);
#pragma unroll
        for (int e = 0; e < KP; ++e) { s[e * ROWS + r] = inf; i[e * ROWS + r] = -1; }
#pragma unroll
        for (int g = 0; g < NG; ++g) { gmax[g] = inf; gpos[g] = 0; }
        bound = inf;
    }
    // cold path: v beat the bound -> it replaces the current overall worst entry
    __device__ __forceinline__ void insert(int r, float v, int32_t j) {
        int gs = 0; float gm = gmax[0];
#pragma unroll
        for (int g = 1; g < NG; ++g) if (gmax[g] > gm) { gm = gmax[g]; gs = g; }
        int ps = gpos[0];
#pragma unroll
        for (int g = 1; g < NG; ++g) if (g == gs) ps = gpos[g];
        const int base = (gs * 8) * ROWS + r;
        s[base + ps * ROWS] = v; i[base + ps * ROWS] = j;
        float m = s[base]; int mp = 0;
#pragma unroll
        for (int e = 1; e < 8; ++e) {
            const float x = s[base + e * ROWS];
            if (x > m) { m = x; mp = e; }
        }
        float b = m;
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            if (g == gs) { gmax[g] = m; gpos[g] = mp; }
            else b = fmaxf(b, gmax[g]);
        }
        bound = b;
    }
};

struct KbTcArgs {
    const void* d_operand; int64_t ld_operand; int32_t d_cols_padded;
    const kb_rowmeta* d_rowmeta; int64_t nk, q_row0, nq;
    float* cand_score; int32_t* cand_idx; int32_t* row_thr;
    const KbPiece* pieces; const int32_t* piece_start;
    const uint32_t* d_arrive; const uint32_t* d_epoch; int64_t rows_per_src; int32_t self_rank;
};
int kb_knn_tc_launch(kb_ctx* ctx, const KbKnnPlan& p, const KbTcArgs& a);
