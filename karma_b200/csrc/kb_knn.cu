// kb_knn.cu -- kNN driver: plan, SIMT candidate kernel (K4-simt), candidate merge + exact rerank +
// certification (K5), exact side path for rows beyond the tensor range (K4x) and the exact pass over
// all keys for rows that could not be certified (K6).  The tcgen05 candidate kernel is in kb_knn_tc.cu.
//
// Replaces the neighbour search inside umap.UMAP(...).fit_transform at
// /root/reference/karma/kmer.py:285-290 (euclidean metric, the point itself is
// neighbour 0).  The profile rows are counts/len(key) (kmer.py:120,:213), so
// with integer counts c, n_i = sum c_i^2, g_ij = sum c_i c_j, l = len(key):
//     d2_ij = n_i/l_i^2 + n_j/l_j^2 - 2 g_ij / (l_i l_j)
// K4 gets g_ij exactly (integer Gram, fp32 accumulation below 2^24) and ranks by
// the fp32 norm expansion; K5 recomputes the kept candidates exactly:
//     d2_ij = sum_c (c_ic*l_j - c_jc*l_i)^2 / (l_i*l_j)^2       (fp64, integer terms)
#include "kb_knn.cuh"
#include <cub/cub.cuh>
#include <math.h>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <algorithm>

// ---------------------------------------------------------------------------------------------
// host: plan
// ---------------------------------------------------------------------------------------------
namespace {

struct Band { int64_t t_lo, cnt; };

// What a piece costs on top of its tile visits (list set-up, cold first tile, descriptor and row-record loads, write-back),
// in tile visits.  Measured on 50k x 1088: 132 visits in 2 pieces per CTA pair take 0.767 ms, 66 visits in 5.2 pieces 0.455 ms
// against 5.56 us per visit for one long sweep: about 1.5 visits per piece.
// (of 17 k-blocks; wider rows make a visit longer, not a piece dearer).
inline double piece_cost(const KbKnnPlan& p) { return p.piece_cost; }

struct Sched {
    std::vector<std::vector<KbPiece>> per_worker;
    std::vector<int32_t> slot_count;
    int slots = 0;
    int64_t n_pieces = 0;
    double makespan = 0.0;
};

// unit (round r, group g).
// All keys local (nq == nk): band (sd_g + r) % S, rotated to start at the diagonal tile when r == 0.
// Query shard (the other shards arrive over NVLink in the order q+1, q+2, ..., q-1): the sweep of a group is a
// rotation of the key tiles that starts inside the local shard (at the group's diagonal tile, or earlier, see LEAD) and
// runs upwards with wrap-around, cut into S equal bands -- so tiles are needed in exactly the order in which their
// shards land, and the tile that straddles the start of the local shard (it needs rows of rank q-1, the LAST to
// arrive) comes after all the shards instead of first.
// A piece visits tile(i) = (t_lo + ((i + shift) mod cnt)) mod n_tiles.
inline void unit_of(const KbKnnPlan& p, int64_t q_row0, int S, int r, int64_t g, KbPiece* u) {
    int64_t td = (q_row0 + g * p.cl * p.bm) / p.bn;
    if (td >= p.n_tiles) td = p.n_tiles - 1;
    if (p.shard) {
        const int64_t n = p.n_tiles;
        int64_t t_start = (q_row0 + p.bn - 1) / p.bn;                       // first tile fully inside the local rows ...
        if ((t_start + 1) * p.bn > q_row0 + p.nq || t_start >= n) t_start = q_row0 / p.bn;   // ... if there is one
        if (t_start >= n) t_start = n - 1;
        // A group starts at its own diagonal tile (its rows' nearest neighbours are mostly there: tight bounds from the
        // first tile on) unless that leaves fewer than LEAD local tiles before the first tile of the next shard is due --
        // then it starts that much earlier, so that nobody waits for the first arrival.
        constexpr int64_t LEAD = 32;
        int64_t local = (q_row0 + p.nq) / p.bn - t_start;                   // tiles fully inside the local rows
        if (local < 1) local = 1;
        int64_t off_d = (td - t_start + n) % n;                             // the diagonal in rotated coordinates
        if (off_d >= local) off_d = (off_d == n - 1) ? 0 : local - 1;       // (it is one of the two straddling tiles)
        const int64_t o = std::min<int64_t>(off_d, std::max<int64_t>(0, local - LEAD));
        const int64_t rho_lo = (n * r) / S, cnt = (n * (r + 1)) / S - rho_lo;   // equal bands of the group's rotated order
        u->group = (int32_t)g; u->slot = 0; u->t_lo = (int32_t)((t_start + o + rho_lo) % n); u->cnt = (int32_t)cnt;
        u->shift = 0;
        u->i_lo = 0; u->i_cnt = (int32_t)cnt; u->pad = 0;
        return;
    }
    int sd = (int)((td * S) / p.n_tiles);
    while (sd + 1 < S && (p.n_tiles * (sd + 1)) / S <= td) ++sd;
    while (sd > 0 && (p.n_tiles * sd) / S > td) --sd;
    const int s = (sd + r) % S;
    const int64_t t_lo = (p.n_tiles * s) / S;
    const int64_t cnt = (p.n_tiles * (s + 1)) / S - t_lo;
    u->group = (int32_t)g; u->slot = 0; u->t_lo = (int32_t)t_lo; u->cnt = (int32_t)cnt;
    u->shift = (r == 0) ? (int32_t)(td - t_lo) : 0;
    u->i_lo = 0; u->i_cnt = (int32_t)cnt; u->pad = 0;
}

// kind 0: whole units dealt round-robin (round-major).  kind 1: every round's tile visits are cut into
// `workers` equal contiguous ranges (group-major), so that all workers finish every band together.
void build_sched(const KbKnnPlan& p, int64_t q_row0, int S, int kind, Sched* out) {
    const int W = p.workers;
    out->per_worker.assign(W, {});
    out->slot_count.assign((size_t)p.groups, 0);
    std::vector<double> load(W, 0.0);
    int64_t u_lin = 0;
    for (int r = 0; r < S; ++r) {
        if (kind == 0) {
            for (int64_t g = 0; g < p.groups; ++g, ++u_lin) {
                KbPiece u; unit_of(p, q_row0, S, r, g, &u);
                if (u.cnt == 0) continue;
                u.slot = out->slot_count[g]++;
                const int w = (int)(u_lin % W);
                out->per_worker[w].push_back(u);
                load[w] += u.i_cnt + piece_cost(p);
            }
        } else {
            int64_t V = 0;
            for (int64_t g = 0; g < p.groups; ++g) { KbPiece u; unit_of(p, q_row0, S, r, g, &u); V += u.cnt; }
            const int rot = (int)(((int64_t)r * W) / S);                 // decorrelates the floor/ceil pattern of the cuts
            int64_t pos = 0;                                             // position in the round's sequence
            int j = 0;                                                   // current range
            int64_t j_end = (V * (j + 1)) / W;
            for (int64_t g = 0; g < p.groups; ++g) {
                KbPiece u; unit_of(p, q_row0, S, r, g, &u);
                int64_t done = 0;
                while (done < u.cnt) {
                    while (pos >= j_end && j + 1 < W) { ++j; j_end = (V * (j + 1)) / W; }
                    int64_t take = u.cnt - done;
                    if (j + 1 < W && pos + take > j_end) take = j_end - pos;
                    KbPiece pc = u;
                    pc.i_lo = (int32_t)done; pc.i_cnt = (int32_t)take;
                    pc.slot = out->slot_count[g]++;
                    const int w = (j + rot) % W;
                    out->per_worker[w].push_back(pc);
                    load[w] += take + piece_cost(p);
                    done += take; pos += take;
                }
            }
        }
    }
    out->slots = 0; out->n_pieces = 0; out->makespan = 0.0;
    for (int64_t g = 0; g < p.groups; ++g) out->slots = std::max(out->slots, (int)out->slot_count[g]);
    for (int w = 0; w < W; ++w) { out->n_pieces += (int64_t)out->per_worker[w].size(); out->makespan = std::max(out->makespan, load[w]); }
}

// min_bands[kind]: fewest key bands a schedule of that kind may use; sync_only: the key set is far beyond the L2, so
// concurrent workers must sweep the same key tiles at the same time (whole bands dealt round-robin only).
void choose_sched(const KbKnnPlan& p, int64_t q_row0, const int* min_bands, bool sync_only, Sched* best, int* best_S, int* best_kind) {
    static const int cand[] = {1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 14, 16, 20, 24, 28, 32, 40, 48, 64};
    const int max_slots = KB_KNN_MAX_CAND / p.kp;
    bool have = false;
    for (int S : cand) {
        if (S > p.n_tiles || S > max_slots) break;
        for (int kind = 0; kind < 2; ++kind) {
            if (sync_only && kind == 1) continue;
            if (S < min_bands[kind] && S < p.n_tiles && S < max_slots) continue;
            Sched s;
            build_sched(p, q_row0, S, kind, &s);
            if (s.slots > max_slots) continue;
            // fewer pieces win ties: every piece costs a list set-up and a write-back
            if (!have || s.makespan < best->makespan * 0.995) { *best = std::move(s); *best_S = S; *best_kind = kind; have = true; }
        }
    }
    if (!have) { build_sched(p, q_row0, 1, 0, best); *best_S = 1; *best_kind = 0; }
}

}  // namespace

int kb_knn_plan(int sm_count, int impl, int64_t nq, int64_t nk, int64_t q_row0, int32_t dp, int32_t k, int64_t n_flag, KbKnnPlan* p) {
    if (k < 1 || nq < 1 || nk < 1 || k > nk) { kb_set_error("kNN: need 1 <= k <= nk and nq >= 1"); return KB_EINVAL; }
    memset(p, 0, sizeof(*p));
    p->impl = impl;
    if (k > KB_KNN_K_MAX) {
        // no candidate kernel: every row goes through the exact pass over all keys (kb_knn_fixup)
        p->impl = 0; p->kp = 0; p->slots = 0;
    } else {
        // candidates kept per (row, slot): k plus a margin against fp32 ranking noise; K5 certifies every
        // row against the margin actually available, so the margin is a matter of speed, not of correctness
        p->kp = (k <= 2) ? 8 : (k <= 10 ? 16 : (k <= 18 ? 24 : (k <= 26 ? 32 : (k <= 42 ? 48 : 64))));
        if (impl == KB_KNN_TC) { p->bm = 128; p->bn = 256; }
        else { p->bm = 64; p->bn = 64; }
        p->m_blocks = (nq + p->bm - 1) / p->bm;
        p->n_tiles = (nk + p->bn - 1) / p->bn;
        p->nq = nq;
        p->piece_cost = std::min(1.5, std::max(0.25, 1.5 * 1088.0 / (double)dp));
        p->shard = (q_row0 > 0 || nq < nk) ? 1 : 0;
        if (impl == KB_KNN_TC) {
            // CTA pairs (k4_tc2), also for a lone query block: the second CTA of its pair has no live rows
            p->cl = 2;
            p->groups = (p->m_blocks + 1) / 2;
            int64_t w = sm_count / 2 > 0 ? sm_count / 2 : 1;
            const int64_t visits = p->groups * p->n_tiles;
            if (w > visits) w = visits;
            p->workers = (int)w;
            Sched s; int S = 1, kind = 0;
            // B200: 126 MB of L2.  A key set that fills a good part of it is swept in bands that all workers share
            // (measured in place, i.e. with the L2 cold after K1-K3: 50k x 1088 keys = 109 MB, one band cut into
            // ranges 3.30 ms, three whole bands dealt round-robin 3.13 ms); beyond the L2 only whole bands are dealt.
            const double l2_mb = 120.0;
            const double key_bytes = (double)nk * dp * 2.0;
            const bool sync_only = key_bytes > l2_mb * 1e6;
            const bool shard = p->shard != 0;                        // arrival order: at least 4 bands
            const int min_bands[2] = {key_bytes > 0.5 * l2_mb * 1e6 ? 2 : (shard ? 4 : 1),
                                      (key_bytes > 0.5 * l2_mb * 1e6 || shard) ? 4 : 1};
            choose_sched(*p, q_row0, min_bands, sync_only, &s, &S, &kind);
            p->slots = s.slots; p->bands = S; p->sched_kind = kind; p->n_pieces = s.n_pieces; p->makespan = s.makespan;
        } else {
            // SIMT: grid (m_blocks, slots); enough slots to fill the machine, at most 8 tiles per... keep it simple
            p->cl = 1; p->groups = p->m_blocks; p->workers = 0;
            int64_t want = ((int64_t)sm_count * 2 + p->m_blocks - 1) / p->m_blocks;
            const int64_t max_slots = KB_KNN_MAX_CAND / p->kp < 32 ? KB_KNN_MAX_CAND / p->kp : 32;
            if (want > max_slots) want = max_slots;
            if (want > p->n_tiles) want = p->n_tiles;
            if (want < 1) want = 1;
            p->slots = (int)want; p->bands = (int)want;
        }
    }
    int64_t off = 0;
    const int64_t cand = nq * (int64_t)p->slots * p->kp;
    p->off_score = off;   off += kb_round_up(cand * (int64_t)sizeof(float), 256);
    p->off_idx = off;     off += kb_round_up(cand * (int64_t)sizeof(int32_t), 256);
    p->off_rowthr = off;  off += kb_round_up(nq * (int64_t)sizeof(int32_t), 256);
    p->off_xidx = off;    off += (n_flag > 0 && p->kp) ? kb_round_up(nq * p->kp * (int64_t)sizeof(int32_t), 256) : 0;
    p->off_xd2 = off;     off += (n_flag > 0 && p->kp) ? kb_round_up(nq * p->kp * (int64_t)sizeof(double), 256) : 0;
    p->off_uncert = off;  off += kb_round_up((nq + 4) * (int64_t)sizeof(int32_t), 256);    // [0] count, [1] Gram entries recomputed by K5, [4..] rows
    p->total = off;
    return KB_OK;
}

void kb_knn_plan_pieces(const KbKnnPlan& p, int64_t q_row0, KbPiece* pieces, int32_t* piece_start, int32_t* slot_count) {
    Sched s;
    build_sched(p, q_row0, p.bands, p.sched_kind, &s);      // same inputs -> the schedule the plan chose
    int64_t at = 0;
    for (int w = 0; w < p.workers; ++w) {
        piece_start[w] = (int32_t)at;
        for (const KbPiece& pc : s.per_worker[w]) pieces[at++] = pc;
    }
    piece_start[p.workers] = (int32_t)at;
    for (int64_t g = 0; g < p.groups; ++g) slot_count[g] = s.slot_count[g];
}

// Per-context cache of plans and (tensor path) uploaded piece tables [pieces | piece_start | slot_count],
// keyed by the plan inputs: planning walks every (band, group) unit, which is not free for a million rows.
struct KbKnnEntry {
    bool used;
    int impl; int64_t nq, nk, q_row0, n_flag; int32_t k, dp; int sm;
    KbKnnPlan plan;
    void* d; int64_t off_start, off_slots;
    uint64_t stamp;
};
struct KbKnnCache { KbKnnEntry e[8]; uint64_t clock; };

void kb_knn_cache_free(kb_ctx* c) {
    KbKnnCache* cache = reinterpret_cast<KbKnnCache*>(c->knn_cache);
    if (!cache) return;
    for (auto& t : cache->e) if (t.d) cudaFree(t.d);
    free(cache);
    c->knn_cache = nullptr;
}

static int plan_cached(kb_ctx* ctx, int impl, int64_t nq, int64_t nk, int64_t q_row0, int32_t dp, int32_t k, int64_t n_flag, KbKnnEntry** out) {
    if (!ctx->knn_cache) {
        ctx->knn_cache = calloc(1, sizeof(KbKnnCache));
        if (!ctx->knn_cache) { kb_set_error("out of host memory"); return KB_EINVAL; }
    }
    KbKnnCache* cache = reinterpret_cast<KbKnnCache*>(ctx->knn_cache);
    KbKnnEntry* lru = &cache->e[0];
    for (auto& t : cache->e) {
        if (t.used && t.impl == impl && t.nq == nq && t.nk == nk && t.q_row0 == q_row0 && t.dp == dp && t.k == k && t.n_flag == n_flag &&
            t.sm == ctx->sm_count) {
            t.stamp = ++cache->clock; *out = &t; return KB_OK;
        }
        if (t.stamp < lru->stamp) lru = &t;
    }
    KbKnnPlan p;
    int rc = kb_knn_plan(ctx->sm_count, impl, nq, nk, q_row0, dp, k, n_flag, &p);
    if (rc) return rc;
    if (lru->d) { KB_CUDA(cudaStreamSynchronize(ctx->stream)); KB_CUDA(cudaFree(lru->d)); lru->d = nullptr; }
    lru->used = true; lru->impl = impl; lru->nq = nq; lru->nk = nk; lru->q_row0 = q_row0; lru->n_flag = n_flag; lru->k = k; lru->dp = dp;
    lru->sm = ctx->sm_count; lru->plan = p; lru->stamp = ++cache->clock;
    *out = lru;
    return KB_OK;
}

// tensor path: build the piece table on the host and upload it synchronously (once per shape; warm up
// before capturing a CUDA graph)
static int table_cached(kb_ctx* ctx, KbKnnEntry* e) {
    if (e->d) return KB_OK;
    const KbKnnPlan& p = e->plan;
    std::vector<KbPiece> pieces((size_t)p.n_pieces);
    std::vector<int32_t> start((size_t)p.workers + 1), slots((size_t)p.groups);
    kb_knn_plan_pieces(p, e->q_row0, pieces.data(), start.data(), slots.data());
    const int64_t off_start = kb_round_up(p.n_pieces * (int64_t)sizeof(KbPiece), 256);
    const int64_t off_slots = off_start + kb_round_up((p.workers + 1) * (int64_t)sizeof(int32_t), 256);
    const int64_t bytes = off_slots + kb_round_up(p.groups * (int64_t)sizeof(int32_t), 256);
    void* dv = nullptr;
    KB_CUDA(cudaMalloc(&dv, (size_t)bytes));
    uint8_t* d = reinterpret_cast<uint8_t*>(dv);
    KB_CUDA(cudaMemcpy(d, pieces.data(), pieces.size() * sizeof(KbPiece), cudaMemcpyHostToDevice));
    KB_CUDA(cudaMemcpy(d + off_start, start.data(), start.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    KB_CUDA(cudaMemcpy(d + off_slots, slots.data(), slots.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    e->d = dv; e->off_start = off_start; e->off_slots = off_slots;
    return KB_OK;
}

namespace {

__global__ void __launch_bounds__(256)
k4_init(int32_t* __restrict__ row_thr, int64_t nq, int32_t* __restrict__ uncert, int mark_all) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nq) {
        row_thr[j] = 0x7f800000;                              // +inf as an ordered-int key
        if (mark_all) uncert[4 + j] = (int32_t)j;
    }
    if (j == 0) { uncert[0] = mark_all ? (int32_t)nq : 0; uncert[1] = 0; }   // [1]: Gram entries K5 took from the operand rows
}

// ---------------------------------------------------------------------------
// K4-simt: 64x64 score tiles on the CUDA cores (checker / small inputs)
// dynamic shared memory: KP*64 floats + KP*64 ints (the lists)
// ---------------------------------------------------------------------------
template <int KP>
__global__ void __launch_bounds__(256)
k4_simt(const __half* __restrict__ op, int64_t ld, int32_t dp,
        const kb_rowmeta* __restrict__ rowmeta,
        int64_t nk, int64_t q_row0, int64_t nq, int splits, int64_t n_tiles,
        float* __restrict__ cand_score, int32_t* __restrict__ cand_idx) {
    constexpr int BM = 64, BN = 64, BK = 32;
    // operand tiles and the score tile share storage (the score tile is written
    // only after the last k-step of a tile has been consumed)
    __shared__ __align__(16) float ab[2 * BK * (BM + 4)];
    float (*As)[BM + 4] = reinterpret_cast<float (*)[BM + 4]>(ab);
    float (*Bs)[BN + 4] = reinterpret_cast<float (*)[BN + 4]>(ab + BK * (BM + 4));
    float (*tile)[BN + 1] = reinterpret_cast<float (*)[BN + 1]>(ab);
    static_assert(BM * (BN + 1) <= 2 * BK * (BM + 4), "score tile must fit in the operand tiles");
    extern __shared__ __align__(16) uint8_t dyn[];
    float* ls = reinterpret_cast<float*>(dyn);
    int32_t* li = reinterpret_cast<int32_t*>(dyn + KP * BM * sizeof(float));
    __shared__ float2 cms[BN];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int s = blockIdx.y;
    const int64_t t_lo = n_tiles * s / splits, t_hi = n_tiles * (s + 1) / splits;

    KbRowList<KP, BM> list(ls, li);
    float my_len = 1.f;
    if (tid < BM) {
        list.init(tid);
        const int64_t q = m0 + tid;
        if (q < nq) my_len = (float)rowmeta[q_row0 + q].key_len;
    }
    const int lrow = tid >> 2, lseg = (tid & 3) * 8;
    for (int64_t t = t_lo; t < t_hi; ++t) {
        const int64_t n0 = t * BN;
        float acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
        if (tid < BN) cms[tid] = kb_load_cm(rowmeta, n0 + tid, nk);
        for (int k0 = 0; k0 < dp; k0 += BK) {
            uint4 va = make_uint4(0, 0, 0, 0), vb = make_uint4(0, 0, 0, 0);
            if (m0 + lrow < nq) va = *reinterpret_cast<const uint4*>(op + (q_row0 + m0 + lrow) * ld + k0 + lseg);
            if (n0 + lrow < nk) vb = *reinterpret_cast<const uint4*>(op + (n0 + lrow) * ld + k0 + lseg);
            const __half2* ha = reinterpret_cast<const __half2*>(&va);
            const __half2* hb = reinterpret_cast<const __half2*>(&vb);
            __syncthreads();
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 fa = __half22float2(ha[e]), fb = __half22float2(hb[e]);
                As[lseg + 2 * e][lrow] = fa.x; As[lseg + 2 * e + 1][lrow] = fa.y;
                Bs[lseg + 2 * e][lrow] = fb.x; Bs[lseg + 2 * e + 1][lrow] = fb.y;
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < BK; ++kk) {
                const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
                const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
                const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(av[x], bv[y], acc[x][y]);
            }
        }
        __syncthreads();
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) tile[ty * 4 + x][tx * 4 + y] = acc[x][y];
        __syncthreads();
        if (tid < BM) {
            for (int c = 0; c < BN; ++c) {
                const float sc = kb_score(tile[tid][c], cms[c], my_len);
                if (sc < list.bound) list.insert(tid, sc, (int32_t)(n0 + c));
            }
        }
        __syncthreads();
    }
    if (tid < BM && m0 + tid < nq) {
        const int64_t base = ((m0 + tid) * splits + s) * KP;
        for (int e = 0; e < KP; ++e) { cand_score[base + e] = ls[e * BM + tid]; cand_idx[base + e] = li[e * BM + tid]; }
    }
}

// ---------------------------------------------------------------------------
// K5: merge the per-slot candidate lists by score, rerank exactly, order, certify, emit.
// One warp per query row.  Lane l holds merged candidates l and l+32 (KP <= 64).
// ---------------------------------------------------------------------------
struct K5Peers { int32_t n; int32_t* const* idx; float* const* dist; };

#ifndef KB_K5_ALWAYS_DOT
#define KB_K5_ALWAYS_DOT 0     // 1: recompute every Gram entry from the operand rows (the pre-r02 rerank; A/B and checks)
#endif

// MAXC: candidates per lane the merge holds (slots*KP <= 32*MAXC; the launcher picks the smallest that fits)
template <int KP, int MAXC>
__global__ void __launch_bounds__(256)
k5_merge_rerank(const __half* __restrict__ op, int64_t ld, int32_t dp,
                const kb_rowmeta* __restrict__ rowmeta, int64_t q_row0, int64_t nq, int slots, int32_t k,
                const int32_t* __restrict__ slot_count, int rows_per_group,
                const float* __restrict__ cand_score, const int32_t* __restrict__ cand_idx,
                const int32_t* __restrict__ extra_idx, const double* __restrict__ extra_d2,
                int32_t* __restrict__ out_idx, float* __restrict__ out_dist, double* __restrict__ out_d2,
                int32_t* __restrict__ uncert, K5Peers peers) {
    constexpr int NS = (KP + 31) / 32;                       // merged candidates per lane
    const int lane = threadIdx.x & 31;
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= nq) return;
    const int my_slots = slot_count ? slot_count[q / rows_per_group] : slots;
    const int total = my_slots * KP;
    const float INF = __int_as_float(0x7f800000);
    // ---- 1. every lane takes candidates lane, lane+32, ... ; KP rounds of warp arg-min
    float cs[MAXC]; int32_t ci[MAXC];
    const int64_t cbase = q * (int64_t)slots * KP;
#pragma unroll
    for (int u = 0; u < MAXC; ++u) {
        const int e = lane + 32 * u;
        if (e < total) { cs[u] = cand_score[cbase + e]; ci[u] = cand_idx[cbase + e]; }
        else { cs[u] = INF; ci[u] = -1; }
        if (ci[u] < 0) cs[u] = INF;
    }
    int32_t my_idx[NS]; float my_sc[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) { my_idx[s] = -1; my_sc[s] = INF; }
    float m_last = INF;                                       // score of the KP-th merged candidate (+inf: fewer exist)
    for (int r = 0; r < KP; ++r) {
        float best = INF; int32_t bidx = 0x7fffffff; int bu = -1;
#pragma unroll
        for (int u = 0; u < MAXC; ++u)
            if (ci[u] >= 0 && (cs[u] < best || (cs[u] == best && ci[u] < bidx))) { best = cs[u]; bidx = ci[u]; bu = u; }
        // warp arg-min over (score, idx): two integer min-reductions (order-preserving key of the score, then the
        // index among the lanes that hold that score) instead of a 5-step shuffle ladder over three values
        const int32_t kb_ = __float_as_int(best);
        const int32_t kbest = kb_ >= 0 ? kb_ : kb_ ^ 0x7fffffff;
        const int32_t wk = __reduce_min_sync(0xffffffffu, kbest);
        const int32_t wi = __reduce_min_sync(0xffffffffu, kbest == wk ? bidx : 0x7fffffff);
        const int wl = __ffs(__ballot_sync(0xffffffffu, kbest == wk && bidx == wi)) - 1;
        const float wb = __int_as_float(wk >= 0 ? wk : wk ^ 0x7fffffff);
        if (wi == 0x7fffffff) break;                          // nothing left anywhere
        if (lane == wl) {
#pragma unroll
            for (int u = 0; u < MAXC; ++u) if (u == bu) ci[u] = -1;   // consume
        }
#pragma unroll
        for (int s = 0; s < NS; ++s) if (r == lane + 32 * s) { my_idx[s] = wi; my_sc[s] = wb; }
        if (r == KP - 1) m_last = wb;
    }
    // ---- 2. exact-side-path extras (rows the tensor path cannot score exactly): lane e also
    //         holds extra candidates e, e+32 with their exact d2.  A flagged QUERY keeps only extras.
    const int32_t self = (int32_t)(q_row0 + q);
    const kb_rowmeta mq = rowmeta[self];
    const bool q_flagged = (mq.flags & 3) != 0;
    int32_t x_idx[NS]; double x_d2[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) { x_idx[s] = -1; x_d2[s] = 0.0; }
    int n_extra = 0; double x_max = 0.0;
    if (extra_idx) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const int e = lane + 32 * s;
            if (e < KP) { x_idx[s] = extra_idx[q * KP + e]; x_d2[s] = extra_d2[q * KP + e]; }
            n_extra += __popc(__ballot_sync(0xffffffffu, x_idx[s] >= 0));
            double xm = x_idx[s] >= 0 ? x_d2[s] : 0.0;
            for (int o = 16; o > 0; o >>= 1) xm = fmax(xm, __shfl_xor_sync(0xffffffffu, xm, o));
            x_max = fmax(x_max, xm);
        }
        if (q_flagged) {
#pragma unroll
            for (int s = 0; s < NS; ++s) my_idx[s] = -1;
        }
    }
    // self must be a candidate: it replaces the last merged slot if it is missing
    bool has_self_l = false;
#pragma unroll
    for (int s = 0; s < NS; ++s) has_self_l |= (my_idx[s] == self || x_idx[s] == self);
    const unsigned has_self = __ballot_sync(0xffffffffu, has_self_l);
    if (!has_self) {
#pragma unroll
        for (int s = 0; s < NS; ++s) if (lane + 32 * s == KP - 1) my_idx[s] = self;
    }
    // ---- 3. exact distances.
    //   sum_c (a_c*lj - b_c*lq)^2 = lj^2*n_q + lq^2*n_j - 2*lj*lq*g,  g = sum_c a_c*b_c.
    //   Rows that reach this point are unflagged: counts <= 2048 and n < 2^24, hence g <= sqrt(n_q*n_j) < 2^24 is an
    //   integer the candidate kernels hold EXACTLY (fp32 accumulation of integer products), and the score they
    //   stored is s = RN(g*cm_x + RN(l_q*cm_y)) -- one FMUL, one FFMA (kb_score), both reproducible here.  So the
    //   Gram entry is read back out of the score instead of being recomputed from two 2*dp-byte operand rows:
    //   g0 = rint((s - t)/cm_x); RN(g*cm_x + t) is monotone in g, so when g0 reproduces s and g0-1, g0+1 do not,
    //   g0 is the only integer that maps to s, i.e. the Gram entry itself.  Candidates for which that test fails
    //   (score spacing coarser than |cm_x|: very long contigs against short keys) take the operand rows (the
    //   fp32 FMA chain below IS the exact integer dot product for unflagged rows).
    //   The three terms are exact integers in fp64 (< 2^53), so d2 has one rounding (the division).
    const __half* qrow = op + (int64_t)self * ld;
    const double lq = (double)mq.key_len;
    const float lqf = (float)mq.key_len;
    double my_d2[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) my_d2[s] = 0.0;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int32_t j = my_idx[s];
        bool need_dot = false;
        kb_rowmeta mj; mj.sqnorm = 0.0; mj.key_len = 1; mj.cm_x = -1.f; mj.cm_y = 0.f;
        if (lane + 32 * s < KP && j >= 0 && j != self) {      // d2(self) = 0 exactly
            mj = rowmeta[j];
            const float t = __fmul_rn(lqf, mj.cm_y);
            const float sc = my_sc[s];
            const float g = (float)rint(((double)sc - (double)t) / (double)mj.cm_x);
            const bool unique = g >= 0.f && g < 16777216.f && __fmaf_rn(g, mj.cm_x, t) == sc &&
                                __fmaf_rn(g + 1.f, mj.cm_x, t) != sc && __fmaf_rn(g - 1.f, mj.cm_x, t) != sc;
            if (unique && !KB_K5_ALWAYS_DOT) {
                const double lj = (double)mj.key_len;
                const double num = lj * lj * mq.sqnorm + lq * lq * mj.sqnorm - 2.0 * (lj * lq) * (double)g;
                my_d2[s] = num / ((lq * lj) * (lq * lj));
            } else {
                need_dot = true;
            }
        }
        unsigned todo = __ballot_sync(0xffffffffu, need_dot);
        while (todo) {                                        // all lanes cooperate on one candidate at a time
            const int e = __ffs(todo) - 1;
            todo &= todo - 1;
            const int32_t jj = __shfl_sync(0xffffffffu, j, e);
            const __half* krow = op + (int64_t)jj * ld;
            float g0 = 0.f, g1 = 0.f;
            for (int c = 8 * lane; c < dp; c += 256) {
                const uint4 a = *reinterpret_cast<const uint4*>(qrow + c);
                const uint4 b = *reinterpret_cast<const uint4*>(krow + c);
                const __half2* ha = reinterpret_cast<const __half2*>(&a);
                const __half2* hb = reinterpret_cast<const __half2*>(&b);
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    const float2 fa = __half22float2(ha[x]), fb = __half22float2(hb[x]);
                    g0 = fmaf(fa.x, fb.x, g0);
                    g1 = fmaf(fa.y, fb.y, g1);
                }
            }
            float g = g0 + g1;
            for (int o = 16; o > 0; o >>= 1) g += __shfl_xor_sync(0xffffffffu, g, o);
            if (lane == e) {
                const double lj = (double)mj.key_len;
                const double num = lj * lj * mq.sqnorm + lq * lq * mj.sqnorm - 2.0 * (lj * lq) * (double)g;
                my_d2[s] = num / ((lq * lj) * (lq * lj));
                atomicAdd(&uncert[1], 1);
            }
        }
    }
    // ---- 4. order: self first, then (d2, idx); rank by counting over both item sets
    bool valid_a[NS], valid_b[NS]; double key_a[NS], key_b[NS]; int rank_a[NS], rank_b[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const bool in = lane + 32 * s < KP;
        valid_a[s] = in && my_idx[s] >= 0;
        valid_b[s] = in && x_idx[s] >= 0;
        key_a[s] = (my_idx[s] == self) ? -1.0 : my_d2[s];
        key_b[s] = (x_idx[s] == self) ? -1.0 : x_d2[s];
        rank_a[s] = 0; rank_b[s] = 0;
    }
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        for (int e = 0; e < 32 && e + 32 * t < KP; ++e) {
            const int32_t oj = __shfl_sync(0xffffffffu, my_idx[t], e);
            const double od = __shfl_sync(0xffffffffu, key_a[t], e);
            const int32_t xj = __shfl_sync(0xffffffffu, x_idx[t], e);
            const double xd = __shfl_sync(0xffffffffu, key_b[t], e);
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const bool same = (s == t) && (e == lane);
                if (oj >= 0) {
                    if (!same && (od < key_a[s] || (od == key_a[s] && oj < my_idx[s]))) ++rank_a[s];
                    if (od < key_b[s] || (od == key_b[s] && oj < x_idx[s])) ++rank_b[s];
                }
                if (xj >= 0) {
                    if (xd < key_a[s] || (xd == key_a[s] && xj < my_idx[s])) ++rank_a[s];
                    if (!same && (xd < key_b[s] || (xd == key_b[s] && xj < x_idx[s]))) ++rank_b[s];
                }
            }
        }
    }
    int n_valid = 0;
    double dk = -2.0;                                          // d2 key of the k-th neighbour
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        n_valid += __popc(__ballot_sync(0xffffffffu, valid_a[s])) + __popc(__ballot_sync(0xffffffffu, valid_b[s]));
        if (valid_a[s] && rank_a[s] == k - 1) dk = key_a[s];
        if (valid_b[s] && rank_b[s] == k - 1) dk = key_b[s];
    }
    for (int o = 16; o > 0; o >>= 1) dk = fmax(dk, __shfl_xor_sync(0xffffffffu, dk, o));
    const int64_t grow = (int64_t)self * k;                   // row in the peers' gathered arrays
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        if (valid_a[s] && rank_a[s] < k) {
            const float dd = (float)sqrt(my_d2[s]);
            out_idx[q * k + rank_a[s]] = my_idx[s];
            out_dist[q * k + rank_a[s]] = dd;
            if (out_d2) out_d2[q * k + rank_a[s]] = my_d2[s];
            for (int pr = 0; pr < peers.n; ++pr) { peers.idx[pr][grow + rank_a[s]] = my_idx[s]; peers.dist[pr][grow + rank_a[s]] = dd; }
        }
        if (valid_b[s] && rank_b[s] < k) {
            const float dd = (float)sqrt(x_d2[s]);
            out_idx[q * k + rank_b[s]] = x_idx[s];
            out_dist[q * k + rank_b[s]] = dd;
            if (out_d2) out_d2[q * k + rank_b[s]] = x_d2[s];
            for (int pr = 0; pr < peers.n; ++pr) { peers.idx[pr][grow + rank_b[s]] = x_idx[s]; peers.dist[pr][grow + rank_b[s]] = dd; }
        }
    }
    // fewer valid candidates than k -> mark the rest
    for (int e = n_valid + lane; e < k; e += 32) {
        out_idx[q * k + e] = -1;
        out_dist[q * k + e] = INF;
        if (out_d2) out_d2[q * k + e] = (double)INF;
        for (int pr = 0; pr < peers.n; ++pr) { peers.idx[pr][grow + e] = -1; peers.dist[pr][grow + e] = INF; }
    }
    // ---- 5. certificate.  Every key that is not among the merged candidates has an fp32 score >= m_last.
    //   s_k = exact score of the k-th neighbour (s = l_q*d2 - n_q/l_q); a key j with a_j = l_q*n_j/l_j^2 > Y^2,
    //   Y = c + sqrt(c^2 + s_k), c^2 = n_q/l_q, has an exact score above s_k whatever its Gram entry is
    //   (Cauchy-Schwarz); for all other keys the fp32 evaluation error is at most E = 2^-22*(Y^2 + 2cY)
    //   (three roundings of 2^-24 on terms bounded by Y^2 and 2cY, a third on top for safety).
    //   Flagged keys only come through the extras (exact): if that list is full, the k-th neighbour must
    //   not be farther than its last entry.
    if (lane == 0) {
        // a flagged QUERY needs exact distances to every key: that is the exact pass (K6), which spreads one row over
        // many CTAs -- K4x only serves ordinary queries (their distances to the few flagged keys)
        bool ok = !q_flagged;
        if (!q_flagged) {
            if (n_valid < k) ok = (m_last == INF);
            else if (m_last != INF) {
                const double d2k = dk < 0.0 ? 0.0 : dk;
                const double c2 = mq.sqnorm / lq;
                const double sk = lq * d2k - c2;
                const double c = sqrt(c2);
                const double Y = c + sqrt(fmax(c2 + sk, 0.0));
                const double E = 2.384185791015625e-07 * (Y * Y + 2.0 * c * Y);
                // stated ties (SURVEY 8c, north_star): a key within 1e-5 relative of the k-th distance may stand in
                // for it; a quarter of that is granted here, so an unseen key is at worst 2.5e-6 closer (relative
                // in d2) than the k-th neighbour returned.  At d2 = 0 (exact duplicates) nothing is granted.
                const double tie = 2.5e-6 * lq * d2k;
                ok = sk + E < (double)m_last + tie;
            }
            if (ok && n_extra >= KP && n_valid >= k && dk > x_max) ok = false;
        }
        if (!ok) {
            const int pos = atomicAdd(&uncert[0], 1);
            uncert[4 + pos] = (int32_t)q;
        }
    }
}

// ---------------------------------------------------------------------------
// K4x: exact side path.  Rows whose counts do not fit the tensor path exactly
// (flags bit0: a count > 2048, bit1: sum c^2 >= 2^24 -- contigs beyond ~130 kb, long
// homopolymers) are "flagged": masked out of the Gram kernel and handled here from their
// true u32 counts (exact 64-bit integer Gram entries, fp64 only for the final d2).  Four query rows per CTA:
//   unflagged query -> exact d2 to every FLAGGED key; the KP best go to K5 as extra candidates
//   flagged query   -> nothing here: K5 lists it for the exact pass over all keys (K6, kb_knn_fixup)
// ---------------------------------------------------------------------------
// d2 = (l_j^2 n_i + l_i^2 n_j - 2 l_i l_j g) / (l_i l_j)^2 from the exact integers n_i, n_j (sum c^2) and g (sum c_i c_j).
// While every term stays below 2^51 the numerator is exact in fp64 (one rounding, the division); beyond that (key
// lengths in the thousands against contigs of hundreds of kb) it is formed in 128-bit integers first.
__device__ __forceinline__ double kb_d2_from_gram(double ni, int32_t li, double nj, int32_t lj, unsigned long long g) {
    const double dli = (double)li, dlj = (double)lj;
    const double a = dlj * dlj * ni, b = dli * dli * nj, c = 2.0 * (dli * dlj) * (double)g;
    const double den = (dli * dlj) * (dli * dlj);
    const double lim = 2251799813685248.0;                    // 2^51
    if (a < lim && b < lim && c < lim) return (a + b - c) / den;
    const unsigned __int128 A = (unsigned __int128)((unsigned long long)lj * (unsigned long long)lj) * (unsigned long long)ni;
    const unsigned __int128 B = (unsigned __int128)((unsigned long long)li * (unsigned long long)li) * (unsigned long long)nj;
    const unsigned __int128 C = (unsigned __int128)(2ull * (unsigned long long)li * (unsigned long long)lj) * g;
    const unsigned __int128 num = A + B >= C ? A + B - C : 0;               // Cauchy-Schwarz: never negative
    const double hi = (double)(unsigned long long)(num >> 64), lo = (double)(unsigned long long)num;
    return (hi * 18446744073709551616.0 + lo) / den;
}

__device__ __forceinline__ int find_slot(const int32_t* __restrict__ rows, int n, int32_t row) {
    int lo = 0, hi = n - 1;
    while (lo <= hi) {
        const int mid = (lo + hi) >> 1;
        const int32_t v = rows[mid];
        if (v == row) return mid;
        if (v < row) lo = mid + 1; else hi = mid - 1;
    }
    return -1;
}

// QB: query rows per CTA (4: every flagged key row read serves four queries; 1 when four rows of dp counts do not fit
// the shared memory, i.e. beyond ~10k columns)
template <int KP, int QB>
__global__ void __launch_bounds__(256)
k4x_exact(const __half* __restrict__ op, int64_t ld, int32_t dp, const kb_rowmeta* __restrict__ rowmeta,
          int64_t nk, int64_t q_row0, int64_t nq,
          const int32_t* __restrict__ flag_rows, const uint32_t* __restrict__ flag_counts, int64_t ld_fc,
          int32_t fc_cols, int32_t n_flag,
          int32_t* __restrict__ extra_idx, double* __restrict__ extra_d2) {
    extern __shared__ __align__(16) uint32_t qrows[];         // QB x dp exact counts of the query rows
    __shared__ double wl_d[8][QB][KP];                        // per warp and query: running KP best flagged keys
    __shared__ int32_t wl_i[8][QB][KP];
    __shared__ double q_n[QB]; __shared__ int32_t q_l[QB]; __shared__ int32_t q_ok[QB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double DINF = __longlong_as_double(0x7ff0000000000000LL);
    const bool vec = (ld_fc & 3) == 0 && (reinterpret_cast<uintptr_t>(flag_counts) & 15) == 0;
    const int nc = fc_cols < dp ? fc_cols : dp;
    const int n4 = vec ? (nc >> 2) : 0;
    for (int64_t qb = (int64_t)blockIdx.x * QB; qb < nq; qb += (int64_t)gridDim.x * QB) {
        __syncthreads();
        if (threadIdx.x < QB) {
            const int64_t q = qb + threadIdx.x;
            int ok = 0;
            if (q < nq) {
                const kb_rowmeta mq = rowmeta[q_row0 + q];
                // a flagged QUERY is listed by K5 for the exact pass over all keys (K6); nothing to propose here
                ok = (mq.flags & 3) == 0;
                q_n[threadIdx.x] = mq.sqnorm; q_l[threadIdx.x] = mq.key_len;
            }
            q_ok[threadIdx.x] = ok;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < QB; ++i) {
            const int64_t q = qb + i;
            if (q >= nq) continue;
            if (!q_ok[i]) {
                for (int e = threadIdx.x; e < KP; e += 256) { extra_idx[q * KP + e] = -1; extra_d2[q * KP + e] = DINF; }
                continue;
            }
            const __half* src = op + (q_row0 + q) * ld;
            for (int c = threadIdx.x; c < dp; c += 256) qrows[i * dp + c] = (uint32_t)__half2float(src[c]);
        }
        for (int e = threadIdx.x; e < 8 * QB * KP; e += 256) { (&wl_d[0][0][0])[e] = DINF; (&wl_i[0][0][0])[e] = -1; }
        __syncthreads();
        // lane i < QB keeps the list of query i of this warp: worst entry (value, position) in registers
        double thr = DINF; int pos = 0;
        const bool mine = lane < QB && q_ok[lane < QB ? lane : 0] && qb + lane < nq;
        for (int64_t t = warp; t < n_flag; t += 8) {
            const int32_t j = flag_rows[t];
            const kb_rowmeta mj = rowmeta[j];
            if (mj.flags & 8) continue;                        // padding row of a multi-rank gather
            // exact integer Gram entries g_i = sum_c a_ic*b_c (u32 x u32 -> u64 multiply-adds)
            unsigned long long g[QB];
#pragma unroll
            for (int i = 0; i < QB; ++i) g[i] = 0ull;
            const uint32_t* krow = flag_counts + t * ld_fc;    // keys are the flagged rows, in flag_rows order
            const uint4* k4 = reinterpret_cast<const uint4*>(krow);
            for (int c = lane; c < n4; c += 32) {
                const uint4 b = __ldg(k4 + c);
#pragma unroll
                for (int i = 0; i < QB; ++i) {
                    const uint4 a = reinterpret_cast<const uint4*>(qrows + i * dp)[c];
                    g[i] += (unsigned long long)a.x * b.x; g[i] += (unsigned long long)a.y * b.y;
                    g[i] += (unsigned long long)a.z * b.z; g[i] += (unsigned long long)a.w * b.w;
                }
            }
            for (int c = (n4 << 2) + lane; c < nc; c += 32) {
                const uint32_t b = __ldg(krow + c);
#pragma unroll
                for (int i = 0; i < QB; ++i) g[i] += (unsigned long long)qrows[i * dp + c] * b;
            }
#pragma unroll
            for (int i = 0; i < QB; ++i)
                for (int o = 16; o > 0; o >>= 1) g[i] += __shfl_xor_sync(0xffffffffu, g[i], o);
            if (mine) {
                unsigned long long gm = g[0];
#pragma unroll
                for (int i = 1; i < QB; ++i) if (lane == i) gm = g[i];
                const double d2 = kb_d2_from_gram(q_n[lane], q_l[lane], mj.sqnorm, mj.key_len, gm);
                if (d2 < thr || (d2 == thr && wl_i[warp][lane][pos] < 0)) {
                    wl_d[warp][lane][pos] = d2; wl_i[warp][lane][pos] = j;
                    double m = -1.0; int mp = 0;
                    for (int e = 0; e < KP; ++e) {
                        const double x = wl_i[warp][lane][e] < 0 ? DINF : wl_d[warp][lane][e];
                        if (x > m) { m = x; mp = e; }
                    }
                    thr = m; pos = mp;
                }
            }
        }
        __syncthreads();
        // merge the 8 warp lists of query `warp` (warps 0..QB-1): KP rounds of arg-min over 8*KP entries
        if (warp < QB && q_ok[warp] && qb + warp < nq) {
            const int64_t q = qb + warp;
            for (int r = 0; r < KP; ++r) {
                double best = DINF; int32_t bi = 0x7fffffff; int bslot = -1;
                for (int e = lane; e < 8 * KP; e += 32) {
                    const int32_t ii = wl_i[e / KP][warp][e % KP];
                    const double dd = wl_d[e / KP][warp][e % KP];
                    if (ii >= 0 && (dd < best || (dd == best && ii < bi))) { best = dd; bi = ii; bslot = e; }
                }
                for (int o = 16; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const int32_t oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    const int os = __shfl_xor_sync(0xffffffffu, bslot, o);
                    if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; bslot = os; }
                }
                if (lane == 0) {
                    extra_idx[q * KP + r] = (bslot >= 0) ? bi : -1;
                    extra_d2[q * KP + r] = (bslot >= 0) ? best : DINF;
                    if (bslot >= 0) wl_i[bslot / KP][warp][bslot % KP] = -1;
                }
                __syncwarp();
            }
        }
    }
}

// ---------------------------------------------------------------------------
// K6: exact pass over ALL keys for the rows K5 could not certify (and for every row when
// k > KB_KNN_K_MAX).  k6_dist: one CTA per (K6_QB listed queries, chunk of keys); a warp takes one key
// row at a time and produces its exact d2 to the K6_QB queries (4; 2 or 1 when four rows of dp counts do not fit the
// shared memory: -k 7 has 16384 columns).  The rows are then ordered by a segmented radix sort on (d2, key index);
// k6_emit writes the first k of every segment.
// ---------------------------------------------------------------------------
template <int K6_QB>
__global__ void __launch_bounds__(256)
k6_dist(const __half* __restrict__ op, int64_t ld, int32_t dp, const kb_rowmeta* __restrict__ rowmeta,
        int64_t nk, int64_t q_row0, const int32_t* __restrict__ rows, int64_t row_lo, int64_t n_rows,
        const int32_t* __restrict__ flag_rows, const uint32_t* __restrict__ flag_counts, int64_t ld_fc,
        int32_t fc_cols, int32_t n_flag, int64_t keys_per_cta,
        double* __restrict__ d2_out, int32_t* __restrict__ idx_out) {
    // K6_QB x dp query counts: as floats (exact <= 2^24) when no listed row of this CTA is flagged -- then the fp32 dot
    // product against an ordinary key IS the exact integer Gram entry --, as u32 when one is (integer path for every key)
    extern __shared__ __align__(16) float qs[];
    uint32_t* qu = reinterpret_cast<uint32_t*>(qs);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t b0 = (int64_t)blockIdx.x * K6_QB;           // first listed row of this CTA (relative to row_lo)
    const double DINF = __longlong_as_double(0x7ff0000000000000LL);
    int32_t selfs[K6_QB]; double lqs[K6_QB], nqs[K6_QB]; bool qf[K6_QB], live[K6_QB];
    bool cta_f = false;
#pragma unroll
    for (int i = 0; i < K6_QB; ++i) {
        live[i] = b0 + i < n_rows;
        selfs[i] = live[i] ? (int32_t)(q_row0 + rows[row_lo + b0 + i]) : 0;
        const kb_rowmeta m = rowmeta[selfs[i]];
        lqs[i] = (double)m.key_len; nqs[i] = m.sqnorm; qf[i] = live[i] && (m.flags & 3) != 0;
        cta_f |= qf[i];
    }
#pragma unroll
    for (int i = 0; i < K6_QB; ++i) {
        if (qf[i]) {
            const int slot = find_slot(flag_rows, n_flag, selfs[i]);
            for (int c = threadIdx.x; c < dp; c += 256)
                qu[i * dp + c] = (slot >= 0 && c < fc_cols) ? flag_counts[(int64_t)slot * ld_fc + c] : 0u;
        } else if (cta_f) {
            for (int c = threadIdx.x; c < dp; c += 256) qu[i * dp + c] = (uint32_t)__half2float(op[(int64_t)selfs[i] * ld + c]);
        } else {
            for (int c = threadIdx.x; c < dp; c += 256) qs[i * dp + c] = __half2float(op[(int64_t)selfs[i] * ld + c]);
        }
    }
    __syncthreads();
    const bool fvec = (ld_fc & 3) == 0 && (reinterpret_cast<uintptr_t>(flag_counts) & 15) == 0;
    const int nfc = fc_cols < dp ? fc_cols : dp;
    const int64_t j_lo = (int64_t)blockIdx.y * keys_per_cta;
    const int64_t j_hi = (j_lo + keys_per_cta < nk) ? j_lo + keys_per_cta : nk;
    for (int64_t j = j_lo + warp; j < j_hi; j += 8) {
        const kb_rowmeta mj = rowmeta[j];
        const bool kf = (mj.flags & 3) != 0;
        const bool pad = (mj.flags & 8) != 0;
        const bool any_f = kf || cta_f;
        unsigned long long gi[K6_QB];                         // exact Gram entries (after the reduction: in every lane)
#pragma unroll
        for (int i = 0; i < K6_QB; ++i) gi[i] = 0ull;
        if (!pad) {
            if (any_f) {
                // a flagged row is involved: exact 64-bit integer Gram entries from the true counts
                if (kf) {
                    const int slot = find_slot(flag_rows, n_flag, (int32_t)j);
                    if (slot >= 0) {
                        const uint32_t* krow = flag_counts + (int64_t)slot * ld_fc;
                        const int n4 = (fvec && cta_f) ? (nfc >> 2) : 0;
                        const uint4* k4 = reinterpret_cast<const uint4*>(krow);
                        for (int c = lane; c < n4; c += 32) {
                            const uint4 b = __ldg(k4 + c);
#pragma unroll
                            for (int i = 0; i < K6_QB; ++i) {
                                const uint4 a = reinterpret_cast<const uint4*>(qu + i * dp)[c];
                                gi[i] += (unsigned long long)a.x * b.x; gi[i] += (unsigned long long)a.y * b.y;
                                gi[i] += (unsigned long long)a.z * b.z; gi[i] += (unsigned long long)a.w * b.w;
                            }
                        }
                        for (int c = (n4 << 2) + lane; c < nfc; c += 32) {
                            const uint32_t b = __ldg(krow + c);
#pragma unroll
                            for (int i = 0; i < K6_QB; ++i)
                                gi[i] += (unsigned long long)(cta_f ? qu[i * dp + c] : __float2uint_rn(qs[i * dp + c])) * b;
                        }
                    }
                } else {
                    // ordinary key (fp16 counts, exact integers <= 2048) against u32 query rows: 8 columns per load
                    const uint4* k8 = reinterpret_cast<const uint4*>(op + j * ld);
                    for (int c = lane; c < (dp >> 3); c += 32) {
                        const uint4 b = __ldg(k8 + c);
                        const __half2* hb = reinterpret_cast<const __half2*>(&b);
                        const float2 f0 = __half22float2(hb[0]), f1 = __half22float2(hb[1]), f2 = __half22float2(hb[2]), f3 = __half22float2(hb[3]);
                        const uint32_t b0 = (uint32_t)f0.x, b1 = (uint32_t)f0.y, b2 = (uint32_t)f1.x, b3 = (uint32_t)f1.y;
                        const uint32_t b4 = (uint32_t)f2.x, b5 = (uint32_t)f2.y, b6 = (uint32_t)f3.x, b7 = (uint32_t)f3.y;
#pragma unroll
                        for (int i = 0; i < K6_QB; ++i) {
                            const uint4 a0 = reinterpret_cast<const uint4*>(qu + i * dp)[2 * c];
                            const uint4 a1 = reinterpret_cast<const uint4*>(qu + i * dp)[2 * c + 1];
                            gi[i] += (unsigned long long)a0.x * b0; gi[i] += (unsigned long long)a0.y * b1;
                            gi[i] += (unsigned long long)a0.z * b2; gi[i] += (unsigned long long)a0.w * b3;
                            gi[i] += (unsigned long long)a1.x * b4; gi[i] += (unsigned long long)a1.y * b5;
                            gi[i] += (unsigned long long)a1.z * b6; gi[i] += (unsigned long long)a1.w * b7;
                        }
                    }
                }
            } else {
                // unflagged x unflagged: the fp32 dot product is the exact integer Gram entry
                float g[K6_QB];
#pragma unroll
                for (int i = 0; i < K6_QB; ++i) g[i] = 0.f;
                const __half* krow = op + j * ld;
                for (int c = 8 * lane; c < dp; c += 256) {
                    const uint4 b = *reinterpret_cast<const uint4*>(krow + c);
                    const __half2* hb = reinterpret_cast<const __half2*>(&b);
#pragma unroll
                    for (int x = 0; x < 4; ++x) {
                        const float2 fb = __half22float2(hb[x]);
#pragma unroll
                        for (int i = 0; i < K6_QB; ++i) {
                            g[i] = fmaf(qs[i * dp + c + 2 * x], fb.x, g[i]);
                            g[i] = fmaf(qs[i * dp + c + 2 * x + 1], fb.y, g[i]);
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < K6_QB; ++i) gi[i] = (unsigned long long)g[i];   // per-lane partial sums are exact integers
            }
        }
#pragma unroll
        for (int i = 0; i < K6_QB; ++i)
            for (int o = 16; o > 0; o >>= 1) gi[i] += __shfl_xor_sync(0xffffffffu, gi[i], o);
        if (lane < K6_QB) {
            // lane i finishes listed row i
            unsigned long long gm = gi[0]; double nq_ = nqs[0], lq_ = lqs[0]; int32_t self_ = selfs[0]; bool live_ = live[0];
#pragma unroll
            for (int i = 1; i < K6_QB; ++i) if (lane == i) { gm = gi[i]; nq_ = nqs[i]; lq_ = lqs[i]; self_ = selfs[i]; live_ = live[i]; }
            if (live_) {
                double d2;
                if (pad) d2 = DINF;
                else if ((int32_t)j == self_) d2 = -1.0;                      // the point itself sorts first
                else d2 = kb_d2_from_gram(nq_, (int32_t)lq_, mj.sqnorm, mj.key_len, gm);
                d2_out[(b0 + lane) * nk + j] = d2;
                idx_out[(b0 + lane) * nk + j] = (int32_t)j;
            }
        }
    }
}

__global__ void __launch_bounds__(256)
k6_emit(const double* __restrict__ d2_sorted, const int32_t* __restrict__ idx_sorted, int64_t nk,
        const int32_t* __restrict__ rows, int64_t row_lo, int64_t n_rows, int32_t k,
        int32_t* __restrict__ out_idx, float* __restrict__ out_dist, double* __restrict__ out_d2) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_rows * k) return;
    const int64_t b = t / k; const int e = (int)(t % k);
    const int64_t q = rows[row_lo + b];
    double d2 = d2_sorted[b * nk + e];
    int32_t j = idx_sorted[b * nk + e];
    if (d2 < 0.0) d2 = 0.0;                                    // self
    if (isinf(d2)) j = -1;
    out_idx[q * k + e] = j;
    out_dist[q * k + e] = (float)sqrt(d2);
    if (out_d2) out_d2[q * k + e] = d2;
}

__global__ void k6_segments(int64_t nk, int64_t n, int64_t* __restrict__ seg) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) seg[i] = i * nk;
}

template <int KP>
int run_simt(kb_ctx* ctx, const KbKnnPlan& p, const __half* op, int64_t ld, int32_t dp,
             const kb_rowmeta* rowmeta, int64_t nk, int64_t q_row0, int64_t nq, uint8_t* ws) {
    dim3 grid((unsigned)p.m_blocks, (unsigned)p.slots);
    auto kern = k4_simt<KP>;
    const size_t smem = (size_t)KP * 64 * 8;
    static bool attr_set[16] = {false};
    if (!attr_set[ctx->device & 15]) {
        KB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[ctx->device & 15] = true;
    }
    kern<<<grid, 256, smem, ctx->stream>>>(op, ld, dp, rowmeta, nk, q_row0, nq, p.slots, p.n_tiles,
                                           reinterpret_cast<float*>(ws + p.off_score),
                                           reinterpret_cast<int32_t*>(ws + p.off_idx));
    ctx->launches++;
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}

template <int KP>
int run_rerank(kb_ctx* ctx, const KbKnnPlan& p, const __half* op, int64_t ld, int32_t dp,
               const kb_rowmeta* rowmeta, int64_t q_row0, int64_t nq, int32_t k, uint8_t* ws, bool extras,
               const int32_t* slot_count, int32_t* d_idx, float* d_dist, double* d_d2, K5Peers peers) {
    const int64_t grid = (nq + 7) / 8;
    const int per_lane = (p.slots * KP + 31) / 32;
#define K5_LAUNCH(MC)                                                                                              \
    k5_merge_rerank<KP, MC><<<(unsigned)grid, 256, 0, ctx->stream>>>(                                              \
        op, ld, dp, rowmeta, q_row0, nq, p.slots, k, slot_count, p.bm * p.cl,                                      \
        reinterpret_cast<const float*>(ws + p.off_score), reinterpret_cast<const int32_t*>(ws + p.off_idx),        \
        extras ? reinterpret_cast<const int32_t*>(ws + p.off_xidx) : nullptr,                                      \
        extras ? reinterpret_cast<const double*>(ws + p.off_xd2) : nullptr, d_idx, d_dist, d_d2,                   \
        reinterpret_cast<int32_t*>(ws + p.off_uncert), peers)
    if (per_lane <= 1) K5_LAUNCH(1);
    else if (per_lane <= 2) K5_LAUNCH(2);
    else if (per_lane <= 4) K5_LAUNCH(4);
    else if (per_lane <= 8) K5_LAUNCH(8);
    else K5_LAUNCH(KB_KNN_MAX_CAND / 32);
#undef K5_LAUNCH
    ctx->launches++;
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}

template <int KP, int QB>
int launch_exact(kb_ctx* ctx, const KbKnnPlan& p, const __half* op, int64_t ld, int32_t dp, const kb_rowmeta* rowmeta,
                 int64_t nk, int64_t q_row0, int64_t nq, const int32_t* flag_rows, const uint32_t* flag_counts,
                 int64_t ld_fc, int32_t fc_cols, int32_t n_flag, uint8_t* ws) {
    auto kern = k4x_exact<KP, QB>;
    const size_t smem = (size_t)QB * dp * sizeof(uint32_t);
    KB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t blocks = (nq + QB - 1) / QB;
    const int64_t grid = blocks < (int64_t)ctx->sm_count * 8 ? blocks : (int64_t)ctx->sm_count * 8;
    kern<<<(unsigned)grid, 256, smem, ctx->stream>>>(op, ld, dp, rowmeta, nk, q_row0, nq, flag_rows, flag_counts, ld_fc,
                                                     fc_cols, n_flag, reinterpret_cast<int32_t*>(ws + p.off_xidx),
                                                     reinterpret_cast<double*>(ws + p.off_xd2));
    ctx->launches++;
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}

template <int KP>
int run_exact(kb_ctx* ctx, const KbKnnPlan& p, const __half* op, int64_t ld, int32_t dp, const kb_rowmeta* rowmeta,
              int64_t nk, int64_t q_row0, int64_t nq, const int32_t* flag_rows, const uint32_t* flag_counts,
              int64_t ld_fc, int32_t fc_cols, int32_t n_flag, uint8_t* ws) {
    if ((size_t)4 * dp * sizeof(uint32_t) <= 160 * 1024) return launch_exact<KP, 4>(ctx, p, op, ld, dp, rowmeta, nk, q_row0, nq, flag_rows, flag_counts, ld_fc, fc_cols, n_flag, ws);
    return launch_exact<KP, 1>(ctx, p, op, ld, dp, rowmeta, nk, q_row0, nq, flag_rows, flag_counts, ld_fc, fc_cols, n_flag, ws);
}

#define KB_KP_SWITCH(kp, CALL)                 \
    switch (kp) {                              \
        case 8: rc = CALL(8); break;           \
        case 16: rc = CALL(16); break;         \
        case 24: rc = CALL(24); break;         \
        case 32: rc = CALL(32); break;         \
        case 48: rc = CALL(48); break;         \
        default: rc = CALL(64); break;         \
    }

int check_args(kb_ctx* ctx, int& impl, int32_t k, const void* d_operand, int64_t ld_operand, int32_t d_cols_padded,
               const kb_rowmeta* d_rowmeta, int64_t nk, int64_t q_row0, int64_t nq, const int32_t* d_flag_rows,
               const uint32_t* d_flag_counts, int64_t ld_flag_counts, int32_t flag_cols, int64_t n_flag,
               int32_t* d_idx, float* d_dist, void* d_workspace, int64_t workspace_bytes, KbKnnEntry** ent) {
    KB_CHECK_ARG(ctx && d_operand && d_rowmeta && d_idx && d_dist && d_workspace, "null pointer");
    KB_CHECK_ARG(d_cols_padded > 0 && (d_cols_padded % 64) == 0 && ld_operand >= d_cols_padded && (ld_operand % 8) == 0,
                 "operand columns must be padded to a multiple of 64");
    KB_CHECK_ARG(((uintptr_t)d_operand % 16) == 0, "operand must be 16-byte aligned");
    KB_CHECK_ARG(q_row0 >= 0 && nq >= 1 && q_row0 + nq <= nk, "query rows must be a sub-range of the keys");
    KB_CHECK_ARG(nk < (1LL << 31), "more than 2^31 keys");
    if (impl == KB_KNN_AUTO) impl = (nk >= 512) ? KB_KNN_TC : KB_KNN_SIMT;
    KB_CHECK_ARG(impl == KB_KNN_SIMT || impl == KB_KNN_TC, "impl");
    KB_CHECK_ARG(n_flag >= 0 && n_flag < (1LL << 31) && (n_flag == 0 || (d_flag_rows && d_flag_counts && ld_flag_counts >= flag_cols)),
                 "flagged-row side inputs");
    int rc = plan_cached(ctx, impl, nq, nk, q_row0, d_cols_padded, k, n_flag, ent);
    if (rc) return rc;
    const KbKnnPlan* p = &(*ent)->plan;
    if (p->slots * p->kp > KB_KNN_MAX_CAND) { kb_set_error("internal: too many candidates per row"); return KB_EUNSUPPORTED; }
    if (workspace_bytes < p->total) { kb_set_error("kNN workspace: need %lld bytes, got %lld", (long long)p->total, (long long)workspace_bytes); return KB_EWORKSPACE; }
    KB_CHECK_ARG(((uintptr_t)d_workspace % 256) == 0, "workspace must be 256-byte aligned");
    return KB_OK;
}

}  // namespace

extern "C" int64_t kb_knn_workspace_bytes(kb_ctx* ctx, int64_t nq, int64_t nk, int64_t q_row0, int32_t d_cols_padded, int32_t k, int impl, int64_t n_flag) {
    int64_t best = 0;
    for (int im = KB_KNN_SIMT; im <= KB_KNN_TC; ++im) {
        if (impl != KB_KNN_AUTO && impl != im) continue;
        KbKnnPlan p;
        if (ctx) {
            KbKnnEntry* ent = nullptr;
            int rc = plan_cached(ctx, im, nq, nk, q_row0, d_cols_padded, k, n_flag, &ent);
            if (rc) return rc;
            p = ent->plan;
        } else {
            int rc = kb_knn_plan(148, im, nq, nk, q_row0, d_cols_padded, k, n_flag, &p);   // no context: a 148-SM B200
            if (rc) return rc;
        }
        if (p.total > best) best = p.total;
    }
    return best;
}

// host-only view of the schedule (tests, diagnostics): fills out[0..7] = kp, slots, bands, kind, workers, pieces,
// makespan*1000, ideal*1000 (tile visits per worker)
extern "C" int kb_knn_plan_info(int sm_count, int impl, int64_t nq, int64_t nk, int64_t q_row0, int32_t d_cols_padded, int32_t k, int64_t* out) {
    KbKnnPlan p;
    int rc = kb_knn_plan(sm_count, impl, nq, nk, q_row0, d_cols_padded, k, 0, &p);
    if (rc) return rc;
    out[0] = p.kp; out[1] = p.slots; out[2] = p.bands; out[3] = p.sched_kind; out[4] = p.workers; out[5] = p.n_pieces;
    out[6] = (int64_t)(p.makespan * 1000.0);
    out[7] = p.workers ? (int64_t)(1000.0 * (double)p.groups * (double)p.n_tiles / p.workers) : 0;
    return KB_OK;
}

// host-only: the piece table itself, for coverage checks.  pieces: int32[n_pieces*8] (KbPiece), piece_start:
// int32[workers+1], slot_count: int32[groups]
extern "C" int kb_knn_plan_table(int sm_count, int impl, int64_t nq, int64_t nk, int64_t q_row0, int32_t d_cols_padded, int32_t k,
                                 int32_t* pieces, int32_t* piece_start, int32_t* slot_count) {
    KbKnnPlan p;
    int rc = kb_knn_plan(sm_count, impl, nq, nk, q_row0, d_cols_padded, k, 0, &p);
    if (rc) return rc;
    if (p.impl != KB_KNN_TC) { kb_set_error("piece tables belong to the tensor kernel"); return KB_EINVAL; }
    kb_knn_plan_pieces(p, q_row0, reinterpret_cast<KbPiece*>(pieces), piece_start, slot_count);
    return KB_OK;
}

extern "C" int kb_knn_uncertified_ptr(kb_ctx* ctx, int64_t nq, int64_t nk, int64_t q_row0, int32_t d_cols_padded, int32_t k, int impl, int64_t n_flag,
                                      void* d_workspace, const uint32_t** d_count) {
    KB_CHECK_ARG(ctx && d_workspace && d_count, "null pointer");
    if (impl == KB_KNN_AUTO) impl = (nk >= 512) ? KB_KNN_TC : KB_KNN_SIMT;
    KbKnnEntry* ent = nullptr;
    int rc = plan_cached(ctx, impl, nq, nk, q_row0, d_cols_padded, k, n_flag, &ent);
    if (rc) return rc;
    const KbKnnPlan& p = ent->plan;
    *d_count = reinterpret_cast<const uint32_t*>(reinterpret_cast<uint8_t*>(d_workspace) + p.off_uncert);
    return KB_OK;
}

extern "C" int kb_knn(kb_ctx* ctx, int impl, int32_t k,
                      const void* d_operand, int64_t ld_operand, int32_t d_cols_padded,
                      const kb_rowmeta* d_rowmeta,
                      int64_t nk, int64_t q_row0, int64_t nq,
                      const int32_t* d_flag_rows, const uint32_t* d_flag_counts, int64_t ld_flag_counts,
                      int32_t flag_cols, int64_t n_flag,
                      int32_t* d_idx, float* d_dist, double* d_d2,
                      void* d_workspace, int64_t workspace_bytes, const kb_knn_xchg* xchg) {
    KbKnnEntry* ent = nullptr;
    int rc = check_args(ctx, impl, k, d_operand, ld_operand, d_cols_padded, d_rowmeta, nk, q_row0, nq, d_flag_rows,
                        d_flag_counts, ld_flag_counts, flag_cols, n_flag, d_idx, d_dist, d_workspace, workspace_bytes, &ent);
    if (rc) return rc;
    const KbKnnPlan& p = ent->plan;
    uint8_t* ws = reinterpret_cast<uint8_t*>(d_workspace);
    const __half* op = reinterpret_cast<const __half*>(d_operand);
    int32_t* uncert = reinterpret_cast<int32_t*>(ws + p.off_uncert);

    k4_init<<<(unsigned)((nq + 255) / 256), 256, 0, ctx->stream>>>(reinterpret_cast<int32_t*>(ws + p.off_rowthr), nq, uncert,
                                                                   p.impl == 0 ? 1 : 0);
    ctx->launches++;
    KB_CUDA(cudaGetLastError());
    if (p.impl == 0) {
        KB_CHECK_ARG(!xchg || xchg->n_peers == 0, "peer result stores need k <= 60");
        return KB_OK;                                         // k > KB_KNN_K_MAX: kb_knn_fixup does all rows
    }
    const int32_t* slot_count = nullptr;
    {
        KbTimer t(ctx, 4);
        if (impl == KB_KNN_TC) {
            rc = table_cached(ctx, ent);
            if (rc) return rc;
            const uint8_t* d = reinterpret_cast<const uint8_t*>(ent->d);
            slot_count = reinterpret_cast<const int32_t*>(d + ent->off_slots);
            KbTcArgs a;
            a.d_operand = d_operand; a.ld_operand = ld_operand; a.d_cols_padded = d_cols_padded;
            a.d_rowmeta = d_rowmeta; a.nk = nk; a.q_row0 = q_row0; a.nq = nq;
            a.cand_score = reinterpret_cast<float*>(ws + p.off_score);
            a.cand_idx = reinterpret_cast<int32_t*>(ws + p.off_idx);
            a.row_thr = reinterpret_cast<int32_t*>(ws + p.off_rowthr);
            a.pieces = reinterpret_cast<const KbPiece*>(d);
            a.piece_start = reinterpret_cast<const int32_t*>(d + ent->off_start);
            a.d_arrive = xchg ? xchg->d_arrive : nullptr;
            a.d_epoch = xchg ? xchg->d_epoch : nullptr;
            a.rows_per_src = xchg ? xchg->rows_per_src : 0;
            a.self_rank = xchg ? xchg->self_rank : 0;
            rc = kb_knn_tc_launch(ctx, p, a);
        } else {
            KB_CHECK_ARG(!xchg || !xchg->d_arrive, "the SIMT kernel does not wait for peer shards");
#define CALL(KP) run_simt<KP>(ctx, p, op, ld_operand, d_cols_padded, d_rowmeta, nk, q_row0, nq, ws)
            KB_KP_SWITCH(p.kp, CALL)
#undef CALL
        }
        if (rc) return rc;
    }
    const bool extras = n_flag > 0;
    if (extras) {
        KbTimer t(ctx, 6);
#define CALL(KP) run_exact<KP>(ctx, p, op, ld_operand, d_cols_padded, d_rowmeta, nk, q_row0, nq, d_flag_rows, d_flag_counts, ld_flag_counts, flag_cols, (int32_t)n_flag, ws)
        KB_KP_SWITCH(p.kp, CALL)
#undef CALL
        if (rc) return rc;
    }
    {
        KbTimer t(ctx, 5);
        K5Peers peers;
        peers.n = xchg ? xchg->n_peers : 0;
        peers.idx = xchg ? xchg->d_peer_idx : nullptr;
        peers.dist = xchg ? xchg->d_peer_dist : nullptr;
#define CALL(KP) run_rerank<KP>(ctx, p, op, ld_operand, d_cols_padded, d_rowmeta, q_row0, nq, k, ws, extras, slot_count, d_idx, d_dist, d_d2, peers)
        KB_KP_SWITCH(p.kp, CALL)
#undef CALL
    }
    return rc;
}

extern "C" int64_t kb_knn_fixup(kb_ctx* ctx, int impl, int32_t k,
                                const void* d_operand, int64_t ld_operand, int32_t d_cols_padded,
                                const kb_rowmeta* d_rowmeta,
                                int64_t nk, int64_t q_row0, int64_t nq,
                                const int32_t* d_flag_rows, const uint32_t* d_flag_counts, int64_t ld_flag_counts,
                                int32_t flag_cols, int64_t n_flag,
                                int32_t* d_idx, float* d_dist, double* d_d2,
                                void* d_workspace, int64_t workspace_bytes) {
    KbKnnEntry* ent = nullptr;
    int rc = check_args(ctx, impl, k, d_operand, ld_operand, d_cols_padded, d_rowmeta, nk, q_row0, nq, d_flag_rows,
                        d_flag_counts, ld_flag_counts, flag_cols, n_flag, d_idx, d_dist, d_workspace, workspace_bytes, &ent);
    if (rc) return rc;
    const KbKnnPlan& p = ent->plan;
    uint8_t* ws = reinterpret_cast<uint8_t*>(d_workspace);
    const int32_t* uncert = reinterpret_cast<const int32_t*>(ws + p.off_uncert);
    int32_t n_rows = 0;
    KB_CUDA(cudaMemcpyAsync(&n_rows, uncert, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    KB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (n_rows <= 0) return 0;
    if (n_rows > nq) n_rows = (int32_t)nq;
    const __half* op = reinterpret_cast<const __half*>(d_operand);
    const int32_t* rows = uncert + 4;
    // batches sized for ~1 GB of scratch: (d2 f64 + idx i32) x 2 (sort double buffers) per (row, key)
    int64_t batch = (1LL << 30) / (nk * 24);
    // listed rows per CTA: as many (4, 2, 1) as fit the shared memory with their dp counts each
    const int qb = (size_t)4 * d_cols_padded * sizeof(float) <= 200 * 1024 ? 4 : ((size_t)2 * d_cols_padded * sizeof(float) <= 200 * 1024 ? 2 : 1);
    if ((size_t)qb * d_cols_padded * sizeof(float) > 227 * 1024) { kb_set_error("exact pass: %d columns do not fit the shared memory", (int)d_cols_padded); return KB_EUNSUPPORTED; }
    if (batch < qb) batch = qb;
    batch = batch / qb * qb;
    if (batch > n_rows) batch = kb_round_up(n_rows, qb);
    cudaMemPool_t pool;
    rc = kb_pool_get(ctx, &pool);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    double *d2a = nullptr, *d2b = nullptr; int32_t *ia = nullptr, *ib = nullptr; int64_t* seg = nullptr; void* tmp = nullptr;
    const size_t cells = (size_t)batch * (size_t)nk;
    KB_CUDA(cudaMallocFromPoolAsync((void**)&d2a, cells * 8, pool, st));
    KB_CUDA(cudaMallocFromPoolAsync((void**)&d2b, cells * 8, pool, st));
    KB_CUDA(cudaMallocFromPoolAsync((void**)&ia, cells * 4, pool, st));
    KB_CUDA(cudaMallocFromPoolAsync((void**)&ib, cells * 4, pool, st));
    KB_CUDA(cudaMallocFromPoolAsync((void**)&seg, (size_t)(batch + 1) * 8, pool, st));
    size_t tmp_bytes = 0;
    cub::DeviceSegmentedRadixSort::SortPairs(nullptr, tmp_bytes, d2a, d2b, ia, ib, (int64_t)cells, (int)batch, seg, seg + 1, 0, 64, st);
    KB_CUDA(cudaMallocFromPoolAsync(&tmp, tmp_bytes ? tmp_bytes : 16, pool, st));
    const size_t smem = (size_t)qb * d_cols_padded * sizeof(float);
    if (qb == 4) { KB_CUDA(cudaFuncSetAttribute(k6_dist<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); }
    else if (qb == 2) { KB_CUDA(cudaFuncSetAttribute(k6_dist<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); }
    else { KB_CUDA(cudaFuncSetAttribute(k6_dist<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); }
    {
        KbTimer t(ctx, 6);
        for (int64_t lo = 0; lo < n_rows; lo += batch) {
            const int64_t nb = (n_rows - lo < batch) ? n_rows - lo : batch;
            const int64_t q_ctas = (nb + qb - 1) / qb;
            int64_t key_ctas = ((int64_t)ctx->sm_count * 8 + q_ctas - 1) / q_ctas;        // enough CTAs to fill the GPU
            if (key_ctas > (nk + 63) / 64) key_ctas = (nk + 63) / 64;
            if (key_ctas < 1) key_ctas = 1;
            if (key_ctas > 65535) key_ctas = 65535;
            const int64_t keys_per_cta = (nk + key_ctas - 1) / key_ctas;
#define K6_LAUNCH(QB)                                                                                                 \
    k6_dist<QB><<<dim3((unsigned)q_ctas, (unsigned)key_ctas), 256, smem, st>>>(                                        \
        op, ld_operand, d_cols_padded, d_rowmeta, nk, q_row0, rows, lo, nb, d_flag_rows, d_flag_counts,                \
        ld_flag_counts, flag_cols, (int32_t)n_flag, keys_per_cta, d2a, ia)
            if (qb == 4) K6_LAUNCH(4); else if (qb == 2) K6_LAUNCH(2); else K6_LAUNCH(1);
#undef K6_LAUNCH
            ctx->launches++;
            KB_CUDA(cudaGetLastError());
            k6_segments<<<(unsigned)((nb + 256) / 256), 256, 0, st>>>(nk, nb, seg);
            ctx->launches++;
            // stable LSD radix sort on the fp64 keys: ties keep ascending key index
            KB_CUDA(cub::DeviceSegmentedRadixSort::SortPairs(tmp, tmp_bytes, d2a, d2b, ia, ib, (int64_t)(nb * nk), (int)nb, seg, seg + 1, 0, 64, st));
            ctx->launches += 2;
            k6_emit<<<(unsigned)((nb * k + 255) / 256), 256, 0, st>>>(d2b, ib, nk, rows, lo, nb, k, d_idx, d_dist, d_d2);
            ctx->launches++;
            KB_CUDA(cudaGetLastError());
        }
    }
    KB_CUDA(cudaFreeAsync(d2a, st)); KB_CUDA(cudaFreeAsync(d2b, st)); KB_CUDA(cudaFreeAsync(ia, st));
    KB_CUDA(cudaFreeAsync(ib, st)); KB_CUDA(cudaFreeAsync(seg, st)); KB_CUDA(cudaFreeAsync(tmp, st));
    KB_CUDA(cudaStreamSynchronize(st));
    return n_rows;
}
