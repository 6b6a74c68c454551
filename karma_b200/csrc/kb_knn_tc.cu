// kb_knn_tc.cu -- K4: distance GEMM on tcgen05 tensor cores with a fused per-row
// top-k' epilogue (sm_100a only).
//
// Replaces the O(N^2 D) neighbour search inside umap.UMAP(...).fit_transform at
// /root/reference/karma/kmer.py:285-290.
//
//   G = C_q * C_k^T     C = raw k-mer counts as fp16 (exact <= 2048), fp32 accumulate
//                       in TMEM (exact integer Gram while sum c^2 < 2^24)
//   score_ij = fma(G_ij, -2/l_j, l_i * n_j/l_j^2)   ( = l_i*d2_ij - n_i/l_i )
//
// k4_tc2: persistent CTA pairs (clusters of 2, one CTA per SM), 6 warps per CTA, ONE 2-CTA MMA per pair:
//   warp 0      TMA producer (both CTAs): the CTA's 128 query rows x 64 (A) and its half of the key tile,
//               128 rows x 64 (B), fp16 boxes, SWIZZLE_128B, STAGES-deep mbarrier ring (32 KB per stage)
//   warp 1      TMEM allocator (both CTAs) + single-thread tcgen05.mma issuer in the leader CTA
//               (cta_group::2, kind::f16, M=256 N=256 K=16), accumulators double buffered in TMEM
//               (2 x 256 columns per SM)
//   warps 2-5   epilogue of the CTA's own 128 rows: tcgen05.ld 32 lanes x 32 columns, one thread per
//               query row; running top-KP list per row in shared memory
// Work = a host-built table of pieces per CTA pair (kb_knn.cuh: KbPiece): a group of two adjacent 128-row
// query blocks against a run of key tiles; each piece writes KP candidates per row into its slot, merged and
// exactly reranked by K5 (kb_knn.cu).  A group whose second block has no live rows (an odd number of query
// blocks, or a query range of at most 128 rows) still runs as a pair; the idle CTA's rows are never written.
// With a peer-memory exchange the TMA producer (and the epilogue, for the key records) waits for the arrival
// flag of the rank that owns a key row before touching it, so the sweep starts on the local shard while the
// other shards are still in flight over NVLink.
//
// Roofline: tensor pipe.  Algorithmic flops = 2 * nq * nk * D.
#include "kb_knn.cuh"
#include <cuda.h>

namespace {

constexpr int BM = 128, BN = 256, BK = 64;
constexpr int A_BYTES = BM * BK * 2;          // 16 KB
constexpr int B_BYTES = BN * BK * 2;          // 32 KB
constexpr int NUM_THREADS = 192;
constexpr uint32_t TMEM_COLS = 512;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped kernel, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    uint32_t it = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++it & 0x3ff) == 0 && clock64() - t0 > 90000000000LL) {      // ~45 s: longer than the wait for a peer's shard
            printf("kb_knn_tc: mbarrier wait timed out (tag %d, block %d, thread %d)\n", tag, blockIdx.x, threadIdx.x);
            __trap();
        }
    }
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"):
// rows are 128 B apart, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);            // start address          [0,14)
    d |= (uint64_t)1 << 16;                              // leading byte offset    [16,30) (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                    // stride byte offset     [32,46)
    d |= (uint64_t)1 << 46;                              // descriptor version     [46,48)
    d |= (uint64_t)2 << 61;                              // SWIZZLE_128B           [61,64)
    return d;
}

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

struct TcParams {
    int64_t nk, q_row0, nq;
    int slots;                        // candidate lists per query row (stride of cand_*)
    int k_blocks;                     // Dp / 64
    int32_t n_tiles;                  // ceil(nk / BN)
    const kb_rowmeta* rowmeta;
    float* cand_score;
    int32_t* cand_idx;
    int32_t* row_thr;                 // per query row: best known KP-th score (ordered-int key), shared by all pieces
    const KbPiece* pieces;
    const int32_t* piece_start;       // per CTA pair
    const uint32_t* arrive;           // peer exchange (nullable): arrive[r] >= *epoch once rank r's shard has landed
    const uint32_t* epoch;
    int64_t rows_per_src;
    int32_t self_rank;
};

__device__ __forceinline__ KbPiece load_piece(const KbPiece* p) {
    const int4 a = __ldg(reinterpret_cast<const int4*>(p)), b = __ldg(reinterpret_cast<const int4*>(p) + 1);
    KbPiece pc;
    pc.group = a.x; pc.slot = a.y; pc.t_lo = a.z; pc.cnt = a.w; pc.shift = b.x; pc.i_lo = b.y; pc.i_cnt = b.z; pc.pad = 0;
    return pc;
}
__device__ __forceinline__ int64_t piece_tile(const KbPiece& pc, int i, int32_t n_tiles) {
    int t = i + pc.shift;
    if (t >= pc.cnt) t -= pc.cnt;
    t += pc.t_lo;
    if (t >= n_tiles) t -= n_tiles;                          // a shard's band may wrap round the end of the key set
    return (int64_t)t;
}

// Wait (bounded) until the shard of the rank owning key row `row` has arrived.  `seen` caches the answer.
__device__ __forceinline__ void wait_row_arrived(const TcParams& p, uint32_t epoch, int64_t row, uint32_t& seen, int tag) {
    if (row >= p.nk) row = p.nk - 1;
    const int src = (int)(row / p.rows_per_src);
    if (src == p.self_rank || ((seen >> src) & 1u)) return;
    const uint32_t* f = p.arrive + src;
    const long long t0 = clock64();
    uint32_t it = 0;
    while (true) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        if ((int32_t)(v - epoch) >= 0) break;
        if ((++it & 0xff) == 0 && clock64() - t0 > 60000000000LL) {        // ~30 s
            printf("kb_knn_tc: shard of rank %d never arrived (tag %d, block %d): flag %u, epoch %u\n", src, tag, blockIdx.x, v, epoch);
            __trap();
        }
        __nanosleep(64);
    }
    seen |= 1u << src;
}

// order-preserving float <-> int key (atomicMin on signed ints)
__device__ __forceinline__ int32_t f2key(float f) { const int32_t i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__device__ __forceinline__ float key2f(int32_t k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

// =====================================================================================
// k4_tc2: ONE 2-CTA MMA per CTA pair (tcgen05.mma.cta_group::2, M=256 N=256 K=16).  Each CTA
// keeps its 128 query rows (A) and HALF of the key tile (128 B rows) in shared memory: 32 KB
// per stage, so the ring is up to 6 deep, and the tensor core reads B once for both SMs.  The leader CTA (cluster
// rank 0) issues the MMAs; every TMA of either CTA signals the leader's "full" barrier
// (.cta_group::2 TMA with the peer-masked barrier address); the leader's commits are multicast
// to both CTAs' "stage empty" and "accumulator full" barriers; both CTAs' epilogue warps arrive
// on the leader's "accumulator empty" barrier.  Measured against two 1-CTA MMAs per pair with the key tile multicast
// to both CTAs: +0.4 % at 1088 columns, +10 % at 5120 (profiles/r01/k4_variants.md).
// =====================================================================================
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;        // clears the cluster-rank bit of a shared address: the even CTA
constexpr int STAGE2_BYTES = A_BYTES + B_BYTES / 2;  // 32 KB per CTA and stage
constexpr uint32_t IDESC2 = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);

__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint32_t leader_bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_f16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_2sm_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void mbar_arrive_rank(uint32_t bar, uint32_t rank) {   // arrive on CTA `rank`'s copy of `bar`
    asm volatile("{\n\t.reg .b32 ra;\n\t"
                 "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
                 "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}" ::"r"(bar), "r"(rank) : "memory");
}

// QCAP: pending list insertions per query row (k4_tc2)
template <int KP, int STAGES, int QCAP>
struct Smem2 {
    static constexpr int OFF_STAGES = 0;
    static constexpr int OFF_LIST_S = STAGES * STAGE2_BYTES;
    static constexpr int OFF_LIST_I = OFF_LIST_S + KP * BM * 4;
    static constexpr int OFF_QUEUE = OFF_LIST_I + KP * BM * 4;           // QCAP x BM x {score, key index}
    static constexpr int OFF_COLMETA = OFF_QUEUE + QCAP * BM * 8;
    static constexpr int OFF_BARS = OFF_COLMETA + BN * 8;
    static constexpr int OFF_TMEM_SLOT = OFF_BARS + (2 * STAGES + 4) * 8;
    static constexpr int TOTAL = OFF_TMEM_SLOT + 16;
    // 224 KB at most: with a peer exchange the tiny flag kernels of kb_xchg.cu (1 KB of system shared memory each) must
    // find room on an SM NEXT TO a resident CTA of this persistent kernel -- it waits for the very flags they raise
    static_assert(TOTAL <= 229376, "leave 4 KB of the SM's 228 KB to the exchange's flag kernels");
};

template <int KP, int STAGES, int QCAP>
__global__ void __launch_bounds__(NUM_THREADS, 1)
k4_tc2(const __grid_constant__ CUtensorMap tmap, const TcParams p) {
    using L = Smem2<KP, STAGES, QCAP>;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0 && (sbase & 1023u)) {
        printf("kb_knn_tc2: dynamic shared memory is not 1024-byte aligned (0x%x)\n", sbase);
        __trap();
    }
    const uint32_t bar_full = sbase + L::OFF_BARS;            // used in the leader CTA only
    const uint32_t bar_empty = bar_full + STAGES * 8;
    const uint32_t bar_tfull = bar_empty + STAGES * 8;
    const uint32_t bar_tempty = bar_tfull + 2 * 8;             // used in the leader CTA only
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + L::OFF_TMEM_SLOT);
    const int cta_rank = (int)cluster_ctarank();
    const bool leader = cta_rank == 0;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        // accumulator empty: 4 epilogue warps of each of the two CTAs
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + 8 * a, 1); mbar_init(bar_tempty + 8 * a, 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {                                          // both CTAs, same warp id
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32((const void*)tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int worker = blockIdx.x / 2;
    const int32_t pc_lo = p.piece_start[worker], pc_hi = p.piece_start[worker + 1];
    const uint32_t epoch = p.arrive ? *p.epoch : 0u;

    if (warp == 0) {
        // ================= TMA producer (both CTAs) =================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            uint32_t seen = 0;
            for (int32_t pi = pc_lo; pi < pc_hi; ++pi) {
                const KbPiece pc = load_piece(p.pieces + pi);
                const int32_t arow = (int32_t)(p.q_row0 + ((int64_t)pc.group * 2 + cta_rank) * BM);
                for (int i = pc.i_lo; i < pc.i_lo + pc.i_cnt; ++i) {
                    const int32_t brow = (int32_t)(piece_tile(pc, i, p.n_tiles) * BN) + 128 * cta_rank;   // my half of the key tile
                    if (p.arrive) {
                        wait_row_arrived(p, epoch, brow, seen, 11);
                        wait_row_arrived(p, epoch, (int64_t)brow + 127, seen, 11);
                        asm volatile("fence.proxy.async;" ::: "memory");
                    }
                    for (int kb = 0; kb < p.k_blocks; ++kb) {
                        mbar_wait(bar_empty + 8 * stage, phase ^ 1, 11);
                        const uint32_t sa = sbase + L::OFF_STAGES + stage * STAGE2_BYTES;
                        const uint32_t fb = (bar_full + 8 * stage) & PEER_MASK;          // the leader's barrier
                        if (leader) mbar_expect_tx(bar_full + 8 * stage, 2 * STAGE2_BYTES);   // both CTAs' bytes
                        tma_load_2d_2sm(sa, &tmap, kb * BK, arow, fb);
                        tma_load_2d_2sm(sa + A_BYTES, &tmap, kb * BK, brow, fb);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (leader CTA only) =================
        if (leader && lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int32_t pi = pc_lo; pi < pc_hi; ++pi) {
                const KbPiece pc = load_piece(p.pieces + pi);
                for (int i = 0; i < pc.i_cnt; ++i) {
                    mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1, 12);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                    for (int kb = 0; kb < p.k_blocks; ++kb) {
                        mbar_wait(bar_full + 8 * stage, phase, 13);
                        tc_fence_after();
                        const uint32_t sa = sbase + L::OFF_STAGES + stage * STAGE2_BYTES;
                        const uint64_t adesc = make_smem_desc(sa);
                        const uint64_t bdesc = make_smem_desc(sa + A_BYTES);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k)
                            umma_f16_2sm(d_tmem, adesc + 2 * k, bdesc + 2 * k, IDESC2, (kb | k) != 0);
                        umma_commit_2sm_mc(bar_empty + 8 * stage, (uint16_t)0x3);   // both CTAs' stage is free
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit_2sm_mc(bar_tfull + 8 * acc, (uint16_t)0x3);          // both CTAs' epilogues may read
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
            }
        }
    } else {
        // ================= epilogue: warps 2..5 of both CTAs (each its own 128 rows) =================
        const int quad = warp & 3;
        const int r = quad * 32 + lane;
        const int et = threadIdx.x - 64;
        KbRowList<KP, BM> list(reinterpret_cast<float*>(smem + L::OFF_LIST_S),
                               reinterpret_cast<int32_t*>(smem + L::OFF_LIST_I));
        const float4* cm4 = reinterpret_cast<const float4*>(smem + L::OFF_COLMETA);
        float2* cm_s = reinterpret_cast<float2*>(smem + L::OFF_COLMETA);
        // Elements that beat the row's bound are not inserted one by one as they turn up (the 32 rows of a warp
        // find theirs at different columns, so every insertion would run for the whole warp): they are queued per
        // row in shared memory and drained for all rows of the warp together, at the end of the tile or when a
        // queue runs full.  The bound is refreshed at every drain.
        float2* queue = reinterpret_cast<float2*>(smem + L::OFF_QUEUE) + r;    // entry j of this row at queue[j * BM]
        int acc = 0; uint32_t acc_phase = 0;
        uint32_t seen = 0;
        for (int32_t pi = pc_lo; pi < pc_hi; ++pi) {
            const KbPiece pc = load_piece(p.pieces + pi);
            const int64_t q = ((int64_t)pc.group * 2 + cta_rank) * BM + r;
            const bool live = q < p.nq;
            const float li = live ? (float)p.rowmeta[p.q_row0 + q].key_len : 1.f;
            list.init(r);
            float thr = __int_as_float(0x7f800000);
            int cnt = 0;                                      // queued entries of this row
            auto drain = [&]() {
                const int n_it = __reduce_max_sync(0xffffffffu, cnt);
                for (int j = 0; j < n_it; ++j) {
                    if (j < cnt) {
                        const float2 e = queue[j * BM];
                        if (e.x < thr) {
                            list.insert(r, e.x, __float_as_int(e.y));
                            thr = fminf(thr, list.bound);
                        }
                    }
                }
                cnt = 0;
            };
            for (int i = pc.i_lo; i < pc.i_lo + pc.i_cnt; ++i) {
                const int64_t n0 = piece_tile(pc, i, p.n_tiles) * BN;
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (p.arrive) { wait_row_arrived(p, epoch, n0 + et, seen, 15); wait_row_arrived(p, epoch, n0 + et + 128, seen, 15); }
                cm_s[et] = kb_load_cm(p.rowmeta, n0 + et, p.nk);
                cm_s[et + 128] = kb_load_cm(p.rowmeta, n0 + et + 128, p.nk);
                if (live) thr = fminf(thr, key2f(__ldcg(p.row_thr + q)));
                asm volatile("bar.sync 1, 128;" ::: "memory");
                mbar_wait(bar_tfull + 8 * acc, acc_phase, 14);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN);
#pragma unroll 1
                for (int c = 0; c < BN / 32; ++c) {
                    uint32_t v[32];
                    tmem_ld32(taddr + c * 32, v);
                    tmem_ld_wait();
                    float sc[32];
                    float m0 = thr, m1 = thr, m2 = thr, m3 = thr;
#pragma unroll
                    for (int x = 0; x < 32; x += 2) {
                        const float4 cm = cm4[c * 16 + (x >> 1)];
                        sc[x] = fmaf(__uint_as_float(v[x]), cm.x, li * cm.y);
                        sc[x + 1] = fmaf(__uint_as_float(v[x + 1]), cm.z, li * cm.w);
                    }
#pragma unroll
                    for (int x = 0; x < 32; x += 4) {
                        m0 = fminf(m0, sc[x]); m1 = fminf(m1, sc[x + 1]);
                        m2 = fminf(m2, sc[x + 2]); m3 = fminf(m3, sc[x + 3]);
                    }
                    if (__any_sync(0xffffffffu, fminf(fminf(m0, m1), fminf(m2, m3)) < thr)) {
                        // queue this chunk's candidates (predicated, no divergence)
                        const int cnt0 = cnt;
                        const int32_t idx0 = (int32_t)(n0 + c * 32);
#pragma unroll
                        for (int x = 0; x < 32; ++x) {
                            if (sc[x] < thr) {
                                if (cnt < QCAP) queue[cnt * BM] = make_float2(sc[x], __int_as_float(idx0 + x));
                                ++cnt;
                            }
                        }
                        if (__any_sync(0xffffffffu, cnt > QCAP)) {
                            // some row found more than its queue holds (a cold list: nearly everything passes and the rows of
                            // the warp insert in step anyway): take the earlier entries in, then this chunk element by element
                            cnt = cnt0;
                            drain();
#pragma unroll
                            for (int x = 0; x < 32; ++x) {
                                if (sc[x] < thr) {
                                    list.insert(r, sc[x], idx0 + x);
                                    thr = fminf(thr, list.bound);
                                }
                            }
                        } else if (__any_sync(0xffffffffu, cnt > QCAP / 2)) {
                            drain();
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_rank(bar_tempty + 8 * acc, 0);   // the leader's barrier
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                drain();                                      // (the accumulator is already released: the MMA runs ahead)
                if (live && list.bound < __int_as_float(0x7f800000)) atomicMin(p.row_thr + q, f2key(list.bound));
            }
            if (live) {
                const int64_t base = (q * p.slots + pc.slot) * KP;
#pragma unroll
                for (int e = 0; e < KP; ++e) {
                    p.cand_score[base + e] = list.s[e * BM + r];
                    p.cand_idx[base + e] = list.i[e * BM + r];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

template <int KP, int STAGES, int QCAP>
int launch_tc2(kb_ctx* ctx, const CUtensorMap& tmap, const TcParams& prm, int workers) {
    using L = Smem2<KP, STAGES, QCAP>;
    auto kern = k4_tc2<KP, STAGES, QCAP>;
    static bool attr_set[16] = {false};
    if (!attr_set[ctx->device & 15]) {
        KB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
        attr_set[ctx->device & 15] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(workers * 2));
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = L::TOTAL;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    KB_CUDA(cudaLaunchKernelEx(&cfg, kern, tmap, prm));
    ctx->launches++;
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}

// shared memory: 32 KB stages next to the lists and the insertion queues (16 entries per row = 16 KB; 12 for 16-wide
// lists): 6 stages up to 16-wide lists, 5 for 24 / 32, 4 for 48 / 64 (n_neighbors 27..60).  Wide rows (>= 2560 columns:
// long MMA tiles, light epilogue) with 24-wide lists trade most of the queue for the sixth stage.
template <int KP>
int launch_tc_kp(kb_ctx* ctx, const CUtensorMap& tmap, const TcParams& prm, int workers) {
    constexpr int ST2 = KP <= 16 ? 6 : (KP <= 32 ? 5 : 4);
    constexpr int Q2 = KP == 16 ? 12 : 16;
    if constexpr (KP == 24) { if (prm.k_blocks >= 40) return launch_tc2<24, 6, 4>(ctx, tmap, prm, workers); }
    return launch_tc2<KP, ST2, Q2>(ctx, tmap, prm, workers);
}

}  // namespace

int kb_knn_tc_launch(kb_ctx* ctx, const KbKnnPlan& p, const KbTcArgs& a) {
    if (!ctx->encode_tiled) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        KB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) { kb_set_error("cuTensorMapEncodeTiled not available from the driver"); return KB_ECUDA; }
        ctx->encode_tiled = fn;
    }
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {(cuuint64_t)a.d_cols_padded, (cuuint64_t)a.nk};
    const cuuint64_t gstride[1] = {(cuuint64_t)a.ld_operand * 2};
    const cuuint32_t box[2] = {BK, 128};
    const cuuint32_t estr[2] = {1, 1};
    CUresult cr = ((EncodeTiledFn)ctx->encode_tiled)(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(a.d_operand),
                                                    gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { kb_set_error("cuTensorMapEncodeTiled failed (%d)", (int)cr); return KB_ECUDA; }
    TcParams prm;
    prm.nk = a.nk; prm.q_row0 = a.q_row0; prm.nq = a.nq;
    prm.slots = p.slots;
    prm.k_blocks = a.d_cols_padded / BK;
    prm.n_tiles = (int32_t)((a.nk + BN - 1) / BN);
    prm.rowmeta = a.d_rowmeta;
    prm.cand_score = a.cand_score; prm.cand_idx = a.cand_idx; prm.row_thr = a.row_thr;
    prm.pieces = a.pieces; prm.piece_start = a.piece_start;
    prm.arrive = a.d_arrive; prm.epoch = a.d_epoch; prm.rows_per_src = a.rows_per_src > 0 ? a.rows_per_src : 1;
    prm.self_rank = a.self_rank;
    switch (p.kp) {
        case 8: return launch_tc_kp<8>(ctx, tmap, prm, p.workers);
        case 16: return launch_tc_kp<16>(ctx, tmap, prm, p.workers);
        case 24: return launch_tc_kp<24>(ctx, tmap, prm, p.workers);
        case 32: return launch_tc_kp<32>(ctx, tmap, prm, p.workers);
        case 48: return launch_tc_kp<48>(ctx, tmap, prm, p.workers);
        default: return launch_tc_kp<64>(ctx, tmap, prm, p.workers);
    }
}
