// kb_count.cu -- K1: per-contig k-mer counting (sm_100a).
//
// Replaces KmerClustering.__count_kmer_occurence (/root/reference/karma/kmer.py:56-92)
// and the window generator __kmers_of_seq (kmer.py:181-197) for windows made of
// A/C/G/T only.  Windows that contain any other byte ("exotic": kmer.py has no
// alphabet, so 'N', lowercase ... get string-keyed columns of their own) are
// only tallied per contig here; kb_exotic.cu enumerates them.
//
// Layout / algorithm
//   bases   uint8[sumL]  ASCII, contigs back to back          (HBM, read once)
//   counts  u32 [n][ld]  one row per contig                   (HBM, written once)
//   Persistent grid, dynamic queue (one atomic counter, rows taken in small batches).  One WARP
//   owns one contig when the histogram is <= 8 KB (5p6, 4+5, k <= 5), one CTA when it is
//   16-64 KB (5+6, k = 6, 7); the histogram (cols x u32) lives in shared memory.
//   A warp walks "spans" of 31 x 16 bytes: lane l loads the aligned 128-bit vector of bytes
//   [A0+16l, A0+16l+16), converts it bit-parallel to 2-bit codes (validated through a PRMT
//   lookup of "ACGT") and takes the 8 halo bases it needs from lane l+1 by shuffle; lane 31
//   only serves as halo.  The next span's vector is already in flight while the current one is
//   binned.  5-/6-/k-mer codes are shifted out of a 48-bit register pair; increments are
//   branch-free shared-memory reductions (windows that must not count go to a dummy word).
//   The string-palindrome test of the 16 six-windows is three XOR/shift masks compressed to
//   one bit per window.  The row is flushed with coalesced 128-bit streaming stores (histogram
//   cleared in the same pass).  Column presence (kmer.py:146-179 "observed k-mers") is
//   optional here: the whole-path pass lets K3 derive it from the rows it reads anyway.
//   Contigs longer than the LongPolicy threshold are queued on the device as (row, first
//   chunk) pairs; a second kernel deals the flat list of chunks to the whole grid (k-1 halo,
//   global red.add merge).
//
// Roofline: HBM.  Algorithmic bytes per contig = L (bases) + 4*cols (row).
#include "kb_common.cuh"
#include <cstdlib>
#include <cstring>
#include <climits>
#include <type_traits>

// Scheduling of the dynamic queue (warp-per-contig kernel):
//   contigs longer than `threshold` bases take the split path, `chunk` window starts per work item;
//   contigs longer than `first` (and <= threshold) are handed out BEFORE all others, `rows1` rows per
//   ticket, and binned by a whole CTA each, so that a 15 kb contig cannot become the tail of the launch;
//   the remaining contigs are taken `batch` consecutive rows at a time, one warp each.
// Defaults: threshold 64 kb, chunk 16 kb, first 4 kb.
struct LongPolicy { int64_t first, threshold, chunk; int batch, rows1; };

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int SPAN = 31 * 16;          // bytes of new window starts per warp span (lane 31 = halo only)

// 4 ASCII bytes -> 8 bits of 2-bit codes (first byte most significant).  `xinv` gets a
// non-zero byte wherever the input byte is not one of A/C/G/T.
//   code = ((b>>1) ^ (b>>2)) & 3   maps A,C,G,T -> 0,1,2,3 (and garbage for other bytes),
//   PRMT looks the code up in "ACGT" and the XOR with the input exposes every other byte.
__device__ __forceinline__ uint32_t codes4(uint32_t w, uint32_t& xinv) {
    const uint32_t t = ((w >> 1) ^ (w >> 2)) & 0x03030303u;
    const uint32_t sel = (t & 0x3u) | ((t >> 4) & 0x30u) | ((t >> 8) & 0x300u) | ((t >> 12) & 0x3000u);
    xinv = __byte_perm(0x54474341u, 0u, sel) ^ w;
    return (t * 0x40100401u) >> 24;                            // c0<<6 | c1<<4 | c2<<2 | c3
}
// per-byte "non-zero" -> 4 bits, first byte most significant
__device__ __forceinline__ uint32_t badbits4(uint32_t x) {
    const uint32_t y = (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
    return (((y >> 7) * 0x08040201u) >> 24) & 0xFu;
}

// Branch-free conditional increment: windows that must not count are steered to a
// per-thread dummy word behind the histogram (ptxas turns a predicated ATOMS into a
// branch; a select + unconditional reduction is shorter and never diverges).
__device__ __forceinline__ void red_shared_inc_if(uint32_t saddr, uint32_t dummy, uint32_t pred) {
    const uint32_t a = pred ? saddr : dummy;
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(a) : "memory");
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t saddr) {
    uint16_t v;
    asm("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(saddr));       // read-only table: free to be hoisted
    return v;
}

template <int KA, int KB, bool PALB>
struct Bins {
    static constexpr int A = 1 << (2 * KA);
    static constexpr int B = (KB == 0) ? 0 : (PALB ? (1 << KB) : (1 << (2 * KB)));  // pal: 4^(KB/2)=2^KB
    static constexpr int TOTAL = A + B;
};

// kmer.py:172-177 column order of "5p6" (sorted(): a palindromic 6-mer follows its 5-mer prefix):
//   column(5-mer code c) = c + #{palindromic 6-mers sorting before it}
//   column(palindromic 6-mer of rank r = 16*x1+4*x2+x3) = 272*x1 + 69*x2 + 21*x3 + 1
// (closed forms checked against sorted() in tests/test_oracle_golden.py::test_full_column_set_ka6).
__device__ __forceinline__ uint32_t sorted_col_5mer(uint32_t c) {
    const uint32_t d1 = c >> 8, d2 = (c >> 6) & 3u;
    const int cc = (int)(c & 63u) - (int)d2;
    const uint32_t t = cc <= 0 ? 0u : (uint32_t)min(4, (cc + 19) / 20);
    return c + 16u * d1 + 4u * d2 + t;
}
__device__ __forceinline__ uint32_t sorted_col_pal6(uint32_t r) {
    return 272u * (r >> 4) + 69u * ((r >> 2) & 3u) + 21u * (r & 3u) + 1u;
}
// SORTED mode: byte offsets of the histogram words in kmer.py's column order, 1024 entries for the
// 5-mer codes followed by 64 for the palindromic 6-mer ranks (u16, 2176 bytes of shared memory)
constexpr int LUT_BYTES = 2304;        // 1088 x u16, padded to keep the histogram 256-byte aligned
__device__ __forceinline__ void fill_lut(uint16_t* lut, int tid, int nthreads) {
    for (int c = tid; c < 1024; c += nthreads) lut[c] = (uint16_t)(4u * sorted_col_5mer((uint32_t)c));
    for (int r = tid; r < 64; r += nthreads) lut[1024 + r] = (uint16_t)(4u * sorted_col_pal6((uint32_t)r));
}

// What a warp needs to know about the piece of a contig it is binning (warp-uniform):
//   base0  absolute byte address of the first window start of the piece (beg + lo)
//   endv   absolute end of the contig: vectors at or beyond it are not loaded
//   cntA   number of window starts of component A counted from base0 (0 if the contig is too short)
//   cntB   same for component B
struct Piece {
    int64_t base0, endv;
    int cntA, cntB;
};
template <int KA, int KB>
__device__ __forceinline__ Piece make_piece(int64_t beg, int64_t L, int64_t lo, int64_t hi) {
    Piece p;
    p.base0 = beg + lo;
    p.endv = beg + L;
    const int64_t cap = 1 << 30;
    int64_t a = ((hi < L - KA + 1) ? hi : (L - KA + 1)) - lo;
    a = a < 0 ? 0 : (a > cap ? cap : a);
    p.cntA = (int)a;
    int64_t b = 0;
    if (KB > 0) {
        b = ((hi < L - KB + 1) ? hi : (L - KB + 1)) - lo;
        b = b < 0 ? 0 : (b > cap ? cap : b);
    }
    p.cntB = (int)b;
    return p;
}

__device__ __forceinline__ uint4 load_vec(const uint8_t* __restrict__ bases, int64_t A, int64_t endv) {
    uint4 v = make_uint4(0, 0, 0, 0);
    if (A < endv) v = __ldg(reinterpret_cast<const uint4*>(bases + A));
    return v;
}

// Bin the windows of one span.  v = this lane's vector (bytes [A, A+16), A = A0 + 16*lane, zero when
// not loaded), d = (int)(A - base0): window w of this lane is window number d + w of the piece.
// h32/d32/lut32 are shared-memory byte addresses (histogram, this thread's dummy word, offset table).
// Returns the lane's tally of in-range windows that hold a non-ACGT byte.
template <int KA, int KB, bool PALB, bool SORTED>
__device__ __forceinline__ uint32_t bin_span(uint4 v, bool loaded, int d, int cntA, int cntB,
                                             uint32_t h32, uint32_t d32, uint32_t lut32, int lane) {
    constexpr int KMAX = (KB > KA) ? KB : KA;
    static_assert(KMAX <= 7, "8 halo bases and the shift arithmetic below cover k <= 7");
    static_assert(!SORTED || (KA == 5 && KB == 6 && PALB), "sorted layout is the 5p6 mode");
    static_assert(!PALB || KB == 6, "palindromic component implemented for 6-mers");
    constexpr uint32_t BINS_A = Bins<KA, KB, PALB>::A;
    uint32_t x0, x1, x2, x3;
    const uint32_t own = (codes4(v.x, x0) << 24) | (codes4(v.y, x1) << 16) | (codes4(v.z, x2) << 8) | codes4(v.w, x3);
    const uint32_t nxt = __shfl_down_sync(FULL, own, 1);                 // lane+1's 16 bases: the first 8 are my halo
    // 24 bases: base j at bits [2*(23-j), 2*(23-j)+2)
    const uint64_t codes = ((uint64_t)own << 16) | (uint64_t)(nxt >> 16);
    // non-ACGT bytes are rare: the per-base bad mask is only built when some lane saw one
    uint32_t bad = 0;                                                    // base j at bit 23-j
    const bool inv = loaded && ((x0 | x1 | x2 | x3) != 0);
    if (__any_sync(FULL, inv)) {
        const uint32_t b16 = loaded ? ((badbits4(x0) << 12) | (badbits4(x1) << 8) | (badbits4(x2) << 4) | badbits4(x3)) : 0u;
        const uint32_t nb = __shfl_down_sync(FULL, b16, 1);
        bad = (b16 << 8) | (nb >> 8);
    }
    const int nwin = (lane == 31) ? 0 : 16;                              // lane 31 is halo only
    const int wlo = min(max(-d, 0), 16);
    uint32_t exotic = 0;
    // ---- component A: window w <-> bit 23-w
    {
        const int whi = min(max(cntA - d, 0), nwin);
        const uint32_t rA = whi > wlo ? (1u << (24 - wlo)) - (1u << (24 - whi)) : 0u;
        uint32_t BA = bad;
#pragma unroll
        for (int s = 1; s < KA; ++s) BA |= bad << s;
        const uint32_t okA = rA & ~BA;
        exotic += __popc(rA & BA);
        // byte offsets first (table loads in flight together), 8 windows at a time
#pragma unroll
        for (int g = 0; g < 16; g += 8) {
            uint32_t off[8];
#pragma unroll
            for (int x = 0; x < 8; ++x) {
                const int sh = 2 * (24 - KA - (g + x));                  // code = codes >> sh, sh >= 4
                if constexpr (SORTED) off[x] = lds_u16(lut32 + ((uint32_t)(codes >> (sh - 1)) & (2u * (BINS_A - 1))));
                else off[x] = (uint32_t)(codes >> (sh - 2)) & (4u * (BINS_A - 1));
            }
#pragma unroll
            for (int x = 0; x < 8; ++x) red_shared_inc_if(h32 + off[x], d32, okA & (1u << (23 - g - x)));
        }
    }
    if constexpr (KB > 0) {
        const int whi = min(max(cntB - d, 0), nwin);
        const uint32_t rB = whi > wlo ? (1u << (24 - wlo)) - (1u << (24 - whi)) : 0u;
        uint32_t BB = bad;
#pragma unroll
        for (int s = 1; s < KB; ++s) BB |= bad << s;
        const uint32_t okB = rB & ~BB;
        exotic += __popc(rB & BB);
        if constexpr (PALB) {
            // string palindrome x1x2x3x3x2x1 (kmer.py:46-54), all 16 windows at once:
            // field j of X_d is zero iff base j == base j+d; window w is a palindrome iff
            // base w==w+5, w+1==w+4, w+2==w+3.  np: bit 2*(23-w) set <=> NOT a palindrome.
            const uint64_t X5 = codes ^ (codes << 10), X3 = codes ^ (codes << 6), X1 = codes ^ (codes << 2);
            const uint64_t np = (X5 | (X5 >> 1)) | ((X3 | (X3 >> 1)) << 2) | ((X1 | (X1 >> 1)) << 4);
            // windows 0..15 sit at the even bits 46..16: compress them to one bit per window (w at bit 15-w)
            uint32_t e = ~(uint32_t)(np >> 16) & 0x55555555u;
            e = (e | (e >> 1)) & 0x33333333u; e = (e | (e >> 2)) & 0x0F0F0F0Fu;
            e = (e | (e >> 4)) & 0x00FF00FFu; e = (e | (e >> 8)) & 0x0000FFFFu;
            uint32_t pm = e & (okB >> 8);                               // valid palindromic windows (~1/64 of all)
            while (__any_sync(FULL, pm != 0)) {                         // warp-uniform trip count: no divergence
                const int b = pm ? 31 - __clz(pm) : 0;                  // window 15-b
                const uint32_t r = (uint32_t)(codes >> (12 + 2 * b)) & 63u;   // x1x2x3 of bases w..w+2: bits [2*(21-w), ..+6)
                uint32_t off;
                if constexpr (SORTED) off = lds_u16(lut32 + 2048u + 2u * r);
                else off = 4u * (BINS_A + r);
                red_shared_inc_if(h32 + off, d32, pm != 0);
                pm &= ~(1u << b);
            }
        } else {
#pragma unroll
            for (int w = 0; w < 16; ++w) {
                const int sh = 2 * (24 - KB - w);
                const uint32_t off = (uint32_t)(codes >> (sh - 2)) & (4u * ((1u << (2 * KB)) - 1));
                red_shared_inc_if(h32 + 4u * BINS_A + off, d32, okB & (1u << (23 - w)));
            }
        }
    }
    return exotic;
}

// Warp-cooperative accumulation of one piece: spans A_first, A_first + A_stride, ... (16-byte aligned
// absolute addresses; A_stride is a multiple of SPAN) until the piece's windows are exhausted.
// `v` holds the first span's vector of this lane on entry; on exit it holds the vector at `A_after`
// (the first span of whatever the warp does next; pass a negative address for "nothing").
template <int KA, int KB, bool PALB, bool SORTED>
__device__ __forceinline__ uint32_t accumulate_piece(const uint8_t* __restrict__ bases, const Piece& p, int64_t A_first,
                                                     int64_t A_stride, uint4& v, int64_t A_after, int64_t endv_after,
                                                     uint32_t h32, uint32_t d32, uint32_t lut32, int lane) {
    uint32_t exotic = 0;
    const int nwin = (KB > 0 && p.cntB > p.cntA) ? p.cntB : p.cntA;
    int d0 = (int)(A_first - p.base0);
    int64_t A0 = A_first;
    const int dstride = (int)A_stride;
    if (d0 >= nwin) {                                                    // nothing to bin (contig shorter than k, or no span for this warp)
        if (A_after >= 0) v = load_vec(bases, A_after + 16 * lane, endv_after);
        return 0;
    }
    while (true) {                                                       // warp-uniform trip count
        const bool more = d0 + dstride < nwin;
        const int64_t An = more ? A0 + A_stride : A_after;
        uint4 vn = make_uint4(0, 0, 0, 0);
        if (An >= 0) vn = load_vec(bases, An + 16 * lane, more ? p.endv : endv_after);   // in flight while this span is binned
        const int64_t A = A0 + 16 * lane;
        exotic += bin_span<KA, KB, PALB, SORTED>(v, A < p.endv, d0 + 16 * lane, p.cntA, p.cntB, h32, d32, lut32, lane);
        v = vn;
        if (!more) break;
        d0 += dstride; A0 += A_stride;
    }
    return exotic;
}

__device__ __forceinline__ uint32_t warp_sum(uint32_t v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// Flush one histogram (group of NT threads, this thread = tid) to a count row with 128-bit
// stores and clear it.  TRACK: collect presence bits (bit 4*it+j for vector tid+it*NT, element j).
template <int COLS, int NT, bool TRACK>
__device__ __forceinline__ void flush_row(uint32_t* hist, uint32_t* __restrict__ row_out, int tid, uint64_t& pres) {
    constexpr int VEC = COLS / 4;
    constexpr int ITERS = (VEC + NT - 1) / NT;
    static_assert(COLS % 4 == 0, "row flush is 128-bit");
    static_assert(ITERS * 4 <= 64, "presence bits live in one 64-bit register");
    uint4* out = reinterpret_cast<uint4*>(row_out);
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int i = tid + it * NT;
        if (i < VEC) {
            const uint4 r = *reinterpret_cast<uint4*>(hist + 4 * i);
            *reinterpret_cast<uint4*>(hist + 4 * i) = make_uint4(0, 0, 0, 0);
            __stcs(out + i, r);                                          // streaming: the row is not re-read here
            if constexpr (TRACK)
                pres |= (uint64_t)((r.x != 0) | ((r.y != 0) << 1) | ((r.z != 0) << 2) | ((r.w != 0) << 3)) << (4 * it);
        }
    }
}

template <int COLS, int NT>
__device__ __forceinline__ void publish_presence(uint32_t* __restrict__ presence, int tid, uint64_t pres) {
    constexpr int VEC = COLS / 4;
    constexpr int ITERS = (VEC + NT - 1) / NT;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int i = tid + it * NT;
        if (i < VEC) {
#pragma unroll
            for (int j = 0; j < 4; ++j)          // check before writing: thousands of warps storing to the same 1088 words cost ~80 us
                if (((pres >> (4 * it + j)) & 1) && __ldcg(presence + 4 * i + j) == 0u) presence[4 * i + j] = 1u;
        }
    }
}

// ---- fused K1+K3 (kb_count_profile): when the column dictionary is the full ACGT set (the optimistic pass), the
// row never goes to HBM as u32 counts: the flush turns the shared-memory histogram straight into the fp64 profile
// row (count / len(key), kmer.py:120,:213), the fp16 kNN operand row and the 32-byte row record.
struct FuseOut {
    const int32_t* key_len;
    double* profile; int64_t ld_profile;       // nullable
    __half* operand; int64_t ld_operand;       // nullable
    kb_rowmeta* rowmeta;                       // nullable
    uint32_t* flags_or;                        // nullable
    int64_t n_alloc;                           // rows [n, n_alloc) of operand / rowmeta are written as gather padding
};

// count / len in IEEE fp64, correctly rounded, without a division per element: q = x*rcp, one residual correction
// (Markstein): exact for every (count, len) pair this path can see (checked exhaustively for count <= 300000,
// len <= 3000 and on 4e8 random pairs up to 2^31 / 2^20 against the true quotient).
__device__ __forceinline__ double quot(uint32_t x, double len, double rcp) {
    const double a = __uint2double_rn(x);
    const double q = a * rcp;
    const double r = fma(-len, q, a);
    return fma(r, rcp, q);
}

template <int COLS, int NT>
__device__ __forceinline__ void flush_fused(uint32_t* hist, int tid, int64_t row, const FuseOut& f, double len, double rcp,
                                            unsigned long long& sq, uint32_t& mx, uint64_t& pres) {
    constexpr int VEC = COLS / 4;
    constexpr int ITERS = (VEC + NT - 1) / NT;
    static_assert(COLS % 4 == 0 && ITERS * 4 <= 64, "row flush is 128-bit; presence bits live in one 64-bit register");
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int i = tid + it * NT;
        if (i < VEC) {
            const uint4 r = *reinterpret_cast<uint4*>(hist + 4 * i);
            *reinterpret_cast<uint4*>(hist + 4 * i) = make_uint4(0, 0, 0, 0);
            sq += (unsigned long long)r.x * r.x + (unsigned long long)r.y * r.y + (unsigned long long)r.z * r.z +
                  (unsigned long long)r.w * r.w;
            mx = max(max(mx, r.x), max(r.y, max(r.z, r.w)));
            pres |= (uint64_t)((r.x != 0) | ((r.y != 0) << 1) | ((r.z != 0) << 2) | ((r.w != 0) << 3)) << (4 * it);
            if (f.profile) {
                double2 a, b;
                a.x = quot(r.x, len, rcp); a.y = quot(r.y, len, rcp);
                b.x = quot(r.z, len, rcp); b.y = quot(r.w, len, rcp);
                double* q = f.profile + row * f.ld_profile + 4 * i;
                if ((f.ld_profile & 1) == 0) {
                    __stcs(reinterpret_cast<double2*>(q), a); __stcs(reinterpret_cast<double2*>(q) + 1, b);
                } else {
                    q[0] = a.x; q[1] = a.y; q[2] = b.x; q[3] = b.y;
                }
            }
            if (f.operand) {
                const __half2 h0 = __floats2half2_rn((float)min(r.x, 2048u), (float)min(r.y, 2048u));
                const __half2 h1 = __floats2half2_rn((float)min(r.z, 2048u), (float)min(r.w, 2048u));
                uint2 pk;
                pk.x = *reinterpret_cast<const uint32_t*>(&h0);
                pk.y = *reinterpret_cast<const uint32_t*>(&h1);
                *reinterpret_cast<uint2*>(f.operand + row * f.ld_operand + 4 * i) = pk;
            }
        }
    }
    if (f.operand)                                                       // zero padding of the operand row
        for (int64_t c = COLS + tid; c < f.ld_operand; c += NT) f.operand[row * f.ld_operand + c] = __float2half_rn(0.f);
}

__device__ __forceinline__ void write_rowmeta(const FuseOut& f, int64_t row, unsigned long long sq, uint32_t mx, int32_t klen) {
    const int flags = (mx > 2048u ? 1 : 0) | (sq >= (1ull << 24) ? 2 : 0) | (mx == 0 ? 4 : 0);
    if (f.rowmeta) {
        const double len = (double)klen;
        kb_rowmeta m;
        m.sqnorm = (double)sq; m.key_len = klen; m.flags = flags;
        if (flags & 3) { m.cm_x = 0.f; m.cm_y = __int_as_float(0x7f800000); }          // K4 never proposes the row
        else { m.cm_x = (float)(-2.0 / len); m.cm_y = (float)((double)sq / (len * len)); }
        m.reserved[0] = m.reserved[1] = 0;
        f.rowmeta[row] = m;
    }
    if (f.flags_or && flags) atomicOr(f.flags_or, (uint32_t)flags);
}

__device__ __forceinline__ void write_padding_rows(const FuseOut& f, int64_t n, int tid, int nthreads) {
    for (int64_t row = n; row < f.n_alloc; ++row) {
        if (f.operand)
            for (int64_t c = tid; c < f.ld_operand; c += nthreads) f.operand[row * f.ld_operand + c] = __float2half_rn(0.f);
        if (tid == 0 && f.rowmeta) {
            kb_rowmeta m;
            m.sqnorm = 0.0; m.key_len = 1; m.flags = 11;
            m.cm_x = 0.f; m.cm_y = __int_as_float(0x7f800000);
            m.reserved[0] = m.reserved[1] = 0;
            f.rowmeta[row] = m;
        }
    }
}

// presence bits of one flush layout (NT threads) -> per-column bytes
template <int COLS, int NT>
__device__ __forceinline__ void presence_to_bytes(uint8_t* col, int tid, uint64_t pres) {
    constexpr int VEC = COLS / 4;
    constexpr int ITERS = (VEC + NT - 1) / NT;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int i = tid + it * NT;
        if (i < VEC) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if ((pres >> (4 * it + j)) & 1) col[4 * i + j] = 1;
        }
    }
}
// per-CTA column bytes -> presence vector: a CTA that saw every column proves the dictionary complete with one
// store (bit 1 of presence[COLS]); otherwise per-column stores, checked before writing
template <int COLS>
__device__ __forceinline__ void publish_bytes(const uint8_t* col, uint32_t* __restrict__ presence, int* s_cnt, int tid, int nthreads) {
    int mine = 0;
    for (int c = tid; c < COLS; c += nthreads) mine += col[c];
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(FULL, mine, o);
    if ((tid & 31) == 0 && mine) atomicAdd(s_cnt, mine);
    __syncthreads();
    if (*s_cnt == COLS) {
        if (tid == 0 && !(__ldcg(presence + COLS) & 2u)) atomicOr(presence + COLS, 2u);
    } else {
        for (int c = tid; c < COLS; c += nthreads)
            if (col[c] && __ldcg(presence + c) == 0u) presence[c] = 1u;
    }
}

// scratch (int32 words): [0] next row, [1] unused, [2..3] exotic total (u64),
//   [4..5] u64: (number of long contigs << 32) | total number of chunks,
//   [6 + 2i], [7 + 2i]: row and first chunk number of the i-th long contig (ascending in both)
__device__ __forceinline__ void queue_long(int32_t* scratch, int64_t row, int64_t L, int64_t chunk) {
    const unsigned long long n_chunks = (unsigned long long)((L + chunk - 1) / chunk);
    const unsigned long long old = atomicAdd(reinterpret_cast<unsigned long long*>(scratch + 4), (1ull << 32) | n_chunks);
    const uint32_t slot = (uint32_t)(old >> 32);
    scratch[6 + 2 * slot] = (int32_t)row;
    scratch[7 + 2 * slot] = (int32_t)(uint32_t)old;
}

// ---- histograms <= 8 KB: one WARP per contig, 8 independent warps per CTA -- after a first phase in
// which the whole CTA bins the longer contigs together.
// Queue tickets [0, nb1) are "class 1" batches of lp.rows1 rows, taken per CTA: contigs longer than
// lp.threshold are queued for the split kernel, contigs longer than lp.first are binned by all 8 warps
// into one histogram (a single warp needs 2-3 us per span with its scheduler shared: a 15 kb contig
// would take 60-90 us alone).  The tickets after that are per warp: the remaining contigs, lp.batch
// consecutive rows at a time, no block barriers.
template <int KA, int KB, bool PALB, bool SORTED, int WARPS, bool TRACK, int MINB, bool FUSE>
__global__ void __launch_bounds__(WARPS * 32, MINB)
k1_count_warp(const uint8_t* __restrict__ bases, const int64_t* __restrict__ offsets, int64_t n,
              uint32_t* __restrict__ counts, int64_t ld, uint32_t* __restrict__ exotic_out,
              uint32_t* __restrict__ presence, int32_t* scratch, LongPolicy lp, FuseOut fuse) {
    constexpr int COLS = Bins<KA, KB, PALB>::TOTAL;
    constexpr int THREADS = WARPS * 32;
    extern __shared__ __align__(16) uint32_t smem_hist[];
    __shared__ int64_t s_ticket;
    __shared__ int64_t s_beg[32], s_len[32];
    __shared__ int32_t s_row[32];
    __shared__ int s_n;
    __shared__ uint32_t s_red[WARPS];
    __shared__ unsigned long long s_sq[WARPS];
    __shared__ uint32_t s_mx[WARPS];
    __shared__ int s_cnt;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t* lut = reinterpret_cast<uint16_t*>(smem_hist);            // SORTED: u16 byte offsets
    uint32_t* hist0 = smem_hist + (SORTED ? LUT_BYTES / 4 : 0);         // warp 0's histogram: the shared one of phase 1
    uint32_t* hist = hist0 + warp * (COLS + 32);                        // + one dummy word per lane
    if constexpr (SORTED) fill_lut(lut, threadIdx.x, THREADS);
    for (int i = lane; i < COLS; i += 32) hist[i] = 0;
    const uint32_t h32 = (uint32_t)__cvta_generic_to_shared(hist);
    const uint32_t h32_0 = (uint32_t)__cvta_generic_to_shared(hist0);
    const uint32_t d32 = h32 + 4u * (COLS + lane);
    const uint32_t lut32 = (uint32_t)__cvta_generic_to_shared(lut);
    const int64_t nb1 = (n + lp.rows1 - 1) / lp.rows1;
    uint64_t pres = 0, pres1 = 0;

    // ================= phase 1: the CTA as a whole =================
    int64_t t;
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) s_ticket = (int64_t)atomicAdd(&scratch[0], 1);
        __syncthreads();
        t = s_ticket;
        if (t >= nb1) break;
        if (warp == 0) {
            const int64_t r = lp.rows1 * t + lane;
            int64_t beg = 0, L = 0;
            if (lane < lp.rows1 && r < n) { beg = offsets[r]; L = offsets[r + 1] - beg; }
            if (L > lp.threshold) {
                queue_long(scratch, r, L, lp.chunk);                     // the split kernel red.adds into the zeroed row
                if (exotic_out) exotic_out[r] = 0;
            }
            // rows to zero (split path) and rows to bin now, compacted in row order
            const unsigned m_long = __ballot_sync(FULL, L > lp.threshold);
            const unsigned m_mid = __ballot_sync(FULL, L > lp.first && L <= lp.threshold);
            const unsigned m_all = m_long | m_mid;
            if ((m_all >> lane) & 1u) {
                const int pos = __popc(m_all & ((1u << lane) - 1u));
                s_beg[pos] = beg;
                s_len[pos] = (L > lp.threshold) ? -1 : L;
                s_row[pos] = (int32_t)r;
            }
            if (lane == 0) s_n = __popc(m_all);
        }
        __syncthreads();
        const int cnt = s_n;
        for (int i = 0; i < cnt; ++i) {
            const int64_t row = s_row[i], beg = s_beg[i], L = s_len[i];
            uint32_t* out = counts + row * ld;
            if (L < 0) {
                for (int j = threadIdx.x; j < COLS / 4; j += THREADS) reinterpret_cast<uint4*>(out)[j] = make_uint4(0, 0, 0, 0);
                continue;
            }
            const Piece p = make_piece<KA, KB>(beg, L, 0, L);
            const int64_t A_first = (beg & ~int64_t(15)) + (int64_t)SPAN * warp;
            uint4 v = load_vec(bases, A_first + 16 * lane, p.endv);
            const uint32_t ex = warp_sum(accumulate_piece<KA, KB, PALB, SORTED>(bases, p, A_first, (int64_t)SPAN * WARPS, v, -1, 0,
                                                                                h32_0, d32, lut32, lane));
            if (lane == 0) s_red[warp] = ex;
            __syncthreads();                                             // all reductions done, s_red visible
            if (threadIdx.x == 0) {
                uint32_t ex_total = 0;
                for (int w = 0; w < WARPS; ++w) ex_total += s_red[w];
                if (exotic_out) exotic_out[row] = ex_total;
                if (ex_total) {
                    atomicAdd(reinterpret_cast<unsigned long long*>(scratch + 2), (unsigned long long)ex_total);
                    if (presence) presence[COLS] = 1u;                   // "some window holds a non-ACGT byte"
                }
            }
            if constexpr (FUSE) {
                const int32_t klen = fuse.key_len[row];
                const double len = (double)klen;
                unsigned long long sq = 0; uint32_t mx = 0;
                flush_fused<COLS, THREADS>(hist0, threadIdx.x, row, fuse, len, 1.0 / len, sq, mx, pres1);
                for (int o = 16; o > 0; o >>= 1) {
                    sq += __shfl_xor_sync(FULL, sq, o);
                    mx = max(mx, __shfl_xor_sync(FULL, mx, o));
                }
                if (lane == 0) { s_sq[warp] = sq; s_mx[warp] = mx; }
                __syncthreads();
                if (threadIdx.x == 0) {
                    for (int w = 1; w < WARPS; ++w) { sq += s_sq[w]; mx = max(mx, s_mx[w]); }
                    write_rowmeta(fuse, row, sq, mx, klen);
                }
            } else {
                flush_row<COLS, THREADS, TRACK>(hist0, out, threadIdx.x, pres1);
                __syncthreads();
            }
        }
    }
    if constexpr (TRACK && !FUSE) publish_presence<COLS, THREADS>(presence, threadIdx.x, pres1);

    // ================= phase 2: every warp on its own =================
    bool have_ticket = (warp == 0);                                      // the ticket that ended phase 1 is a class-2 ticket
    while (true) {
        if (!have_ticket) {
            t = 0;
            if (lane == 0) t = (int64_t)atomicAdd(&scratch[0], 1);
            t = __shfl_sync(FULL, t, 0);
        }
        have_ticket = false;
        const int64_t row0 = (t - nb1) * lp.batch;
        if (row0 >= n) break;
        const int nb = (int)((n - row0 < lp.batch) ? n - row0 : lp.batch);
        int64_t my_off = 0;
        if (lane <= nb) my_off = offsets[row0 + lane];                  // batch <= 31
        int32_t my_len = 1;
        if constexpr (FUSE) { if (lane < nb) my_len = fuse.key_len[row0 + lane]; }
        int64_t beg = __shfl_sync(FULL, my_off, 0);
        uint4 v = make_uint4(0, 0, 0, 0);
        bool have_v = false;                                             // v holds the first span of contig c
        for (int c = 0; c < nb; ++c) {
            const int64_t end = __shfl_sync(FULL, my_off, c + 1);
            const int64_t L = end - beg;
            if (L > lp.first) {
                have_v = false;                                          // done in phase 1
            } else {
                if (!have_v) v = load_vec(bases, (beg & ~int64_t(15)) + 16 * lane, end);
                // the next contig of the batch starts where this one ends: its first span is prefetched
                int64_t A_after = -1, endv_after = 0;
                if (c + 1 < nb) {
                    const int64_t end2 = __shfl_sync(FULL, my_off, c + 2);
                    if (end2 - end <= lp.first) { A_after = end & ~int64_t(15); endv_after = end2; }
                }
                const int64_t row = row0 + c;
                const Piece p = make_piece<KA, KB>(beg, L, 0, L);
                const uint32_t ex = accumulate_piece<KA, KB, PALB, SORTED>(bases, p, beg & ~int64_t(15), SPAN, v, A_after, endv_after,
                                                                           h32, d32, lut32, lane);
                const uint32_t ex_total = warp_sum(ex);
                if (lane == 0) {
                    if (exotic_out) exotic_out[row] = ex_total;
                    if (ex_total) {
                        atomicAdd(reinterpret_cast<unsigned long long*>(scratch + 2), (unsigned long long)ex_total);
                        if (presence) presence[COLS] = 1u;
                    }
                }
                __syncwarp();
                if constexpr (FUSE) {
                    const int32_t klen = __shfl_sync(FULL, my_len, c);
                    const double len = (double)klen;
                    unsigned long long sq = 0; uint32_t mx = 0;
                    flush_fused<COLS, 32>(hist, lane, row, fuse, len, 1.0 / len, sq, mx, pres);
                    for (int o = 16; o > 0; o >>= 1) {
                        sq += __shfl_xor_sync(FULL, sq, o);
                        mx = max(mx, __shfl_xor_sync(FULL, mx, o));
                    }
                    if (lane == 0) write_rowmeta(fuse, row, sq, mx, klen);
                } else {
                    flush_row<COLS, 32, TRACK>(hist, counts + row * ld, lane, pres);
                }
                __syncwarp();
                have_v = A_after >= 0;
            }
            beg = end;
        }
    }
    if constexpr (TRACK && !FUSE) publish_presence<COLS, 32>(presence, lane, pres);
    if constexpr (FUSE) {
        // column presence of this CTA: both flush layouts -> bytes (the histograms are idle now) -> one store if complete
        __syncthreads();
        uint8_t* col = reinterpret_cast<uint8_t*>(hist0);
        for (int c = threadIdx.x; c < COLS; c += THREADS) col[c] = 0;
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
        presence_to_bytes<COLS, THREADS>(col, threadIdx.x, pres1);
        presence_to_bytes<COLS, 32>(col, lane, pres);
        __syncthreads();
        if (presence) publish_bytes<COLS>(col, presence, &s_cnt, threadIdx.x, THREADS);
        if (blockIdx.x == 0) write_padding_rows(fuse, n, threadIdx.x, THREADS);
    }
}

// ---- one CTA per contig (histograms of 16-64 KB)
template <int KA, int KB, bool PALB, bool SORTED, int THREADS, bool TRACK, bool FUSE>
__global__ void __launch_bounds__(THREADS)
k1_count_cta(const uint8_t* __restrict__ bases, const int64_t* __restrict__ offsets, int64_t n,
             uint32_t* __restrict__ counts, int64_t ld, uint32_t* __restrict__ exotic_out,
             uint32_t* __restrict__ presence, int32_t* scratch, LongPolicy lp, FuseOut fuse) {
    constexpr int COLS = Bins<KA, KB, PALB>::TOTAL;
    constexpr int NW = THREADS / 32;
    extern __shared__ __align__(16) uint32_t smem_hist[];
    __shared__ uint32_t s_red[NW];
    __shared__ unsigned long long s_sq[NW];
    __shared__ uint32_t s_mx[NW];
    __shared__ int s_cnt;
    __shared__ int64_t s_row;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t* lut = reinterpret_cast<uint16_t*>(smem_hist);
    uint32_t* hist = smem_hist + (SORTED ? LUT_BYTES / 4 : 0);
    if constexpr (SORTED) fill_lut(lut, threadIdx.x, THREADS);
    for (int i = threadIdx.x; i < COLS; i += THREADS) hist[i] = 0;
    const uint32_t h32 = (uint32_t)__cvta_generic_to_shared(hist);
    const uint32_t d32 = h32 + 4u * (COLS + threadIdx.x);
    const uint32_t lut32 = (uint32_t)__cvta_generic_to_shared(lut);
    uint64_t pres = 0;
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) s_row = (int64_t)atomicAdd(&scratch[0], 1);
        __syncthreads();
        const int64_t row = s_row;
        if (row >= n) break;
        const int64_t beg = offsets[row];
        const int64_t L = offsets[row + 1] - beg;
        uint32_t* out = counts + row * ld;
        if (L > lp.threshold) {
            if (threadIdx.x == 0) {
                queue_long(scratch, row, L, lp.chunk);
                if (exotic_out) exotic_out[row] = 0;
            }
            for (int i = threadIdx.x; i < COLS / 4; i += THREADS) reinterpret_cast<uint4*>(out)[i] = make_uint4(0, 0, 0, 0);
            continue;
        }
        const Piece p = make_piece<KA, KB>(beg, L, 0, L);
        const int64_t A_first = (beg & ~int64_t(15)) + (int64_t)SPAN * warp;
        uint4 v = load_vec(bases, A_first + 16 * lane, p.endv);
        const uint32_t ex = warp_sum(accumulate_piece<KA, KB, PALB, SORTED>(bases, p, A_first, (int64_t)SPAN * NW, v, -1, 0,
                                                                            h32, d32, lut32, lane));
        if (lane == 0) s_red[warp] = ex;
        __syncthreads();                                         // all atomics done, s_red visible
        if (threadIdx.x == 0) {
            uint32_t ex_total = 0;
            for (int i = 0; i < NW; ++i) ex_total += s_red[i];
            if (exotic_out) exotic_out[row] = ex_total;
            if (ex_total) {
                atomicAdd(reinterpret_cast<unsigned long long*>(scratch + 2), (unsigned long long)ex_total);
                if (presence) presence[COLS] = 1u;
            }
        }
        if constexpr (FUSE) {
            const int32_t klen = fuse.key_len[row];
            const double len = (double)klen;
            unsigned long long sq = 0; uint32_t mx = 0;
            flush_fused<COLS, THREADS>(hist, threadIdx.x, row, fuse, len, 1.0 / len, sq, mx, pres);
            for (int o = 16; o > 0; o >>= 1) {
                sq += __shfl_xor_sync(FULL, sq, o);
                mx = max(mx, __shfl_xor_sync(FULL, mx, o));
            }
            if (lane == 0) { s_sq[warp] = sq; s_mx[warp] = mx; }
            __syncthreads();
            if (threadIdx.x == 0) {
                for (int w = 1; w < NW; ++w) { sq += s_sq[w]; mx = max(mx, s_mx[w]); }
                write_rowmeta(fuse, row, sq, mx, klen);
            }
        } else {
            flush_row<COLS, THREADS, TRACK>(hist, out, threadIdx.x, pres);
        }
    }
    if constexpr (TRACK && !FUSE) publish_presence<COLS, THREADS>(presence, threadIdx.x, pres);
    if constexpr (FUSE) {
        __syncthreads();
        uint8_t* col = reinterpret_cast<uint8_t*>(hist);
        for (int c = threadIdx.x; c < COLS; c += THREADS) col[c] = 0;
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
        presence_to_bytes<COLS, THREADS>(col, threadIdx.x, pres);
        __syncthreads();
        if (presence) publish_bytes<COLS>(col, presence, &s_cnt, threadIdx.x, THREADS);
        if (blockIdx.x == 0) write_padding_rows(fuse, n, threadIdx.x, THREADS);
    }
}

// ---- split path: the flat list of chunks of all long contigs is dealt to the grid in contiguous ranges
template <int KA, int KB, bool PALB, bool SORTED, int THREADS>
__global__ void __launch_bounds__(THREADS)
k1_count_long(const uint8_t* __restrict__ bases, const int64_t* __restrict__ offsets,
              uint32_t* __restrict__ counts, int64_t ld, uint32_t* __restrict__ exotic_out,
              uint32_t* __restrict__ presence, int32_t* scratch, LongPolicy lp) {
    constexpr int COLS = Bins<KA, KB, PALB>::TOTAL;
    constexpr int NW = THREADS / 32;
    extern __shared__ __align__(16) uint32_t smem_hist[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long packed = *reinterpret_cast<const unsigned long long*>(scratch + 4);
    const int64_t n_long = (int64_t)(packed >> 32);
    const int64_t total = (int64_t)(packed & 0xffffffffull);
    if (total == 0) return;
    // my contiguous range of chunk numbers
    const int64_t per = (total + gridDim.x - 1) / gridDim.x;
    int64_t w = per * blockIdx.x;
    const int64_t w_end = (w + per < total) ? w + per : total;
    if (w >= w_end) return;
    uint16_t* lut = reinterpret_cast<uint16_t*>(smem_hist);
    uint32_t* hist = smem_hist + (SORTED ? LUT_BYTES / 4 : 0);
    if constexpr (SORTED) fill_lut(lut, threadIdx.x, THREADS);
    for (int i = threadIdx.x; i < COLS; i += THREADS) hist[i] = 0;
    __syncthreads();
    const uint32_t h32 = (uint32_t)__cvta_generic_to_shared(hist);
    const uint32_t d32 = h32 + 4u * (COLS + threadIdx.x);
    const uint32_t lut32 = (uint32_t)__cvta_generic_to_shared(lut);
    // the list is ascending in the first chunk number: find the contig that owns chunk w
    int64_t lo_i = 0, hi_i = n_long - 1;
    while (lo_i < hi_i) {
        const int64_t mid = (lo_i + hi_i + 1) >> 1;
        if ((int64_t)(uint32_t)scratch[7 + 2 * mid] <= w) lo_i = mid; else hi_i = mid - 1;
    }
    int64_t li = lo_i;
    while (w < w_end) {
        const int64_t row = scratch[6 + 2 * li];
        const int64_t first = (int64_t)(uint32_t)scratch[7 + 2 * li];
        const int64_t beg = offsets[row];
        const int64_t L = offsets[row + 1] - beg;
        const int64_t n_chunks = (L + lp.chunk - 1) / lp.chunk;
        int64_t c = w - first;
        for (; c < n_chunks && w < w_end; ++c, ++w) {
            const int64_t lo = c * lp.chunk;
            const int64_t hi = (lo + lp.chunk < L) ? lo + lp.chunk : L;
            const Piece p = make_piece<KA, KB>(beg, L, lo, hi);
            const int64_t A_first = ((beg + lo) & ~int64_t(15)) + (int64_t)SPAN * warp;
            uint4 v = load_vec(bases, A_first + 16 * lane, p.endv);
            const uint32_t ex = warp_sum(accumulate_piece<KA, KB, PALB, SORTED>(bases, p, A_first, (int64_t)SPAN * NW, v, -1, 0,
                                                                                h32, d32, lut32, lane));
            if (lane == 0 && ex) {
                if (exotic_out) atomicAdd(&exotic_out[row], ex);
                atomicAdd(reinterpret_cast<unsigned long long*>(scratch + 2), (unsigned long long)ex);
                if (presence) presence[COLS] = 1u;
            }
            __syncthreads();
            uint32_t* out = counts + row * ld;
            for (int i = threadIdx.x; i < COLS; i += THREADS) {
                const uint32_t x = hist[i];
                if (x) {
                    atomicAdd(&out[i], x);
                    hist[i] = 0;
                    if (presence) presence[i] = 1u;
                }
            }
            __syncthreads();
        }
        ++li;
    }
}

template <int KA, int KB, bool PALB, bool SORTED>
int launch(kb_ctx* ctx, const uint8_t* d_bases, const int64_t* d_offsets, int64_t n,
           uint32_t* d_counts, int64_t ld, uint32_t* d_exotic, uint32_t* d_presence, int track, const FuseOut* fuse) {
    constexpr int COLS = Bins<KA, KB, PALB>::TOTAL;
    constexpr bool WARP_PER_CONTIG = COLS <= 2048;
    constexpr int WARPS = 8;
    constexpr int THREADS = (COLS > 8192) ? 256 : 128;            // CTA-per-contig / split kernels
    // scratch: counter, exotic total, long-contig list (at most n entries of 2 words)
    const int64_t need = 2 * n + 8;
    if (ctx->k1_scratch_cap < need) {
        if (ctx->d_k1_scratch) KB_CUDA(cudaFree(ctx->d_k1_scratch));
        ctx->d_k1_scratch = nullptr; ctx->k1_scratch_cap = 0;
        KB_CUDA(cudaMalloc(&ctx->d_k1_scratch, (size_t)need * sizeof(int32_t)));
        ctx->k1_scratch_cap = need;
    }
    KB_CUDA(cudaMemsetAsync(ctx->d_k1_scratch, 0, 8 * sizeof(int32_t), ctx->stream));
    const size_t smem_one = (size_t)(COLS + THREADS) * sizeof(uint32_t) + (SORTED ? LUT_BYTES : 0);   // histogram + dummy words (+ offset table)
    LongPolicy lp{4096, 1 << 16, 1 << 14, 4, 32};
    const bool tr = track && d_presence && !fuse;
    FuseOut fo;
    memset(&fo, 0, sizeof(fo));
    if (fuse) {
        fo = *fuse;
        lp.threshold = INT64_MAX;                                 // fused rows are never split: the longer contigs are binned by whole CTAs
    }
    if constexpr (WARP_PER_CONTIG) {
        // 4 CTAs of 8 warps per SM (64 registers, no spills) beat 5 (48 registers): 0.088 vs 0.095 ms at 50k contigs
        // (the fused kernel: 0.141 ms with 4 CTAs per SM / 64 registers, 0.146 ms with 3 CTAs / 85 registers)
        auto k1 = fuse ? k1_count_warp<KA, KB, PALB, SORTED, WARPS, false, 4, true>
                       : (tr ? k1_count_warp<KA, KB, PALB, SORTED, WARPS, true, 4, false> : k1_count_warp<KA, KB, PALB, SORTED, WARPS, false, 4, false>);
        const size_t smem = (size_t)(COLS + 32) * sizeof(uint32_t) * WARPS + (SORTED ? LUT_BYTES : 0);
        static int per_sm_cache[16][3] = {{0}};                // per device and variant: attribute set + occupancy known
        int& per_sm = per_sm_cache[ctx->device & 15][fuse ? 2 : (tr ? 1 : 0)];
        if (per_sm == 0) {
            KB_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            KB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k1, WARPS * 32, smem));
        }
        if (per_sm < 1) { kb_set_error("k1_count_warp does not fit on an SM"); return KB_ECUDA; }
        const int64_t resident_warps = (int64_t)ctx->sm_count * per_sm * WARPS;
        if (n < 8 * resident_warps) lp.batch = 2;
        if (n < 4 * resident_warps) lp.batch = 1;
        if (n < 2 * resident_warps) lp.rows1 = 8;                // few contigs: finer class-1 tickets keep every CTA busy
        int64_t grid = (int64_t)ctx->sm_count * per_sm;         // persistent: one resident wave
        const int64_t want = (n + WARPS - 1) / WARPS;
        if (grid > want) grid = want;
        if (grid < 1) grid = 1;
        KbTimer t(ctx, 0);
        k1<<<(unsigned)grid, WARPS * 32, smem, ctx->stream>>>(d_bases, d_offsets, n, d_counts, ld, d_exotic,
                                                              d_presence, ctx->d_k1_scratch, lp, fo);
        ctx->launches++;
    } else {
        auto k1 = fuse ? k1_count_cta<KA, KB, PALB, SORTED, THREADS, false, true>
                       : (tr ? k1_count_cta<KA, KB, PALB, SORTED, THREADS, true, false> : k1_count_cta<KA, KB, PALB, SORTED, THREADS, false, false>);
        static int per_sm_cache[16][3] = {{0}};
        int& per_sm = per_sm_cache[ctx->device & 15][fuse ? 2 : (tr ? 1 : 0)];
        if (per_sm == 0) {
            KB_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_one));
            KB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k1, THREADS, smem_one));
        }
        if (per_sm < 1) { kb_set_error("k1_count_cta does not fit on an SM"); return KB_ECUDA; }
        int64_t grid = (int64_t)ctx->sm_count * per_sm;
        if (grid > n) grid = n;
        if (grid < 1) grid = 1;
        if (!fuse && n < 2 * (int64_t)ctx->sm_count * per_sm) lp = LongPolicy{16384, 16384, 8192, 1, 32};
        KbTimer t(ctx, 0);
        k1<<<(unsigned)grid, THREADS, smem_one, ctx->stream>>>(d_bases, d_offsets, n, d_counts, ld, d_exotic,
                                                               d_presence, ctx->d_k1_scratch, lp, fo);
        ctx->launches++;
    }
    KB_CUDA(cudaGetLastError());
    if (!fuse) {
        auto k1l = k1_count_long<KA, KB, PALB, SORTED, THREADS>;
        static bool attr_set[16] = {false};
        if (!attr_set[ctx->device & 15]) {
            KB_CUDA(cudaFuncSetAttribute(k1l, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_one));
            attr_set[ctx->device & 15] = true;
        }
        KbTimer t(ctx, 1);
        k1l<<<(unsigned)(ctx->sm_count * 2), THREADS, smem_one, ctx->stream>>>(d_bases, d_offsets, d_counts, ld,
                                                                              d_exotic, d_presence,
                                                                              ctx->d_k1_scratch, lp);
        ctx->launches++;
    }
    KB_CUDA(cudaGetLastError());
    return KB_OK;
}

template <class F>
int dispatch_mode(const KbMode& m, F&& f) {
    if (m.permute) return f(std::integral_constant<int, 0>{});     // kmer.py's sorted() column order
    if (m.ka == 5 && m.kb == 6) return f(std::integral_constant<int, 1>{});
    if (m.ka == 4 && m.kb == 5) return f(std::integral_constant<int, 2>{});
    if (m.kb == 0) {
        switch (m.ka) {
            case 1: return f(std::integral_constant<int, 11>{});
            case 2: return f(std::integral_constant<int, 12>{});
            case 3: return f(std::integral_constant<int, 13>{});
            case 4: return f(std::integral_constant<int, 14>{});
            case 5: return f(std::integral_constant<int, 15>{});
            case 6: return f(std::integral_constant<int, 16>{});
            case 7: return f(std::integral_constant<int, 17>{});
        }
    }
    kb_set_error("count mode not built");
    return KB_EUNSUPPORTED;
}

}  // namespace

static int launch_any(kb_ctx* ctx, const KbMode& m, const uint8_t* d_bases, const int64_t* d_offsets, int64_t n, uint32_t* d_counts,
                      int64_t ld, uint32_t* d_exotic, uint32_t* d_presence, int track, const FuseOut* fuse) {
#define KB_ARGS ctx, d_bases, d_offsets, n, d_counts, ld, d_exotic, d_presence, track, fuse
    return dispatch_mode(m, [&](auto tag) -> int {
        constexpr int T = decltype(tag)::value;
        if constexpr (T == 0) return launch<5, 6, true, true>(KB_ARGS);
        else if constexpr (T == 1) return launch<5, 6, false, false>(KB_ARGS);
        else if constexpr (T == 2) return launch<4, 5, false, false>(KB_ARGS);
        else return launch<T - 10, 0, false, false>(KB_ARGS);
    });
#undef KB_ARGS
}

int kb_launch_count_kernels(kb_ctx* ctx, const KbMode& m, const uint8_t* d_bases,
                            const int64_t* d_offsets, int64_t n, uint32_t* d_counts,
                            int64_t ld, uint32_t* d_exotic, uint32_t* d_presence, int track) {
    return launch_any(ctx, m, d_bases, d_offsets, n, d_counts, ld, d_exotic, d_presence, track, nullptr);
}

extern "C" int kb_count_profile(kb_ctx* ctx, int mode, const uint8_t* d_bases, const int64_t* d_offsets, const int32_t* d_key_len,
                                int64_t n, int64_t n_alloc, double* d_profile, int64_t ld_profile, void* d_operand, int64_t ld_operand,
                                kb_rowmeta* d_rowmeta, uint32_t* d_exotic, uint32_t* d_presence, uint32_t* d_flags_or) {
    KB_CHECK_ARG(ctx && (n == 0 || (d_bases && d_offsets && d_key_len)), "null pointer");
    KbMode m;
    int rc = kb_mode_describe(mode, &m);
    if (rc) return rc;
    KB_CHECK_ARG(n >= 0 && n < (1LL << 31) - 2 && n_alloc >= n, "contig count");
    KB_CHECK_ARG(((uintptr_t)d_bases % 16) == 0, "bases must be 16-byte aligned");
    KB_CHECK_ARG(!d_profile || (ld_profile >= m.cols && ((uintptr_t)d_profile % 16) == 0), "profile ld/alignment");
    KB_CHECK_ARG(!d_operand || (ld_operand >= m.cols && (ld_operand % 64) == 0 && ((uintptr_t)d_operand % 16) == 0),
                 "operand ld must be a multiple of 64 and >= columns");
    if (n_alloc == 0) return KB_OK;
    KB_CUDA(cudaSetDevice(ctx->device));
    FuseOut f;
    f.key_len = d_key_len; f.profile = d_profile; f.ld_profile = ld_profile;
    f.operand = reinterpret_cast<__half*>(d_operand); f.ld_operand = ld_operand;
    f.rowmeta = d_rowmeta; f.flags_or = d_flags_or; f.n_alloc = n_alloc;
    return launch_any(ctx, m, d_bases, d_offsets, n, nullptr, 0, d_exotic, d_presence, 0, &f);
}
