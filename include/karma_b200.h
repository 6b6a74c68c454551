/* karma_b200.h -- C ABI of libkarma_b200.so (sm_100a).
 *
 * B200-native replacement for ONE hot path of lmfaber/karma: the per-contig
 * k-mer profile matrix of karma/kmer.py and the exact kNN graph over it.
 * The reference is pure Python and has NO FFI of its own; every entry point
 * below therefore cites the Python function it replaces (paths relative to the
 * reference tree, /root/reference/karma/).  INTEGRATION.md shows the ctypes
 * binding a karma maintainer would add.
 *
 * Conventions
 *  - plain C: pointers + sizes, no exceptions, no Python/torch types.
 *  - every function returns 0 on success or a negative KB_E* code; the text of
 *    the last error on the calling thread is at kb_last_error().
 *  - "d_" pointers are device memory on the context's GPU, "h_" pointers host.
 *  - all work is enqueued on the context's stream (kb_set_stream); functions
 *    that return values to the host synchronise that stream first and say so.
 *  - a context is not thread-safe; distinct contexts are independent.
 *  - there is NO CPU fallback: without a usable sm_100 GPU kb_create fails.
 */
#ifndef KARMA_B200_H
#define KARMA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define KB_API __attribute__((visibility("default")))
#else
#define KB_API
#endif

typedef struct kb_ctx kb_ctx;

/* Per-contig record of the kNN stage, produced by kb_normalise, consumed by kb_knn.
 * One 32-byte record per row, so that a row shard travels in ONE exchange step. */
typedef struct kb_rowmeta {
    double  sqnorm;   /* sum_c count^2 (exact integer)                                   */
    int32_t key_len;  /* len(header key incl. '>'), what kmer.py:213 divides by          */
    int32_t flags;    /* bit0: some count > 2048 (fp16 operand saturated)
                         bit1: sqnorm >= 2^24 (fp32 Gram not exact)
                         bit2: all-zero row (kmer.py:250-258 exits)
                         bit3: padding row of a multi-rank gather (never a neighbour)     */
    float   cm_x;     /* -2/key_len            } score of this row as a KEY in K4:        */
    float   cm_y;     /* sqnorm/key_len^2      } fma(g_ij, cm_x, l_i*cm_y) = l_i*d2_ij - n_i/l_i;
                         +inf when flags & 11: the tensor path never proposes the row      */
    int32_t reserved[2];
} kb_rowmeta;

/* error codes */
#define KB_OK            0
#define KB_EINVAL       -1   /* bad argument                                  */
#define KB_ECUDA        -2   /* CUDA runtime/driver error (see kb_last_error) */
#define KB_ENOGPU       -3   /* no sm_100 device                               */
#define KB_EUNSUPPORTED -4   /* valid request this build cannot serve          */
#define KB_EWORKSPACE   -5   /* workspace too small                            */
#define KB_EOVERFLOW    -6   /* a count exceeds what the kNN operand can hold exactly */

/* column modes (what the count matrix columns mean)
 *  KB_MODE_5P6       kmer.py's default "-k 5p6": 5-mers + STRING-palindromic
 *                    6-mers (kmer.py:46-54,69-81), columns in kmer.py's
 *                    sorted() order over ACGT (kmer.py:172-177): 1088 columns.
 *  KB_MODE_DENSE_5_6 1024 5-mer codes then 4096 6-mer codes (5120 columns);
 *                    the north-star throughput shape, NOT kmer.py's columns.
 *  KB_MODE_DENSE_4_5 256 + 1024 = 1280 columns.
 *  KB_MODE_K(k)      integer k (kmer.py:83-85), 4^k columns in code order
 *                    (== sorted() order for ACGT), 1 <= k <= 7; k = 8..16 through
 *                    kb_kmer_sorted_collect (columns = the observed k-mers).
 * Codes are base-4 big-endian with A=0 C=1 G=2 T=3 (uppercase only: kmer.py
 * has no alphabet, any other byte makes an "exotic" window, see kb_count). */
#define KB_MODE_5P6        0
#define KB_MODE_DENSE_5_6  1
#define KB_MODE_DENSE_4_5  2
#define KB_MODE_K(k)       (16 + (k))
/* OR-ed into kb_count's mode: d_presence then receives only [D] ("a non-ACGT byte was seen");
 * the per-column words are left alone (kb_normalise can derive them from the rows it reads). */
#define KB_COUNT_NO_COLUMNS 0x100

/* kNN implementations */
#define KB_KNN_AUTO   0
#define KB_KNN_SIMT   1   /* CUDA-core tile kernel (checker / small inputs)    */
#define KB_KNN_TC     2   /* tcgen05 + TMA + TMEM distance GEMM, fused top-k   */

KB_API int         kb_version(void);
KB_API const char* kb_last_error(void);

/* Number of count-matrix columns of a mode, or KB_EINVAL. */
KB_API int kb_mode_columns(int mode);

/* Context bound to one GPU (one process per GPU).  Fails with KB_ENOGPU when
 * the device is absent or is not compute capability 10.x. */
KB_API int kb_create(kb_ctx** out, int device);
KB_API int kb_destroy(kb_ctx* ctx);
/* cudaStream_t to enqueue on (e.g. torch.cuda.current_stream().cuda_stream). */
KB_API int kb_set_stream(kb_ctx* ctx, void* cuda_stream);

/* ---- K1: counting ---------------------------------------------------------
 * Replaces KmerClustering.__count_kmer_occurence (kmer.py:56-92) and the
 * window enumeration __kmers_of_seq (kmer.py:181-197) for ACGT-only windows.
 *
 *  d_bases    uint8[total]  the sequences' bytes back to back (values of the
 *                           dict karma.py:40-61 builds); the allocation must be
 *                           16-byte aligned and readable up to
 *                           round_up(total,16)+16 bytes.
 *  d_offsets  int64[n+1]    contig i is bases[offsets[i] .. offsets[i+1])
 *  d_counts   uint32[n*ld]  out: row i = counts of contig i, columns per mode;
 *                           fully overwritten (no need to zero).  ld >= D.
 *  d_exotic   uint32[n]     out (nullable): windows of contig i that contain a
 *                           byte other than A/C/G/T.  kmer.py gives such windows
 *                           their own string-keyed columns; they are NOT counted
 *                           in d_counts (see kb_exotic_*).
 *  d_presence uint32[D+1]   out (nullable): [c] non-zero iff column c is non-zero
 *                           in some row (kmer.py:146-179 "observed k-mers");
 *                           [D] non-zero iff some window holds a non-ACGT byte.
 *                           Must be zeroed by the caller (accumulates, so a
 *                           multi-call / multi-rank OR/MAX is possible).
 * Contigs longer than an internal threshold are split across CTAs and merged.
 */
KB_API int kb_count(kb_ctx* ctx, int mode,
             const uint8_t* d_bases, const int64_t* d_offsets, int64_t n,
             uint32_t* d_counts, int64_t ld,
             uint32_t* d_exotic, uint32_t* d_presence);

/* Totals of the most recent kb_count on this context (synchronises the stream):
 * number of contigs that took the long-contig split path and the sum of d_exotic. */
KB_API int kb_count_stats(kb_ctx* ctx, int64_t* n_long, int64_t* exotic_total);

/* ---- K1x: exotic windows ---------------------------------------------------
 * kmer.py has no alphabet (kmer.py:72-73): 'N', lowercase, '\r' ... make their
 * own k-mer columns, ordered by Python string comparison.  kb_exotic_collect
 * enumerates every window with a non-ACGT byte, packs it as a 54-bit key
 * (6 x 9 bits, big-endian, byte+1, zero padded: key order == string order),
 * and reduces to unique keys and (row,key) counts, all on the GPU.
 * Synchronises the stream.  n_keys / n_entries are written to the host.      */
KB_API int kb_exotic_collect(kb_ctx* ctx, int mode,
                      const uint8_t* d_bases, const int64_t* d_offsets, int64_t n,
                      const uint32_t* d_exotic,
                      int64_t* n_keys, int64_t* n_entries);
/* Copy results of the last kb_exotic_collect to host arrays:
 *  h_keys  uint64[n_keys] ascending;  entries sorted by (key,row):
 *  h_entry_row int32, h_entry_key int32 (index into h_keys), h_entry_count uint32 */
KB_API int kb_exotic_fetch(kb_ctx* ctx, uint64_t* h_keys,
                    int32_t* h_entry_row, int32_t* h_entry_key, uint32_t* h_entry_count);
/* Scatter the collected entries into a count matrix:
 *  d_key_col int32[n_keys] destination column of each unique key. */
KB_API int kb_exotic_scatter(kb_ctx* ctx, const int32_t* d_key_col,
                      uint32_t* d_counts, int64_t ld);

/* ---- integer k >= 8: sorted k-mer counting ---------------------------------------------
 * kmer.py:83-85 accepts any integer -k; beyond k = 7 the 4^k bins leave shared memory, and kmer.py's columns are
 * the OBSERVED k-mers anyway (kmer.py:146-179).  kb_kmer_sorted_collect turns every k-window of every contig,
 * whatever bytes it holds, into a 128-bit key (8 bits per character, big-endian; 1 <= k <= 16), sorts, and
 * reduces to the unique keys (ascending == Python sorted() order) and the (row, key, count) entries, on the GPU.
 * Synchronises.  kb_kmer_sorted_fetch copies the unique keys out (hi = characters 0..7, lo = 8..15);
 * kb_exotic_scatter then writes the counts into a zeroed matrix (d_key_col: destination column of each key). */
KB_API int kb_kmer_sorted_collect(kb_ctx* ctx, int k, const uint8_t* d_bases, const int64_t* d_offsets, int64_t n,
                           int64_t* n_keys, int64_t* n_entries);
KB_API int kb_kmer_sorted_fetch(kb_ctx* ctx, uint64_t* h_keys_hi, uint64_t* h_keys_lo);

/* ---- K2: column compaction -------------------------------------------------
 * Replaces the sorted(set) column dictionary of __extract_kmers
 * (kmer.py:146-179): out[:, colmap[c]] = in[:, c] for colmap[c] >= 0; columns
 * of `out` that no source maps to are zero-filled. */
KB_API int kb_compact(kb_ctx* ctx, const uint32_t* d_in, int64_t ld_in, int32_t d_cols_in,
               const int32_t* d_colmap, int64_t n,
               uint32_t* d_out, int64_t ld_out, int32_t d_cols_out);

/* ---- K3: normalise / convert ----------------------------------------------
 * Replaces fill_array_for_contig + the scatter loop (kmer.py:108-122,
 * :206-233): profile[i,c] = (double)count[i,c] / (double)key_len[i], where
 * key_len[i] = len(header key incl. '>') (kmer.py:213).  Also emits what the
 * kNN consumes.  Any output may be NULL.
 *  d_profile  double[n*ld_profile]
 *  d_operand  fp16 [n_alloc*ld_operand]  raw counts as fp16 (exact <= 2048), columns
 *                                   [d_cols, ld_operand) zero-filled;
 *                                   ld_operand % 64 == 0
 *  d_rowmeta  kb_rowmeta[n_alloc]   squared norm, key length, flags and K4 constants per row
 *  n_alloc    >= n: rows [n, n_alloc) of operand/rowmeta are written as gather padding
 *             (zero counts, flags 1|2|8) so that equal-size shards can be exchanged
 *  d_presence uint32[d_cols+1] (accumulates; zero it first): [c] != 0 iff column c is
 *             non-zero in some row -- OR bit1 of [d_cols] is set, which proves that EVERY
 *             column is present (one CTA saw them all and skipped the per-column stores)
 *  d_flags_or uint32[1] (accumulates): OR of kb_rowmeta.flags over rows [0,n) */
KB_API int kb_normalise(kb_ctx* ctx, const uint32_t* d_counts, int64_t ld, int32_t d_cols,
                 const int32_t* d_key_len, int64_t n, int64_t n_alloc,
                 double* d_profile, int64_t ld_profile,
                 void* d_operand, int64_t ld_operand,
                 kb_rowmeta* d_rowmeta, uint32_t* d_presence, uint32_t* d_flags_or);

/* ---- K1+K3 fused ------------------------------------------------------------
 * kb_count followed by kb_normalise in ONE kernel, for inputs whose column dictionary is the full ACGT set of
 * the mode (what a real assembly gives: validate with d_presence / d_exotic afterwards, and fall back to
 * kb_count + kb_exotic_* + kb_compact + kb_normalise when a column is missing or a non-ACGT byte was seen).
 * The u32 count rows never go to HBM: every contig's shared-memory histogram is turned straight into its
 * fp64 profile row (count / key_len, bit-identical to kb_normalise), its fp16 operand row and its row record.
 * Arguments as in kb_count / kb_normalise; ld_profile / ld_operand >= the mode's column count; contigs of any
 * length (no split path: the longer ones are binned by whole CTAs).  n == 0 with n_alloc > 0 writes padding only. */
KB_API int kb_count_profile(kb_ctx* ctx, int mode, const uint8_t* d_bases, const int64_t* d_offsets, const int32_t* d_key_len,
                     int64_t n, int64_t n_alloc, double* d_profile, int64_t ld_profile, void* d_operand, int64_t ld_operand,
                     kb_rowmeta* d_rowmeta, uint32_t* d_exotic, uint32_t* d_presence, uint32_t* d_flags_or);

/* OR of kb_rowmeta.flags over rows [0,n) (padding rows, bit3, excluded) into *d_out:
 * lets the host validate a whole pass by reading one word. */
KB_API int kb_rowmeta_flags_or(kb_ctx* ctx, const kb_rowmeta* d_rowmeta, int64_t n, uint32_t* d_out);

/* ---- K4 + K5: exact kNN ----------------------------------------------------
 * Replaces the neighbour search inside umap.UMAP(...).fit_transform at
 * kmer.py:285-290 (euclidean metric over the profile rows, the point itself
 * included as neighbour 0; any n_neighbors the reference's CLI accepts,
 * cmd_parser.py:101-107).  Queries are a row range of the (possibly gathered)
 * key set: query q is key row q_row0 + q.
 *
 * Candidate search: integer Gram matrix of the raw counts on the tensor cores
 * (fp16 in, fp32 accumulate: exact while counts <= 2048 and sqnorm < 2^24),
 * distances by norm expansion, per-row running top-k' in the epilogue
 * (k' = 8..64 for k <= 60).  Then K5 reranks the k' candidates exactly:
 *   d2 = sum_c (c_ic*l_j - c_jc*l_i)^2 / (l_i*l_j)^2 = (l_j^2 n_i + l_i^2 n_j - 2 l_i l_j g_ij) / (l_i*l_j)^2   (fp64)
 * with the integer Gram entry g_ij read back out of the candidate's fp32 score when exactly one integer maps to
 * that score (the common case: no second pass over the operand rows), recomputed from the operand rows otherwise;
 * orders by (self first, d2, index) and CERTIFIES every row: with s = l_i*d2 - n_i/l_i the
 * exact score of its k-th neighbour, B the k'-th best fp32 score (every key that is not a
 * candidate scored >= B) and E = 2^-22*(Y^2 + 2cY), c^2 = n_i/l_i, Y = c + sqrt(c^2 + s), a bound
 * on the fp32 evaluation error of any key that could still beat s, the row is final iff
 * s + E < B + 2.5e-6*l_i*d2_k (a quarter of the stated-ties tolerance of 1e-5 relative on d2; nothing at
 * d2 = 0).  Rows that fail (more than k'-k near-ties: long contigs, mass duplicates) and
 * every row when k > 60 are listed in the workspace and redone by kb_knn_fixup with exact
 * distances to ALL keys.
 * d_dist receives sqrt(d2) as float (UMAP's knn_dists), d_d2 (nullable) the fp64 squared
 * distances.
 * Exact side path (K4x): rows whose flags bit0/bit1 are set cannot be scored exactly by
 * the tensor path; they are masked there and handled from their true counts (exact 64-bit integer
 * Gram entries): an ordinary query gets its exact distances to every flagged key as extra candidates;
 * a flagged QUERY is always listed for kb_knn_fixup (exact distances to all keys):
 *  d_flag_rows   int32[n_flag]  ascending key-row indices of ALL flagged rows
 *  d_flag_counts uint32[n_flag*ld_flag_counts]  their count rows (flag_cols columns)
 * (both NULL / 0 when no row is flagged).
 * Multi-GPU (peer-memory exchange, see kb_xchg_*): d_arrive/d_epoch (nullable) make the TMA
 * producer wait until arrive[r] >= *epoch before it touches a key row of source rank
 * r = row / rows_per_src; peer_idx/peer_dist (n_peers device pointers, nullable) are the
 * peers' gathered result arrays: K5 stores row q_row0+q there as well (stores over NVLink).
 * kb_knn only enqueues.  kb_knn_fixup synchronises the stream, returns the number of rows it
 * had to redo (0 in the common case: then it is a read of one word) or a negative error. */
/* ctx may be NULL (then a 148-SM B200 is assumed: the number of candidate lists depends on the SM count) */
KB_API int64_t kb_knn_workspace_bytes(kb_ctx* ctx, int64_t nq, int64_t nk, int64_t q_row0, int32_t d_cols_padded, int32_t k, int impl, int64_t n_flag);
typedef struct kb_knn_xchg {
    const uint32_t* d_arrive;     /* uint32[world]: arrive[r] = epoch of the last shard pushed by rank r */
    const uint32_t* d_epoch;      /* uint32[1]: epoch of the current pass                                   */
    int64_t rows_per_src;         /* rows of the gathered key set per source rank                           */
    int32_t n_peers;              /* entries of peer_idx / peer_dist (0: none)                              */
    int32_t self_rank;            /* this rank: its own rows are always there                               */
    int32_t* const* d_peer_idx;   /* device array of n_peers pointers: peers' all_idx [world*rows_per_src, k] */
    float* const* d_peer_dist;    /* device array of n_peers pointers: peers' all_dist                      */
} kb_knn_xchg;
KB_API int kb_knn(kb_ctx* ctx, int impl, int32_t k,
           const void* d_operand, int64_t ld_operand, int32_t d_cols_padded,
           const kb_rowmeta* d_rowmeta,
           int64_t nk, int64_t q_row0, int64_t nq,
           const int32_t* d_flag_rows, const uint32_t* d_flag_counts, int64_t ld_flag_counts,
           int32_t flag_cols, int64_t n_flag,
           int32_t* d_idx, float* d_dist, double* d_d2,
           void* d_workspace, int64_t workspace_bytes, const kb_knn_xchg* xchg);
KB_API int64_t kb_knn_fixup(kb_ctx* ctx, int impl, int32_t k,
           const void* d_operand, int64_t ld_operand, int32_t d_cols_padded,
           const kb_rowmeta* d_rowmeta,
           int64_t nk, int64_t q_row0, int64_t nq,
           const int32_t* d_flag_rows, const uint32_t* d_flag_counts, int64_t ld_flag_counts,
           int32_t flag_cols, int64_t n_flag,
           int32_t* d_idx, float* d_dist, double* d_d2,
           void* d_workspace, int64_t workspace_bytes);
/* Number of uncertified rows recorded by the last kb_knn in this workspace: a device word the
 * caller may copy back with its other validation words instead of calling kb_knn_fixup. */
KB_API int kb_knn_uncertified_ptr(kb_ctx* ctx, int64_t nq, int64_t nk, int64_t q_row0, int32_t d_cols_padded, int32_t k, int impl, int64_t n_flag,
                           void* d_workspace, const uint32_t** d_count);
/* Host-only views of the tensor kernel's work schedule (tests, diagnostics): kb_knn_plan_info fills
 * out[0..7] = candidate width k', lists per row, key bands, schedule kind, workers (CTA pairs), pieces,
 * 1000 x tile visits of the busiest worker, 1000 x the ideal; kb_knn_plan_table the table itself:
 * pieces int32[pieces*8] = {group, slot, t_lo, cnt, shift, i_lo, i_cnt, 0}, piece_start int32[workers+1],
 * slot_count int32[groups]. */
KB_API int kb_knn_plan_info(int sm_count, int impl, int64_t nq, int64_t nk, int64_t q_row0, int32_t d_cols_padded, int32_t k, int64_t* out);
KB_API int kb_knn_plan_table(int sm_count, int impl, int64_t nq, int64_t nk, int64_t q_row0, int32_t d_cols_padded, int32_t k,
                      int32_t* pieces, int32_t* piece_start, int32_t* slot_count);

/* ---- peer-memory exchange of the kNN stage (GPUs of one node; NVLink / NVSwitch) ----------------
 * SURVEY 8e: the one exchange step of the path.  Every rank owns an "arena" (device memory, same layout
 * on every rank, mapped by its peers through CUDA IPC).  The first 1 KB is the control block (epoch and
 * arrival / done / results flags); the caller lays out the gathered arrays behind it.
 *   kb_xchg_create   allocates the arena and returns the 64-byte IPC handle to hand to the peers
 *   kb_xchg_attach   maps the peers' arenas (handles: world x 64 bytes, indexed by rank)
 *   kb_xchg_peer_ptr base address of a peer's arena in THIS process (peer == rank: the local arena)
 * A pass (all calls only enqueue; the whole pass may be captured in a CUDA graph):
 *   kb_xchg_begin    on the context stream, first thing: epoch += 1, tell the peers that this rank no longer
 *                    reads what they pushed for the previous pass
 *   kb_xchg_push     on `stream` (a side stream ordered after K3): wait until every peer is done with the
 *                    previous pass, copy this rank's shard of every region -- bytes [off + rank*shard_bytes,
 *                    +shard_bytes) -- into every peer's arena (copy engines, three peers at a time, nearest-following
 *                    rank first), then arrive[rank] = epoch there
 *   kb_knn(..xchg..) sweeps the local shard first and waits for arrive[r] before the first key row of rank r
 *   kb_xchg_finish   on the context stream after K5: copy this rank's record (rec_words u32 at
 *                    rec_off + rank*rec_words*4) to every peer, raise the results flag everywhere and wait
 *                    until every peer's results and record have landed here
 * All waits are bounded (a dead peer traps the kernel after ~30 s instead of hanging the GPU). */
typedef struct kb_xchg kb_xchg;
KB_API int kb_xchg_create(kb_ctx* ctx, int world, int rank, int64_t bytes, kb_xchg** out, void** d_local, uint8_t* handle64);
KB_API int kb_xchg_attach(kb_xchg* x, const uint8_t* handles);
KB_API int kb_xchg_peer_ptr(kb_xchg* x, int peer, void** d_ptr);
KB_API int kb_xchg_flags(kb_xchg* x, const uint32_t** d_arrive, const uint32_t** d_epoch);
KB_API int kb_xchg_destroy(kb_xchg* x);
/* once after kb_xchg_attach: memset this rank's shard of every region in every peer's arena and synchronise, so that
 * the peer mappings of a fresh multi-gigabyte arena are set up before the first pass */
KB_API int kb_xchg_warm(kb_xchg* x, int n_regions, const int64_t* region_off, const int64_t* shard_bytes);
KB_API int kb_xchg_begin(kb_xchg* x);
KB_API int kb_xchg_push(kb_xchg* x, void* stream, int n_regions, const int64_t* region_off, const int64_t* shard_bytes);
KB_API int kb_xchg_finish(kb_xchg* x, int64_t rec_off, int32_t rec_words);

/* ---- FASTA reader / packer (host only) --------------------------------------------
 * Replaces read_fasta_file (karma.py:40-61) and the dict -> buffer marshalling: same
 * record rules (first line is a header, key = first space-delimited token INCLUDING
 * '>', universal newlines, line endings stripped from sequence lines, the last record
 * always emitted).  kb_fasta_open reads and sizes the file; kb_fasta_fill writes
 *  h_bases uint8[total_bases], h_offsets int64[n+1], h_key_len int32[n],
 *  h_keys uint8[total_key_bytes] (keys back to back), h_key_offsets int64[n+1]
 * (h_bases / h_keys / h_key_offsets may be NULL).  Non-ASCII files are rejected. */
typedef struct kb_fasta kb_fasta;
KB_API int kb_fasta_open(const char* path, kb_fasta** out, int64_t* n_records, int64_t* total_bases,
                  int64_t* total_key_bytes);
KB_API int kb_fasta_fill(kb_fasta* f, uint8_t* h_bases, int64_t* h_offsets, int32_t* h_key_len,
                  uint8_t* h_keys, int64_t* h_key_offsets);
KB_API int kb_fasta_close(kb_fasta* f);

/* ---- read graph from salmon equivalence classes (SURVEY 8f rank 3; separate path) -----
 * Replaces the loops of ReadGraph.from_equivalence_classes (read_graph.py:61-148).
 * kb_eq_open parses eq_classes.txt (read_graph.py:75-82: contig count, ignored line, names,
 * then "first<TAB>id...<TAB>count" lines) into CSR arrays; kb_eq_fill copies them out:
 *  h_names uint8[name_bytes], h_name_off int64[n+1], h_class_off int64[C+1], h_ids int32[n_ids],
 *  h_counts int64[C], h_skip uint8[C] (1 iff the first token is "1": read_graph.py:102 skips
 *  those classes when pairing).
 * kb_readgraph_build (device inputs, synchronises): d_totals uint64[n_contigs] receives the
 * reads per contig (read_graph.py:86-93); the unique contig pairs with their shared read
 * counts and weights ((shared/totA)+(shared/totB))/2 are kept in the context in exactly the
 * order networkx's graph.edges() yields them in the reference; kb_readgraph_fetch copies
 * them to the host (edges with shared == 0 are included; the reference drops them). */
typedef struct kb_eq kb_eq;
KB_API int kb_eq_open(const char* path, kb_eq** out, int64_t* n_contigs, int64_t* n_classes, int64_t* n_ids,
               int64_t* name_bytes);
KB_API int kb_eq_fill(kb_eq* q, uint8_t* h_names, int64_t* h_name_off, int64_t* h_class_off, int32_t* h_ids,
               int64_t* h_counts, uint8_t* h_skip);
KB_API int kb_eq_close(kb_eq* q);
KB_API int kb_readgraph_build(kb_ctx* ctx, int64_t n_contigs, int64_t n_classes, const int64_t* d_class_off,
                       const int32_t* d_ids, const int64_t* d_counts, const uint8_t* d_skip,
                       uint64_t* d_totals, int64_t* n_edges);
KB_API int kb_readgraph_fetch(kb_ctx* ctx, int32_t* h_a, int32_t* h_b, double* h_weight, uint64_t* h_shared);

/* ---- connection weights between groups of contigs (SURVEY 8f rank 4; follows the read graph) ----
 * Replaces the itertools.product loops of calc_connections_between_mcl_subclusters
 * (karma.py:103-118) and ReadGraph.calc_distance_between_subgraphs (read_graph.py:359-373).
 * Inputs (device): the undirected edge list (every edge once) with float64 weights, and per node
 * a ROW role (group, position in that group's node list) and a COLUMN role, -1 = none.  For every
 * pair of groups (ga < gb) joined by at least one edge the result holds
 *   weight  = the weights of the joining edges added in product order (row position major, column
 *             position minor): the reference's float64 running sum, bit for bit,
 *   edges   = number of joining edges,
 *   over    = number of edges at which the running sum exceeded `cutoff` (how often karma.py:116-117
 *             appends the pair),
 * ordered by (ga, gb) = itertools.combinations order.  Sub-cluster partition: both roles = the node's
 * sub-cluster.  Two node lists: row role = (0, index in nodes_a), column role = (1, index in nodes_b).
 * A node must not occur twice in one list.  n_groups > every group id, max_pos >= every position.
 * kb_links_build synchronises and keeps the result in the context; kb_links_fetch copies it out
 * (any output pointer may be NULL). */
KB_API int kb_links_build(kb_ctx* ctx, int64_t n_edges, const int32_t* d_a, const int32_t* d_b, const double* d_weight,
                   int64_t n_nodes, const int32_t* d_row_group, const int32_t* d_row_pos,
                   const int32_t* d_col_group, const int32_t* d_col_pos,
                   int64_t n_groups, int64_t max_pos, double cutoff, int64_t* n_pairs);
KB_API int kb_links_fetch(kb_ctx* ctx, int32_t* h_group_a, int32_t* h_group_b, double* h_weight, int64_t* h_edges,
                   int64_t* h_over);

/* ---- K7: UMAP's fuzzy simplicial set over the exact kNN lists (the stage after K5/K6) ----
 * Replaces umap.umap_.fuzzy_simplicial_set(knn_indices=, knn_dists=) of umap-learn 0.3.x, the graph that
 * UMAP.fit builds from the lists at kmer.py:285-290 (rules frozen in oracle/umap_graph_oracle.py):
 * smooth_knn_dist (rho, 64-step bisection for sigma, the 1e-3 mean floors), the membership strengths
 * exp(-(d - rho)/sigma) (self -> 0, d <= rho -> 1, index -1 skipped, zeros dropped) and the fuzzy union
 * mix*(A + A^T - A*A^T) + (1 - mix)*A*A^T with zeros dropped.  All arithmetic is fp64.
 *  d_idx   int32[n*k]   neighbour lists, row-major; entries in [-1, n), no index twice in a row (KB_EINVAL)
 *  d_dist  float[n*k]   their distances
 *  d_sigma, d_rho  double[n]  out
 * kb_fuzzy_graph_build synchronises and returns the number of stored entries; the CSR (rows = n, column
 * indices ascending within a row) stays in the context until the next build.  kb_fuzzy_graph_fetch enqueues
 * copies of it into the caller's device buffers (any may be NULL): d_indptr int64[n+1], d_indices int32[nnz],
 * d_data double[nnz]. */
KB_API int kb_fuzzy_graph_build(kb_ctx* ctx, int64_t n, int32_t k, const int32_t* d_idx, const float* d_dist,
                         double local_connectivity, double set_op_mix_ratio, double* d_sigma, double* d_rho,
                         int64_t* nnz);
KB_API int kb_fuzzy_graph_fetch(kb_ctx* ctx, int64_t* d_indptr, int32_t* d_indices, double* d_data);

/* ---- K8: UMAP's layout optimisation over the fuzzy graph (the stage after K7) ----
 * Replaces the tail of umap.umap_.simplicial_set_embedding of umap-learn 0.3.9: the pruning of weights below
 * max / n_epochs, make_epochs_per_sample and optimize_layout (head = tail = the embedding).  umap's loop is sequential;
 * this one is epoch-synchronous and deterministic (rules frozen in oracle/umap_layout_oracle.py, optimize_layout_sync):
 * umap's fp64 schedule (so every kept edge's sample counts are umap's), every sample of epoch n reads the positions of
 * the start of the epoch, negative samples come from a counter-based hash of (seed, kept edge, epoch, sample), and the
 * fp64 gradient coordinates are rounded to int64 at 2^-32 and summed exactly: the same inputs and seed give the same
 * bits whatever the launch shape.  The moves of a vertex within an epoch are summed, not applied one by one.
 *  nnz       the length of d_indices / d_data; nothing beyond it is read
 *  d_indptr  int64[n+1], d_indices int32[nnz], d_data double[nnz]   the graph; indptr from 0 to nnz and never
 *            decreasing, indices in [0, n), data finite and > 0 (KB_EINVAL otherwise)
 *  dim       n_components, 1..64 (KB_EUNSUPPORTED above)
 *  d_embedding float[n*dim]   in: the initial layout (finite, KB_EINVAL otherwise); out: the result
 *  d_samples int64[2*nnz] (nullable): per kept edge in CSR order (rows 0 .. nnz_kept-1), the
 *            positive and negative samples it drew
 *  nnz_kept  out (host): the edges left after pruning
 * Inputs whose worst-case per-vertex, per-epoch sum could leave int64 at 2^-32 are refused (KB_EUNSUPPORTED):
 * max total kept degree x (2 + ceil(2 * rate)) x 4 x initial_alpha x 2^32 >= 2^62.
 * Synchronises once, to validate; the n_epochs epochs are then enqueued without a host synchronisation. */
KB_API int kb_umap_layout(kb_ctx* ctx, int64_t n, int64_t nnz, const int64_t* d_indptr, const int32_t* d_indices, const double* d_data,
                   int32_t dim, int32_t n_epochs, double a, double b, double gamma, double initial_alpha,
                   double negative_sample_rate, uint64_t seed, float* d_embedding, int64_t* d_samples, int64_t* nnz_kept);

/* ---- K9: HDBSCAN's mutual-reachability MST (device) and its clusters (host) ----
 * Replaces hdbscan.HDBSCAN(min_cluster_size=m).fit(embedding) of hdbscan 0.8.22 (kmer.py:296-301), metric euclidean,
 * alpha 1, eom selection; the reference of record is scikit-learn 1.9.0's port of its tree code (rules frozen in
 * oracle/hdbscan_oracle.py).  d(i, j) = RN(sqrt(sum_c (x_ic - x_jc)^2)) in fp64 from the float32 coordinates, in
 * coordinate order, no FMA; core_i = the core_k-th smallest of {d(i, j) : all j}, d(i, i) = 0 and duplicates counted
 * (hdbscan's min_samples = m is core_k = m + 1); w(i, j) = max(core_i, core_j, d(i, j)).  Edges are totally ordered
 * by (w, min(i, j), max(i, j)), so the MST is unique: it is the exact MST (hdbscan 0.8.22 defaults to an approximate
 * one), whatever the execution order.
 * kb_hdbscan_mst (device pointers; Boruvka over the implicit complete graph, one host read per round):
 *  d_x       float[n*dim]   the points, row-major, finite (KB_EINVAL otherwise); n >= 2
 *  dim       1..64, core_k 1..min(n, 128) (KB_EINVAL below 1 or above n, KB_EUNSUPPORTED above 64 / 128)
 *  d_core    double[n]      out: core distances
 *  d_edges   int32[(n-1)*2] out: the MST's edges, each (min, max), sorted by (w, min, max)
 *  d_weights double[n-1]    out: their weights
 * Synchronises once per round; the sorted edges are enqueued on the context stream when it returns.
 * kb_hdbscan_labels (host pointers, no GPU): scikit-learn's make_single_linkage, _condense_tree, _compute_stability,
 * _get_clusters (eom, allow_single_cluster), _do_labelling and get_probabilities over such a sorted spanning tree,
 * with their fp64 operation order.  KB_EINVAL for an index outside [0, n), an edge not (min, max), edges out of
 * (w, min, max) order, a negative or non-finite weight, a cycle, or min_cluster_size < 2.
 *  labels int32[n] (-1 = noise; clusters numbered in the order of their condensed-tree ids), probabilities double[n],
 *  n_clusters out.  It also returns KB_EINVAL, with a message naming an internal inconsistency, if its own tree walk
 *  contradicts itself; a valid tree never does. */
KB_API int kb_hdbscan_mst(kb_ctx* ctx, int64_t n, int32_t dim, const float* d_x, int32_t core_k,
                   double* d_core, int32_t* d_edges /* [n-1][2], (min,max) */, double* d_weights /* [n-1] */);
KB_API int kb_hdbscan_labels(int64_t n, const int32_t* edges, const double* weights, int32_t min_cluster_size,
                   int32_t allow_single_cluster, int32_t* labels, double* probabilities, int64_t* n_clusters);

/* ---- K10: UMAP's spectral initialisation over the pruned fuzzy graph (the stage between K7 and K8) ----
 * Replaces umap.spectral.spectral_layout of umap-learn 0.3.9 (init="spectral"), disconnected graphs included (rules
 * frozen in oracle/umap_spectral_oracle.py).  The graph (as for kb_umap_layout: indptr from 0 to nnz, indices in
 * [0, n), data finite and > 0, else KB_EINVAL; symmetric, as K7 builds it) is pruned with K8's rule, w >= max / n_epochs
 * (n_epochs 0: no pruning, for a graph pruned already).  Its weakly connected components are labelled in the order of
 * their smallest vertex (scipy's connected_components).
 *  - A connected graph, and every component of at least 2 * dim vertices of a disconnected one, is solved: the unit
 *    eigenvectors of the dim smallest non-trivial eigenvalues of L = I - D^-1/2 W D^-1/2, each with its largest-|.|
 *    entry positive.  fp64 Lanczos with full reorthogonalisation and thick restart on D^-1/2 W D^-1/2, the trivial
 *    vector D^1/2 1 deflated; every returned Ritz pair has a residual estimate ||M v - theta v|| <= 1e-9.  A solve that
 *    needs more than 500 restarts leaves its component not converged (status 2: umap's ARPACK fallback, a draw); a
 *    repeated wanted eigenvalue (a uniform ring, a clique) is found only through rounding and may end so.
 *  - Components of fewer than 2 * dim vertices take uniform draws (status 0).
 *  - Meta points (n_comp > 1): with n_comp > 2 * dim, scikit-learn 1.9.0's spectral embedding of the components'
 *    float32 centroids (numpy's float32 mean, bit for bit) under exp(-d^2), over its global max; this needs the data
 *    (KB_EINVAL without), refuses more than 65536 components (KB_EUNSUPPORTED: n_comp^2 fp64 of dense affinity), and
 *    an affinity that underflows to 0 (KB_EUNSUPPORTED); a meta solve that does not converge is KB_EINVAL.  With
 *    2 <= n_comp <= 2 * dim, the rows of [eye(k), 0; -eye(k), 0], k = ceil(n_comp / 2).
 *  - range[c] = half the smallest positive euclidean distance from meta point c to the others, fp64 in coordinate
 *    order without FMA (umap takes it from a dot-product expansion; DESIGN §3 K10); 10 for a connected graph.
 * The same inputs give the same bits: fixed-order reductions, integer atomics only.
 * kb_spectral_build (device pointers; synchronises; keeps the result in the context until the next build):
 *  dim      1..64 (KB_EUNSUPPORTED above); a connected graph needs n > dim + 1 (KB_EINVAL)
 *  d_x      nullable: the data, row-major n x x_cols, x_dtype 1 float32 or 2 float64 (every value is cast to
 *           float32 first, as umap's check_array does; not finite -> KB_EINVAL); x_dtype 0: none
 *  n_comp   out: the number of components
 * kb_spectral_fetch (any pointer may be NULL): h_size int32[n_comp], h_status int32[n_comp] (0 draw, 1 solved,
 *  2 not converged), h_range double[n_comp], h_stats int64[6] (Lanczos steps and restarts over the components, the
 *  meta solve's steps and restarts, component rounds, 0); device copies enqueued on the context stream: d_labels
 *  int32[n], d_meta double[n_comp*dim] (n_comp > 1), d_vectors double[n*dim] (row i: vertex i's entries of its
 *  component's vectors; zero where not solved), d_centroids double[n_comp*x_cols] (n_comp > 2 * dim).
 * kb_spectral_assemble: the float32 [n, dim] layout spectral_layout returns, with umap's arithmetic: solved,
 *  fp32(v * (range / max|v|) + meta) (fp32(v) when connected); otherwise fp32((-range + 2 range u) + meta) (no meta
 *  when connected), u = d_u[i*dim + d], the uniform [0, 1) draws of random_state.uniform for vertex i's component,
 *  row i = vertex i (d_u may be NULL when every component is solved).  Enqueued on the context stream. */
KB_API int kb_spectral_build(kb_ctx* ctx, int64_t n, int64_t nnz, const int64_t* d_indptr, const int32_t* d_indices,
                   const double* d_data, int32_t n_epochs, int32_t dim, const void* d_x, int32_t x_dtype, int64_t x_cols,
                   int64_t* n_comp);
KB_API int kb_spectral_fetch(kb_ctx* ctx, int32_t* h_size, int32_t* h_status, double* h_range, int64_t* h_stats,
                   int32_t* d_labels, double* d_meta, double* d_vectors, double* d_centroids);
KB_API int kb_spectral_assemble(kb_ctx* ctx, const double* d_u, float* d_out);

/* ---- K11: MCL of many groups of a read graph in one call ----
 * Replaces karma's `mcl - --abc -o -` per k-mer cluster (Mcl.run_pipe); the semantics are this library's definition,
 * frozen in oracle/mcl_oracle.py (DESIGN §3 K11 lists the parts that rest on memory of mcl 14-137, unpinned).
 * Group g's abc stream is the edges with both ends in g, in edge order; its nodes are numbered by first appearance
 * (a before b).  A = adjacency + loops A[j,j] = max_i A[i,j]; M = A / column sums; until g's chaos
 * max_j (max_i M[i,j] / sum_i M[i,j]^2 - 1) < 1e-4, each iteration expands (M*M, terms in ascending k), prunes every
 * column (cutoff 1/7000, the 900 largest, recovery up to 1000 entries or 90 % of the mass; ties by row), inflates
 * (x^inflation) and renormalises.  fp64, no FMA, every sum a left fold in ascending rows: the same inputs give the same
 * bits.  Every group iterates until its own convergence, so its result does not depend on the other groups.
 * Interpretation: attractors M[a,a] > 0, systems = connected attractors numbered by their smallest attractor, each node
 * to the smallest system it reaches (alone if none); clusters ordered by size desc, then smallest member.
 * kb_mcl_build (device pointers; synchronises once per iteration; keeps the result on the host side of the context):
 *  d_a, d_b int32[n_edges]  edge ends in [0, n_nodes); d_w double[n_edges]
 *  d_group  int32[n_nodes]  group ids in [-1, n_groups), -1 = in no group
 *  inflation finite and > 1
 *  KB_EINVAL for an index or group id out of range, and inside a group for a self-edge, a pair listed twice or a weight
 *  that is not finite and > 0; also for a group that has not converged after 1000 iterations (the message names it).
 *  n_cols out: the nodes in streams; nnz out: the entries of the final matrix.
 * kb_mcl_fetch (host pointers, any may be NULL): h_local int32[n_nodes] (stream index, -1 outside every stream),
 *  h_cluster int32[n_nodes] (cluster number within the group, in output order; -1 outside), h_n_clusters,
 *  h_iterations, h_overlap int64[n_groups] (overlap: nodes reaching attractors of several systems), and the final
 *  matrix: h_colptr int64[n_cols + 1] (columns group by group, stream index within), h_rows int32[nnz] (stream
 *  indices, ascending per column), h_vals double[nnz]. */
KB_API int kb_mcl_build(kb_ctx* ctx, int64_t n_nodes, int64_t n_edges, const int32_t* d_a, const int32_t* d_b,
                   const double* d_w, const int32_t* d_group, int64_t n_groups, double inflation, int64_t* n_cols,
                   int64_t* nnz);
KB_API int kb_mcl_fetch(kb_ctx* ctx, int32_t* h_local, int32_t* h_cluster, int64_t* h_n_clusters, int64_t* h_iterations,
                   int64_t* h_overlap, int64_t* h_colptr, int32_t* h_rows, double* h_vals);

/* Per-stage device times.  With timing enabled every launch of a stage is bracketed
 * by a CUDA-event pair on the context stream (a ring of 128 pairs per stage).
 * kb_stage_ms synchronises, returns the mean duration (ms) and the number of launches
 * recorded since the last read, and resets the stage.
 *  which: 0 count, 1 count-long, 2 compact, 3 normalise, 4 knn-gemm, 5 rerank, 6 exact side path,
 *         7 read-graph build, 8 group-pair connection weights, 9 K9 core distances, 10 K9 Boruvka rounds (one launch
 *         recorded per round), 11 K9 edge sort, 12 K10 components (validation, pruning, component rounds, labels and
 *         the permuted CSR), 13 K10 eigensolve (every component solve, host Ritz steps included), 14 K10 meta-embedding
 *         (centroids, affinity, the meta solve, data ranges), 15 K11 set-up (validation, labelling, the initial matrix),
 *         16 K11 iteration (one launch recorded per iteration) */
KB_API int kb_enable_timing(kb_ctx* ctx, int on);
KB_API int kb_stage_ms(kb_ctx* ctx, int which, float* mean_ms, int* n_launches);
/* Number of kernels this library launched since the context was created (a CUB device-wide call counts as one). */
KB_API int64_t kb_launch_count(kb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* KARMA_B200_H */
