/*
 * swb200.h -- C ABI of libswb200.so: B200-native score-only Smith-Waterman/Gotoh.
 *
 * The drop-in boundary is the reference's own GPU header, algoGPU.h:5-9 (three extern "C"
 * functions: two host byte sequences in, one int local-alignment score out) plus the fourth symbol
 * of SmithDiagonalGPUrefactored.cu:174.  Those four names are declared in include/algoGPU.h and
 * exported by the library with the reference's exact signatures; TestFileWithGPU.cpp:82,87,92
 * links against them unchanged (INTEGRATION.md).  Everything below is additive: runtime scoring
 * parameters (the reference hard-codes them per file, main.cpp:20-23), error codes (the reference
 * has no error channel), device-resident inputs, batches, banded alignment, multi-GPU stripes.
 *
 * Plain C, plain pointers and sizes; no C++ or torch types cross this boundary.
 */
#ifndef SWB200_H
#define SWB200_H

#include <stdint.h>

#if defined(__GNUC__)
#define SWB200_API __attribute__((visibility("default")))
#else
#define SWB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* MATCH / MISMATCH / G_INIT / G_EXT of main.cpp:20-23, as data.  A gap of length k costs
 * gap_init + (k-1)*gap_ext (main.cpp:57-58).  Limits: |match|,|mismatch| <= 100,
 * 0 <= gap_ext, gap_init <= 100, match + gap_init <= 127, mismatch <= 0 <= match. */
typedef struct {
  int match;
  int mismatch;
  int gap_init;
  int gap_ext;
} swb200_params;

/* Kernel selection; all zero = automatic.  Exposed for benchmarking and tests. */
typedef struct {
  int lanes;       /* 0 auto (packed 16-bit, 32-bit re-run if the score leaves the s16 range), 16, 32 */
  int rows;        /* R: DP rows per sub-lane, one of 1,2,3,4,6,8,10,12,14,16 (batch kernel: 2,4,6,8,10,12,16); 0 auto */
  int config;      /* pair engine: 0 auto, 1 = one warp per scheduler (4 warps/CTA, slack step), 2 = two (8 warps/CTA), 3 = one, no
                      slack step; measurement variants for packed 16-bit lanes: 4 = 1 plus a slack step inside each thread,
                      5 = 1 with the boundary chunk fetched by cp.async.bulk + mbarrier, 6 = 12 warps/CTA (rows <= 10);
                      7 = the CTA-chained engine (csrc/swb_chain.cuh: one band per warp, four consecutive bands per CTA handed
                      over through shared memory; plain 16-bit lanes, one GPU, rows 1,2,3,4,6,8) -- what "auto" picks for
                      fill-dominated pairs such as 100 000 x 100 000.
                      banded calls with a 64-diagonal band: 0 = 4 threads per pair (default), 8 = 8 threads per pair, 16 = 16
                      threads per pair, 2 = 2 threads per pair; ignored for wider bands */
  int ctas;        /* thread blocks (<= co-resident limit); 0 auto */
  int no_linear;   /* 1 = keep the affine kernel even when gap_init == gap_ext */
  int orient;      /* 0 auto (stripe the longer sequence across lanes), 1 = stripe seq1, 2 = stripe seq2 */
  int rebase;      /* 16-bit lanes relative to a moving base (scores beyond 32767 at the packed rate): 0 auto, 1 force, -1 never */
  int two_sided;   /* forward sweep on the top half of the rows + reversed sweep on the bottom half: 0 auto, 1 force, -1 never */
} swb200_options;

/* Return codes (legacy names have no error channel: they print and abort instead). */
#define SWB200_OK 0
#define SWB200_ERR_CUDA (-1)      /* a CUDA call failed; see swb200_last_error() */
#define SWB200_ERR_ARG (-2)       /* bad argument or parameter outside the documented limits */
#define SWB200_ERR_ALPHABET (-3)  /* batch calls only: a byte other than A,C,G,T */
#define SWB200_ERR_TIMEOUT (-4)   /* a boundary hand-off never arrived (peer GPU gone) */
#define SWB200_ERR_NOMEM (-5)
#define SWB200_ERR_RANGE (-6)     /* score does not fit the requested lane width */

SWB200_API const char* swb200_last_error(void);
SWB200_API int swb200_device_count(void);

/* Debugging / measurement switches.  Each has an environment variable that is read ONCE, at the first call
 * into the library (the scoring calls never call getenv); swb200_configure changes them afterwards:
 *   "spin_limit" (SWB200_SPIN_LIMIT)  polls before a waiting warp gives up and the call returns SWB200_ERR_TIMEOUT
 *   "debug" (SWB200_DEBUG)            "1": print the post-mortem of a timed-out hand-off to stderr
 *   "prof" (SWB200_PROF)              "1": per-warp cycle counters of the pair engine to stderr; any other value: a file
 *                                     that receives one JSON line per launch; "": off
 *   "dbg" (SWB200_DBG)                timing experiments only (1 = no boundary stores, 2 = no boundary polls: WRONG scores)
 *   "dump_final" (SWB200_DUMP_FINAL)  file receiving the two middle boundary rows of a two-sided sweep
 *   "batch_chunk_bytes" (SWB200_BATCH_CHUNK_BYTES)  chunk size of the host batch calls' copy/compute pipeline (0 = default)
 *   "ring_min_cells" (SWB200_RING_MIN_CELLS)  host-buffer pairs with at least this many cells use all devices chosen
 *                                     with swb200_set_devices (default 2e11)
 *   "chain" (SWB200_CHAIN)            "0": the planner never picks the CTA-chained engine (launch config 7) by itself
 *   "align_block_rows" (SWB200_ALIGN_BLOCK_ROWS)  swb200_align's traceback in blocks of this many span rows, a positive
 *                                     multiple of 256 (SWB200_ERR_ARG otherwise), even when the whole rectangle fits;
 *                                     "0" (default): blocks only when the rectangle's directions do not fit in device memory */
SWB200_API int swb200_configure(const char* key, const char* value);

/* Diagnostic (needs no GPU): the kernel variant the planner picks for an n x m pair on `sms` SMs in all (148 per B200):
 * out = {mode, rows, launch config, two_sided}, *est_cycles its cost estimate.  lanes: 16 = packed 16-bit, 17 = packed
 * 16-bit re-based, 32 = 32-bit. */
SWB200_API int swb200_plan(long long n, long long m, const swb200_params* p, const swb200_options* opt, int lanes, int sms,
                           int allow_two_sided, int out[4], double* est_cycles);

/* ---- several GPUs from one host process ------------------------------------------------------------
 * The reference's caller is a single-threaded C++ loop (TestFileWithGPU.cpp:57-94).  swb200_set_devices(G) makes
 * the HOST-buffer entry points below (and therefore the four legacy names) use devices 0 .. G-1:
 *   - a pair with at least "ring_min_cells" cells (swb200_configure) is spread over an in-process ring of the G
 *     GPUs (one host thread per GPU for the duration of the call, peer access over NVLink, swept from both ends);
 *   - the host batch calls (swb200_score_batch, swb200_score_banded_batch, swb200_score_batch_packed,
 *     swb200_score_banded_batch_packed, swb200_align_batch) cut the batch into G contiguous ranges of pairs, one
 *     copy/compute pipeline per GPU, no communication; swb200_last_run(NULL, ..) then reports cells and launches summed
 *     over the GPUs and the longest device time.
 * Results are identical for every G.  count 0 or 1 = one GPU (the default).  Needs peer access between the devices. */
SWB200_API int swb200_set_devices(int count);
SWB200_API int swb200_get_devices(void);

/* ---- one pair, HOST buffers: the call behind the four legacy names ------------------------------
 * seq1/seq2: raw bytes, not NUL-terminated, caller-owned, never modified (algoGPU.h:5-9).
 * n = len(seq1), m = len(seq2); n == 0 or m == 0 scores 0.  p == NULL means 1/-1/1/1. */
SWB200_API int swb200_score(const unsigned char* seq1, int n, const unsigned char* seq2, int m,
                 const swb200_params* p, int* score_out);
SWB200_API int swb200_score_ex(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                    const swb200_params* p, const swb200_options* opt, int* score_out);

/* ---- handle API: sequences already resident in HBM ------------------------------------------------ */
typedef struct swb200_ctx swb200_ctx;
SWB200_API int swb200_ctx_create(int device, swb200_ctx** ctx_out);
SWB200_API void swb200_ctx_destroy(swb200_ctx* ctx);

/* d_seq1/d_seq2: DEVICE pointers to raw bytes.  stream: a cudaStream_t (NULL = default stream).
 * All kernels are enqueued on `stream`; the call returns after the 16-byte result came back. */
SWB200_API int swb200_score_device(swb200_ctx* ctx, const unsigned char* d_seq1, long long n,
                        const unsigned char* d_seq2, long long m, const swb200_params* p,
                        const swb200_options* opt, void* stream, int* score_out);

/* ---- score AND end cell (SURVEY.md 8(f) row 4; the reference is score-only, README.md:6) -----------
 * i_end / j_end: 1-based positions in seq2 / seq1 of the last aligned pair of the best local alignment,
 * i.e. the cell (i, j) of main.cpp's H matrix that holds the maximum; among several such cells the one with
 * the smallest j, then the smallest i.  Score 0 gives (0, 0).  One pass of the 32-bit tracking kernel;
 * needs match * min(n, m) < 2^20 (SWB200_ERR_RANGE otherwise). */
SWB200_API int swb200_score_end(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                     const swb200_params* p, int* score_out, long long* i_end, long long* j_end);
SWB200_API int swb200_score_end_device(swb200_ctx* ctx, const unsigned char* d_seq1, long long n,
                            const unsigned char* d_seq2, long long m, const swb200_params* p, void* stream,
                            int* score_out, long long* i_end, long long* j_end);

/* Score, START cell and end cell: span_out = {i_start, j_start, i_end, j_end}, 1-based and inclusive (i in seq2, j in
 * seq1); the end cell as in swb200_score_end, the start cell the one closest to it (largest j_start, then largest
 * i_start) among the optimal alignments that end there.  Two passes: the tracking kernel, then the anchored
 * recurrence over the reversed prefixes.  All zero when the score is 0.  Same limits as swb200_score_end. */
SWB200_API int swb200_score_span(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                      const swb200_params* p, int* score_out, long long span_out[4]);
SWB200_API int swb200_score_span_device(swb200_ctx* ctx, const unsigned char* d_seq1, long long n,
                             const unsigned char* d_seq2, long long m, const swb200_params* p, void* stream,
                             int* score_out, long long span_out[4]);

/* ---- the alignment itself (SURVEY.md 8(f) row 4, second half; the reference is score-only, README.md:6) ----------
 * Score, span (as swb200_score_span) and an extended CIGAR of the best local alignment between the start and the end
 * cell, read from the start cell: "<count>=" matches, "<count>X" mismatches, "<count>I" bases of seq1 against a gap,
 * "<count>D" bases of seq2 against a gap.  Contract: re-scoring the CIGAR over the span with the costs of
 * main.cpp:28-33,57-58 (MATCH / MISMATCH per pair, G_INIT for the first character of a gap, G_EXT for each further
 * one) gives exactly *score_out -- the library checks this itself before it returns.  Which of several equally good
 * alignments is reported: at every cell diagonal before gap in seq2 (E) before gap in seq1 (F); a gap counts as
 * extended only where extending is strictly better than opening.
 * Three passes: end cell, start cell, then the anchored recurrence over the span rectangle with 4 bits of traceback
 * direction per cell kept in HBM (0.5 byte per cell: the 100 000 x 100 000 pair takes 5 GB) and a walk back through them.
 * When the whole rectangle's directions do not fit in free device memory, the third pass runs in blocks of rows: a
 * forward sweep keeps only the boundary row between blocks (16 bytes per span column each), then the walk goes back
 * block by block, recomputing each block from the row above it over the columns left of the walk.  Score, span and
 * CIGAR are byte for byte those of the one-block traceback; the cost is about one more sweep over the span.
 * SWB200_ERR_NOMEM only when not even a block of 256 rows plus the boundary rows fits.  "align_block_rows"
 * (swb200_configure) forces the blocked path.  cigar_out may be NULL to ask for the length only (*cigar_len_out,
 * without the terminating NUL).  Same limits as swb200_score_end. */
SWB200_API int swb200_align(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                            const swb200_params* p, int* score_out, long long span_out[4], char* cigar_out,
                            long long cigar_cap, long long* cigar_len_out);
SWB200_API int swb200_align_device(swb200_ctx* ctx, const unsigned char* d_seq1, long long n, const unsigned char* d_seq2,
                                   long long m, const swb200_params* p, void* stream, int* score_out, long long span_out[4],
                                   char* cigar_out, long long cigar_cap, long long* cigar_len_out);

/* What the last swb200_score*_ call on this context actually ran. */
typedef struct {
  int lanes;            /* 16 or 32 */
  int rebased;          /* 1 if the 16-bit lanes were relative to a moving base */
  int two_sided;        /* 1 if the pair was swept from both ends (two half problems + combination kernel) */
  int linear;           /* 1 if the gap_init == gap_ext kernel was used */
  int rows;             /* R */
  int config;
  int ctas, warps;      /* launch shape */
  int bands;            /* DP bands of the pair */
  int engine_launches;  /* wavefront kernels launched (2 when an s16 run was repeated in s32) */
  int aux_launches;     /* encode / presence kernels launched */
  long long cells;      /* n*m */
  float engine_ms;      /* device time of the last wavefront kernel (CUDA events on its stream) */
} swb200_run_info;
SWB200_API int swb200_last_run(swb200_ctx* ctx, swb200_run_info* info);

/* ---- batches of independent pairs (reads vs windows) ----------------------------------------------
 * The reference scores pairs one call at a time (TestFileWithGPU.cpp:57-94); a batch call scores
 * npairs independent pairs in one kernel, several pairs per warp, nothing leaving the registers.
 * Pair k is seq1_all[off1[k] .. off1[k]+len1[k]) vs seq2_all[off2[k] .. off2[k]+len2[k]).
 * Limits: bytes must be A,C,G,T; min(len1[k], len2[k]) <= 1024 and match*min(len) <= 32766 - match for every
 * pair (SWB200_ERR_RANGE otherwise; such pairs: swb200_score).  Empty sequences score 0.
 * Every host batch call (HOST buffers, here and below) checks its arguments, lengths, parameters and these limits before
 * it touches a device, so a bad call fails with SWB200_ERR_ARG / SWB200_ERR_RANGE on any machine. */
SWB200_API int swb200_score_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                                  const unsigned char* seq2_all, const long long* off2, const int* len2,
                                  long long npairs, const swb200_params* p, const swb200_options* opt,
                                  int* scores_out);

/* The same for HOST batches that are already in the resident 2-bit format (32 symbols per 64-bit word, symbol k at bits
 * 2*(k%32), codes (c >> 1) & 3, i.e. A,C,G,T -> 0,1,3,2; per pair q_stride words of the SHORTER sequence and t_stride words
 * of the longer one; strides from swb200_batch_strides): a quarter of the bytes cross PCIe and no pack kernel runs.
 * swb200_pack_batch_host converts raw bytes into that layout on the host (format conversion only -- nothing is scored on
 * the CPU); it writes the same words as the device packer.  q_len / t_len: the packed lengths (q_len[k] <= t_len[k]). */
SWB200_API int swb200_batch_strides(int max_short, int max_long, long long* q_stride, long long* t_stride);
SWB200_API int swb200_pack_batch_host(const unsigned char* seq1_all, const long long* off1, const int* len1,
                                      const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                                      long long q_stride, long long t_stride, unsigned long long* q_words,
                                      unsigned long long* t_words, int* q_len, int* t_len);
SWB200_API int swb200_score_batch_packed(const unsigned long long* q_words, long long q_stride,
                                         const unsigned long long* t_words, long long t_stride, const int* q_len,
                                         const int* t_len, long long npairs, const swb200_params* p,
                                         const swb200_options* opt, int* scores_out);

/* Banded batches (swb200_score_banded_batch below) from HOST words in the same 2-bit format.  seq1 (columns) and seq2
 * (rows) keep their roles: stride1 words of seq1 and stride2 words of seq2 per pair (swb200_banded_strides), len1 / len2
 * as given by the caller.  swb200_pack_banded_host is the format conversion on the host. */
SWB200_API int swb200_banded_strides(int max_len1, int max_len2, long long* stride1, long long* stride2);
SWB200_API int swb200_pack_banded_host(const unsigned char* seq1_all, const long long* off1, const int* len1,
                                       const unsigned char* seq2_all, const long long* off2, const int* len2,
                                       long long npairs, long long stride1, long long stride2,
                                       unsigned long long* words1, unsigned long long* words2);
SWB200_API int swb200_score_banded_batch_packed(const unsigned long long* words1, long long stride1,
                                                const unsigned long long* words2, long long stride2, const int* len1,
                                                const int* len2, long long npairs, int band_lo, int band_hi,
                                                const swb200_params* p, const swb200_options* opt, int* scores_out);

/* Device-resident form: pack once (2-bit codes in HBM, the resident format), score many times.
 * All pointers are DEVICE pointers; max_short / max_long bound min(len1,len2) / max(len1,len2) over the
 * batch; total_cells (sum of len1*len2) is only recorded for swb200_last_run.  d_scores: npairs ints.
 * keep_order = 0: the shorter sequence of each pair is striped across lanes (full DP, swb200_batch_score);
 * keep_order = 1: seq1 stays the column sequence, seq2 the row sequence (needed by the banded kernel, where
 * j - i matters); max_short / max_long then bound len1 / len2. */
typedef struct swb200_batch swb200_batch;
SWB200_API int swb200_batch_pack_device(swb200_ctx* ctx, const unsigned char* d_seq1_all, const long long* d_off1,
                                        const int* d_len1, const unsigned char* d_seq2_all, const long long* d_off2,
                                        const int* d_len2, long long npairs, int max_short, int max_long,
                                        long long total_cells, int keep_order, void* stream,
                                        swb200_batch** batch_out);
SWB200_API int swb200_batch_score(swb200_batch* batch, const swb200_params* p, const swb200_options* opt,
                                  void* stream, int* d_scores);

/* Batches whose shorter side is over 1024 (gene / contig pairs, long reads without a band, database search with long
 * queries): the same scores as swb200_score_ex gives each pair, from one multi-band kernel.  One warp per pair; the shorter
 * sequence is cut into bands of 64*R rows swept one after the other over the whole longer one, the bottom row of a band
 * carried to the next through a per-warp row in device memory; warps take the next pair from a counter, so a ragged batch
 * keeps every warp busy.  Argument form and limits are swb200_score_batch's without the 1024 cap: bytes A,C,G,T
 * (SWB200_ERR_ALPHABET), match*min(len) <= 32766 - match (SWB200_ERR_RANGE); the longer side is limited by int and by
 * the boundary rows, (max(len) rounded up to 32) * 4 bytes per resident warp (SWB200_ERR_NOMEM).  Both calls run this
 * kernel for any shorter side, also one of 1024 or less.  opt->rows picks R (2,4,6,8,10,12,16; 0: the smallest R with
 * 64*R >= the longest shorter side, else 16; other values SWB200_ERR_ARG); opt->no_linear as in swb200_score_batch; other
 * option fields are ignored.  All checks run before a device is touched.  swb200_last_run reports config 332, rows R and
 * bands = the band count of the tallest pair.  The host call packs and scores in chunks of whole waves of resident warps
 * and shards over swb200_set_devices like swb200_score_batch; the device call takes a batch packed with keep_order = 0
 * (SWB200_ERR_ARG for keep_order = 1). */
SWB200_API int swb200_score_long_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                                       const unsigned char* seq2_all, const long long* off2, const int* len2,
                                       long long npairs, const swb200_params* p, const swb200_options* opt,
                                       int* scores_out);
SWB200_API int swb200_batch_score_long(swb200_batch* batch, const swb200_params* p, const swb200_options* opt,
                                       void* stream, int* d_scores);
SWB200_API void swb200_batch_free(swb200_batch* batch);

/* ---- batch alignment: score, span and CIGAR for every pair of a batch -------------------------------------------------
 * For every pair k the same score, span {i_start, j_start, i_end, j_end} and alignment that swb200_align(seq1[k], seq2[k])
 * returns for that pair alone (same tie rules), one thread per pair on the device: end cell, start cell, then the anchored
 * recurrence over the span rectangle with 4 bits of traceback direction per cell and the walk back through them.  Limits
 * and errors are those of swb200_score_batch (bytes A,C,G,T: SWB200_ERR_ALPHABET; min(len1,len2) <= 1024: SWB200_ERR_ARG;
 * match*min(len) <= 32766 - match: SWB200_ERR_RANGE); pairs outside them go through swb200_align.  Score 0 (and an
 * empty sequence) gives span (0,0,0,0) and no operations.
 * Operations: count << 4 | op with op 7 '=', 8 'X', 1 'I' (a base of seq1 against a gap), 2 'D' (a base of seq2 against a
 * gap) -- BAM's numbering -- first operation first.  Pair k's operations go to ops_out[k*ops_stride ...], ops_count[k] of
 * them; a pair that needs more than ops_stride gets ops_count[k] = -(its count), nothing is written for it, and the call
 * still succeeds (len1 + len2 operations always suffice; the host call returns that pair's slot zero-filled).  When gap_ext > gap_init the recurrence never extends a gap,
 * so two neighbouring gap characters are two gaps and are reported as two operations ("1I1I"); otherwise the operations
 * are exactly swb200_align's CIGAR.  Every alignment is re-scored on the device with the costs of main.cpp:28-33,57-58
 * before the call returns; a mismatch fails the call with SWB200_ERR_CUDA ("internal: ...").
 * The host call copies and packs in chunks and, after swb200_set_devices(G), gives each GPU a contiguous range of pairs
 * (results identical for every G).  spans_out: 4 ints per pair.  opt is reserved (NULL). */
SWB200_API int swb200_align_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                                  const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                                  const swb200_params* p, const swb200_options* opt, int* scores_out, int* spans_out,
                                  unsigned int* ops_out, int ops_stride, int* ops_count);
/* The same for a device-resident batch packed with keep_order = 0; every output pointer is a DEVICE pointer. */
SWB200_API int swb200_batch_align(swb200_batch* batch, const swb200_params* p, const swb200_options* opt, void* stream,
                                  int* d_scores, int* d_spans, unsigned int* d_ops, int ops_stride, int* d_ops_count);

/* Batch alignment without the 1024 cap: for every pair k the score, span and operations that swb200_align returns for
 * that pair alone, with swb200_align_batch's tie rules, output format, ops_stride overflow rule (ops_count = -n; the host
 * call zero-fills that slot), "1I1I" split when gap_ext > gap_init (the one documented difference from swb200_align) and
 * device re-score (SWB200_ERR_CUDA "internal: ..." on a mismatch).  One warp per pair, the shorter sequence cut into bands
 * of 256 rows (DESIGN.md section 4e); short pairs are accepted too.  Limits and errors are swb200_score_long_batch's, so
 * every score can be checked against it: bytes A,C,G,T (SWB200_ERR_ALPHABET); match*min(len) <= 32766 - match
 * (SWB200_ERR_RANGE).  SWB200_ERR_NOMEM when the boundary rows, or direction storage for the largest span the batch can
 * have (4 bits per cell of max(len) x max(min(len)), in 256-row bands), cannot be allocated: swb200_align, whose blocked
 * traceback needs no such storage, is the route for those pairs.  All argument checks run before a device is touched.
 * The host call packs in chunks and shards over swb200_set_devices like swb200_align_batch (results identical for every
 * G).  swb200_last_run: config 320, lanes 32, rows 8, bands = the band count of the tallest pair, cells summed over the
 * three passes.  opt is reserved (NULL). */
SWB200_API int swb200_align_long_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                                       const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                                       const swb200_params* p, const swb200_options* opt, int* scores_out, int* spans_out,
                                       unsigned int* ops_out, int ops_stride, int* ops_count);
/* The same for a device-resident batch packed with keep_order = 0 (SWB200_ERR_ARG for keep_order = 1); every output
 * pointer is a DEVICE pointer. */
SWB200_API int swb200_batch_align_long(swb200_batch* batch, const swb200_params* p, const swb200_options* opt, void* stream,
                                       int* d_scores, int* d_spans, unsigned int* d_ops, int ops_stride, int* d_ops_count);

/* ---- banded batches (long reads): cell (i,j), i = row in seq2, j = column in seq1, is scored iff
 * band_lo <= j - i <= band_hi; everything outside the band is H=E=F=0 and excluded from the max.  The reference
 * has no banded mode; semantics = main.cpp:57-63 restricted to the band (oracle: oracle_gotoh_banded).
 * The band holds W = band_hi - band_lo + 1 diagonals, W = 64, 128, 256 or 512; any other width is SWB200_ERR_ARG.  The
 * 16-bit range rule match*min(len) <= 32766 - match (SWB200_ERR_RANGE) does not depend on W.  swb200_last_run reports
 * bands = W and config 204 / 208 / 216 / 202 (W = 64: the layout options.config picks) or 2128 / 2256 / 2512 (W = 128 /
 * 256 / 512: W / 16 threads per pair, options.config ignored). */
/* One banded pair (the batch call with npairs = 1). */
SWB200_API int swb200_score_banded(const unsigned char* seq1, int n, const unsigned char* seq2, int m, int band_lo,
                                   int band_hi, const swb200_params* p, int* score_out);
SWB200_API int swb200_score_banded_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                                         const unsigned char* seq2_all, const long long* off2, const int* len2,
                                         long long npairs, int band_lo, int band_hi, const swb200_params* p,
                                         const swb200_options* opt, int* scores_out);
SWB200_API int swb200_batch_score_banded(swb200_batch* batch, int band_lo, int band_hi, const swb200_params* p,
                                         const swb200_options* opt, void* stream, int* d_scores);

/* Banded batch alignment: score, span and CIGAR of the best local alignment all of whose cells lie in the band B
 * (band_lo <= j - i <= band_hi; every aligned pair and every gap position counts as a cell).  For every pair k:
 *   score      exactly swb200_score_banded_batch's (oracle_gotoh_banded);
 *   end cell   among in-band cells holding the score, the smallest j, then the smallest i;
 *   start cell the anchored recurrence over the reversed prefixes seq1[..j_end], seq2[..i_end], cells outside the
 *              mirrored band (j_end - i_end) - band_hi .. (j_end - i_end) - band_lo unreachable; ties to the largest
 *              j_start, then the largest i_start;
 *   operations the anchored recurrence over the span rectangle inside B, 4 direction bits per cell (diagonal before E
 *              before F; a gap extends only where extending is strictly better than opening), walked back from the end
 *              cell.  Every cell of the walk lies in B.
 * Output format, '='/'X' split, ops_stride overflow (ops_count = -n; the host call zero-fills that slot), the "1I1I"
 * split when gap_ext > gap_init, the device re-score and its SWB200_ERR_CUDA ("internal: ...") are swb200_align_batch's.
 * When B covers the whole pair (band_lo <= -(len2-1), band_hi >= len1-1) the result is swb200_align_batch's.
 * Limits and errors are swb200_score_banded_batch's: bytes A,C,G,T (SWB200_ERR_ALPHABET); W = band_hi - band_lo + 1
 * in {64, 128, 256, 512} (SWB200_ERR_ARG); match*min(len) <= 32766 - match (SWB200_ERR_RANGE), so every accepted pair can be checked against
 * the score-only call.  All argument checks run before a device is touched.  One warp per pair on the device; the host
 * call packs in chunks and shards over swb200_set_devices like swb200_align_batch.  opt is reserved (NULL).
 * swb200_last_run: lanes 32, bands = W, config 310 / 311 / 312 / 313 for W = 64 / 128 / 256 / 512. */
SWB200_API int swb200_align_banded_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                                         const unsigned char* seq2_all, const long long* off2, const int* len2,
                                         long long npairs, int band_lo, int band_hi, const swb200_params* p,
                                         const swb200_options* opt, int* scores_out, int* spans_out,
                                         unsigned int* ops_out, int ops_stride, int* ops_count);
/* The same for a device-resident batch packed with keep_order = 1 (SWB200_ERR_ARG for keep_order = 0); every output
 * pointer is a DEVICE pointer. */
SWB200_API int swb200_batch_align_banded(swb200_batch* batch, int band_lo, int band_hi, const swb200_params* p,
                                         const swb200_options* opt, void* stream, int* d_scores, int* d_spans,
                                         unsigned int* d_ops, int ops_stride, int* d_ops_count);

/* ---- seeded synthetic inputs, generated in HBM (SURVEY.md 8d) -----------------------------------------
 * The portable counter-based generator of concurrentproject_b200/rng.py and oracle/gotoh_oracle.c on the device,
 * bit-identical to both: symbol k of stream s = 2 bits of mix64(seed, s, k / 32) -> "ACGT".  Replaces the reference
 * harness's unseeded rand() % 4 (TestFileWithGPU.cpp:25-36).  All pointers are DEVICE pointers on `device`.
 *   gen_random      length symbols of one stream (rng.random_acgt)
 *   gen_read_pairs  BASELINE config 4, pairs first_pair .. first_pair+npairs-1 (global ids, so shards of one batch are
 *                   generated independently): window = window_len random bases; even pairs: the read is a substring
 *                   of the window with 5 % substitutions and 1 % indels, odd pairs: read_len random bases
 *                   (rng.read_pair).  d_reads: npairs*read_len bytes, d_windows: npairs*window_len bytes.
 *   gen_long_pairs  BASELINE config 5: seq1 = len random bases, seq2 = the same stretch with 10 % substitutions and
 *                   2 % short indels, cut to len (rng.long_pair).  d_seq1, d_seq2: npairs*len bytes each. */
SWB200_API int swb200_gen_random_device(int device, unsigned long long seed, unsigned long long stream_id, long long length,
                                        unsigned char* d_out, void* stream);
SWB200_API int swb200_gen_read_pairs_device(int device, unsigned long long seed, long long first_pair, long long npairs,
                                            int read_len, int window_len, unsigned char* d_reads, unsigned char* d_windows,
                                            void* stream);
SWB200_API int swb200_gen_long_pairs_device(int device, unsigned long long seed, long long first_pair, long long npairs,
                                            int len, unsigned char* d_seq1, unsigned char* d_seq2, void* stream);

/* ---- one very long pair over a ring of GPUs ------------------------------------------------------
 * All warps of all GPUs form one ring of DP bands (DESIGN.md): the last warp of GPU g pushes its
 * boundary stream straight into GPU g+1's memory (peer stores over NVLink), so neighbouring GPUs
 * are pipelined at single-entry granularity.  One swb200_ring per GPU; with one process per GPU the
 * 64-byte handles travel over any side channel (torch.distributed all_gather in ring.py).
 *   create   allocates this rank's inbound boundary buffer for streamed sequences up to
 *            max_stream_len (the shorter of the two sequences) and returns its CUDA IPC handle
 *   connect  maps the NEXT rank's buffer ((rank+1) % world); connect_local does the same for rings
 *            that live in this process (single-process multi-GPU, tests)
 *   score    collective: every rank passes the same two device-resident sequences and the same
 *            parameters/options (options.lanes must be 16 or 32); returns THIS rank's partial
 *            best score and the raw status bits (1 = left the s16 range, 2 = hand-off timed out).
 *            The pair's score is the max over ranks; if any rank reports bit 1, repeat with lanes=32.
 * A ring serves 16383 calls. */
typedef struct swb200_ring swb200_ring;
SWB200_API int swb200_ring_create(swb200_ctx* ctx, int rank, int world, long long max_stream_len,
                                  swb200_ring** ring_out, unsigned char handle_out[64]);
SWB200_API int swb200_ring_connect(swb200_ring* ring, const unsigned char next_handle[64]);
SWB200_API int swb200_ring_connect_local(swb200_ring* ring, swb200_ring* next);
/* Optional: map rank 0's region as well (its IPC handle, or its ring when it lives in this process).  With a root a
 * long pair is swept from BOTH ends (two half problems, each a ring over all GPUs; half as many bands in a row, so
 * half the pipeline fill); the ranks that own the two last bands store the two middle boundary rows into the root's
 * memory.  After swb200_ring_score_device has returned on EVERY rank (the caller's barrier), rank 0 calls
 * swb200_ring_combine and folds its result into the max over the ranks' partial scores.  Without a root the ring
 * sweeps one-sided as before. */
SWB200_API int swb200_ring_connect_root(swb200_ring* ring, const unsigned char root_handle[64]);
SWB200_API int swb200_ring_connect_root_local(swb200_ring* ring, swb200_ring* root);
SWB200_API int swb200_ring_combine_pending(swb200_ring* ring);    /* 1 if the last score call was two-sided */
SWB200_API int swb200_ring_combine(swb200_ring* ring, void* stream, int* crossing_score_out);
SWB200_API int swb200_ring_score_device(swb200_ring* ring, const unsigned char* d_seq1, long long n,
                                        const unsigned char* d_seq2, long long m, const swb200_params* p,
                                        const swb200_options* opt, void* stream, int* partial_score_out,
                                        int* status_out);
SWB200_API void swb200_ring_destroy(swb200_ring* ring);

#ifdef __cplusplus
}
#endif
#endif /* SWB200_H */
