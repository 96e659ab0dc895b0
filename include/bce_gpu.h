/*
 * bce_gpu.h -- C ABI of the B200 compression front end for BCE v0.4.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  The reference (akamiru/bce) has no
 * runtime plugin interface; its seams are the libdivsufsort C API and the
 * policy_coder / policy_unbwt template parameters of BCE<> (bce.cpp:1111).  Each
 * entry point below names the reference interface it replaces.  INTEGRATION.md shows
 * the few lines a maintainer adds to bce.cpp to bind them.
 *
 * Conventions: plain pointers and sizes, no C++ / torch types; the caller owns every
 * buffer it passes; functions return 0 or a negative BCE_GPU_E_* code (never throw,
 * never exit); one context per GPU; a context is not thread-safe; all host pointers
 * may be pageable or pinned memory.  Domain: 1 <= n < 2^31 (bce.cpp:374, saidx_t).
 *
 * There is no CPU fallback behind this header: every function runs CUDA kernels for
 * sm_100a and fails with BCE_GPU_E_NODEVICE / BCE_GPU_E_CUDA when it cannot.
 */
#ifndef BCE_GPU_H
#define BCE_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BCE_GPU_ABI_VERSION 1

enum {
  BCE_GPU_OK = 0,
  BCE_GPU_E_ARG = -1,        /* bad argument (NULL, n == 0, n >= 2^31, ...) */
  BCE_GPU_E_NOMEM = -2,      /* host or device allocation failed */
  BCE_GPU_E_CUDA = -3,       /* a CUDA call or kernel failed; see bce_gpu_last_error */
  BCE_GPU_E_STATE = -4,      /* call sequence violated (e.g. cse_next before cse_begin) */
  BCE_GPU_E_FRONTIER = -5,   /* CSE node frontier outgrew the device memory set aside for it */
  BCE_GPU_E_INTERNAL = -6,   /* internal consistency check failed (watchdog, invariant) */
  BCE_GPU_E_NODEVICE = -7    /* no usable CUDA device */
};

typedef struct bce_gpu_ctx bce_gpu_ctx;

/* One emitted count = the five arguments of policy_coder::set(s, k, c1, c2, cs) at the
 * reference's only call site, bce.cpp:1302:  (_0x0 - min, max - min + 1, _0x, _x1, _x). */
typedef struct bce_tuple {
  uint32_t sym, k, c1, c2, cs;
} bce_tuple;

/* A batch of emitted counts.  tuples[i] points into pinned host memory owned by the
 * context.  Two buffers alternate: a batch stays valid until the call AFTER the next
 * bce_gpu_cse_next* returns (or the next cse_begin / close), so a consumer can work on batch j
 * while the next call fetches batch j+1 (host coders overlapped with the GPU, SURVEY.md 8f-1).
 * Stream i = wavelet level i = coder_[i] (bce.cpp:1124).  Concatenating the batches of
 * one stream gives exactly the sequence of set() calls the reference makes on coder_[i]:
 * ascending round of the do..while (bce.cpp:1246), ascending position inside a round. */
typedef struct bce_cse_batch {
  const bce_tuple *tuples[8];
  size_t count[8];
  int done;                  /* 1 = the level loop terminated (bce.cpp:1371), no more batches */
} bce_cse_batch;

/* Counters and device timings of the last front-end call (bench / roofline input). */
typedef struct bce_gpu_stats {
  uint32_t n;
  uint32_t sort_rounds;          /* prefix-doubling rounds, round 0 = initial 8-byte sort */
  uint64_t sort_m[48];           /* elements sorted in round r */
  uint32_t sort_passes[48];      /* radix passes run in round r */
  uint64_t radix_launches;       /* onesweep pass launches in total */
  uint64_t radix_elems;          /* sum over those launches of elements moved */
  uint64_t cse_visits;           /* node visits (8(n-1) for primitive input) */
  uint64_t cse_tuples;           /* emitted counts, all streams */
  uint64_t cse_rounds;           /* rounds of the level loop */
  uint64_t cse_launches;         /* launches of the level-loop kernel */
  uint64_t cse_peak_frontier;    /* max nodes in one round, all levels */
  uint64_t gpu_launches;         /* kernels launched by the last call */
  float ms_h2d, ms_d2h;          /* host<->device copies */
  float ms_pack, ms_radix, ms_rerank, ms_rekey, ms_bwt_gather;   /* stage A (BWT) */
  float ms_wavelet, ms_cse;                                       /* stage B */
  float ms_unbwt_bytes, ms_unbwt_chase;                           /* inverse */
  float ms_bwt_total, ms_cse_total, ms_total;
  float ms_cse_narrow;           /* part of ms_cse spent in the narrow-frontier (cluster) kernel */
  uint32_t cse_rounds_narrow;    /* rounds run by it */
  float ms_radix_kernel;         /* sum over launches of radix_onesweep_kernel alone (event pairs) */
  uint64_t cse_words;            /* 32-bit words emitted (5 per count raw, 1-2 packed) */
  uint64_t sort_local_elems;     /* elements of rounds >= 1 ordered by the tile-local sort instead of radix passes
                                    (sort_passes[r] then holds the passes an LSD sort of those keys would take) */
  uint64_t sort_fallback_elems;  /* ... of which went through the radix sort after all (groups crossing tiles) */
  uint32_t sort_radix_passes[48];/* radix passes actually run over the whole working set of round r (0 when the
                                    tile-local sort took the round) */
  uint32_t unbwt_dicts;          /* dictionaries inverted by bce_gpu_unbwt_many (bce_gpu_unbwt: 1) */
  uint32_t unbwt_serial;         /* ... of which took its serial path (unbwt_many: exact powers, damaged dictionaries;
                                    bce_gpu_unbwt: words that are no rank directory, walked on the host) */
  float ms_coder;                /* bce_gpu_compress_many_archives: the range coders' launch */
  float ms_decoder;              /* bce_gpu_decompress_many: the decode loop's launch */
} bce_gpu_stats;

/* ---- lifecycle ---------------------------------------------------------------- */
int bce_gpu_open(int device, bce_gpu_ctx **out);
void bce_gpu_close(bce_gpu_ctx *ctx);
int bce_gpu_abi_version(void);
const char *bce_gpu_error_string(int code);
const char *bce_gpu_last_error(const bce_gpu_ctx *ctx);
int bce_gpu_get_stats(const bce_gpu_ctx *ctx, bce_gpu_stats *out);
/* cap on the scratch arena in bytes (0 = default: a share of free device memory) */
int bce_gpu_set_scratch_limit(bce_gpu_ctx *ctx, size_t bytes);
/* Tuning options of a context (value 0 = back to the default).  Results never depend on them.
 *   EMIT_BATCH_BYTES  target size of one batch of emitted counts handed back by cse_next* (default
 *                     1 GiB; small values force many batches -- used by the tests of the draining path)
 *   LOCAL_SORT_MIN    working sets of the suffix sort below this many rotations take the plain
 *                     radix path instead of the tile-local sort (default 2^20)
 *   RESIDENT_CHECKSUM 1 = front_resident also sums the words it emits (see bce_gpu_resident_checksum)
 *   SLOT_ENTER_NODES  the level loop keeps frontiers of at least this many nodes per round in its slot layout
 *                     (default 2,000,000; inputs below 8x this never use it; small values: tests)
 *   MID_ENTER_NODES   frontiers of at most this many nodes per round (and more than the cluster kernels take) run in
 *                     the one-barrier-per-round kernel (default 400,000, at most ~515,000; 1 = never)
 *   NO_NARROW_KERNELS 1 = the cluster / one-CTA kernels for frontiers of a few thousand nodes are not used (tests:
 *                     the other kernels then see every frontier size) */
enum { BCE_GPU_OPT_EMIT_BATCH_BYTES = 1, BCE_GPU_OPT_LOCAL_SORT_MIN = 2, BCE_GPU_OPT_RESIDENT_CHECKSUM = 3,
       BCE_GPU_OPT_SLOT_ENTER_NODES = 4, BCE_GPU_OPT_MID_ENTER_NODES = 5, BCE_GPU_OPT_NO_NARROW_KERNELS = 6 };
int bce_gpu_set_option(bce_gpu_ctx *ctx, int option, uint64_t value);

/* Page-locked host memory for the caller's input and output buffers (File::File reads the whole file into one
 * buffer, bce.cpp:842-856: read it into this and the upload is one DMA transfer instead of staged copies).
 * Any host pointer is accepted everywhere; this is an optimisation, not a requirement. */
void *bce_gpu_host_alloc(bce_gpu_ctx *ctx, size_t bytes);
void bce_gpu_host_free(bce_gpu_ctx *ctx, void *p);

/* ---- stage A: suffix sort / BWT ------------------------------------------------
 * Replaces File::rotate (bce.cpp:858-894) and File::bwt with its divbwt call into
 * libdivsufsort (bce.cpp:896-910, call :901, splice :902).
 *   L_out[r]   = T[(SA[r] - 1) mod n], rows = cyclic rotations of T in sorted order
 *   offset_out = SA[0] = smallest start index of a least rotation  (File::offset_)
 *   SA_out     = optional (may be NULL), n entries; identical rotations by ascending index
 * The BWT also stays resident on the device for a following bce_gpu_cse_begin(L=NULL). */
int bce_gpu_bwt(bce_gpu_ctx *ctx, const uint8_t *T, uint32_t n,
                uint8_t *L_out, uint32_t *offset_out, uint32_t *SA_out);

/* ---- stage B1: wavelet matrix ---------------------------------------------------
 * Replaces the RankFile constructor body (bce.cpp:944-972) and Rank::build (:138-145).
 * L = BWT bytes on the host, or NULL to use the BWT left on the device by bce_gpu_bwt.
 * ranks_out (optional): 8 host arrays of n/32+1 words in the layout of Rank::rank_
 * (bce.cpp:149: [32 data bits | 32-bit cumulative rank]).  C_out[i] = zeros of level
 * (i+7)%8 as computed by BCE::encode (bce.cpp:1128). */
int bce_gpu_wavelet(bce_gpu_ctx *ctx, const uint8_t *L, uint32_t n,
                    uint64_t *const ranks_out[8], uint32_t C_out[8]);

/* ---- stage B2: CSE level loop ---------------------------------------------------
 * Replaces BCE::code(mode = 1) (bce.cpp:1236-1373) including its pArray queues
 * (:226-356) and the root set-up in BCE::encode (:1124-1130, :1238-1240).
 * cse_begin builds the wavelet matrix (as bce_gpu_wavelet) and the root frontier;
 * cse_next runs rounds on the device and hands back the next batch of emitted counts. */
int bce_gpu_cse_begin(bce_gpu_ctx *ctx, const uint8_t *L, uint32_t n, uint32_t C_out[8]);
int bce_gpu_cse_next(bce_gpu_ctx *ctx, bce_cse_batch *out);

/* ---- packed emission (what `bce -c` / `bce -s` of this repository use) ----------------
 * Instead of the five raw arguments (20 B) the device can emit what the host coder consumes:
 *   BCE_EMIT_CODER  one word  [ctx:10 @10|k:5 @5|sym:5]  with ctx = the context index of
 *                   AdaptiveCoder::get_context (bce.cpp:671-677) for the stream's configured
 *                   context bits cfg288[stream][k]; when the reference would halve k > 31
 *                   (bce.cpp:507-510) nb times: [ctx|0|sym'] -- k field 0, a count's k is at least 2 --
 *                   followed by two words [low[0..10) @10|nb:5 @5|k':5] and [low >> 10] with the nb low
 *                   bits of the symbol (coded uniformly, LSB first).  Every word is below 2^20:
 *                   bce_gpu_cse_next_words20 hands the same words back as 20 bits each (3/8 less over PCIe)
 *   BCE_EMIT_SCAN   one word  [esc|nb:5 @26|q2:8 @18|q1:8 @10|k:5 @5|sym:5], q = (c << 8) / cs,
 *                   halving rule of ScanCoder::set (bce.cpp:737-744)
 * set_emit_mode applies to the following cse_begin / compress_front calls of the context.
 * cfg288: 9 x 32 context-bit table (rows 0..7 are used), NULL = default table. */
enum { BCE_EMIT_RAW = 0, BCE_EMIT_CODER = 1, BCE_EMIT_SCAN = 2 };
typedef struct bce_cse_words {
  const uint32_t *words[8];   /* pinned host memory, valid as bce_cse_batch: until the call after the next */
  size_t count[8];            /* words */
  int done;
} bce_cse_words;
int bce_gpu_set_emit_mode(bce_gpu_ctx *ctx, int mode, const uint8_t *cfg288);
int bce_gpu_cse_next_words(bce_gpu_ctx *ctx, bce_cse_words *out);
/* BCE_EMIT_CODER only: the batch as 20 bits per word, packed on the device before the copy: word j of stream i
 * is bits 20 j .. 20 j + 19 of the little-endian bit string bytes[i] (two words in 5 bytes; with o = 5 (j / 2):
 * even j = b[o] | b[o+1] << 8 | (b[o+2] & 15) << 16, odd j = b[o+2] >> 4 | b[o+3] << 4 | b[o+4] << 12).
 * At least 8 bytes past the last word are readable. */
typedef struct bce_cse_words20 {
  const uint8_t *bytes[8];    /* pinned host memory, valid as bce_cse_batch: until the call after the next */
  size_t count[8];            /* words (20 bits each) */
  int done;
} bce_cse_words20;
int bce_gpu_cse_next_words20(bce_gpu_ctx *ctx, bce_cse_words20 *out);

/* ---- `bce -s`: counts bucketed on the device ------------------------------------------------
 * ScanCoder::set (bce.cpp:737-744) appends every symbol to stat_[k][(q2 << 16) | q1]; its flush
 * (:751-800) needs, per (k, key), the symbols in insertion order, and the keys of one k in the order
 * of their first appearance (it walks an unordered_map).  In BCE_EMIT_SCAN mode this call returns a
 * batch already bucketed -- a stable device sort of the batch's words by (k, q1, q2):
 *   syms[i]     one byte per count, bucket after bucket, insertion order inside a bucket
 *   buckets[i]  one record per (k, key) present in the batch, in no particular order:
 *               key = k | q1 << 5 | q2 << 13, start = index of its first byte in syms[i], first =
 *               position in the batch's stream of the count that opened the bucket
 *   halvings[i] how often the reference would have added log 2 for k > 31 (:738-741)
 * so the host only appends runs of bytes and runs the unchanged flush.  Same validity as bce_cse_words. */
typedef struct bce_scan_bucket {
  uint32_t key, start, first, reserved;
} bce_scan_bucket;
typedef struct bce_scan_buckets {
  const uint8_t *syms[8];
  size_t count[8];
  const bce_scan_bucket *buckets[8];
  size_t nbuckets[8];
  uint64_t halvings[8];
  int done;
} bce_scan_buckets;
int bce_gpu_cse_next_buckets(bce_gpu_ctx *ctx, bce_scan_buckets *out);

/* ---- fused front end -------------------------------------------------------------
 * bce_gpu_bwt + bce_gpu_cse_begin without the BWT leaving the device: what
 * `RankFile file{...}` (bce.cpp:1411) plus the start of BCE::encode do.  Follow with
 * bce_gpu_cse_next until done. */
int bce_gpu_compress_front(bce_gpu_ctx *ctx, const uint8_t *T, uint32_t n,
                           uint32_t *offset_out, uint32_t C_out[8]);

/* ---- many small inputs in one call ------------------------------------------------------
 * The whole front end (bce_gpu_compress_front and every batch of the level loop) for k inputs at once: one CTA per
 * input, a grid of them per launch, for corpora of many small files where per-call costs dominate.  Input i is
 * T[starts[i] .. starts[i+1]) with 1 <= size <= BCE_GPU_MANY_MAX_N (starts: k + 1 offsets, k >= 1); any other size,
 * k = 0 or the BCE_EMIT_SCAN mode is BCE_GPU_E_ARG.  Emission follows the context's mode (BCE_EMIT_RAW: 5 words per
 * count as bce_tuple, BCE_EMIT_CODER).  out[i] (k entries) receives input i's offset and C[8] (as compress_front),
 * and its whole streams: words[s] / count[s] point into pinned host memory that stays valid as a bce_cse_words
 * batch does -- until the call after the next bce_gpu_compress_many.  The words of one call share one arena of
 * BCE_GPU_OPT_EMIT_BATCH_BYTES (never less than one input's worst case); an input that did not fit has done = 0 and
 * nothing else set: submit it again.  Which inputs are done depends on timing, what a done input holds does not.
 * Stats: cse_visits, cse_rounds, cse_words, cse_tuples of the done inputs; ms_h2d, ms_cse_total (the launch),
 * ms_d2h, ms_total; n = the largest input. */
#define BCE_GPU_MANY_MAX_N 65536u
typedef struct bce_many_result {
  uint32_t offset;
  uint32_t C[8];
  int done;
  const uint32_t *words[8];
  size_t count[8];            /* words */
} bce_many_result;
int bce_gpu_compress_many(bce_gpu_ctx *ctx, const uint8_t *T, const uint64_t *starts, uint32_t k,
                          bce_many_result *out);

/* The same k inputs (T, starts and limits as bce_gpu_compress_many) to finished archives: out[i] is the archive of
 * input i, the uint16 words `bce -c` writes for it with the table cfg288 (9 x 32 context bits, NULL = the default
 * table; a cell above 5 is BCE_GPU_E_ARG).  The front end runs as in BCE_EMIT_CODER mode, then one launch runs every
 * input's eight range coders and its header coder (row 8 of cfg288) on the device; only the archives cross PCIe.
 * The context's emission mode and table are neither read nor changed.  words points into pinned host memory that
 * stays valid until the call after the next bce_gpu_compress_many / bce_gpu_compress_many_archives; an input with
 * done = 0 did not fit this call's arenas: submit it again.  Stats as bce_gpu_compress_many, plus ms_coder (the
 * coder launch); ms_d2h is the archives' copy; gpu_launches counts both launches. */
typedef struct bce_many_archive {
  const uint16_t *words;
  size_t nwords;
  int done;
} bce_many_archive;
int bce_gpu_compress_many_archives(bce_gpu_ctx *ctx, const uint8_t *T, const uint64_t *starts, uint32_t k,
                                   const uint8_t *cfg288, bce_many_archive *out);

/* Start uploading the NEXT input while the level loop of the current one still runs (its batches are being
 * fetched with bce_gpu_cse_next*): legal once bce_gpu_compress_front / bce_gpu_bwt of the current input has returned
 * -- the text is not read after the BWT exists.  A following bce_gpu_compress_front / bce_gpu_bwt with the same T
 * and n finds the text on the device; any other input is uploaded as usual.  T must stay unchanged until then;
 * only page-locked memory (bce_gpu_host_alloc) can be copied asynchronously, for pageable T this is a no-op. */
int bce_gpu_prefetch_input(bce_gpu_ctx *ctx, const uint8_t *T, uint32_t n);

/* ---- device-resident variant (measurement) ---------------------------------------
 * stage_input copies T to the device; front_resident then runs stage A + B entirely in
 * HBM (counts are written to device memory, nothing crosses PCIe) and returns the number
 * of emitted counts.  Used for the `value` leg of bench.py. */
int bce_gpu_stage_input(bce_gpu_ctx *ctx, const uint8_t *T, uint32_t n);
int bce_gpu_front_resident(bce_gpu_ctx *ctx, uint32_t *offset_out, uint64_t *tuples_out);
/* Proof that the resident run emitted what the hosted run hands back: per stream i, over the words
 * w_0, w_1, ... in emission order (the words bce_gpu_cse_next* would have returned for the mode set with
 * bce_gpu_set_emit_mode),  sum[i] = SUM w_j  and  wsum[i] = SUM w_j * (2 j + 1),  both mod 2^64.
 * Needs BCE_GPU_OPT_RESIDENT_CHECKSUM = 1 before front_resident (one extra read of the emitted words). */
int bce_gpu_resident_checksum(bce_gpu_ctx *ctx, uint64_t sum[8], uint64_t wsum[8]);

/* ---- inverse --------------------------------------------------------------------
 * Replaces unbwt::bytewise::unbwt (bce.cpp:1043-1103): wavelet -> bytes (:1050-1085),
 * inverse_bw_transform(..., idx = 1) from libdivsufsort (:1091), rotate by offset (:1093).
 * ranks: 8 host arrays of n/32+1 words, layout of bce.cpp:149, as they are after
 * Rank::finalize (:187-194): both the data bits and the cumulative ranks are read.  offset < n (else BCE_GPU_E_ARG).
 * The text is unbwt::bitwise (bce.cpp:999-1038) with the host decoder's clamps (unbwt_serial, `bce -ds`), for any words:
 *   out[(n - 1 - k + offset) mod n] = byte of row s_k,   s_0 = 0,   s_{k+1} = the descent from s_k
 * where every bit and ones_before is read at min(pos, n), the row keeps its 32-bit value and zeros_j = n - ones_j(n).
 * Words that are a true rank directory (base of word 0 is 0, base of word i+1 = base of word i + its data bits, for
 * i < n/32: every archive writer's) are inverted on the device, exact powers included (LF then has several cycles);
 * any other words (damaged archives) by the same walk on the host.  Stats: ms_unbwt_bytes (check, L and LF),
 * ms_unbwt_chase, gpu_launches; unbwt_dicts = 1, unbwt_serial = 1 when the host walk ran. */
int bce_gpu_unbwt(bce_gpu_ctx *ctx, const uint64_t *const ranks[8],
                  uint32_t offset, uint32_t n, uint8_t *out);

/* Inverse BWT of k dictionaries of 1 .. BCE_GPU_MANY_MAX_N rows at once, one CTA each (archives of many small files).
 * ranks: dictionary i's 8 levels of n[i]/32+1 words (layout of bce.cpp:149, after Rank::finalize), level 0 first,
 * dictionaries back to back in order; offset[i] <= n[i]; out: the k texts back to back (sum of n[i] bytes).
 * Text i = unbwt::bitwise (bce.cpp:999-1038) of dictionary i with positions clamped to [0, n] as the host decoder's
 * DecodeRank does -- defined for any words: bce_gpu_unbwt's contract above.  k = 0, n[i] = 0 or n[i] > BCE_GPU_MANY_MAX_N: BCE_GPU_E_ARG.
 * Stats: n = the largest dictionary; ms_h2d, ms_unbwt_chase (the launch), ms_d2h, ms_total; gpu_launches;
 * unbwt_dicts, unbwt_serial. */
int bce_gpu_unbwt_many(bce_gpu_ctx *ctx, const uint64_t *ranks, const uint32_t *n, const uint32_t *offset,
                       uint32_t k, uint8_t *out);

/* The whole decoder of k small archives on the device: archive i = words[starts[i] .. starts[i+1]) (uint16 words,
 * starts: k + 1 offsets that never decrease) whose header claims n[i] bytes, 1 <= n[i] <= BCE_GPU_MANY_MAX_N (the
 * caller reads n from the header).  out receives the texts back to back (sum of n[i] bytes); status[i] = 0, or
 * BCE_GPU_E_ARG where the host decoder (decode_to_ranks) rejects archive i -- a header that does not claim n[i]
 * included -- and text i is then zero.  Text i is what `bce -ds` makes of archive i, damaged archives included.
 * One launch decodes every archive (one CTA of 8 warps each, a warp per level), a second inverts the accepted ones
 * (bce_gpu_unbwt_many's kernel); only archives go up and only texts come down.  k = 0, n[i] = 0, n[i] above the
 * limit or decreasing starts: BCE_GPU_E_ARG.  Stats: n = the largest archive; cse_visits / cse_rounds of the
 * accepted archives; unbwt_dicts (accepted archives) and unbwt_serial; ms_h2d, ms_decoder, ms_unbwt_chase, ms_d2h,
 * ms_total; gpu_launches. */
int bce_gpu_decompress_many(bce_gpu_ctx *ctx, const uint16_t *words, const uint64_t *starts, const uint32_t *n,
                            uint32_t k, uint8_t *out, int *status);

#ifdef __cplusplus
}
#endif
#endif
