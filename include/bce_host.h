/*
 * bce_host.h -- C interface of the host half of the compressor (libbce_host.so):
 * the adaptive range coders and the archive writer that consume the counts emitted by
 * the GPU front end (include/bce_gpu.h).  Behaviour follows BCE::encode, bce.cpp:1117-1167,
 * and AdaptiveCoder<31> / ScanCoder<31>, bce.cpp:484-834; archives are bit-exact drop-ins.
 * Used by the `bce` tool and, through ctypes, by the tests.
 */
#ifndef BCE_HOST_H
#define BCE_HOST_H

#include <stddef.h>
#include <stdint.h>

#include "bce_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bce_archive_writer bce_archive_writer;

/* cfg288: 9 x 32 context-bit table or NULL for the default (bce.cpp:713-724).
 * C[i] as returned by bce_gpu_cse_begin / compress_front; it is coded first on stream i
 * (coder_[i].set(C[i], n + 1), bce.cpp:1129). */
bce_archive_writer *bce_archive_begin(uint32_t n, const uint32_t C[8], const uint8_t *cfg288);
/* feed one batch (all 8 streams); threads > 1 codes the streams concurrently (one thread per
 * stream at most, like the reference's omp parallel for over the 8 levels, bce.cpp:1250). */
int bce_archive_feed(bce_archive_writer *w, const bce_cse_batch *batch, int threads);
/* same for BCE_EMIT_CODER word batches (the config must be the one given to bce_gpu_set_emit_mode) */
int bce_archive_feed_words(bce_archive_writer *w, const bce_cse_words *batch, int threads);
/* Overlapped form: begin hands the batch to one persistent coder thread per stream and returns at once (the
 * reference forks its eight coders inside the level loop, bce.cpp:1250-1252, :1302); wait blocks until the
 * batch is coded.  The batch's memory must stay valid until then; one batch in flight at a time. */
int bce_archive_begin_words(bce_archive_writer *w, const bce_cse_words *batch);
int bce_archive_begin_words20(bce_archive_writer *w, const bce_cse_words20 *batch);   /* bce_gpu_cse_next_words20 batches */
int bce_archive_wait(bce_archive_writer *w);
/* flush, header (n, offset, sizes), concatenate; *words is malloc'd (bce_host_free). */
int bce_archive_finish(bce_archive_writer *w, uint32_t offset, uint16_t **words, size_t *nwords);
void bce_archive_abort(bce_archive_writer *w);

/* `bce -s`: collect the same counts per context and derive the 288-byte config.
 * Prints the reference's nine "Result size" lines. */
typedef struct bce_scan bce_scan;
bce_scan *bce_scan_begin(void);
int bce_scan_feed(bce_scan *s, const bce_cse_batch *batch);
int bce_scan_feed_words(bce_scan *s, const bce_cse_words *batch);   /* BCE_EMIT_SCAN batches */
int bce_scan_feed_buckets(bce_scan *s, const bce_scan_buckets *batch);   /* bce_gpu_cse_next_buckets batches */
int bce_scan_finish(bce_scan *s, uint8_t cfg288_out[288]);

/* whole pipelines over a memory buffer, GPU front end + host coders */
int bce_compress_buffer(bce_gpu_ctx *ctx, const uint8_t *T, uint32_t n, const uint8_t *cfg288,
                        int threads, uint16_t **words, size_t *nwords);
int bce_scan_buffer(bce_gpu_ctx *ctx, const uint8_t *T, uint32_t n, uint8_t cfg288_out[288]);
/* k inputs of 1 .. BCE_GPU_MANY_MAX_N bytes (T, starts as bce_gpu_compress_many) -> k archives, the same bytes
 * bce_compress_buffer makes of each: words[i] is malloc'd (bce_host_free), nwords[i] its length.  Calls of at least
 * BCE_HOST_MANY_DEVICE_CODERS inputs run through bce_gpu_compress_many_archives (range coders on the device; `threads`
 * unused); smaller ones through bce_gpu_compress_many, with up to `threads` inputs coded at once, one host thread per
 * input.  Either way inputs are resubmitted until all are done.  On an error no archive is left allocated. */
#define BCE_HOST_MANY_DEVICE_CODERS 256u
int bce_compress_many(bce_gpu_ctx *ctx, const uint8_t *T, const uint64_t *starts, uint32_t k, const uint8_t *cfg288,
                      int threads, uint16_t *words[], size_t nwords[]);

/* k archives (uint16 words; archive i = words[starts[i] .. starts[i+1])) -> k texts on the caller's context.
 * Archives of n <= BCE_GPU_MANY_MAX_N go in groups of up to 64 MiB of text.  A group of at least
 * BCE_HOST_MANY_DEVICE_DECODERS archives is decoded and inverted on the device (bce_gpu_decompress_many); a smaller
 * one is decoded one archive per thread (up to `threads` at once, levels serial), then every inverse in one
 * bce_gpu_unbwt_many call.  Larger archives: the 8-level-thread decoder and bce_gpu_unbwt on ctx.  Whichever path
 * runs, text i is what `bce -ds` makes of archive i (both inverses keep unbwt_serial's contract, bce_gpu.h), damaged
 * archives the decoder accepts included; the environment variable BCE_HOST_MANY_DEVICE_DECODERS overrides the
 * threshold (measurements).
 * status[i] = 0 or archive i's own error (BCE_GPU_E_ARG for a damaged archive); out[i] / nout[i] malloc'd
 * (bce_host_free) where status[i] == 0.  A non-zero return (arguments, CUDA, memory) leaves nothing allocated. */
/* n, the text size an archive's header claims (what bce_gpu_decompress_many needs): 0, or BCE_GPU_E_ARG for a header
 * that cannot be read. */
int bce_archive_size(const uint16_t *words, size_t nwords, uint32_t *n);
#define BCE_HOST_MANY_DEVICE_DECODERS 64u
int bce_decompress_many(bce_gpu_ctx *ctx, const uint16_t *words, const uint64_t *starts, uint32_t k, int threads,
                        uint8_t *out[], size_t nout[], int status[]);

/* host-side packer with the device's word formats (mode = BCE_EMIT_CODER / BCE_EMIT_SCAN);
 * words must hold 3 * count entries; returns the number of words written */
size_t bce_host_pack_counts(int mode, const uint8_t *cfg288, int stream, const bce_tuple *t, size_t count,
                            uint32_t *words);

/* `bce -d` (low_memory = 0: inverse BWT on the GPU through bce_gpu_unbwt) and `bce -ds`
 * (low_memory = 1: serial unbwt::bitwise on the host, no GPU needed) over an archive in memory.
 * *out is malloc'd (bce_host_free). */
int bce_decode_buffer(const uint16_t *words, size_t nwords, int low_memory, uint8_t **out, size_t *nout);

const uint8_t *bce_host_default_config(void);   /* 288 bytes */
void bce_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif
