/* zipc_b200.h -- C ABI of libzipc_b200.so: the B200-native DEFLATE / zlib / ZIP hot path of zipc.
 *
 * The reference (dbuenzli/zipc) is pure OCaml and has no FFI; its boundary for this path is the
 * module signature src/zipc_deflate.mli plus the documented plug point Zipc.File.make
 * (src/zipc.mli:26-28,100-121).  Each entry point below names the reference function(s) it
 * replaces.  The OCaml binding a maintainer adds on top (ocaml/zipc_cuda_stubs.c) and the ctypes
 * binding used by the tests (zipc_b200/_lib.py) are shown in INTEGRATION.md.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes, int status returns (ZIPC_OK = 0).
 *  - Batch calls return a call-level status (argument / CUDA / memory failures) and a per-member
 *    status[]: one bad member never poisons the batch.
 *  - Per-member messages are the reference's exact English strings: zipc_b200_strerror().
 *  - Host-pointer calls copy inputs to the device and results back inside the call; `_dev`
 *    variants take device pointers (same device as the ctx) and leave results on the device.
 *  - The library never retains caller pointers after a call returns.
 *  - A ctx is bound to one CUDA device and is single-owner (one call in flight); several ctxs
 *    (one per GPU) may be driven from different host threads or processes.
 *  - There is no CPU fallback: without a CUDA device every compute entry returns
 *    ZIPC_ERR_NO_DEVICE / ZIPC_ERR_CUDA.
 */
#ifndef ZIPC_B200_H
#define ZIPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ------------------------------------------------------------------------ */
enum {
  ZIPC_OK = 0,
  ZIPC_ERR_CORRUPTED = 1,      /* "Corrupted data stream"                 zipc_deflate.ml:233   */
  ZIPC_ERR_SIZE_EXCEEDED = 2,  /* "Expected decompression size exceeded"  zipc_deflate.ml:29    */
  ZIPC_ERR_ZLIB_METHOD = 3,    /* "Unknown compression method (%d)"       zipc_deflate.ml:728   */
  ZIPC_ERR_ZLIB_WINDOW = 4,    /* "Window size too large"                 zipc_deflate.ml:729   */
  ZIPC_ERR_ZLIB_DICT = 5,      /* "Preset dictionary unsupported"         zipc_deflate.ml:730   */
  ZIPC_ERR_CHECKSUM = 6,       /* "Checksum mismatch, expected %lx found %lx)"  :103-104        */
  ZIPC_ERR_NOMEM = 7,
  ZIPC_ERR_INVALID_ARG = 8,    /* maps to OCaml Invalid_argument                                */
  ZIPC_ERR_CUDA = 9,           /* no analogue in the reference; see zipc_b200_last_error()      */
  ZIPC_ERR_NO_DEVICE = 10,
  ZIPC_ERR_DST_TOO_SMALL = 11, /* caller's output arena is too small; needed size is reported   */
  ZIPC_ERR_ZIP_ZIP64 = 20,     /* zipc.ml:290 */
  ZIPC_ERR_ZIP_MULTIPART = 21, /* zipc.ml:291 */
  ZIPC_ERR_ZIP_EOCD = 22,      /* zipc.ml:292 */
  ZIPC_ERR_ZIP_NO_EOCD = 23,   /* zipc.ml:293-294 */
  ZIPC_ERR_ZIP_SHORT = 24,     /* zipc.ml:296 */
  ZIPC_ERR_ZIP_TRUNC_CD = 25,  /* zipc.ml:297 */
  ZIPC_ERR_ZIP_CDFH = 26,      /* zipc.ml:298 */
  ZIPC_ERR_ZIP_LFH = 27,       /* zipc.ml:299 */
  ZIPC_ERR_ZIP_COUNT = 28,     /* zipc.ml:231-232 */
  ZIPC_ERR_ZIP_PATH_LEN = 29,  /* zipc.ml:234-235 */
  ZIPC_ERR_ZIP_SIZE = 30,      /* zipc.ml:130-133 */
  ZIPC_ERR_ZIP_ENCRYPTED = 31, /* zipc.ml:129 */
  ZIPC_ERR_ZIP_FORMAT = 32,    /* zipc.ml:128 */
  ZIPC_ERR_ZIP_CD_OFFSET = 33, /* zipc.ml:550 */
  ZIPC_ERR_ZIP_CD_SIZE = 34    /* zipc.ml:551 */
};

/* crc_op (zipc_deflate.ml:210) selecting the checksum fused with a codec call */
enum { ZIPC_CK_NONE = 0, ZIPC_CK_ADLER32 = 1, ZIPC_CK_CRC32 = 2 };
/* type level (zipc_deflate.mli:123-126) */
enum { ZIPC_LEVEL_NONE = 0, ZIPC_LEVEL_FAST = 1, ZIPC_LEVEL_DEFAULT = 2, ZIPC_LEVEL_BEST = 3 };
/* Adler-32 flavour.  REF_COMPAT reproduces the reference's signed Int32.rem
 * (zipc_deflate.ml:95,196) bit for bit; RFC1950 is the standard checksum.  They agree whenever
 * every 5552-byte chunk has mean byte < 115 (ordinary text). */
enum { ZIPC_ADLER_REF_COMPAT = 0, ZIPC_ADLER_RFC1950 = 1 };

#define ZIPC_SIZE_UNKNOWN ((size_t)-1) /* ?decompressed_size omitted */

typedef struct zipc_b200_ctx zipc_b200_ctx;

/* ---- library / context --------------------------------------------------------------------- */
const char *zipc_b200_version(void);
/* Exact reference message for a status (printf patterns left in place). */
const char *zipc_b200_strerror(int status);
/* Number of CUDA devices visible (0 if none / no driver). */
int zipc_b200_device_count(void);
/* Create / destroy a context bound to CUDA device `device`. */
int zipc_b200_ctx_create(int device, zipc_b200_ctx **ctx);
void zipc_b200_ctx_destroy(zipc_b200_ctx *ctx);
/* Text of the last CUDA / internal failure on this ctx ("" if none). */
const char *zipc_b200_last_error(const zipc_b200_ctx *ctx);
/* The CUDA stream (cudaStream_t) all of this ctx's work is launched on; for event timing. */
void *zipc_b200_ctx_stream(zipc_b200_ctx *ctx);
/* Number of kernels this ctx has launched so far (bench.py's gpu_launches). */
uint64_t zipc_b200_ctx_launches(const zipc_b200_ctx *ctx);
/* Diagnostics counters: 0 = kernels launched, 1 = large streams inflated in parallel inside the stream, 2 = large streams
 * whose parallel decoding did not check out and that were decoded by the serial path instead. */
uint64_t zipc_b200_ctx_counter(const zipc_b200_ctx *ctx, int which);
/* Diagnostics: when enabled, every call brackets its dominant kernel (CRC tiles / Adler chunks / inflate /
 * deflate) with CUDA events on the ctx stream; zipc_b200_ctx_kernel_ms returns the duration of the last
 * bracketed kernel in milliseconds (it waits for that kernel), or a negative value if none. */
void zipc_b200_ctx_profile(zipc_b200_ctx *ctx, int enable);
float zipc_b200_ctx_kernel_ms(zipc_b200_ctx *ctx);
/* Pinned host memory helpers: buffers from here are DMA'd directly, others are staged. */
int zipc_b200_host_alloc(size_t bytes, void **ptr);
void zipc_b200_host_free(void *ptr);
/* Device memory helpers for the _dev entry points (plain cudaMalloc / cudaFree / memcpy). */
int zipc_b200_dev_alloc(zipc_b200_ctx *ctx, size_t bytes, void **dptr);
void zipc_b200_dev_free(zipc_b200_ctx *ctx, void *dptr);
int zipc_b200_memcpy_h2d(zipc_b200_ctx *ctx, void *dptr, const void *src, size_t bytes);
int zipc_b200_memcpy_d2h(zipc_b200_ctx *ctx, void *dst, const void *dptr, size_t bytes);
int zipc_b200_sync(zipc_b200_ctx *ctx);

/* ---- checksums ----------------------------------------------------------------------------- */
/* Zipc_deflate.Crc_32.string  (src/zipc_deflate.mli:44, zipc_deflate.ml:161-163) */
int zipc_b200_crc32(zipc_b200_ctx *ctx, const void *src, size_t len, uint32_t *crc);
int zipc_b200_crc32_dev(zipc_b200_ctx *ctx, const void *d_src, size_t len, uint32_t *crc);
/* Asynchronous form: result is written to *d_crc (device memory) on the ctx stream. */
int zipc_b200_crc32_dev_async(zipc_b200_ctx *ctx, const void *d_src, size_t len, uint32_t *d_crc);
/* Zipc_deflate.Adler_32.string  (src/zipc_deflate.mli:71, zipc_deflate.ml:203-205) */
int zipc_b200_adler32(zipc_b200_ctx *ctx, const void *src, size_t len, int mode, uint32_t *adler);
int zipc_b200_adler32_dev(zipc_b200_ctx *ctx, const void *d_src, size_t len, int mode, uint32_t *adler);
/* CRC-32 of n independent ranges (Crc_32.string per member; File.stored_of_binary_string,
 * zipc.ml:171-177).  Host pointers. */
int zipc_b200_crc32_batch(zipc_b200_ctx *ctx, size_t n, const void *const *src, const size_t *len,
                          uint32_t *crc);
/* Host-side combine of checksums of adjacent ranges (multi-GPU / multi-call gather; pure
 * integer GF(2) arithmetic, no device needed):  crc(A||B) from crc(A), crc(B), |B|. */
uint32_t zipc_b200_crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b);
uint32_t zipc_b200_adler32_combine(uint32_t adler_a, uint32_t adler_b, uint64_t len_b); /* RFC1950 */

/* ---- inflate ------------------------------------------------------------------------------- */
/* Zipc_deflate.inflate / inflate_and_crc_32 / inflate_and_adler_32 for n independent streams
 * (src/zipc_deflate.mli:79-102, zipc_deflate.ml:692-718).
 *   checksum_kind   ZIPC_CK_*: checksum of each output, as the reference's crc_op
 *   src[i],src_len[i]  compressed stream i (host memory)
 *   max_out[i]      ?decompressed_size of stream i, or ZIPC_SIZE_UNKNOWN
 *   dst,dst_cap     caller's output arena (host).  Stream i's output is written at dst_off[i]
 *                   (assigned by the library, 16-byte aligned, NOT necessarily in input order: a large batch into a
 *                   pinned arena is laid out in download order, smallest outputs first, so that finished ranges are
 *                   copied out while the kernel still works on the larger streams) with length dst_len[i].
 *                   If dst is NULL or too small the call returns ZIPC_ERR_DST_TOO_SMALL and
 *                   *dst_need holds the arena size to provide; outputs then stay available in
 *                   the ctx until the next call and can be fetched with zipc_b200_fetch().
 *   checksum[i]     checksum of output i (0 for ZIPC_CK_NONE)
 *   status[i]       ZIPC_OK / ZIPC_ERR_CORRUPTED / ZIPC_ERR_SIZE_EXCEEDED
 * A stream is decoded by one warp; LARGE streams (64 KiB of compressed data or more, no index needed; which of a batch's streams is
 * decided by a cost model over the batch, see zipc_b200_inflate_plan; several at a time; with either checksum) are decoded by many:
 * block starts are found by scanning for valid dynamic-block headers, the chunks between them are decoded speculatively
 * with the preceding 32 KiB unknown, and resolved once the chunks are seen to chain up exactly; any doubt (and any error
 * inside the stream) sends the stream back to the one-warp decoder, so results and statuses are those of the serial
 * reference loop (zipc_deflate.ml:593-616, 692-709) either way.
 */
int zipc_b200_inflate_batch(zipc_b200_ctx *ctx, int checksum_kind, int adler_mode, size_t n,
                            const void *const *src, const size_t *src_len, const size_t *max_out,
                            void *dst, size_t dst_cap, size_t *dst_need,
                            size_t *dst_off, size_t *dst_len, uint32_t *checksum, int *status);
/* Which streams of an inflate batch are decoded by many warps each, a few at a time (many_warp[i] = 1), and which by one warp
 * each, all side by side (0): the host-side decision of zipc_b200_inflate_batch (a cost model over the compressed sizes; see
 * DESIGN.md 4.6), exposed for tests and capacity planning.  lanes = streams decoded at a time (0: 12).  Host only, no device
 * needed.  Either way the results are the reference's (zipc_deflate.ml:593-616, 692-709); only the time differs. */
void zipc_b200_inflate_plan(size_t n, const size_t *src_len, size_t lanes, char *many_warp);
/* Copy the outputs of the last batch call out of the ctx (after ZIPC_ERR_DST_TOO_SMALL). */
int zipc_b200_fetch(zipc_b200_ctx *ctx, void *dst, size_t dst_cap);
/* Device-resident form: streams live in one device buffer d_src at src_off[i]; outputs are
 * written to d_dst at dst_off[i] (given by the caller, capacity max_out[i] each, which must be
 * known: ZIPC_SIZE_UNKNOWN is ZIPC_ERR_INVALID_ARG).  Per-stream results are copied back to the host arrays.
 * src_off and dst_off need no alignment.  Stream i is read from [src_off[i], src_off[i] + src_len[i]) only: the bytes
 * after it, whatever they are, never change its result.  Output i is written inside [dst_off[i], dst_off[i] + dst_len[i])
 * on success and inside [dst_off[i], dst_off[i] + max_out[i]) otherwise, never outside, so slots may sit back to back.
 * The device bytes may change between calls (each call reads them afresh). */
int zipc_b200_inflate_batch_dev(zipc_b200_ctx *ctx, int checksum_kind, int adler_mode, size_t n,
                                const void *d_src, const size_t *src_off, const size_t *src_len,
                                void *d_dst, const size_t *dst_off, const size_t *max_out,
                                size_t *dst_len, uint32_t *checksum, int *status);
/* Zipc_deflate.zlib_decompress for n streams (src/zipc_deflate.mli:104-118,
 * zipc_deflate.ml:720-740).  status[i] may also be ZIPC_ERR_ZLIB_* / ZIPC_ERR_CHECKSUM;
 * expect[i]/found[i] carry the two Adler-32 values (the reference's option pair). */
int zipc_b200_zlib_decompress_batch(zipc_b200_ctx *ctx, int adler_mode, size_t n,
                                    const void *const *src, const size_t *src_len,
                                    const size_t *max_out, void *dst, size_t dst_cap,
                                    size_t *dst_need, size_t *dst_off, size_t *dst_len,
                                    uint32_t *expect, uint32_t *found, int *status);
/* Device-resident Zipc_deflate.zlib_decompress (src/zipc_deflate.mli:104-118, zipc_deflate.ml:720-740): arguments and output
 * contract of zipc_b200_inflate_batch_dev (any src_off / dst_off; stream i is read from [src_off[i], src_off[i] + src_len[i])
 * only, so its 4-byte trailer is the last 4 bytes of that range; output inside [dst_off[i], dst_off[i] + max_out[i]);
 * ZIPC_SIZE_UNKNOWN is ZIPC_ERR_INVALID_ARG), results of zipc_b200_zlib_decompress_batch for the same bytes (status, dst_len,
 * expect / found, found = the method on ZIPC_ERR_ZLIB_METHOD; the body is [2, src_len - 2) as in the reference,
 * zipc_deflate.ml:732).  The headers are checked on the device, in the reference's order; a stream whose header is
 * rejected is not decoded and its slot is not written.  adler_mode is ZIPC_ADLER_*. */
int zipc_b200_zlib_decompress_batch_dev(zipc_b200_ctx *ctx, int adler_mode, size_t n,
                                        const void *d_src, const size_t *src_off, const size_t *src_len,
                                        void *d_dst, const size_t *dst_off, const size_t *max_out,
                                        size_t *dst_len, uint32_t *expect, uint32_t *found, int *status);

/* ---- deflate ------------------------------------------------------------------------------- */
/* Zipc_deflate.deflate / crc_32_and_deflate / adler_32_and_deflate for n independent inputs
 * (src/zipc_deflate.mli:128-149, zipc_deflate.ml:1247-1259), i.e. the codec under
 * Zipc.File.deflate_of_binary_string (zipc.ml:179-185).  Output streams are valid RFC 1951 and
 * inflate to the input bit-exactly with the reference's inflate; they are not byte-identical to
 * the reference's streams (DESIGN.md: ratio tolerance per level).
 * One member is compressed by one CTA; a member of 2 MiB or more (ZIPC_B200_SPLIT_MIN) by one CTA per segment of 64 - 256 KiB,
 * each primed with the 32 KiB before it: still one ordinary stream, 5 bytes per segment larger.  Adler-32 (this call with
 * ZIPC_CK_ADLER32, zipc_b200_zlib_compress_batch) is then folded over the blocks of all segments in stream order, which is what the
 * reference's zlib_decompress recomputes from the stream.
 * Arena conventions as for zipc_b200_inflate_batch. */
int zipc_b200_deflate_batch(zipc_b200_ctx *ctx, int level, int checksum_kind, int adler_mode,
                            size_t n, const void *const *src, const size_t *src_len,
                            void *dst, size_t dst_cap, size_t *dst_need,
                            size_t *dst_off, size_t *dst_len, uint32_t *checksum, int *status);
/* Device-resident form: input i is [src_off[i], src_off[i] + src_len[i]) of d_src (any alignment; the bytes around it are
 * never read into the result), output i goes to the caller's slot at dst_off[i] of d_dst, which must be 4-byte aligned
 * (ZIPC_ERR_INVALID_ARG otherwise, before anything runs), with capacity dst_cap_each[i] (zipc_b200_deflate_bound(src_len[i])
 * always suffices).  A member is compressed by one CTA whatever its size (no primed segments).  On success exactly
 * [dst_off[i], dst_off[i] + dst_len[i]) is written; bytes of the slot after dst_len[i] keep their contents.  A slot that is
 * too small gives status[i] = ZIPC_ERR_DST_TOO_SMALL and dst_len[i] = 0, and only bytes inside
 * [dst_off[i], dst_off[i] + dst_cap_each[i]) may have been written; the other members are not affected. */
int zipc_b200_deflate_batch_dev(zipc_b200_ctx *ctx, int level, int checksum_kind, int adler_mode,
                                size_t n, const void *d_src, const size_t *src_off,
                                const size_t *src_len, void *d_dst, const size_t *dst_off,
                                const size_t *dst_cap_each, size_t *dst_len, uint32_t *checksum,
                                int *status);
/* Upper bound of the deflate output for an input of src_len bytes (arena sizing). */
size_t zipc_b200_deflate_bound(size_t src_len);
/* Zipc_deflate.zlib_compress (src/zipc_deflate.mli:151-162, zipc_deflate.ml:1262-1277):
 * 2-byte header, deflate body, big-endian Adler-32 trailer; adler[i] is returned too. */
int zipc_b200_zlib_compress_batch(zipc_b200_ctx *ctx, int level, int adler_mode, size_t n,
                                  const void *const *src, const size_t *src_len,
                                  void *dst, size_t dst_cap, size_t *dst_need,
                                  size_t *dst_off, size_t *dst_len, uint32_t *adler, int *status);
/* Device-resident Zipc_deflate.zlib_compress (src/zipc_deflate.mli:151-162, zipc_deflate.ml:1262-1277): input i is
 * [src_off[i], src_off[i] + src_len[i]) of d_src (any alignment), stream i goes to the caller's slot at dst_off[i] of d_dst
 * (any alignment, unlike zipc_b200_deflate_batch_dev) with capacity dst_cap_each[i]; zipc_b200_zlib_bound(src_len[i])
 * always suffices.  Members are compressed as by zipc_b200_zlib_compress_batch, large ones as primed segments over many
 * CTAs, and the streams and adler[] are byte for byte those it returns for the same batch.  On success exactly
 * [dst_off[i], dst_off[i] + dst_len[i]) is written.  A stream that does not fit its slot gives status[i] =
 * ZIPC_ERR_DST_TOO_SMALL, dst_len[i] = 0, adler[i] = 0, and nothing of its slot is written; the other members are not
 * affected.  adler_mode is ZIPC_ADLER_*; adler may be NULL. */
int zipc_b200_zlib_compress_batch_dev(zipc_b200_ctx *ctx, int level, int adler_mode, size_t n,
                                      const void *d_src, const size_t *src_off, const size_t *src_len,
                                      void *d_dst, const size_t *dst_off, const size_t *dst_cap_each,
                                      size_t *dst_len, uint32_t *adler, int *status);
/* Upper bound of a zlib stream of zipc_b200_zlib_compress_batch(_dev) for an input of src_len bytes, whatever segments the
 * library cuts the input into (slot sizing). */
size_t zipc_b200_zlib_bound(size_t src_len);

/* ---- one large stream as independent segments (BASELINE.json configs 1 and 5) ----------------------- */
/* Zipc_deflate.crc_32_and_deflate for ONE large input, parallel inside the stream: the input is cut into
 * segments of segment_size bytes, each compressed with a fresh window by one CTA; every segment but the last
 * ends with an empty stored block, so the pieces are byte aligned and their concatenation is ONE valid
 * RFC 1951 stream that Zipc_deflate.inflate reads.  index receives nseg + 1 pairs (compressed offset,
 * uncompressed offset), the last pair being the totals.  last_piece = 0 keeps BFINAL off the last segment
 * (the slice is a non-final piece of a stream spread over several GPUs).  crc32 = CRC-32 of the input. */
int zipc_b200_deflate_segmented(zipc_b200_ctx *ctx, int level, const void *src, size_t len, size_t segment_size,
                                int last_piece, void *dst, size_t dst_cap, size_t *dst_len, uint64_t *index,
                                size_t index_cap_pairs, size_t *nseg, uint32_t *crc32);
/* The same with every segment PRIMED with the 32 KiB of input before it (pigz style): matches reach back across segment
 * boundaries, so the stream is as small as one compressed in one piece (plus 5 bytes per segment for the byte-aligning
 * empty stored block) while still being compressed by one CTA per segment.  The result is an ordinary RFC 1951 stream;
 * its segments are NOT independent, so it is decoded like any foreign stream (zipc_b200_inflate_batch: many warps through
 * block-start search and speculation), not by zipc_b200_inflate_segmented.  index as above (informational).  This is what
 * one large payload of Zipc.File.deflate_of_binary_string (src/zipc.ml:179-185) should go through. */
int zipc_b200_deflate_primed(zipc_b200_ctx *ctx, int level, const void *src, size_t len, size_t segment_size,
                             int last_piece, void *dst, size_t dst_cap, size_t *dst_len, uint64_t *index,
                             size_t index_cap_pairs, size_t *nseg, uint32_t *crc32);
/* Zipc_deflate.inflate_and_crc_32 of such a stream WITH its index: segments are decoded in parallel (one
 * warp each).  status = ZIPC_OK or the status of the first bad segment.  Without the index the stream
 * is an ordinary deflate stream (zipc_b200_inflate_batch decodes it serially). */
int zipc_b200_inflate_segmented(zipc_b200_ctx *ctx, const void *src, size_t len, const uint64_t *index, size_t nseg,
                                void *dst, size_t dst_cap, size_t *dst_len, uint32_t *crc32, int *status);

/* ---- ZIP archive layer (zipc.ml) ------------------------------------------------------------ */
/* One archive member: Zipc.Member.t + Zipc.File.t (zipc.ml:145-154,238-242). */
typedef struct {
  const char *path;            /* path_len bytes, not NUL terminated */
  uint32_t path_len;
  int32_t is_dir;
  int32_t mode;                /* Fpath.mode */
  int64_t mtime;               /* POSIX seconds */
  int32_t version_made_by, version_needed, gp_flags;
  int32_t compression;         /* 0 stored, 8 deflate, ... (zipc.ml:25-31) */
  const uint8_t *compressed_bytes;
  uint64_t start;              /* payload offset in compressed_bytes */
  uint64_t compressed_size;
  uint64_t decompressed_size;
  uint32_t crc32;
  uint32_t _pad;
} zipc_b200_member;

/* Zipc.Ptime (zipc.ml:64-125): DOS date/time conversions used by the headers. */
void zipc_b200_ptime_to_dos(int64_t ptime_s, int *dos_date, int *dos_time);
int64_t zipc_b200_ptime_of_dos(int dos_date, int dos_time);

/* Zipc.of_binary_string (zipc.ml:400-438): parse the central directory of an in-memory
 * archive.  Host only.  *members is allocated by the library (free with zipc_b200_free) and its
 * path / compressed_bytes pointers alias `bytes`.  Members come back sorted by path with later
 * duplicates winning, like the reference's map. */
int zipc_b200_zip_parse(const void *bytes, size_t len, zipc_b200_member **members, size_t *n);
/* Zipc.encoding_size (zipc.ml:447-455). */
uint64_t zipc_b200_zip_encoding_size(const zipc_b200_member *members, size_t n);
/* Zipc.to_binary_string (zipc.ml:570-588): lay out LFH + payload, central directory, EOCD in
 * the reference's member order (`first`, default "mimetype", then byte-wise path order).
 * Host only; out must hold zipc_b200_zip_encoding_size bytes. */
int zipc_b200_zip_assemble(const zipc_b200_member *members, size_t n, const char *first,
                           void *out, size_t out_cap, size_t *out_len);
/* ZIP64 (SURVEY.md 8f-4; APPNOTE 4.3.14, 4.3.15, 4.5.3).  The reference rejects ZIP64 archives when reading
 * (zipc.ml:404) and refuses to write what would need it (more than 65,535 members, a size or an offset of 4 GiB or
 * more: zipc.ml:229-235, 130-133, 550-551); ZIPC_ZIP_REFERENCE keeps exactly that behaviour and is what the calls
 * without _ex use.  ZIPC_ZIP_ALLOW_ZIP64 goes beyond the reference: the parser follows a ZIP64 end of central
 * directory locator and takes 64-bit sizes / offsets from the ZIP64 extra fields; the writer emits ZIP64 extra fields,
 * the ZIP64 end of central directory record and its locator where (and only where) a 16/32-bit field overflows, so
 * an archive that fits the classic format comes out byte-identical to the reference's.  ZIPC_ZIP_FORCE_ZIP64 (writer)
 * emits them for every member, as CPython's zipfile does with force_zip64.  The checker for these paths is CPython's
 * zipfile (the reference has no ZIP64). */
enum { ZIPC_ZIP_REFERENCE = 0, ZIPC_ZIP_ALLOW_ZIP64 = 1, ZIPC_ZIP_FORCE_ZIP64 = 2 };
int zipc_b200_zip_parse_ex(const void *bytes, size_t len, unsigned flags, zipc_b200_member **members, size_t *n);
uint64_t zipc_b200_zip_encoding_size_ex(const zipc_b200_member *members, size_t n, const char *first, unsigned flags);
int zipc_b200_zip_assemble_ex(const zipc_b200_member *members, size_t n, const char *first, unsigned flags,
                              void *out, size_t out_cap, size_t *out_len);
/* Batch form of Zipc.File.to_binary_string (zipc.ml:205-225) over parsed members: stored and
 * deflate members are extracted on the GPU and their CRC-32 compared with the directory's.
 * status[i]: ZIPC_OK, ZIPC_ERR_CORRUPTED, ZIPC_ERR_SIZE_EXCEEDED (both "deflate: "-prefixed in
 * the reference), ZIPC_ERR_CHECKSUM (found[i] holds the computed CRC), ZIPC_ERR_ZIP_ENCRYPTED,
 * ZIPC_ERR_ZIP_FORMAT.  Directories yield length 0 / ZIPC_OK. */
int zipc_b200_zip_extract_batch(zipc_b200_ctx *ctx, const zipc_b200_member *members, size_t n,
                                void *dst, size_t dst_cap, size_t *dst_need,
                                size_t *dst_off, size_t *dst_len, uint32_t *found, int *status);
/* Device-resident Zipc.of_binary_string (zipc.ml:400-438): the archive is the len bytes at d_bytes in device memory.
 * Returns what zipc_b200_zip_parse_ex returns for the same bytes and flags: the same status, the same members in the same
 * order (sorted by path, a later duplicate winning) and the same field values, with two differences:
 *   - compressed_bytes is d_bytes, a DEVICE pointer: the payload of a member is at compressed_bytes + start on the device;
 *   - path points into a host copy of the central directory.
 * That copy and the member array are one allocation: free both with one zipc_b200_free(*members).  The call copies only the
 * last 65,577 bytes (EOCD search), the ZIP64 end record if there is one, and the central directory to the host, and reads
 * all local headers with one kernel, however many members there are.  len < 22: ZIPC_ERR_ZIP_SHORT, nothing is read.
 * Members from this call go to zipc_b200_zip_extract_batch_dev only, never to the host-pointer calls. */
int zipc_b200_zip_parse_dev(zipc_b200_ctx *ctx, const void *d_bytes, size_t len, unsigned flags,
                            zipc_b200_member **members, size_t *n);
/* Device-resident Zipc.File.to_binary_string (zipc.ml:205-225) over parsed members: members[i].compressed_bytes + start must
 * be device memory on the ctx's device (members of zipc_b200_zip_parse_dev, or built by the caller, from one archive or
 * several); a member whose compressed_bytes is not (host members passed by mistake) makes the call return
 * ZIPC_ERR_INVALID_ARG before anything runs.  Output i goes to d_dst + dst_off[i], any alignment; its slot holds
 * decompressed_size bytes for a deflate member and compressed_size bytes for a stored one.  Nothing is written for
 * directories, encrypted members and unsupported methods.  status / dst_len / found are those of zipc_b200_zip_extract_batch
 * for the same members (found may be NULL).  Output contract of zipc_b200_inflate_batch_dev: on success exactly
 * [dst_off[i], dst_off[i] + dst_len[i]) is written, on failure writes stay inside the slot, so slots may sit back to back.
 * The device bytes are read anew by every call.  Stored members are copied and checksummed in one pass over their bytes,
 * large ones by many warps. */
int zipc_b200_zip_extract_batch_dev(zipc_b200_ctx *ctx, const zipc_b200_member *members, size_t n,
                                    void *d_dst, const size_t *dst_off, size_t *dst_len, uint32_t *found, int *status);
/* Batch form of Zipc.File.deflate_of_binary_string (zipc.ml:179-185) followed by
 * Zipc.to_binary_string: compress n payloads on the GPU at `level` and emit one archive.
 * paths are normalised as Member.make does (zipc.ml:244-255); mode / mtime may be NULL
 * (defaults 0o644 / DOS epoch). */
int zipc_b200_zip_deflate_archive(zipc_b200_ctx *ctx, int level, size_t n,
                                  const char *const *paths, const uint32_t *path_len,
                                  const void *const *src, const size_t *src_len,
                                  const int32_t *mode, const int64_t *mtime, const char *first,
                                  void *out, size_t out_cap, size_t *out_len);

/* The same with ZIPC_ZIP_* flags (see zipc_b200_zip_parse_ex): with ZIP64 allowed, more than 65,535 members or an archive of
 * 4 GiB or more is written with ZIP64 records instead of being refused (zipc.ml:229-235, 550-551, 574). */
int zipc_b200_zip_deflate_archive_ex(zipc_b200_ctx *ctx, int level, size_t n,
                                     const char *const *paths, const uint32_t *path_len,
                                     const void *const *src, const size_t *src_len,
                                     const int32_t *mode, const int64_t *mtime, const char *first, unsigned flags,
                                     void *out, size_t out_cap, size_t *out_len);

/* ---- box-wide entry points (SURVEY.md 8b "device_mask", 8e) -------------------------------------------------------- */
/* One call drives every selected GPU of the node: a multi-context owns one zipc_b200_ctx (stream, arenas) and one
 * host thread per device.  Batches are partitioned over the devices longest-first by member size (members are
 * independent: no collective on the data path); one buffer is cut into contiguous slices whose checksums are
 * merged on the host.  device_mask: bit d selects CUDA device d; 0 = every visible device.
 * These replace the same reference functions as their single-device forms: a loop of
 * Zipc.File.deflate_of_binary_string / File.to_binary_string over the members of an archive (zipc.ml:179-185,
 * 205-225) and Crc_32.string of one string (zipc_deflate.ml:161-163). */
typedef struct zipc_b200_mctx zipc_b200_mctx;
int zipc_b200_mctx_create(uint64_t device_mask, zipc_b200_mctx **mctx);
void zipc_b200_mctx_destroy(zipc_b200_mctx *mctx);
int zipc_b200_mctx_device_count(const zipc_b200_mctx *mctx);
/* The k-th device's context (owned by the mctx), e.g. for zipc_b200_ctx_launches. */
zipc_b200_ctx *zipc_b200_mctx_ctx(zipc_b200_mctx *mctx, int k);
const char *zipc_b200_mctx_last_error(const zipc_b200_mctx *mctx);
/* Crc_32.string of one host buffer: G contiguous slices, G-1 zipc_b200_crc32_combine steps. */
int zipc_b200_multi_crc32(zipc_b200_mctx *mctx, const void *src, size_t len, uint32_t *crc);
/* zipc_b200_inflate_batch / zipc_b200_deflate_batch over all devices; same arguments and arena conventions
 * (dst_off are offsets into ONE arena; after ZIPC_ERR_DST_TOO_SMALL use zipc_b200_multi_fetch). */
int zipc_b200_multi_inflate_batch(zipc_b200_mctx *mctx, int checksum_kind, int adler_mode, size_t n,
                                  const void *const *src, const size_t *src_len, const size_t *max_out,
                                  void *dst, size_t dst_cap, size_t *dst_need,
                                  size_t *dst_off, size_t *dst_len, uint32_t *checksum, int *status);
int zipc_b200_multi_deflate_batch(zipc_b200_mctx *mctx, int level, int checksum_kind, int adler_mode,
                                  size_t n, const void *const *src, const size_t *src_len,
                                  void *dst, size_t dst_cap, size_t *dst_need,
                                  size_t *dst_off, size_t *dst_len, uint32_t *checksum, int *status);
int zipc_b200_multi_fetch(zipc_b200_mctx *mctx, void *dst, size_t dst_cap);

void zipc_b200_free(void *p);

/* ---- synthetic workloads (SURVEY.md section 8d; integer-only, host side) -------------------- */
void zipc_b200_synth_text(uint64_t seed, void *out, size_t n);  /* text-v1 */
void zipc_b200_synth_rand(uint64_t seed, void *out, size_t n);  /* rand-v1 */

#ifdef __cplusplus
}
#endif
#endif
