// common.cuh -- internals shared by the libzipc_b200 translation units (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include <condition_variable>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/zipc_b200.h"

#define ZIPC_B200_VERSION "0.1.0"

namespace zb {

// ---- GF(2)[x] / P arithmetic for CRC-32 (reflected, P = 0xedb88320; x^0 is bit 31) -----------
// Used on both sides: host (table generation, combine) and device (tile / lane alignment).
constexpr uint32_t kCrcPoly = 0xedb88320u;

__host__ __device__ inline uint32_t gf_mul(uint32_t a, uint32_t b) {
  uint32_t p = 0;
#pragma unroll 8
  for (int i = 0; i < 32; i++) {
    p ^= b & (0u - (a >> 31));
    a <<= 1;
    b = (b >> 1) ^ (kCrcPoly & (0u - (b & 1u)));
  }
  return p;
}

// x^(8*nbytes) mod P, host side (square and multiply over a 64-entry x^(2^k) table).
uint32_t gf_xpow8(uint64_t nbytes);

// ---- grow-only device / pinned buffers ------------------------------------------------------
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes);  // returns ZIPC_OK / ZIPC_ERR_NOMEM; contents are NOT preserved
  void release();
  template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};
struct PinBuf {
  void *p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes);
  void release();
  template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// ---- copy / compute pipelining of one large batch --------------------------------------------
// A large host-pointer batch is cut into groups that run on sub-contexts of the same device (own stream, own arenas), one
// host thread each: the upload of group k + 1 and the download of group k - 1 then run under the kernel of group k.  The
// uploads take turns in group order (a ticket), so that group 0's kernel can start after 1/G of the input has arrived
// instead of all groups' copies sharing the bus and finishing together.
struct UploadGate {
  std::mutex m;
  std::condition_variable cv;
  size_t turn = 0;
  // The groups' deflate kernels run in group order, at most two at a time (the tail of one under the start of the next):
  // group k's kernel waits for the event behind group k - 2's.  Left to itself the block scheduler interleaves the CTAs
  // of all queued kernels, every group finishes at the end, and the downloads have nothing to overlap with (measured).
  std::vector<cudaEvent_t> done;    // behind the deflate kernel of each group
  std::vector<char> launched;       // ... which has been recorded (or will never be) in this batch
};

// ---- device descriptors ---------------------------------------------------------------------
struct CrcSeg {       // one CRC-32 work item: state after running `len` bytes from `init`
  const uint8_t *ptr;
  uint64_t len;
  uint32_t init;
  uint32_t _pad;
};
inline CrcSeg crc_seg(const uint8_t *ptr, uint64_t len) {  // a whole range, from the standard initial state
  CrcSeg s;
  s.ptr = ptr;
  s.len = len;
  s.init = 0xFFFFFFFFu;
  s._pad = 0;
  return s;
}

// One tile of a stored ZIP member for stored_copy_crc (crc32.cu): a member of L bytes is cut into tiles of kStoredTile bytes
// (the last one shorter; a member of 0 bytes is one empty tile).
constexpr uint64_t kStoredTile = 256u << 10;
struct StoredTile {
  const uint8_t *src;
  uint8_t *dst;
  uint64_t len;
  uint64_t after;     // bytes of the member after this tile
  uint32_t member;    // index of the member's CRC word
  uint32_t init;      // 0xFFFFFFFF for the member's first tile, 0 for the others
};

struct AdlerSeg {     // one Adler-32 work item: sums over [ptr, ptr+len)
  const uint8_t *ptr;
  uint32_t len;       // <= 5552
  uint32_t _pad;
};

struct InflateTask {  // one deflate stream to inflate
  const uint8_t *src;
  uint64_t src_len;
  uint8_t *dst;       // may be null in count-only mode
  uint64_t dst_cap;   // ?decompressed_size, or ~0ull when unknown (count-only pass)
  uint32_t flags;     // kInflateSegment: a piece of a segmented stream, ends where its input ends
  uint32_t group;     // progressive download: the group whose counter this stream decrements when it is done
  // speculative decoding of one chunk of a large stream (inflate_kernel<.., SPEC>): decoding starts at the block header at
  // bit start_bit of the stream and stops at the first block boundary at or after stop_bit; dst holds 16-bit symbols
  // (dst_cap counts symbols): a byte, or 0x8000 | w for "byte w of the 32 KiB that precede this chunk's output"
  uint64_t start_bit, stop_bit;
};
constexpr uint32_t kInflateSegment = 1u;
constexpr uint32_t kInflatePartShift = 1, kInflatePartMask = 7u;  // flags bits 1..3: the part of a split upload that carries the stream's bytes (0: no wait)
struct InflateResult {
  uint64_t out_len;
  uint32_t status;
  uint32_t _pad;      // fused Adler-32 of the output when the kernel was asked for it
  uint64_t end_bit;   // (speculative chunks) stream bit position after the last block decoded
  uint32_t final_seen; // (speculative chunks) that block had BFINAL set
  uint32_t _pad2;
};

struct DeflateTask {  // one input to deflate (a ZIP member or an independent segment)
  const uint8_t *src;
  uint64_t src_len;   // < 2^32
  uint8_t *dst;       // 4-byte aligned output slot
  uint64_t dst_cap;
  uint32_t flags;     // kDeflateNotFinal: no BFINAL, end with a byte-aligning empty stored block
  uint32_t blk_off;   // index of this member's first entry in the launch's block-length list (see deflate_launch)
};
constexpr uint32_t kDeflateNotFinal = 1u;
// flags bits 8..15: the member is primed with that many 2048-byte tiles of input that lie right BEFORE src (a segment of a
// larger stream whose matches may reach back into the previous segment's bytes: no window reset, no ratio loss)
constexpr uint32_t kDeflatePrimeShift = 8, kDeflatePrimeMask = 0xFFu, kDeflatePrimeTile = 2048u;
struct DeflateResult {
  uint64_t out_len;
  uint32_t status;
  uint32_t blocks;
};

struct CopyDesc {     // gather: len bytes from src to dst
  const uint8_t *src;
  uint8_t *dst;
  uint64_t len;
};

// ---- zlib framing (RFC 1950) -------------------------------------------------------------------
// The header checks of zlib_decompress in the reference's order (zipc_deflate.ml:722-731): ZIPC_OK or the stream's status;
// *method receives CM on ZIPC_ERR_ZLIB_METHOD (the "%d" of the message).  s holds len bytes (host or device memory).
__host__ __device__ inline int zlib_header_status(const uint8_t *s, uint64_t len, uint32_t *method) {
  if (len < 6) return ZIPC_ERR_CORRUPTED;
  const uint32_t cmf = s[0], flg = s[1];
  if ((256 * cmf + flg) % 31 != 0) return ZIPC_ERR_CORRUPTED;
  if ((cmf & 0x0F) != 8) { *method = cmf & 0x0F; return ZIPC_ERR_ZLIB_METHOD; }
  if ((cmf >> 4) > 7) return ZIPC_ERR_ZLIB_WINDOW;
  if (flg & 0x20) return ZIPC_ERR_ZLIB_DICT;
  return ZIPC_OK;
}
// the big-endian Adler-32 in the last 4 of len >= 4 bytes
__host__ __device__ inline uint32_t zlib_trailer(const uint8_t *s, uint64_t len) {
  return (uint32_t)s[len - 4] << 24 | (uint32_t)s[len - 3] << 16 | (uint32_t)s[len - 2] << 8 | s[len - 1];
}
struct ZlibFrame {    // one stream of zipc_b200_zlib_decompress_batch_dev: the host fills src / len, zlib_frames_kernel the rest
  const uint8_t *src;
  uint64_t len;
  uint32_t status;    // zlib_header_status
  uint32_t method;    // CM when status is ZIPC_ERR_ZLIB_METHOD
  uint32_t expect;    // the trailer when status is ZIPC_OK
  uint32_t _pad;
};

// ---- ZIP archives ------------------------------------------------------------------------------
// The four fields of a local file header (APPNOTE 4.3.7) the parser checks; off comes from the central directory.
struct ZipLfh {
  uint64_t off;
  uint32_t sig, crc, name_len, extra_len;
};
// h: the 30 bytes of a local header (host or device memory, any alignment)
__host__ __device__ inline void zip_lfh_fields(const uint8_t *h, ZipLfh &f) {
  f.sig = (uint32_t)h[0] | (uint32_t)h[1] << 8 | (uint32_t)h[2] << 16 | (uint32_t)h[3] << 24;
  f.crc = (uint32_t)h[14] | (uint32_t)h[15] << 8 | (uint32_t)h[16] << 16 | (uint32_t)h[17] << 24;
  f.name_len = (uint32_t)h[26] | (uint32_t)h[27] << 8;
  f.extra_len = (uint32_t)h[28] | (uint32_t)h[29] << 8;
}
struct ZipEnd {       // what the end records say
  uint64_t count, cd_size, cd_start;
  uint64_t rec64;     // offset of the ZIP64 end record still to read (~0: none)
};
// bytes at the end of an archive that zip_find_end may read: the EOCD (22 bytes + a comment of up to 65,535), the ZIP64
// locator in front of it (20)
constexpr uint64_t kZipTailWindow = 65535 + 22 + 20;

}  // namespace zb

// ---- the context -------------------------------------------------------------------------------
struct zipc_b200_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  std::string last_error;
  uint64_t launches = 0;
  bool profile = false;           // bracket the dominant kernel of each call with events
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool ev_valid = false;

  // constant tables on the device
  uint32_t *d_crc_tabs = nullptr;   // see crc32.cu: strided[4][256] | std[4][256] | xp16[32]
  // work buffers (grow-only)
  zb::DevBuf d_in, d_out, d_desc, d_res, d_scratch, d_scratch2, d_small, d_slots, d_desc2, d_blk;
  zb::DevBuf d_par, d_spec, d_win;   // intra-stream parallel inflate: chunk tables, speculative symbols, windows
  zb::PinBuf h_stage, h_res, h_desc;
  cudaStream_t copy_stream = nullptr;  // progressive downloads (api.cu)
  cudaStream_t upload_stream = nullptr;  // late half of a split upload
  cudaStream_t hi_stream = nullptr;      // high priority: compaction of a pipelined group (zip_api.cu compact)
  uint32_t *d_upflag = nullptr;        // device word: serial number of the last completed late half
  uint32_t upload_serial = 0;
  cudaEvent_t ev_block = nullptr;      // stream_sync of a sub-context
  cudaEvent_t ev_half = nullptr;       // first half of a split upload is through
  cudaEvent_t ev_stage[2] = {nullptr, nullptr};  // the last DMA of each buffer of h_stage (api.cu StageRing)
  bool upload_split_live = false;      // the late half of the current upload is still on its way
  uint32_t *h_word = nullptr;          // mapped host memory: one-word results written by kernels (map_host_word)
  uint32_t *h_gflag = nullptr;         // mapped host memory: group-complete flags written by inflate_kernel

  // intra-stream parallel inflate: the plan of the last large stream decoded speculatively (a count-only pass is followed by
  // the real pass over the same device bytes; `epoch` changes whenever new input is uploaded)
  struct ParPlan {
    const uint8_t *src = nullptr;
    size_t src_len = 0;
    uint64_t epoch = 0;
    std::vector<uint64_t> spec_off, len;
    std::vector<uint32_t> blocks;      // output lengths of the stream's non-empty deflate blocks, in order (Adler-32 is folded per block)
    uint64_t total = 0;
  } par_plan;
  uint64_t epoch = 1;
  zb::DevBuf d_adler;                // adler32.cu: CTA partials + arrival counter of the RFC 1950 reduction
  zb::DevBuf d_adler_chain;          // adler32.cu: tile counter + the two chains of the REF_COMPAT fold (tagged by adler_epoch)
  uint32_t adler_epoch = 0;
  void *adler_ticket_at = nullptr;   // where the counter was last zeroed (the kernel resets it itself afterwards)
  uint64_t par_streams = 0, par_fallbacks = 0;   // diagnostics: large streams decoded in parallel / handed back to the serial path

  // pipelining (multi.cc): a sub-context waits for its turn to upload; the parent owns the sub-contexts
  zb::UploadGate *gate = nullptr;
  size_t gate_ticket = 0;
  bool gate_passed = false;
  bool is_sub = false;
  struct zipc_b200_mctx *pipe = nullptr;
  struct zipc_b200_mctx *par_pool = nullptr;   // lanes of the many-warp inflate: sub-contexts that decode large streams side by side
  uint32_t sm_share = 0;                       // a lane: the SMs its speculative decode spreads over (0 = all)
  cudaEvent_t ev_lanes = nullptr;              // "everything queued on `stream` so far" for the lanes' streams to wait on

  size_t last_total = 0;   // bytes of d_out the last host-pointer call left for zipc_b200_fetch()
};

namespace zb {

int set_cuda_error(zipc_b200_ctx *ctx, cudaError_t e, const char *what);
#define ZB_CUDA(ctx, call)                                        \
  do {                                                            \
    cudaError_t _e = (call);                                      \
    if (_e != cudaSuccess) return zb::set_cuda_error(ctx, _e, #call); \
  } while (0)

// brackets one kernel launch with the ctx's profiling events (no-op unless enabled)
struct KernelTimer {
  zipc_b200_ctx *c;
  explicit KernelTimer(zipc_b200_ctx *ctx) : c(ctx) { if (c->profile) cudaEventRecord(c->ev0, c->stream); }
  ~KernelTimer() { if (c->profile) { cudaEventRecord(c->ev1, c->stream); c->ev_valid = true; } }
};

// RAII device guard
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---- kernels' host launchers (each .cu exports these) -----------------------------------------
// crc32.cu
int crc_tables_upload(zipc_b200_ctx *ctx);
// state-after-init for each segment (device descriptors), results to d_states[nseg]
int crc32_launch_segments(zipc_b200_ctx *ctx, const CrcSeg *d_segs, uint32_t nseg, uint32_t *d_states);
// whole-buffer CRC-32 (final value, init/xorout applied) into *d_crc
int crc32_launch_buffer(zipc_b200_ctx *ctx, const uint8_t *d_src, uint64_t len, uint32_t *d_crc);
// Stored ZIP members: copies len[i] bytes from src[i] to dst[i] (device addresses, any alignment, no overlap) and returns
// the CRC-32 of each (final value) in crc[i] on the host.  Every source byte is read once and written once, in one kernel
// whose warps take tiles of kStoredTile bytes.  Exactly [dst[i], dst[i] + len[i]) is written.  The stream is through on return.
int stored_copy_crc(zipc_b200_ctx *ctx, size_t n, const uint8_t *const *src, uint8_t *const *dst, const uint64_t *len,
                    uint32_t *crc);
// adler32.cu
int adler32_launch_buffer(zipc_b200_ctx *ctx, const uint8_t *d_src, uint64_t len, int mode, uint32_t *h_out);
// per-range Adler-32 for n ranges given as (ptr,len) on the host; results (final values) to h_out
int adler32_ranges(zipc_b200_ctx *ctx, const uint8_t *const *d_ptrs, const uint64_t *lens, size_t n, int mode,
                   uint32_t *h_out);
// Adler-32 of n inputs, each folded block by block as the reference does on both codec sides (state re-packed and the
// 5552-byte chunk grid restarted at every block, :682-690, :1081-1086): member i consists of nblk[i] consecutive
// blocks whose lengths follow each other in blk_len
int adler32_blocked(zipc_b200_ctx *ctx, const uint8_t *const *d_ptrs, const uint32_t *nblk, const uint32_t *blk_len,
                    size_t n, int mode, uint32_t *h_out);
// deflate.cu
// d_blk_lens (may be null): receives the source length of every deflate block of member i at
// d_blk_lens[task.blk_off + b], b < result.blocks -- the ranges the reference checksums one by one (:1081-1086)
int deflate_launch(zipc_b200_ctx *ctx, const DeflateTask *d_tasks, uint32_t n, DeflateResult *d_results, int level,
                   uint32_t *d_blk_lens = nullptr, uint64_t max_src_len = 0 /* level `None: the longest input, sizes the grid */);
// upper bound of the number of deflate blocks the encoder emits for an input of src_len bytes
inline uint32_t deflate_max_blocks(uint64_t src_len) { return (uint32_t)(src_len / 61440) + 2; }
constexpr uint32_t kStoredBlock = 65534;  // source bytes per block at level `None (reference :747-750, :1106-1116)
// zip_api.cu: n independent copies on the device (compaction of per-member output slots)
int gather_launch(zipc_b200_ctx *ctx, const CopyDesc *d_descs, uint32_t n, cudaStream_t stream = nullptr);
// api.cu helpers shared with zip_api.cu
int h2d(zipc_b200_ctx *ctx, void *d, const void *h, size_t bytes);
int d2h(zipc_b200_ctx *ctx, void *h, const void *d, size_t bytes);
// One whole host buffer into ctx->d_in at the host's 16-byte phase; *d: where its bytes begin.  Voids the plans made over the
// old input bytes (ctx->epoch).
int upload_buffer(zipc_b200_ctx *ctx, const void *src, size_t len, const uint8_t **d);
// Allocates ctx->h_word on first use: kernels store one-word results there (word 0: Adler-32, word 1: CRC-32), so that no
// 4-byte copy into a caller's pageable word stalls the host.  The host reads a word after its next wait for the stream.
int map_host_word(zipc_b200_ctx *ctx);
// enqueues the CRC-32 of a device buffer into h_word[1]; host_word_crc32 reads it
int crc32_to_host_word(zipc_b200_ctx *ctx, const uint8_t *d_src, uint64_t len);
uint32_t host_word_crc32(const zipc_b200_ctx *ctx);
// cudaStreamSynchronize; the threads of a pipelined batch (sub-contexts) sleep on a blocking event instead of spinning: there
// are up to 24 of them per process, and a box runs one process per GPU
cudaError_t stream_sync(zipc_b200_ctx *ctx, cudaStream_t s);
// A split upload (api.cu upload_ranges): the first part of a large pinned span goes out on the context's stream, the second
// behind it on upload_stream, followed by a count (ctx->upload_serial + 1) into ctx->d_upflag; a stream whose bytes lie in
// the second part is decoded only after the kernel has seen that count.
struct UploadSplit {
  bool want = false;   // in: the caller can deal with a split
  uintptr_t cut = 0;   // out: host address where the second part begins (0: the upload was not split)
  bool late(const void *p) const { return cut && (uintptr_t)p >= cut; }
};
int upload_ranges(zipc_b200_ctx *ctx, size_t n, const void *const *src, const size_t *len,
                  std::vector<const uint8_t *> &d_ptr, UploadSplit *split = nullptr);
// Progressive download of an inflate batch (api.cu): the streams are sorted by output size into groups that own contiguous
// ranges of the output arena; the decoder counts every group down and raises a flag in mapped host memory when a group is
// complete, and the host starts that range's copy while the kernel works on the larger streams.
struct DownloadPlan {
  uint32_t ngroups = 0;                 // 0: not used, the arena is in member order and comes back with one copy
  std::vector<uint32_t> group_of;       // per stream handed to inflate_core
  std::vector<size_t> goff, gbytes;     // arena range of each group
  uint8_t *dst = nullptr;               // the caller's (pinned) arena
  size_t tail_off = 0, tail_bytes = 0;  // arena range of everything that is not a grouped stream (copied at the end)
  std::vector<char> late;               // per stream handed to inflate_core: 1 if the second part of a split upload carries its input
};
int inflate_core(zipc_b200_ctx *ctx, int ck, int adler_mode, size_t n, const std::vector<const uint8_t *> &d_src,
                 const size_t *src_len, const std::vector<uint8_t *> &d_dst, const std::vector<size_t> &cap,
                 bool count_only, size_t *out_len, uint32_t *checksum, int *status, uint32_t flags = 0,
                 const DownloadPlan *plan = nullptr);
// Lay out the output arena of n members (cap[i] bytes each, 16-byte aligned slots).  grouped[i] != 0 marks the streams that
// go through the inflate kernel.  Fills off / total, and plan when the batch qualifies for a progressive download.
// The streams whose input the second part of a split upload carries (src: their host addresses) form the later groups.
bool progressive_ok(zipc_b200_ctx *ctx, size_t n, const size_t *cap, const size_t *src_len, const char *grouped, void *dst, size_t dst_cap);
int plan_arena(zipc_b200_ctx *ctx, size_t n, const size_t *cap, const void *const *src, const size_t *src_len, const char *grouped,
               const UploadSplit &split, void *dst, size_t dst_cap, std::vector<size_t> &off, size_t &total, DownloadPlan &plan);
// Tail of every host-pointer call that leaves its output in ctx->d_out: keeps `total` for zipc_b200_fetch, reports the layout
// (dst_off, dst_need: may be null) and copies the output into the caller's arena, progressively when `plan` has groups.  Without
// an arena, or with one too small, it returns ZIPC_ERR_DST_TOO_SMALL.  Either way the stream is through when it returns.
int finish_to_host(zipc_b200_ctx *ctx, const std::vector<size_t> &off, size_t total, void *dst, size_t dst_cap, size_t *dst_off,
                   size_t *dst_need, const DownloadPlan *plan = nullptr);
// ZIPC_B200_PIPE_DEBUG=1: time stamps of the stages of a pipelined batch on stderr (group ticket, stage, ms)
void pipe_mark(const zipc_b200_ctx *ctx, const char *stage);
// api.cu / multi.cc: copy / compute pipelining of large host-pointer batches on one device
zipc_b200_mctx *pipeline_for(zipc_b200_ctx *ctx, size_t n, const size_t *len, const void *dst);
int pipeline_create(int device, int depth, zipc_b200_mctx **out);
uint64_t pipeline_launches(const zipc_b200_mctx *m);
int pipeline_deflate_gapped(zipc_b200_mctx *m, int level, size_t n, const void *const *src, const size_t *src_len, const uint32_t *gap,
                            void *dst, size_t dst_cap, size_t *dst_need, size_t *dst_off, size_t *dst_len, uint32_t *crc, int *status);
// zip_api.cu: zipc_b200_deflate_batch on one context with a caller-defined output layout
int deflate_batch_layout(zipc_b200_ctx *ctx, int level, int ck, int adler_mode, size_t n, const void *const *src, const size_t *src_len,
                         void *dst, size_t dst_cap, size_t *dst_need, size_t *dst_off, size_t *dst_len, uint32_t *checksum, int *status,
                         const uint32_t *gap, size_t align);
// host_util.cc: the archive parser in pieces (zipc_b200_zip_parse_ex and zipc_b200_zip_parse_dev share them)
int zip_find_end(const uint8_t *tail, uint64_t tail_at, uint64_t len, unsigned flags, ZipEnd &e);
int zip_read_end64(const uint8_t *rec, uint64_t len, ZipEnd &e);
int zip_check_cd_range(uint64_t len, const ZipEnd &e);
int zip_walk_cd(const uint8_t *cd, uint64_t len, unsigned flags, const ZipEnd &e, std::vector<zipc_b200_member> &ms,
                std::vector<ZipLfh> &lfh);
int zip_parse_finish(std::vector<zipc_b200_member> &ms, const std::vector<ZipLfh> &lfh, int cd_status, uint64_t len,
                     const uint8_t *bytes, const uint8_t *cd, uint64_t cd_size, bool cd_copy, zipc_b200_member **members,
                     size_t *n_out);
// host_util.cc
int zip_assemble_impl(const zipc_b200_member *ms, size_t n, const char *first, void *out_v, size_t out_cap,
                      size_t *out_len, bool copy_payload, uint64_t *payload_off, unsigned flags = 0 /* ZIPC_ZIP_* */);
// inflate.cu
int inflate_launch(zipc_b200_ctx *ctx, const InflateTask *d_tasks, uint32_t n, InflateResult *d_results,
                   bool count_only, int adler_mode /* -1: none */, unsigned int *d_group_count = nullptr,
                   uint32_t *group_flag = nullptr, const uint32_t *d_upflag = nullptr, uint32_t upload_serial = 0);
// intra-stream parallel inflate (a large stream without an index): the three device steps; api.cu orchestrates
// 1. for every chunk k >= 1 of `chunk_bytes` compressed bytes laid from bit first_bit on, the first bit position
//    >= first_bit + 8 * k * chunk_bytes at which a valid dynamic-Huffman block header (of some substance) starts
//    (d_found[k], ~0 if none before the next chunk's own search range ends)
int inflate_find_starts(zipc_b200_ctx *ctx, const uint8_t *d_src, uint64_t src_len, uint64_t first_bit, uint64_t chunk_bytes,
                        uint32_t nchunks, uint64_t *d_found);
// 2. speculative decode of the chunks (tasks carry start_bit / stop_bit, dst = 16-bit symbols)
// d_block_lists (may be null): kSpecBlocks entries per task, the output lengths of the non-empty blocks of every chunk (for Adler-32)
constexpr uint32_t kSpecBlocks = 256;
int inflate_launch_spec(zipc_b200_ctx *ctx, const InflateTask *d_tasks, uint32_t n, InflateResult *d_results, unsigned int *d_block_lists = nullptr);
// 3. resolve: windows chunk by chunk, then every symbol to its byte.  d_spec_off / d_out_off / d_len: per chunk (device).
//    d_windows: 4 * 32768 bytes per chunk of scratch.  *d_bad is set if anything refers to bytes before the stream
int inflate_resolve(zipc_b200_ctx *ctx, const uint16_t *d_spec, const uint64_t *d_spec_off, const uint64_t *d_out_off,
                    const uint64_t *d_len, uint32_t nchunks, uint8_t *d_windows, uint8_t *d_dst, uint32_t *d_bad);

}  // namespace zb
