// api.cu -- context management and the host-facing C ABI of libzipc_b200 (include/zipc_b200.h).
//
// Everything here is plumbing: argument checks, staging host memory to the device, ordering the
// kernel launches of crc32.cu / adler32.cu / inflate.cu / deflate.cu on the ctx stream, and
// returning per-member results.  There is no CPU implementation of any codec step in this file.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <numeric>

#include <thread>

#include "common.cuh"

namespace zb {

uint32_t gf_mul_host(uint32_t a, uint32_t b) { return gf_mul(a, b); }

int set_cuda_error(zipc_b200_ctx *ctx, cudaError_t e, const char *what) {
  if (ctx) {
    ctx->last_error = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
  }
  cudaGetLastError();  // clear the sticky-less error state
  return e == cudaErrorMemoryAllocation ? ZIPC_ERR_NOMEM
         : (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? ZIPC_ERR_NO_DEVICE
                                                                        : ZIPC_ERR_CUDA;
}

cudaError_t stream_sync(zipc_b200_ctx *ctx, cudaStream_t s) {
  if (!ctx->is_sub) return cudaStreamSynchronize(s);
  if (!ctx->ev_block)
    if (cudaError_t e = cudaEventCreateWithFlags(&ctx->ev_block, cudaEventBlockingSync | cudaEventDisableTiming)) return e;
  if (cudaError_t e = cudaEventRecord(ctx->ev_block, s)) return e;
  return cudaEventSynchronize(ctx->ev_block);
}

int map_host_word(zipc_b200_ctx *ctx) {
  if (!ctx->h_word) ZB_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_word), 64, cudaHostAllocMapped));
  return ZIPC_OK;
}

int crc32_to_host_word(zipc_b200_ctx *ctx, const uint8_t *d_src, uint64_t len) {
  if (int st = map_host_word(ctx)) return st;
  return crc32_launch_buffer(ctx, d_src, len, ctx->h_word + 1);
}
uint32_t host_word_crc32(const zipc_b200_ctx *ctx) { return reinterpret_cast<const volatile uint32_t *>(ctx->h_word)[1]; }

int DevBuf::reserve(size_t bytes) {
  if (bytes <= cap) return ZIPC_OK;
  if (p) { cudaFree(p); p = nullptr; cap = 0; }
  size_t want = bytes + bytes / 8 + 4096;
  if (cudaMalloc(&p, want) != cudaSuccess) {
    cudaGetLastError();
    if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); p = nullptr; return ZIPC_ERR_NOMEM; }
    want = bytes;
  }
  cap = want;
  return ZIPC_OK;
}
void DevBuf::release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
int PinBuf::reserve(size_t bytes) {
  if (bytes <= cap) return ZIPC_OK;
  if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
  size_t want = bytes + bytes / 8 + 4096;
  if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); p = nullptr; return ZIPC_ERR_NOMEM; }
  cap = want;
  return ZIPC_OK;
}
void PinBuf::release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }

static bool is_pinned(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

// A copy of pinned host memory, or of no more than 64 KiB, is one DMA; anything else goes through the staging ring.
static bool copy_direct(const void *h, size_t bytes) { return bytes <= (1u << 16) || is_pinned(h); }

// Staging of pageable host memory: two pinned buffers of kStageChunk bytes (ctx->h_stage), used in turn, so that the CPU
// copy into or out of one overlaps the DMA of the other.  The last DMA of buffer i is behind ctx->ev_stage[i]; after a
// download its bytes still have to go on to the host address `to[i]`.  A ring is drained when it goes out of scope, so no
// DMA into or out of the staging buffers outlives the call, whichever way it returns.
static constexpr size_t kStageChunk = 16u << 20;
class StageRing {
  zipc_b200_ctx *c;
  int k = 0;  // the buffer to use next
  bool busy[2] = {false, false};
  uint8_t *to[2] = {nullptr, nullptr};
  size_t to_len[2] = {0, 0};
  uint8_t *buf(int i) const { return c->h_stage.as<uint8_t>() + (size_t)i * kStageChunk; }
  int wait(int i) {
    if (!busy[i]) return ZIPC_OK;
    busy[i] = false;
    ZB_CUDA(c, cudaEventSynchronize(c->ev_stage[i]));
    if (to_len[i]) std::memcpy(to[i], buf(i), to_len[i]);
    to_len[i] = 0;
    return ZIPC_OK;
  }
  int dma(void *dst, const void *src, size_t bytes, cudaMemcpyKind kind) {
    ZB_CUDA(c, cudaMemcpyAsync(dst, src, bytes, kind, c->stream));
    busy[k] = true;
    ZB_CUDA(c, cudaEventRecord(c->ev_stage[k], c->stream));
    k ^= 1;
    return ZIPC_OK;
  }

 public:
  explicit StageRing(zipc_b200_ctx *ctx) : c(ctx) {}
  ~StageRing() { drain(); }
  int open() {
    if (int st = c->h_stage.reserve(2 * kStageChunk)) return st;
    for (cudaEvent_t &e : c->ev_stage)
      if (!e) ZB_CUDA(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return ZIPC_OK;
  }
  // the next buffer, once its last DMA is through
  int next(uint8_t **b) {
    if (int st = wait(k)) return st;
    *b = buf(k);
    return ZIPC_OK;
  }
  // DMA of the first `bytes` of that buffer to device address d
  int upload(void *d, size_t bytes) { return dma(d, buf(k), bytes, cudaMemcpyHostToDevice); }
  // DMA of `bytes` from device address d into the next buffer; they reach host address h once it is needed again
  int download(void *h, const void *d, size_t bytes) {
    if (int st = wait(k)) return st;
    to[k] = static_cast<uint8_t *>(h);
    to_len[k] = bytes;
    return dma(buf(k), d, bytes, cudaMemcpyDeviceToHost);
  }
  // waits for both buffers, the older first
  int drain() {
    const int a = wait(k), b = wait(k ^ 1);
    return a ? a : b;
  }
};

// host -> device, enqueued on the context's stream (a pageable source has been read when this returns)
int h2d(zipc_b200_ctx *ctx, void *d, const void *h, size_t bytes) {
  if (copy_direct(h, bytes)) {
    if (bytes) ZB_CUDA(ctx, cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return ZIPC_OK;
  }
  StageRing ring(ctx);
  if (int st = ring.open()) return st;
  for (size_t off = 0; off < bytes; off += kStageChunk) {
    const size_t m = std::min(kStageChunk, bytes - off);
    uint8_t *s;
    if (int st = ring.next(&s)) return st;
    std::memcpy(s, static_cast<const uint8_t *>(h) + off, m);
    if (int st = ring.upload(static_cast<uint8_t *>(d) + off, m)) return st;
  }
  return ring.drain();
}

// device -> host.  Synchronous on return: the context's stream is through.
int d2h(zipc_b200_ctx *ctx, void *h, const void *d, size_t bytes) {
  if (copy_direct(h, bytes)) {
    if (bytes) ZB_CUDA(ctx, cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
    return ZIPC_OK;
  }
  StageRing ring(ctx);
  if (int st = ring.open()) return st;
  for (size_t off = 0; off < bytes; off += kStageChunk)
    if (int st = ring.download(static_cast<uint8_t *>(h) + off, static_cast<const uint8_t *>(d) + off, std::min(kStageChunk, bytes - off)))
      return st;
  return ring.drain();
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) & ~(a - 1); }
static double now_ms() { timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return t.tv_sec * 1e3 + t.tv_nsec / 1e6; }
static uint64_t env_u64(const char *name, uint64_t dflt) {
  const char *v = std::getenv(name);
  return (v && *v) ? std::strtoull(v, nullptr, 10) : dflt;
}

// Uploads n host ranges into ctx->d_in and returns their device addresses.  Never reads a byte of host memory that
// lies in a page none of the ranges touches: the ranges are sent as ONE span only when, in address order, every gap
// between neighbours is smaller than a page (then each gap byte shares a page with the end of one range or the
// start of the next -- members of an in-memory archive, separated by their local headers) and both ends of the
// span have the same kind of memory (pinned or pageable).  Otherwise every range is copied on its own: pinned ranges
// by DMA, pageable ones packed through the staging buffer.
int upload_ranges(zipc_b200_ctx *ctx, size_t n, const void *const *src, const size_t *len,
                  std::vector<const uint8_t *> &d_ptr, UploadSplit *split) {
  d_ptr.assign(n, nullptr);
  if (split) split->cut = 0;
  ctx->epoch++;  // new input bytes: plans made over the old ones are void
  // pipelined batches: wait for this group's turn on the bus; the next group may go once these bytes have arrived
  struct GatePass {
    zipc_b200_ctx *c;
    bool held = false;
    explicit GatePass(zipc_b200_ctx *ctx) : c(ctx) {
      if (!c->gate || c->gate_passed) return;
      std::unique_lock<std::mutex> lk(c->gate->m);
      c->gate->cv.wait(lk, [&] { return c->gate->turn == c->gate_ticket; });
      held = true;
    }
    ~GatePass() {
      if (!held) return;
      stream_sync(c, c->stream);
      { std::lock_guard<std::mutex> lk(c->gate->m); c->gate->turn++; c->gate_passed = true; }
      c->gate->cv.notify_all();
    }
  } gate_pass(ctx);
  if (!n) return ZIPC_OK;
  uintptr_t lo = ~(uintptr_t)0, hi = 0;
  size_t sum = 0, live = 0;
  for (size_t i = 0; i < n; i++) {
    if (!len[i]) continue;
    if (!src[i]) return ZIPC_ERR_INVALID_ARG;
    uintptr_t a = (uintptr_t)src[i];
    if (a + len[i] < a) return ZIPC_ERR_INVALID_ARG;
    lo = std::min(lo, a); hi = std::max(hi, a + len[i]);
    sum += len[i]; live++;
  }
  if (!sum) {
    if (int st = ctx->d_in.reserve(64)) return st;
    for (size_t i = 0; i < n; i++) d_ptr[i] = ctx->d_in.as<uint8_t>();
    return ZIPC_OK;
  }
  constexpr uintptr_t kMaxGap = 4096;  // < the smallest page size: a gap this small never contains a whole page
  const size_t span = hi - lo;
  bool one_span = span <= sum + live * (kMaxGap - 1);
  if (one_span) {
    std::vector<uint32_t> order;
    order.reserve(live);
    for (size_t i = 0; i < n; i++) if (len[i]) order.push_back((uint32_t)i);
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return (uintptr_t)src[a] < (uintptr_t)src[b]; });
    uintptr_t end = (uintptr_t)src[order[0]] + len[order[0]];
    for (size_t k = 1; k < order.size() && one_span; k++) {
      const uintptr_t a = (uintptr_t)src[order[k]];
      if (a > end && a - end >= kMaxGap) one_span = false;
      end = std::max(end, a + len[order[k]]);
    }
    if (one_span && is_pinned((const void *)lo) != is_pinned((const void *)(hi - 1))) one_span = false;
  }
  if (one_span) {
    size_t pre = lo & 15;  // keep the host alignment so 16-byte paths stay aligned
    if (int st = ctx->d_in.reserve(pre + span + 64)) return st;
    uint8_t *base = ctx->d_in.as<uint8_t>() + pre;
    for (size_t i = 0; i < n; i++) d_ptr[i] = len[i] ? base + ((uintptr_t)src[i] - lo) : base;
    if (split && split->want && span >= (128u << 20) && !ctx->gate && is_pinned((const void *)lo)) {
      // two parts (measured 40.3 GB/s end to end on C3, 36-37 with 3 to 6 parts, whose size-ordered queues each end in a tail
      // of large streams), cut at the first start of a range in the second half of the span: the first part on the context's
      // stream (what follows on that stream may use it), the second behind it on its own stream, its arrival announced
      // through d_upflag
      uintptr_t cut = hi;
      for (size_t i = 0; i < n; i++) { const uintptr_t a = (uintptr_t)src[i]; if (len[i] && a >= lo + span / 2 && a < cut) cut = a; }
      if (cut < hi && cut > lo) {
        if (!ctx->upload_stream) ZB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->upload_stream, cudaStreamNonBlocking));
        if (ctx->upload_split_live) {  // (a call that failed half way left its second part behind: its flag word must not be rewritten under it)
          ZB_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream));
          ctx->upload_split_live = false;
        }
        if (!ctx->h_gflag) ZB_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_gflag), 256 * sizeof(uint32_t), cudaHostAllocMapped));
        if (!ctx->d_upflag) {
          ZB_CUDA(ctx, cudaMalloc(reinterpret_cast<void **>(&ctx->d_upflag), 64));
          ZB_CUDA(ctx, cudaMemset(ctx->d_upflag, 0, 64));
        }
        ctx->upload_serial += 16;  // the count of this upload's second part: serial + 1
        ZB_CUDA(ctx, cudaMemcpyAsync(base, (const void *)lo, cut - lo, cudaMemcpyHostToDevice, ctx->stream));
        if (!ctx->ev_half) ZB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_half, cudaEventDisableTiming));
        ZB_CUDA(ctx, cudaEventRecord(ctx->ev_half, ctx->stream));
        ZB_CUDA(ctx, cudaStreamWaitEvent(ctx->upload_stream, ctx->ev_half, 0));  // one part after the other: each gets the whole bus
        ctx->h_gflag[241] = ctx->upload_serial + 1;  // (above the group flags)
        ZB_CUDA(ctx, cudaMemcpyAsync(base + (cut - lo), (const void *)cut, hi - cut, cudaMemcpyHostToDevice, ctx->upload_stream));
        ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_upflag, &ctx->h_gflag[241], sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->upload_stream));
        ctx->upload_split_live = true;
        split->cut = cut;
        return ZIPC_OK;
      }
    }
    if (int st = h2d(ctx, base, (const void *)lo, span)) return st;
    return ZIPC_OK;
  }
  size_t total = 0, pageable = 0;
  std::vector<size_t> off(n);
  std::vector<char> pin(n, 0);
  for (size_t i = 0; i < n; i++) {
    off[i] = total; total += align_up(len[i], 16);
    if (len[i]) { pin[i] = is_pinned(src[i]) && is_pinned(static_cast<const uint8_t *>(src[i]) + len[i] - 1); if (!pin[i]) pageable += align_up(len[i], 16); }
  }
  if (int st = ctx->d_in.reserve(total + 64)) return st;
  uint8_t *dbase = ctx->d_in.as<uint8_t>();
  // pageable ranges: packed into pinned staging chunk by chunk (CPU copy of chunk k+1 overlaps the DMA of chunk k);
  // consecutive pageable ranges keep consecutive device offsets, so a staged run is one DMA
  if (pageable) {
    StageRing ring(ctx);
    if (int st = ring.open()) return st;
    size_t i = 0, done_in_i = 0;  // next range / bytes of it already staged
    for (;;) {
      while (i < n && (!len[i] || pin[i])) { i++; done_in_i = 0; }
      if (i >= n) break;
      uint8_t *s;
      if (int st = ring.next(&s)) return st;
      // fill this staging buffer with a run of device-contiguous pageable bytes
      const size_t dev_start = off[i] + done_in_i;
      size_t fill = 0;
      while (i < n && fill < kStageChunk) {
        if (!len[i]) { i++; done_in_i = 0; continue; }
        if (pin[i] || off[i] + done_in_i != dev_start + fill) break;
        const size_t m = std::min(len[i] - done_in_i, kStageChunk - fill);
        std::memcpy(s + fill, static_cast<const uint8_t *>(src[i]) + done_in_i, m);
        fill += m; done_in_i += m;
        if (done_in_i == len[i]) {
          const size_t padto = std::min(align_up(len[i], 16) - len[i], kStageChunk - fill);
          std::memset(s + fill, 0, padto);
          if (padto == align_up(len[i], 16) - len[i]) { fill += padto; i++; done_in_i = 0; } else break;
        }
      }
      if (int st = ring.upload(dbase + dev_start, fill)) return st;
    }
    if (int st = ring.drain()) return st;
  }
  for (size_t i = 0; i < n; i++)
    if (len[i] && pin[i]) ZB_CUDA(ctx, cudaMemcpyAsync(dbase + off[i], src[i], len[i], cudaMemcpyHostToDevice, ctx->stream));
  for (size_t i = 0; i < n; i++) d_ptr[i] = dbase + off[i];
  return ZIPC_OK;
}

int upload_buffer(zipc_b200_ctx *ctx, const void *src, size_t len, const uint8_t **d) {
  ctx->epoch++;  // new input bytes: plans made over the old ones are void
  const size_t pre = (uintptr_t)src & 15;  // keep the host alignment so 16-byte paths stay aligned
  if (int st = ctx->d_in.reserve(pre + len + 64)) return st;
  uint8_t *p = ctx->d_in.as<uint8_t>() + pre;
  *d = p;
  return h2d(ctx, p, src, len);
}

static __global__ void make_crc_segs_kernel(const InflateTask *tasks, const InflateResult *res, uint32_t n, CrcSeg *segs) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  CrcSeg s;
  s.ptr = tasks[i].dst;
  s.len = res[i].status == ZIPC_OK ? res[i].out_len : 0;
  s.init = 0xFFFFFFFFu;
  s._pad = 0;
  segs[i] = s;
}
static __global__ void xor_ffffffff_kernel(uint32_t *v, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] ^= 0xFFFFFFFFu;
}
// one thread per zlib stream in device memory (byte loads: any offset)
static __global__ void zlib_frames_kernel(ZlibFrame *f, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ZlibFrame z = f[i];
  zlib_check_frame(z);
  f[i] = z;
}

// The results of both zlib_decompress calls from the frames and the decode of the streams whose header passed (status,
// dst_len and adler[i], the Adler-32 of the output).  A rejected stream gets its frame's status (found: CM on
// ZIPC_ERR_ZLIB_METHOD); a decoded one gets expect / found if it decoded, and ZIPC_ERR_CHECKSUM if they differ.
static void zlib_verdict(size_t n, const ZlibFrame *f, const uint32_t *adler, size_t *dst_len, uint32_t *expect, uint32_t *found,
                         int *status) {
  for (size_t i = 0; i < n; i++) {
    if (f[i].status != ZIPC_OK) {
      status[i] = (int)f[i].status;
      dst_len[i] = 0;
      if (f[i].status == ZIPC_ERR_ZLIB_METHOD && found) found[i] = f[i].method;
    } else if (status[i] == ZIPC_OK) {
      if (expect) expect[i] = f[i].expect;
      if (found) found[i] = adler[i];
      if (adler[i] != f[i].expect) status[i] = ZIPC_ERR_CHECKSUM;
    }
  }
}

// One warp per stream (inflate.cu), for the streams sel (ascending indices into the caller's arrays, which results are
// written at).  All pointers in d_src / d_dst are device addresses.
static int inflate_serial_core(zipc_b200_ctx *ctx, int ck, int adler_mode, const std::vector<uint32_t> &sel,
                               const std::vector<const uint8_t *> &d_src, const size_t *src_len, const std::vector<uint8_t *> &d_dst,
                               const std::vector<size_t> &cap, bool count_only, size_t *out_len, uint32_t *checksum, int *status,
                               uint32_t flags, const DownloadPlan *plan) {
  const size_t n = sel.size();
  if (!n) return ZIPC_OK;
  if (n > 0xFFFFFFF0ull) return ZIPC_ERR_INVALID_ARG;
  static const bool call_debug = env_u64("ZIPC_B200_CALL_DEBUG", 0) != 0;   // host-side time stamps of one call on stderr
  double tm[6] = {0, 0, 0, 0, 0, 0};
  if (call_debug) tm[0] = now_ms();
  const bool grouped = plan && plan->ngroups && !count_only;
  // longest streams first: the tail of the dynamic queue is made of short ones.  With a progressive download the groups
  // go in download order instead (smallest outputs first), so that the copies start early and never run dry.
  // (a radix sort of packed keys -- group, length, index: this runs while the GPU waits, 0.5 ms with std::sort for 10k streams)
  std::vector<uint32_t> order(sel);
  {
    bool fits = n <= 0xFFFFFFu;
    for (size_t j = 0; j < n && fits; j++) fits = src_len[sel[j]] < (1ull << 32);
    if (fits) {
      std::vector<uint64_t> key(n), tmp(n);
      for (size_t j = 0; j < n; j++) {
        const uint32_t i = sel[j];
        const uint64_t g = grouped ? plan->group_of[i] : 0u;                                          // < 256
        const uint64_t len = grouped ? (uint64_t)src_len[i] : 0xFFFFFFFFull - (uint64_t)src_len[i];   // ascending in a group, else longest first
        key[j] = (g << 56) | (len << 24) | (uint64_t)j;
      }
      // least significant digit first over bits 24..63 (the position in sel below them keeps equal keys in input order)
      for (int shift = 24; shift < 64; shift += 8) {
        if (shift == 56 && !grouped) break;
        size_t cnt[257] = {0};
        for (size_t i = 0; i < n; i++) cnt[((key[i] >> shift) & 0xFFu) + 1]++;
        for (int d = 0; d < 256; d++) cnt[d + 1] += cnt[d];
        for (size_t i = 0; i < n; i++) tmp[cnt[(key[i] >> shift) & 0xFFu]++] = key[i];
        key.swap(tmp);
      }
      for (size_t k = 0; k < n; k++) order[k] = sel[key[k] & 0xFFFFFFu];
    } else {
      if (grouped)
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
          return plan->group_of[a] != plan->group_of[b] ? plan->group_of[a] < plan->group_of[b] : src_len[a] < src_len[b]; });
      else
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return src_len[a] > src_len[b]; });
    }
  }
  if (call_debug) tm[1] = now_ms();
  if (int st = ctx->h_desc.reserve(n * sizeof(InflateTask))) return st;
  if (int st = ctx->d_desc.reserve(n * (sizeof(InflateTask) + sizeof(CrcSeg)))) return st;
  if (int st = ctx->d_res.reserve(n * (sizeof(InflateResult) + sizeof(uint32_t)) + 1024)) return st;
  if (int st = ctx->h_res.reserve(n * (sizeof(InflateResult) + sizeof(uint32_t)))) return st;
  InflateTask *ht = ctx->h_desc.as<InflateTask>();
  for (size_t k = 0; k < n; k++) {
    uint32_t i = order[k];
    ht[k].src = d_src[i]; ht[k].src_len = src_len[i];
    ht[k].dst = count_only ? nullptr : d_dst[i];
    ht[k].dst_cap = cap[i] == ZIPC_SIZE_UNKNOWN ? ~0ull : (uint64_t)cap[i];
    ht[k].flags = flags | (grouped && !plan->late.empty() ? (uint32_t)plan->late[i] << kInflatePartShift : 0u);
    ht[k].group = grouped ? plan->group_of[i] : 0u; ht[k].start_bit = 0; ht[k].stop_bit = ~0ull;
  }
  InflateTask *dt = ctx->d_desc.as<InflateTask>();
  CrcSeg *dsegs = reinterpret_cast<CrcSeg *>(dt + n);
  InflateResult *dr = ctx->d_res.as<InflateResult>();
  uint32_t *dck = reinterpret_cast<uint32_t *>(dr + n);
  ZB_CUDA(ctx, cudaMemcpyAsync(dt, ht, n * sizeof(InflateTask), cudaMemcpyHostToDevice, ctx->stream));
  if (call_debug) tm[2] = now_ms();
  const bool adler = !count_only && ck == ZIPC_CK_ADLER32;
  unsigned int *d_gcount = nullptr;
  if (grouped) {
    std::vector<unsigned int> cnt(plan->ngroups, 0u);
    for (uint32_t i : sel) cnt[plan->group_of[i]]++;
    d_gcount = reinterpret_cast<unsigned int *>(dck + n);  // behind the checksums (the buffer has 1 KiB to spare)
    if (!ctx->h_gflag) ZB_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_gflag), 256 * sizeof(uint32_t), cudaHostAllocMapped));
    if (!ctx->copy_stream) ZB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (uint32_t g = 0; g < plan->ngroups; g++) reinterpret_cast<volatile uint32_t *>(ctx->h_gflag)[g] = cnt[g] ? 0u : 1u;
    ZB_CUDA(ctx, cudaMemcpyAsync(d_gcount, cnt.data(), plan->ngroups * sizeof(unsigned int), cudaMemcpyHostToDevice, ctx->stream));
    ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));  // (cnt is pageable: the copy must be over before it goes away)
  }
  const bool late = grouped && !plan->late.empty() && ctx->upload_split_live;
  if (ctx->upload_split_live && !late) {  // nobody will wait for the late half inside the kernel: wait for it here
    ZB_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream));
    ctx->upload_split_live = false;
  }
  if (int st = inflate_launch(ctx, dt, (uint32_t)n, dr, count_only, adler ? adler_mode : -1, d_gcount, grouped ? ctx->h_gflag : nullptr,
                              late ? ctx->d_upflag : nullptr, ctx->upload_serial)) return st;
  bool crc = !count_only && ck == ZIPC_CK_CRC32;
  if (crc) {
    make_crc_segs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(dt, dr, (uint32_t)n, dsegs);
    ctx->launches++;
    if (int st = crc32_launch_segments(ctx, dsegs, (uint32_t)n, dck)) return st;
    xor_ffffffff_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(dck, (uint32_t)n);
    ctx->launches++;
  }
  InflateResult *hr = ctx->h_res.as<InflateResult>();
  uint32_t *hck = reinterpret_cast<uint32_t *>(hr + n);
  ZB_CUDA(ctx, cudaMemcpyAsync(hr, dr, n * sizeof(InflateResult) + (crc ? n * sizeof(uint32_t) : 0),
                               cudaMemcpyDeviceToHost, ctx->stream));
  if (call_debug) tm[3] = now_ms();
  if (grouped) {
    // copy every group's range out as soon as the kernel says the group is complete (or the stream is through: then all are)
    const volatile uint32_t *flag = reinterpret_cast<volatile uint32_t *>(ctx->h_gflag);
    bool through = false;
    for (uint32_t g = 0; g < plan->ngroups; g++) {
      while (!through && !flag[g]) {
        for (int spin = 0; spin < 2000 && !flag[g]; spin++) { }
        if (!flag[g] && cudaStreamQuery(ctx->stream) != cudaErrorNotReady) through = true;
      }
      if (plan->gbytes[g])
        ZB_CUDA(ctx, cudaMemcpyAsync(plan->dst + plan->goff[g], ctx->d_out.as<uint8_t>() + plan->goff[g], plan->gbytes[g],
                                     cudaMemcpyDeviceToHost, ctx->copy_stream));
    }
  }
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  if (late) { ZB_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream)); ctx->upload_split_live = false; }
  if (call_debug) tm[4] = now_ms();
  for (size_t k = 0; k < n; k++) {
    uint32_t i = order[k];
    status[i] = (int)hr[k].status;
    out_len[i] = (size_t)hr[k].out_len;
    if (checksum) checksum[i] = crc && hr[k].status == ZIPC_OK ? hck[k] : 0u;
  }
  if (adler && checksum)  // folded block by block inside the kernel (reference :682-690)
    for (size_t k = 0; k < n; k++) checksum[order[k]] = hr[k].status == ZIPC_OK ? hr[k]._pad : 0u;
  if (call_debug)
    std::fprintf(stderr, "[call] inflate of %zu streams: order %.3f, tasks %.3f, enqueue %.3f, wait %.3f, results %.3f ms\n", n, tm[1] - tm[0],
                 tm[2] - tm[1], tm[3] - tm[2], tm[4] - tm[3], now_ms() - tm[4]);
  return ZIPC_OK;
}

// ---- intra-stream parallel inflate of one large stream (no index): find block starts, decode the chunks speculatively into
// 16-bit symbols, check that the chunks chain up exactly, resolve.  *ok = false means "decode it serially": nothing found,
// a wrong guess, an error inside the stream (the serial decoder then reports the reference's exact status), or a chunk that
// expands more than its symbol buffer allows.  Reference: the serial core zipc_deflate.ml:593-616, 692-709.
// tuning knobs (read on every call, so that tests can vary them): compressed bytes per chunk; smallest stream that is tried
static uint64_t par_chunk_bytes() { return std::max<uint64_t>(4096, env_u64("ZIPC_B200_PAR_CHUNK", 8192)); }
static uint64_t par_min_bytes() { return env_u64("ZIPC_B200_PAR_MIN", 262144); }
// Which streams of a batch go through the many-warp decoder?  It takes a stream in a few host round trips and the decode of its
// longest block on one warp (~4 ms, then ~3 MB of compressed data per ms), a handful of streams at a time, while the one-warp decoder takes
// all streams at once but needs ~1 ms per 12 KB of a stream's compressed data (profiles/r02_lone_stream_probe.txt: 148 streams
// of 360 KiB took 816 ms one after the other and 30 ms side by side).  So: sort by size, and send the k largest streams to the
// many-warp decoder for the k that minimises  sum of their times + the one-warp kernel's time for the rest.
// ZIPC_B200_PAR_MIN, when set, is a plain threshold instead (tests force either path with it); 0 switches the path off.
static void par_select(size_t n, const size_t *src_len, std::vector<char> &take, size_t lanes) {
  take.assign(n, 0);
  const uint64_t base = par_min_bytes();
  if (base == 0) return;
  if (std::getenv("ZIPC_B200_PAR_MIN")) { for (size_t i = 0; i < n; i++) take[i] = src_len[i] >= base; return; }
  const uint64_t floor_bytes = 65536;   // (the block-start search wants a few 8 KiB chunks to work with)
  std::vector<uint32_t> big;
  double rest_bytes = 0;
  for (size_t i = 0; i < n; i++) { rest_bytes += (double)src_len[i]; if (src_len[i] >= floor_bytes && big.size() < 4096) big.push_back((uint32_t)i); }
  if (big.empty()) return;
  std::sort(big.begin(), big.end(), [&](uint32_t a, uint32_t b) { return src_len[a] != src_len[b] ? src_len[a] > src_len[b] : a < b; });
  const double one_warp_bytes_per_ms = 12e3, all_warps_bytes_per_ms = 33e6, many_warp_bytes_per_ms = 3e6, many_warp_fixed_ms = 4.5;
  auto one_warp_kernel_ms = [&](size_t k) {  // the k largest are gone: the largest stream left, or the throughput of the whole GPU
    const double largest = k < big.size() ? (double)src_len[big[k]] : (double)floor_bytes;
    return std::max(largest / one_warp_bytes_per_ms, rest_bytes / all_warps_bytes_per_ms);
  };
  // (`lanes` streams are decoded at a time, each lane a host thread with a sub-context of its own; the streams are dealt out
  // largest first to the least loaded lane, here as in inflate_core)
  double best = one_warp_kernel_ms(0);
  size_t best_k = 0;
  std::vector<double> load(std::max<size_t>(1, lanes), 0.0);
  double spent = 0;
  for (size_t k = 1; k <= big.size(); k++) {
    const double len = (double)src_len[big[k - 1]];
    double &l = *std::min_element(load.begin(), load.end());
    l += many_warp_fixed_ms + len / many_warp_bytes_per_ms;
    spent = std::max(spent, l);
    rest_bytes -= len;
    if (spent >= best) break;  // (it only grows)
    const double t = spent + (k == n ? 0.0 : one_warp_kernel_ms(k));
    if (t < best) { best = t; best_k = k; }
  }
  for (size_t k = 0; k < best_k; k++) take[big[k]] = 1;
}

// Lanes of the many-warp decoder: how many large streams are decoded at a time (host threads with a sub-context each).
// ZIPC_B200_PAR_LANES (default: by the cores this process can count on, 2 .. 12; 1 = one stream after the other).
static size_t par_lane_count() {
  static const size_t v = [] {
    int ndev = 1;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) ndev = 1;
    const uint64_t cores = std::max(1u, std::thread::hardware_concurrency());
    const uint64_t automatic = std::min<uint64_t>(12, std::max<uint64_t>(2, cores / (uint64_t)ndev));
    return (size_t)std::min<uint64_t>(std::max<uint64_t>(1, env_u64("ZIPC_B200_PAR_LANES", automatic)), 32);
  }();
  return v;
}
static zipc_b200_mctx *par_lanes(zipc_b200_ctx *ctx, size_t lanes) {
  if (!ctx->par_pool) {
    if (pipeline_create(ctx->device, (int)lanes, &ctx->par_pool) != ZIPC_OK) { ctx->par_pool = nullptr; return nullptr; }
  }
  return ctx->par_pool;
}

static bool par_debug() { static const bool v = env_u64("ZIPC_B200_PAR_DEBUG", 0) != 0; return v; }

static int par_speculate(zipc_b200_ctx *ctx, const uint8_t *d_src, size_t src_len, bool *ok, uint64_t *passes) {
  *ok = false;
  zipc_b200_ctx::ParPlan &plan = ctx->par_plan;
  if (plan.src == d_src && plan.src_len == src_len && plan.epoch == ctx->epoch && !plan.len.empty()) { *ok = true; return ZIPC_OK; }
  // The key goes with the chunks: a speculation that stops part way (a pass that accepts nothing, no room for the symbols of
  // a re-cut) returns with the chunks of its earlier passes in the plan, which must not pass for the previous stream's.
  plan.src = nullptr; plan.src_len = 0; plan.epoch = 0;
  plan.len.clear(); plan.spec_off.clear(); plan.blocks.clear(); plan.total = 0;
  const uint64_t cb = par_chunk_bytes();
  const uint32_t nch0 = (uint32_t)((src_len + cb - 1) / cb);
  if (nch0 < 4 || src_len > (1ull << 40)) return ZIPC_OK;
  // chunk tables: found starts, tasks, results, then the block lists of the chunks of a pass (reserved once their number is
  // known and the stream has passed the symbol check below: kSpecBlocks 64-bit lengths per chunk)
  const size_t tab = (size_t)nch0 * (sizeof(uint64_t) * 4 + sizeof(InflateTask) + sizeof(InflateResult)) + 256;
  if (int st = ctx->d_par.reserve(tab)) return st;
  if (int st = ctx->h_res.reserve(tab)) return st;
  uint64_t *d_found, *h_found, *d_blk;
  InflateTask *d_tasks;
  InflateResult *d_results, *h_results;
  const uint64_t *h_blk;   // per chunk: the output lengths of its non-empty blocks (the Adler-32 of a zlib stream is folded block by block)
  auto layout = [&] {      // (again after every reserve: it does not keep the buffer where it was)
    d_found = ctx->d_par.as<uint64_t>();
    h_found = ctx->h_res.as<uint64_t>();
    d_tasks = reinterpret_cast<InflateTask *>(ctx->d_par.as<uint64_t>() + 4 * (size_t)nch0);
    d_results = reinterpret_cast<InflateResult *>(d_tasks + nch0);
    h_results = reinterpret_cast<InflateResult *>(ctx->h_res.as<uint64_t>() + 4 * (size_t)nch0);
    d_blk = reinterpret_cast<uint64_t *>(d_results + nch0);
    h_blk = reinterpret_cast<const uint64_t *>(h_results + nch0);
  };
  layout();
  // Passes over what is left of the stream.  A pass: (1) block starts, (2) speculative decode of the chunks between them,
  // (3) the chunks must chain up exactly -- each one ends, at a block boundary, on the very bit where the next one was found
  // to start.  A found start that is an accident of the bits inside a block (rare) breaks the chain, and may have hidden the
  // true start behind it; the chunks before the break stand, and the next pass starts where they end, which IS a block boundary.
  uint64_t from_bit = 0;      // everything before this bit is covered by accepted chunks
  uint64_t spec_used = 0;     // symbols of d_spec taken by accepted chunks
  uint64_t spec_cap = 0;      // symbols d_spec holds (fixed by the first pass: later passes must not move the buffer)
  for (int pass = 0; pass < 16; pass++) {
    ++*passes;
    const double t_begin = par_debug() ? (cudaStreamSynchronize(ctx->stream), now_ms()) : 0;
    const uint64_t left_bits = 8ull * src_len - from_bit;
    const uint32_t nch = (uint32_t)std::min<uint64_t>(nch0, (left_bits + 8 * cb - 1) / (8 * cb));
    std::vector<uint64_t> start;
    start.push_back(from_bit);
    if (nch >= 2) {
      if (int st = inflate_find_starts(ctx, d_src, src_len, from_bit, cb, nch, d_found)) return st;
      ZB_CUDA(ctx, cudaMemcpyAsync(h_found, d_found, (size_t)nch * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
      ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
      for (uint32_t k = 1; k < nch; k++) if (h_found[k] != ~0ull && h_found[k] > start.back()) start.push_back(h_found[k]);
    }
    const double t_found = par_debug() ? now_ms() : 0;
    const uint32_t m = (uint32_t)start.size();
    if (pass == 0 && m < 2) return ZIPC_OK;   // no starts at all (stored / fixed blocks only): one warp it is
    // speculative decode: symbol buffers sized for a 24-fold expansion of every chunk
    std::vector<uint64_t> spec_off(m), capv(m);
    uint64_t need = spec_used;
    for (uint32_t k = 0; k < m; k++) {
      const uint64_t stop = k + 1 < m ? start[k + 1] : 8ull * src_len;
      const uint64_t bytes = (stop - start[k] + 7) / 8;
      capv[k] = (24 * bytes + 65536 + 7) & ~7ull;
      spec_off[k] = need;
      need += capv[k];
    }
    if (pass == 0) {
      spec_cap = need + need / 8 + (8u << 20);   // (room for the re-cut chunks of later passes)
      if (spec_cap > (6ull << 30)) return ZIPC_OK;  // 12 GiB of symbols: leave such streams to the serial path
      if (int st = ctx->d_spec.reserve(spec_cap * 2 + 64)) return st;
    } else if (need > spec_cap) {
      return ZIPC_OK;
    }
    if (int st = ctx->d_par.reserve(tab + (size_t)m * kSpecBlocks * sizeof(uint64_t))) return st;
    if (int st = ctx->h_res.reserve(tab + (size_t)m * kSpecBlocks * sizeof(uint64_t))) return st;
    layout();
    std::vector<InflateTask> tasks(m);
    for (uint32_t k = 0; k < m; k++) {
      InflateTask &t = tasks[k];
      t.src = d_src; t.src_len = src_len;
      t.dst = reinterpret_cast<uint8_t *>(ctx->d_spec.as<uint16_t>() + spec_off[k]);
      t.dst_cap = capv[k]; t.flags = 0; t.group = 0;
      t.start_bit = start[k]; t.stop_bit = k + 1 < m ? start[k + 1] : ~0ull;
    }
    ZB_CUDA(ctx, cudaMemcpyAsync(d_tasks, tasks.data(), m * sizeof(InflateTask), cudaMemcpyHostToDevice, ctx->stream));
    if (int st = inflate_launch_spec(ctx, d_tasks, m, d_results, d_blk)) return st;
    ZB_CUDA(ctx, cudaMemcpyAsync(h_results, d_results, m * sizeof(InflateResult), cudaMemcpyDeviceToHost, ctx->stream));
    ZB_CUDA(ctx, cudaMemcpyAsync(const_cast<uint64_t *>(h_blk), d_blk, (size_t)m * kSpecBlocks * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
    if (par_debug())
      std::fprintf(stderr, "[par] pass %d from bit %llu of %zu bytes: %u nominal chunks, %u block starts: find %.2f ms, speculative decode %.2f ms\n",
                   pass, (unsigned long long)from_bit, src_len, nch, m, t_found - t_begin, now_ms() - t_found);
    // the chain
    uint32_t used = 0;
    bool final_seen = false;
    for (uint32_t k = 0; k < m; k++) {
      const InflateResult &r = h_results[k];
      if (r.status != ZIPC_OK) break;   // (chunk 0 starts at a block boundary for sure: its failure is the stream's)
      used = k + 1;
      if (r.final_seen) { final_seen = true; break; }  // the stream ends here (bytes after the final block are ignored, as in the reference)
      if (k + 1 == m || r.end_bit != start[k + 1]) {
        if (par_debug())
          std::fprintf(stderr, "[par] chunk %u of %u ends at bit %llu, the next start was found at %llu: re-cutting from there\n", k, m,
                       (unsigned long long)r.end_bit, (unsigned long long)(k + 1 < m ? start[k + 1] : 0));
        break;
      }
    }
    if (used == 0) return ZIPC_OK;     // corrupt, or larger than 24 times its compressed size: the serial decoder reports it
    for (uint32_t k = 0; k < used; k++) {
      plan.spec_off.push_back(spec_off[k]); plan.len.push_back(h_results[k].out_len); plan.total += h_results[k].out_len;
      plan.blocks.insert(plan.blocks.end(), h_blk + (size_t)k * kSpecBlocks, h_blk + (size_t)k * kSpecBlocks + std::min<uint32_t>(h_results[k]._pad2, kSpecBlocks));
    }
    if (final_seen) {
      plan.src = d_src; plan.src_len = src_len; plan.epoch = ctx->epoch;
      *ok = true;
      return ZIPC_OK;
    }
    from_bit = h_results[used - 1].end_bit;
    spec_used = spec_off[used - 1] + capv[used - 1];
    if (from_bit >= 8ull * src_len) break;   // ran off the end without a final block
  }
  plan.len.clear(); plan.spec_off.clear(); plan.blocks.clear(); plan.total = 0;
  return ZIPC_OK;
}

static int par_resolve(zipc_b200_ctx *ctx, uint8_t *d_dst, bool *ok, uint64_t *chunks) {
  const zipc_b200_ctx::ParPlan &plan = ctx->par_plan;
  const uint32_t m = (uint32_t)plan.len.size();
  *chunks += m;
  *ok = false;
  const double t_begin = par_debug() ? (cudaStreamSynchronize(ctx->stream), now_ms()) : 0;
  std::vector<uint64_t> tab(3 * (size_t)m);
  uint64_t off = 0;
  for (uint32_t k = 0; k < m; k++) { tab[k] = plan.spec_off[k]; tab[m + k] = off; tab[2 * m + k] = plan.len[k]; off += plan.len[k]; }
  if (int st = ctx->d_win.reserve((size_t)m * 32768 * 2 * 2 + 64)) return st;  // two arrays of 16-bit window maps
  uint64_t *d_tab = ctx->d_par.as<uint64_t>();  // (the chunk tables of the speculation are dead)
  if (int st = ctx->d_small.reserve(256)) return st;
  uint32_t *d_bad = ctx->d_small.as<uint32_t>() + 48;
  ZB_CUDA(ctx, cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  ZB_CUDA(ctx, cudaMemsetAsync(d_bad, 0, sizeof(uint32_t), ctx->stream));
  if (int st = inflate_resolve(ctx, ctx->d_spec.as<uint16_t>(), d_tab, d_tab + m, d_tab + 2 * m, m, ctx->d_win.as<uint8_t>(), d_dst, d_bad)) return st;
  uint32_t bad = 1;
  ZB_CUDA(ctx, cudaMemcpyAsync(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost, ctx->stream));
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  *ok = bad == 0;
  if (par_debug()) std::fprintf(stderr, "[par] resolve of %u chunks (%llu bytes): %.2f ms\n", m, (unsigned long long)plan.total, now_ms() - t_begin);
  return ZIPC_OK;
}

// Core of every inflate entry point.  All pointers in d_src / d_dst are device addresses.  subset (null: all n streams) lists,
// in ascending order, the streams to decode; the results of the others are left as they are.
// cap[i] == ZIPC_SIZE_UNKNOWN is only accepted in a count-only pass (the callers resolve sizes first).
// Large streams are decoded in parallel inside the stream where that works out; everything else (and every stream whose
// parallel decoding does not check out) goes to the warp-per-stream decoder.
int inflate_core(zipc_b200_ctx *ctx, int ck, int adler_mode, size_t n, const std::vector<const uint8_t *> &d_src,
                 const size_t *src_len, const std::vector<uint8_t *> &d_dst, const std::vector<size_t> &cap,
                 bool count_only, size_t *out_len, uint32_t *checksum, int *status, uint32_t flags, const DownloadPlan *plan,
                 const std::vector<uint32_t> *subset) {
  std::vector<uint32_t> rest;  // the selected streams the many-warp decoder has not done
  if (subset) rest = *subset;
  else { rest.resize(n); std::iota(rest.begin(), rest.end(), 0u); }
  std::vector<char> done(n, 0);
  if (flags == 0 && par_min_bytes() != 0 && !(plan && plan->ngroups)) {
    const size_t lanes = ctx->is_sub ? 1 : par_lane_count();
    std::vector<size_t> len(rest.size());
    for (size_t j = 0; j < rest.size(); j++) len[j] = src_len[rest[j]];
    std::vector<char> take;
    par_select(rest.size(), len.data(), take, lanes);
    std::vector<uint32_t> sel;
    for (size_t j = 0; j < rest.size(); j++) if (take[j]) sel.push_back(rest[j]);
    // one stream through the many-warp decoder, on context c (ctx itself, or one of its lanes)
    auto one = [&](zipc_b200_ctx *c, uint32_t i, zipc_b200_ctx::ParCounts &count) -> int {
      bool ok = false;
      if (int st = par_speculate(c, d_src[i], src_len[i], &ok, &count.passes)) {
        if (st != ZIPC_ERR_NOMEM) return st;
        ok = false;  // no room for this stream's symbols (24 x its compressed size): the one-warp decoder needs none
      }
      const uint64_t total = c->par_plan.total;
      if (ok && cap[i] != ZIPC_SIZE_UNKNOWN && total > cap[i]) ok = false;  // the serial decoder reports the exact error
      if (ok && !count_only) {
        if (int st = par_resolve(c, d_dst[i], &ok, &count.chunks)) { if (st != ZIPC_ERR_NOMEM) return st; ok = false; }
        if (ok && checksum) {
          checksum[i] = 0;
          if (ck == ZIPC_CK_CRC32) {
            // (a 4-byte copy into the caller's pageable array would hold up every lane)
            if (int st = crc32_to_host_word(c, d_dst[i], total)) return st;
            ZB_CUDA(c, stream_sync(c, c->stream));
            checksum[i] = host_word_crc32(c);
          } else if (ck == ZIPC_CK_ADLER32) {
            // folded block by block, each block on its own 5552-byte grid with the state re-packed in between, as the reference
            // does while it decodes (zipc_deflate.ml:682-690): the chunks reported the lengths of their blocks
            const uint8_t *base = d_dst[i];
            const uint32_t nb = (uint32_t)c->par_plan.blocks.size();
            uint64_t sum = 0;
            for (uint64_t b : c->par_plan.blocks) sum += b;
            // every byte of an accepted chunk lies in one of its non-empty blocks, whose lengths are 64-bit (one block may
            // output 4 GiB or more), so the lists add up to the output; if they ever did not, the one-warp decoder folds it
            if (sum != total) ok = false;
            else if (int st = adler32_blocked(c, &base, &nb, c->par_plan.blocks.data(), 1, adler_mode, &checksum[i])) return st;
          }
        }
      }
      if (ok) { done[i] = 1; status[i] = ZIPC_OK; out_len[i] = (size_t)total; count.streams++; }
      else count.fallbacks++;
      return ZIPC_OK;
    };
    zipc_b200_mctx *pool = sel.size() >= 2 && lanes >= 2 ? par_lanes(ctx, lanes) : nullptr;
    if (!pool) {
      for (uint32_t i : sel) if (int st = one(ctx, i, ctx->par_counts)) return st;
    } else {
      // Several streams at a time: lane k is a host thread with a sub-context (stream, scratch arenas) of its own.  The streams
      // are dealt out largest first, each to the lane with the least compressed bytes so far (the same deal in the sizing pass and
      // in the real pass of a call without sizes).  The lanes' streams start behind everything queued on ctx's stream -- the
      // upload -- and every lane has waited for its own work when its thread ends.
      std::vector<uint32_t> order(sel);
      std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return src_len[a] > src_len[b]; });
      // every lane keeps the 16-bit symbols of its stream (room for a 24-fold expansion) and two window maps per chunk: as many
      // lanes as fit half of the free device memory with the largest streams on them
      size_t L = std::min(lanes, sel.size());
      {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); free_b = 8ull << 30; }
        auto lane_bytes = [&](uint32_t i) { return 64.0 * (double)src_len[i] + (64u << 20); };
        double need = 0;
        size_t fit = 0;
        while (fit < L && need + lane_bytes(order[fit]) <= 0.5 * (double)free_b) need += lane_bytes(order[fit++]);
        L = std::max<size_t>(1, fit);
      }
      std::vector<std::vector<uint32_t>> mine(L);
      std::vector<uint64_t> load(L, 0);
      for (uint32_t i : order) {
        const size_t k = (size_t)(std::min_element(load.begin(), load.end()) - load.begin());
        mine[k].push_back(i);
        load[k] += src_len[i] + (1u << 20);
      }
      if (ctx->upload_split_live) { ZB_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream)); ctx->upload_split_live = false; }
      if (!ctx->ev_lanes) ZB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_lanes, cudaEventDisableTiming));
      ZB_CUDA(ctx, cudaEventRecord(ctx->ev_lanes, ctx->stream));
      double sel_bytes = 0;
      for (uint32_t i : sel) sel_bytes += (double)src_len[i];
      const double active_bytes = std::max(1.0, sel_bytes * (double)L / (double)sel.size());  // (L of the sel.size() streams at a time)
      std::vector<int> rc(L, ZIPC_OK);
      std::vector<zipc_b200_ctx::ParCounts> counts(L);
      std::vector<std::thread> th;
      auto lane = [&](size_t k) {
        zipc_b200_ctx *c = zipc_b200_mctx_ctx(pool, (int)k);
        cudaSetDevice(ctx->device);
        c->epoch = ctx->epoch;  // (the input's epoch: a plan cached in the sizing pass of this call serves its real pass, and no other call's)
        if (cudaError_t e = cudaStreamWaitEvent(c->stream, ctx->ev_lanes, 0)) { rc[k] = set_cuda_error(c, e, "cudaStreamWaitEvent(lane)"); return; }
        for (uint32_t i : mine[k]) {
          // this stream's share of the SMs for its speculative decode (a CTA of that kernel owns its SM): by its size among the
          // streams that are under way at the same time
          c->sm_share = (uint32_t)std::min<double>(ctx->sm_count, std::max(2.0, ctx->sm_count * (double)src_len[i] / active_bytes));
          if ((rc[k] = one(c, i, counts[k])) != ZIPC_OK) return;
        }
      };
      for (size_t k = 1; k < L; k++) th.emplace_back(lane, k);
      lane(0);
      for (auto &t : th) t.join();
      for (size_t k = 0; k < L; k++) {
        ctx->par_counts.streams += counts[k].streams; ctx->par_counts.fallbacks += counts[k].fallbacks;
        ctx->par_counts.passes += counts[k].passes; ctx->par_counts.chunks += counts[k].chunks;
        if (rc[k]) { ctx->last_error = zipc_b200_last_error(zipc_b200_mctx_ctx(pool, (int)k)); return rc[k]; }
      }
    }
    rest.erase(std::remove_if(rest.begin(), rest.end(), [&](uint32_t i) { return done[i] != 0; }), rest.end());
  }
  return inflate_serial_core(ctx, ck, adler_mode, rest, d_src, src_len, d_dst, cap, count_only, out_len, checksum, status, flags, plan);
}

// ---- progressive download ---------------------------------------------------------------------------------------------------
static constexpr uint32_t kDownloadGroups = 32;

bool progressive_ok(zipc_b200_ctx *ctx, size_t n, const size_t *cap, const size_t *src_len, const char *grouped, void *dst, size_t dst_cap) {
  if (!dst || ctx->is_sub) return false;
  size_t sum = 0, ng = 0;
  for (size_t i = 0; i < n; i++) {
    if (cap[i] == ZIPC_SIZE_UNKNOWN) return false;
    sum += align_up(cap[i], 16);
    if (grouped[i]) { ng++; if (par_min_bytes() && src_len[i] >= par_min_bytes()) return false; }  // (large streams: decoded in parallel)
  }
  return ng >= 1024 && sum >= (64ull << 20) && dst_cap >= sum && is_pinned(dst);
}

int plan_arena(zipc_b200_ctx *ctx, size_t n, const size_t *cap, const void *const *src, const size_t *src_len, const char *grouped,
               const UploadSplit &split, void *dst, size_t dst_cap, std::vector<size_t> &off, size_t &total, DownloadPlan &plan) {
  off.assign(n, 0);
  plan = DownloadPlan{};
  if (!progressive_ok(ctx, n, cap, src_len, grouped, dst, dst_cap)) {
    size_t t = 0;
    for (size_t i = 0; i < n; i++) { off[i] = t; t += align_up(cap[i], 16); }
    total = t;
    return ZIPC_OK;
  }
  // grouped streams: in the order in which the parts of the upload arrive, then by ascending output size; equal counts per group
  std::vector<char> late(n);
  for (size_t i = 0; i < n; i++) late[i] = src_len[i] && split.late(src[i]);
  std::vector<uint32_t> idx;
  for (size_t i = 0; i < n; i++) if (grouped[i]) idx.push_back((uint32_t)i);
  std::sort(idx.begin(), idx.end(), [&](uint32_t a, uint32_t b) {
    return late[a] != late[b] ? late[a] < late[b] : cap[a] != cap[b] ? cap[a] < cap[b] : a < b; });
  const uint32_t G = kDownloadGroups;
  plan.ngroups = G; plan.group_of.assign(n, 0); plan.goff.assign(G, 0); plan.gbytes.assign(G, 0); plan.dst = static_cast<uint8_t *>(dst);
  if (split.cut) plan.late = late;
  size_t t = 0;
  for (size_t r = 0; r < idx.size(); r++) {
    const uint32_t i = idx[r], g = (uint32_t)(r * G / idx.size());
    if (plan.gbytes[g] == 0) plan.goff[g] = t;
    plan.group_of[i] = g;
    off[i] = t;
    t += align_up(cap[i], 16);
    plan.gbytes[g] = t - plan.goff[g];
  }
  plan.tail_off = t;
  for (size_t i = 0; i < n; i++) if (!grouped[i]) { off[i] = t; t += align_up(cap[i], 16); }
  plan.tail_bytes = t - plan.tail_off;
  total = t;
  return ZIPC_OK;
}

int finish_to_host(zipc_b200_ctx *ctx, const std::vector<size_t> &off, size_t total, void *dst, size_t dst_cap, size_t *dst_off,
                   size_t *dst_need, const DownloadPlan *plan) {
  ctx->last_total = total;
  if (dst_off) std::copy(off.begin(), off.end(), dst_off);
  if (dst_need) *dst_need = total;
  if (!dst || dst_cap < total) {
    ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
    return ZIPC_ERR_DST_TOO_SMALL;
  }
  if (!plan || !plan->ngroups) return d2h(ctx, dst, ctx->d_out.p, total);
  // the groups are on their way (inflate_core): copy the rest and wait for all of it
  if (plan->tail_bytes)
    ZB_CUDA(ctx, cudaMemcpyAsync(plan->dst + plan->tail_off, ctx->d_out.as<uint8_t>() + plan->tail_off, plan->tail_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  ZB_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  return ZIPC_OK;
}

void pipe_mark(const zipc_b200_ctx *ctx, const char *stage) {
  static const bool on = env_u64("ZIPC_B200_PIPE_DEBUG", 0) != 0;
  if (on) std::fprintf(stderr, "[pipe] %2zu %-12s %10.3f\n", ctx->gate_ticket, stage, now_ms());
}

// The pipelined sub-contexts of ctx, or null if this batch should run as one piece: it is small, there is no caller arena
// to copy into while kernels run, or ctx is a sub-context itself.  ZIPC_B200_PIPE = most groups (default: by the cores per visible GPU, 4 .. 24; 0 or 1 = off).
zipc_b200_mctx *pipeline_for(zipc_b200_ctx *ctx, size_t n, const size_t *len, const void *dst) {
  if (ctx->is_sub || !dst || n < 1024) return nullptr;
  // Every group is a host thread.  A box runs one process per GPU, so the thread budget of this process is its share of the
  // cores: 24 groups where there are cores to spare (measured on C4, one GPU: 11.8 / 12.6 / 13.0 GB/s end to end with 8 / 16 /
  // 24), fewer when eight processes share 32 cores (N = 8: 51.9 GB/s in all with 8 groups each, 37.1 with 24).
  static const uint64_t depth = [] {
    int ndev = 1;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) ndev = 1;
    const uint64_t cores = std::max(1u, std::thread::hardware_concurrency());
    const uint64_t automatic = std::min<uint64_t>(24, std::max<uint64_t>(4, 2 * cores / (uint64_t)ndev));
    return std::min<uint64_t>(env_u64("ZIPC_B200_PIPE", automatic), 64);
  }();
  if (depth < 2) return nullptr;
  uint64_t total = 0;
  for (size_t i = 0; i < n; i++) total += len[i];
  if (total < (64ull << 20)) return nullptr;
  if (!ctx->pipe && pipeline_create(ctx->device, (int)depth, &ctx->pipe) != ZIPC_OK) { ctx->pipe = nullptr; return nullptr; }
  return ctx->pipe;
}

}  // namespace zb

using namespace zb;

extern "C" {

// The host-side decision of the inflate entry points, for tests and capacity planning (no device needed).
void zipc_b200_inflate_plan(size_t n, const size_t *src_len, size_t lanes, char *many_warp) {
  if (!many_warp || (!src_len && n)) return;
  std::vector<char> take;
  par_select(n, src_len, take, lanes ? lanes : 12);
  for (size_t i = 0; i < n; i++) many_warp[i] = take[i];
}

int zipc_b200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int zipc_b200_ctx_create(int device, zipc_b200_ctx **out) {
  if (!out) return ZIPC_ERR_INVALID_ARG;
  *out = nullptr;
  int n = zipc_b200_device_count();
  if (n <= 0) return ZIPC_ERR_NO_DEVICE;
  if (device < 0 || device >= n) return ZIPC_ERR_INVALID_ARG;
  zipc_b200_ctx *ctx = new (std::nothrow) zipc_b200_ctx();
  if (!ctx) return ZIPC_ERR_NOMEM;
  ctx->device = device;
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  cudaDeviceProp prop;
  if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { int st = set_cuda_error(ctx, e, "ctx_create"); delete ctx; return st; }
  ctx->sm_count = prop.multiProcessorCount;
  if (int st = crc_tables_upload(ctx)) { zipc_b200_ctx_destroy(ctx); return st; }
  *out = ctx;
  return ZIPC_OK;
}

void zipc_b200_ctx_destroy(zipc_b200_ctx *ctx) {
  if (!ctx) return;
  if (ctx->pipe) { zipc_b200_mctx_destroy(ctx->pipe); ctx->pipe = nullptr; }
  if (ctx->par_pool) { zipc_b200_mctx_destroy(ctx->par_pool); ctx->par_pool = nullptr; }
  cudaSetDevice(ctx->device);
  if (ctx->ev_lanes) cudaEventDestroy(ctx->ev_lanes);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  ctx->d_in.release(); ctx->d_out.release(); ctx->d_desc.release(); ctx->d_res.release();
  ctx->d_scratch.release(); ctx->d_scratch2.release(); ctx->d_small.release(); ctx->d_slots.release(); ctx->d_desc2.release(); ctx->d_blk.release();
  ctx->d_par.release(); ctx->d_spec.release(); ctx->d_win.release(); ctx->d_adler.release(); ctx->d_adler_chain.release();
  ctx->h_stage.release(); ctx->h_res.release(); ctx->h_desc.release();
  if (ctx->d_crc_tabs) cudaFree(ctx->d_crc_tabs);
  if (ctx->ev0) { cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1); }
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->upload_stream) cudaStreamDestroy(ctx->upload_stream);
  if (ctx->hi_stream) cudaStreamDestroy(ctx->hi_stream);
  if (ctx->d_upflag) cudaFree(ctx->d_upflag);
  if (ctx->ev_half) cudaEventDestroy(ctx->ev_half);
  for (cudaEvent_t e : ctx->ev_stage) if (e) cudaEventDestroy(e);
  if (ctx->ev_block) cudaEventDestroy(ctx->ev_block);
  if (ctx->h_gflag) cudaFreeHost(ctx->h_gflag);
  if (ctx->h_word) cudaFreeHost(ctx->h_word);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char *zipc_b200_last_error(const zipc_b200_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }
void *zipc_b200_ctx_stream(zipc_b200_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
uint64_t zipc_b200_ctx_launches(const zipc_b200_ctx *ctx) { return ctx ? ctx->launches + (ctx->par_pool ? pipeline_launches(ctx->par_pool) : 0) : 0; }
uint64_t zipc_b200_ctx_counter(const zipc_b200_ctx *ctx, int which) {
  if (!ctx) return 0;
  const zipc_b200_ctx::ParCounts &p = ctx->par_counts;
  return which == 0 ? ctx->launches : which == 1 ? p.streams : which == 2 ? p.fallbacks : which == 3 ? p.passes : which == 4 ? p.chunks : 0;
}
void zipc_b200_ctx_profile(zipc_b200_ctx *ctx, int enable) {
  if (!ctx) return;
  DeviceGuard g(ctx->device);
  if (enable && !ctx->ev0) { cudaEventCreate(&ctx->ev0); cudaEventCreate(&ctx->ev1); }
  ctx->profile = enable != 0;
  ctx->ev_valid = false;
}
float zipc_b200_ctx_kernel_ms(zipc_b200_ctx *ctx) {
  if (!ctx || !ctx->ev_valid) return -1.0f;
  DeviceGuard g(ctx->device);
  float ms = -1.0f;
  if (cudaEventSynchronize(ctx->ev1) != cudaSuccess || cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) != cudaSuccess) {
    cudaGetLastError();
    return -1.0f;
  }
  return ms;
}

int zipc_b200_host_alloc(size_t bytes, void **ptr) {
  if (!ptr) return ZIPC_ERR_INVALID_ARG;
  if (cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); *ptr = nullptr; return ZIPC_ERR_NOMEM; }
  return ZIPC_OK;
}
void zipc_b200_host_free(void *ptr) { if (ptr) cudaFreeHost(ptr); }

int zipc_b200_dev_alloc(zipc_b200_ctx *ctx, size_t bytes, void **dptr) {
  if (!ctx || !dptr) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  ZB_CUDA(ctx, cudaMalloc(dptr, bytes ? bytes : 1));
  return ZIPC_OK;
}
void zipc_b200_dev_free(zipc_b200_ctx *ctx, void *dptr) {
  if (!ctx || !dptr) return;
  DeviceGuard g(ctx->device);
  cudaFree(dptr);
}
int zipc_b200_memcpy_h2d(zipc_b200_ctx *ctx, void *dptr, const void *src, size_t bytes) {
  if (!ctx) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  if (int st = h2d(ctx, dptr, src, bytes)) return st;
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  return ZIPC_OK;
}
int zipc_b200_memcpy_d2h(zipc_b200_ctx *ctx, void *dst, const void *dptr, size_t bytes) {
  if (!ctx) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  return d2h(ctx, dst, dptr, bytes);
}
int zipc_b200_sync(zipc_b200_ctx *ctx) {
  if (!ctx) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  return ZIPC_OK;
}

// ---- checksums -------------------------------------------------------------------------------------
int zipc_b200_crc32_dev_async(zipc_b200_ctx *ctx, const void *d_src, size_t len, uint32_t *d_crc) {
  if (!ctx || !d_crc || (!d_src && len)) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  return crc32_launch_buffer(ctx, static_cast<const uint8_t *>(d_src), len, d_crc);
}

int zipc_b200_crc32_dev(zipc_b200_ctx *ctx, const void *d_src, size_t len, uint32_t *crc) {
  if (!ctx || !crc || (!d_src && len)) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  if (int st = crc32_to_host_word(ctx, static_cast<const uint8_t *>(d_src), len)) return st;
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  *crc = host_word_crc32(ctx);
  return ZIPC_OK;
}

int zipc_b200_crc32(zipc_b200_ctx *ctx, const void *src, size_t len, uint32_t *crc) {
  if (!ctx || !crc || (!src && len)) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  const uint8_t *d;
  if (int st = upload_buffer(ctx, src, len, &d)) return st;
  return zipc_b200_crc32_dev(ctx, d, len, crc);
}

int zipc_b200_adler32_dev(zipc_b200_ctx *ctx, const void *d_src, size_t len, int mode, uint32_t *adler) {
  if (!ctx || !adler || (!d_src && len) || (mode != ZIPC_ADLER_REF_COMPAT && mode != ZIPC_ADLER_RFC1950))
    return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  return adler32_launch_buffer(ctx, static_cast<const uint8_t *>(d_src), len, mode, adler);
}

int zipc_b200_adler32(zipc_b200_ctx *ctx, const void *src, size_t len, int mode, uint32_t *adler) {
  if (!ctx || !adler || (!src && len)) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  const uint8_t *d;
  if (int st = upload_buffer(ctx, src, len, &d)) return st;
  return zipc_b200_adler32_dev(ctx, d, len, mode, adler);
}

int zipc_b200_crc32_batch(zipc_b200_ctx *ctx, size_t n, const void *const *src, const size_t *len, uint32_t *crc) {
  if (!ctx || (n && (!src || !len || !crc))) return ZIPC_ERR_INVALID_ARG;
  if (!n) return ZIPC_OK;
  DeviceGuard g(ctx->device);
  std::vector<const uint8_t *> dp;
  if (int st = upload_ranges(ctx, n, src, len, dp)) return st;
  if (int st = ctx->h_desc.reserve(n * sizeof(CrcSeg))) return st;
  if (int st = ctx->d_desc.reserve(n * sizeof(CrcSeg))) return st;
  if (int st = ctx->d_res.reserve(n * sizeof(uint32_t))) return st;
  CrcSeg *hs = ctx->h_desc.as<CrcSeg>();
  for (size_t i = 0; i < n; i++) hs[i] = crc_seg(dp[i], len[i]);
  ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_desc.p, hs, n * sizeof(CrcSeg), cudaMemcpyHostToDevice, ctx->stream));
  if (int st = crc32_launch_segments(ctx, ctx->d_desc.as<CrcSeg>(), (uint32_t)n, ctx->d_res.as<uint32_t>())) return st;
  ZB_CUDA(ctx, cudaMemcpyAsync(crc, ctx->d_res.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  for (size_t i = 0; i < n; i++) crc[i] ^= 0xFFFFFFFFu;
  return ZIPC_OK;
}

// ---- inflate ---------------------------------------------------------------------------------------
int zipc_b200_inflate_batch(zipc_b200_ctx *ctx, int ck, int adler_mode, size_t n, const void *const *src,
                            const size_t *src_len, const size_t *max_out, void *dst, size_t dst_cap,
                            size_t *dst_need, size_t *dst_off, size_t *dst_len, uint32_t *checksum, int *status) {
  if (!ctx || ck < 0 || ck > 2 || (n && (!src || !src_len || !dst_off || !dst_len || !status)))
    return ZIPC_ERR_INVALID_ARG;
  if (dst_need) *dst_need = 0;
  if (!n) return ZIPC_OK;
  DeviceGuard g(ctx->device);
  // (Not cut into groups on sub-contexts like zipc_b200_deflate_batch: a group's kernel lasts as long as its largest member takes on one warp
  // (~14 ms for 256 KiB), whatever the group's size, so no download can start earlier than that and groups gain nothing:
  // measured 26.5 GB/s in 6 groups against 28.0 GB/s in one piece.  What overlaps instead is the download: plan_arena.)
  std::vector<size_t> cap(n);
  bool any_unknown = false;
  for (size_t i = 0; i < n; i++) { cap[i] = max_out ? max_out[i] : ZIPC_SIZE_UNKNOWN; any_unknown |= cap[i] == ZIPC_SIZE_UNKNOWN; }
  const std::vector<char> all(n, 1);
  UploadSplit split;
  split.want = !any_unknown && progressive_ok(ctx, n, cap.data(), src_len, all.data(), dst, dst_cap);
  std::vector<const uint8_t *> d_src;
  if (int st = upload_ranges(ctx, n, src, src_len, d_src, &split)) return st;
  // resolve unknown output sizes with a count-only pass (no bytes are written)
  std::vector<uint8_t *> d_dst(n, nullptr);
  std::vector<int> cs;
  std::vector<char> was_unknown(n, 0);
  if (any_unknown) {
    std::vector<size_t> cl(n);
    cs.assign(n, ZIPC_OK);
    if (int st = inflate_core(ctx, ZIPC_CK_NONE, adler_mode, n, d_src, src_len, d_dst, cap, true, cl.data(), nullptr, cs.data()))
      return st;
    for (size_t i = 0; i < n; i++)
      if (cap[i] == ZIPC_SIZE_UNKNOWN) { was_unknown[i] = 1; cap[i] = cs[i] == ZIPC_OK ? cl[i] : 0; }
  }
  std::vector<size_t> off;
  size_t total = 0;
  DownloadPlan plan;
  if (int st = plan_arena(ctx, n, cap.data(), src, src_len, all.data(), split, dst, dst_cap, off, total, plan)) return st;
  if (int st = ctx->d_out.reserve(total + 64)) return st;
  d_dst = slot_addrs(ctx->d_out.as<uint8_t>(), off.data(), n);
  if (int st = inflate_core(ctx, ck, adler_mode, n, d_src, src_len, d_dst, cap, false, dst_len, checksum, status, 0, &plan)) {
    if (plan.ngroups && ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);  // no copy into the caller's arena outlives the call
    return st;
  }
  // a stream of unknown size that failed while being sized keeps that (uncapped) verdict
  for (size_t i = 0; i < n; i++)
    if (was_unknown[i] && cs[i] != ZIPC_OK) { status[i] = cs[i]; dst_len[i] = 0; if (checksum) checksum[i] = 0; }
  return finish_to_host(ctx, off, total, dst, dst_cap, dst_off, dst_need, &plan);
}

int zipc_b200_fetch(zipc_b200_ctx *ctx, void *dst, size_t dst_cap) {
  if (!ctx || !dst) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  return finish_to_host(ctx, {}, ctx->last_total, dst, dst_cap, nullptr, nullptr);
}

int zipc_b200_inflate_batch_dev(zipc_b200_ctx *ctx, int ck, int adler_mode, size_t n, const void *d_src_v,
                                const size_t *src_off, const size_t *src_len, void *d_dst_v, const size_t *dst_off,
                                const size_t *max_out, size_t *dst_len, uint32_t *checksum, int *status) {
  if (!ctx || ck < 0 || ck > 2 || (n && (!d_src_v || !src_off || !src_len || !d_dst_v || !dst_off || !max_out || !dst_len || !status)))
    return ZIPC_ERR_INVALID_ARG;
  if (!n) return ZIPC_OK;
  DeviceGuard g(ctx->device);
  ctx->epoch++;  // the caller's device bytes may have changed since the last call
  for (size_t i = 0; i < n; i++) if (max_out[i] == ZIPC_SIZE_UNKNOWN) return ZIPC_ERR_INVALID_ARG;
  return inflate_core(ctx, ck, adler_mode, n, slot_addrs(static_cast<const uint8_t *>(d_src_v), src_off, n), src_len,
                      slot_addrs(static_cast<uint8_t *>(d_dst_v), dst_off, n), std::vector<size_t>(max_out, max_out + n), false,
                      dst_len, checksum, status);
}

int zipc_b200_zlib_decompress_batch(zipc_b200_ctx *ctx, int adler_mode, size_t n, const void *const *src,
                                    const size_t *src_len, const size_t *max_out, void *dst, size_t dst_cap,
                                    size_t *dst_need, size_t *dst_off, size_t *dst_len, uint32_t *expect,
                                    uint32_t *found, int *status) {
  if (!ctx || (n && (!src || !src_len || !dst_off || !dst_len || !status))) return ZIPC_ERR_INVALID_ARG;
  if (dst_need) *dst_need = 0;
  if (!n) return ZIPC_OK;
  // header checks in the reference's order (zipc_deflate.ml:722-731); bad streams become empty tasks
  std::vector<ZlibFrame> f(n);
  std::vector<const void *> body(n);
  std::vector<size_t> blen(n, 0), mo(n, 0);
  for (size_t i = 0; i < n; i++) {
    const uint8_t *s = static_cast<const uint8_t *>(src[i]);
    if (src_len[i] && !s) return ZIPC_ERR_INVALID_ARG;
    f[i] = ZlibFrame{s, src_len[i], 0, 0, 0, 0};
    zlib_check_frame(f[i]);
    body[i] = s;
    if (f[i].status != ZIPC_OK) continue;
    body[i] = s + 2;
    blen[i] = src_len[i] - 4;  // as the reference: two bytes into the trailer (zipc_deflate.ml:732)
    mo[i] = max_out ? max_out[i] : ZIPC_SIZE_UNKNOWN;
  }
  std::vector<uint32_t> ad(n);
  int rc = zipc_b200_inflate_batch(ctx, ZIPC_CK_ADLER32, adler_mode, n, body.data(), blen.data(), mo.data(), dst, dst_cap,
                                   dst_need, dst_off, dst_len, ad.data(), status);
  if (rc != ZIPC_OK && rc != ZIPC_ERR_DST_TOO_SMALL) return rc;
  zlib_verdict(n, f.data(), ad.data(), dst_len, expect, found, status);
  return rc;
}

int zipc_b200_zlib_decompress_batch_dev(zipc_b200_ctx *ctx, int adler_mode, size_t n, const void *d_src_v, const size_t *src_off,
                                        const size_t *src_len, void *d_dst_v, const size_t *dst_off, const size_t *max_out,
                                        size_t *dst_len, uint32_t *expect, uint32_t *found, int *status) {
  if (!ctx || (adler_mode != ZIPC_ADLER_REF_COMPAT && adler_mode != ZIPC_ADLER_RFC1950) ||
      (n && (!d_src_v || !src_off || !src_len || !d_dst_v || !dst_off || !max_out || !dst_len || !status)))
    return ZIPC_ERR_INVALID_ARG;
  if (!n) return ZIPC_OK;
  if (n > 0xFFFFFFF0ull) return ZIPC_ERR_INVALID_ARG;
  for (size_t i = 0; i < n; i++) if (max_out[i] == ZIPC_SIZE_UNKNOWN) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  ctx->epoch++;  // the caller's device bytes may have changed since the last call
  // headers and trailers are read on the device, by one thread per stream, and come back in one copy
  if (int st = ctx->h_res.reserve(n * sizeof(ZlibFrame))) return st;
  if (int st = ctx->d_desc2.reserve(n * sizeof(ZlibFrame))) return st;
  ZlibFrame *hf = ctx->h_res.as<ZlibFrame>(), *df = ctx->d_desc2.as<ZlibFrame>();
  for (size_t i = 0; i < n; i++) hf[i] = ZlibFrame{static_cast<const uint8_t *>(d_src_v) + src_off[i], src_len[i], 0, 0, 0, 0};
  ZB_CUDA(ctx, cudaMemcpyAsync(df, hf, n * sizeof(ZlibFrame), cudaMemcpyHostToDevice, ctx->stream));
  zlib_frames_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(df, (uint32_t)n);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  ZB_CUDA(ctx, cudaMemcpyAsync(hf, df, n * sizeof(ZlibFrame), cudaMemcpyDeviceToHost, ctx->stream));
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  // streams with a bad header are not decoded (their slots stay untouched); the others' bodies are [2, len - 2), as in the
  // reference (zipc_deflate.ml:732)
  const std::vector<ZlibFrame> f(hf, hf + n);  // (h_res is the inflate core's too)
  std::vector<uint32_t> sel;
  std::vector<const uint8_t *> body(n);
  std::vector<size_t> blen(n, 0);
  for (size_t i = 0; i < n; i++) {
    if (f[i].status != ZIPC_OK) continue;
    sel.push_back((uint32_t)i);
    body[i] = f[i].src + 2;
    blen[i] = (size_t)f[i].len - 4;
  }
  std::vector<uint32_t> ad(n);
  if (int rc = inflate_core(ctx, ZIPC_CK_ADLER32, adler_mode, n, body, blen.data(), slot_addrs(static_cast<uint8_t *>(d_dst_v), dst_off, n),
                            std::vector<size_t>(max_out, max_out + n), false, dst_len, ad.data(), status, 0, nullptr, &sel))
    return rc;
  zlib_verdict(n, f.data(), ad.data(), dst_len, expect, found, status);
  return ZIPC_OK;
}

}  // extern "C"
