// zip_api.cu -- deflate / zlib-compress / archive entry points of the C ABI (host orchestration) and the
// device gather that compacts per-member output slots.
//
//   zipc_b200_deflate_batch        <- Zipc_deflate.deflate / crc_32_and_deflate / adler_32_and_deflate
//                                     (reference src/zipc_deflate.ml:1247-1259)
//   zipc_b200_zlib_compress_batch  <- Zipc_deflate.zlib_compress (:1262-1277); _dev: inputs and outputs in device memory
//   zipc_b200_zip_extract_batch    <- Zipc.File.to_binary_string over parsed members (src/zipc.ml:205-225); _dev: members
//                                     and outputs in device memory
//   zipc_b200_zip_parse_dev        <- Zipc.of_binary_string (src/zipc.ml:400-438) of an archive in device memory
//   zipc_b200_zip_deflate_archive  <- Zipc.File.deflate_of_binary_string + Zipc.to_binary_string
//                                     (src/zipc.ml:179-185, 570-588)
#include <algorithm>
#include <cstring>
#include <numeric>

#include "common.cuh"

namespace zb {
namespace {

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) & ~(a - 1); }

// one CTA per copy; 16-byte vectors when both ends allow it, otherwise aligned 32-bit stores fed by funnel-shifted
// aligned loads (payloads land at arbitrary archive offsets: LFH + name bytes in front of each)
__global__ void __launch_bounds__(256) gather_kernel(const CopyDesc *__restrict__ descs, uint32_t n) {
  for (uint32_t k = blockIdx.x; k < n; k += gridDim.x) {
    const CopyDesc d = descs[k];
    if (!d.len) continue;
    if ((((uintptr_t)d.src | (uintptr_t)d.dst) & 15) == 0) {
      const uint4 *s = reinterpret_cast<const uint4 *>(d.src);
      uint4 *t = reinterpret_cast<uint4 *>(d.dst);
      uint64_t nv = d.len >> 4;
      for (uint64_t i = threadIdx.x; i < nv; i += blockDim.x) t[i] = s[i];
      for (uint64_t i = (nv << 4) + threadIdx.x; i < d.len; i += blockDim.x) d.dst[i] = d.src[i];
    } else {
      // bytes up to a word boundary of the destination, then words
      uint64_t head = (4 - ((uintptr_t)d.dst & 3)) & 3;
      if (head > d.len) head = d.len;
      for (uint64_t i = threadIdx.x; i < head; i += blockDim.x) d.dst[i] = d.src[i];
      const uint8_t *sb = d.src + head;
      const uint32_t sh = (uint32_t)((uintptr_t)sb & 3) * 8;
      const uint32_t *s = reinterpret_cast<const uint32_t *>(sb - (sh >> 3));
      uint32_t *t = reinterpret_cast<uint32_t *>(d.dst + head);
      const uint64_t nw = (d.len - head) >> 2;
      if (sh == 0) {
        for (uint64_t i = threadIdx.x; i < nw; i += blockDim.x) t[i] = s[i];
      } else {
        // word i of the destination = bytes [4i + sh/8, 4i + sh/8 + 4) of the aligned source words: s[i+1] holds at
        // least one byte of the range, so it lies inside the source buffer's last touched word
        for (uint64_t i = threadIdx.x; i < nw; i += blockDim.x) t[i] = __funnelshift_r(s[i], s[i + 1], sh);
      }
      for (uint64_t i = head + (nw << 2) + threadIdx.x; i < d.len; i += blockDim.x) d.dst[i] = d.src[i];
    }
  }
}

// one thread per member of an archive in device memory: the fields of its local header (byte loads: any offset).  The host
// hands in only headers that lie inside the archive (off + 30 <= len).
__global__ void zip_lfh_kernel(const uint8_t *__restrict__ archive, ZipLfh *f, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ZipLfh h = f[i];
  zip_lfh_fields(archive + h.off, h);
  f[i] = h;
}

// One thread per member of an archive being written: its local header at lfh_at and its central directory entry at cd_at,
// byte stores at any alignment of out; thread n writes the end records.  The writers are the host assembler's (common.cuh).
__global__ void zip_headers_kernel(const ZipHdr *__restrict__ hdr, uint32_t n, const char *__restrict__ names, ZipTail tail,
                                   uint8_t *__restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const ZipHdr h = hdr[i];
    zip_write_lfh(out + h.lfh_at, h, names + h.name);
    zip_write_cdfh(out + h.cd_at, h, names + h.name);
  } else if (i == n) {
    zip_write_end(out + tail.cd_start + tail.cd_size, tail);
  }
}

// p is device memory of the ctx's device (a host pointer handed to a _dev call by mistake is refused before anything runs)
bool on_device(const zipc_b200_ctx *ctx, const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice && a.device == ctx->device;
}

// File.to_binary_string's dispatch (zipc.ml:205-217): 1 stored, 2 deflate, 0 nothing to extract (a directory, or a member
// whose status this sets: encrypted, unsupported method)
int member_kind(const zipc_b200_member &m, int *status) {
  *status = ZIPC_OK;
  if (m.is_dir) return 0;
  if (m.gp_flags & 1) { *status = ZIPC_ERR_ZIP_ENCRYPTED; return 0; }
  if (m.compression != 0 && m.compression != 8) { *status = ZIPC_ERR_ZIP_FORMAT; return 0; }
  return m.compression == 0 ? 1 : 2;
}

// File.to_binary_string over n members (zipc.ml:205-225) whose payloads are at d_src[i] (device), into d_dst[i]: sets every
// member's status, dst_len and found.  Deflate members go through the inflate core with CRC-32 (plan: the progressive
// download of zipc_b200_zip_extract_batch, or null), then stored members through stored_copy_crc, which copies and checksums
// in one pass; both are checked against the directory's CRC-32.
int extract_members(zipc_b200_ctx *ctx, const zipc_b200_member *ms, size_t n, const std::vector<const uint8_t *> &d_src,
                    const std::vector<uint8_t *> &d_dst, const DownloadPlan *plan, size_t *dst_len, uint32_t *found, int *status) {
  std::vector<uint32_t> inflated, stored;
  std::vector<size_t> slen(n, 0), cap(n, 0);
  std::vector<const uint8_t *> s1;
  std::vector<uint8_t *> d1;
  std::vector<uint64_t> l1;
  for (size_t i = 0; i < n; i++) {
    const zipc_b200_member &m = ms[i];
    dst_len[i] = 0;
    if (found) found[i] = 0;
    const int kind = member_kind(m, &status[i]);
    if (kind == 1) { stored.push_back((uint32_t)i); s1.push_back(d_src[i]); d1.push_back(d_dst[i]); l1.push_back(m.compressed_size); }
    if (kind == 2) { inflated.push_back((uint32_t)i); slen[i] = (size_t)m.compressed_size; cap[i] = (size_t)m.decompressed_size; }
  }
  std::vector<uint32_t> ck(n);
  if (int st = inflate_core(ctx, ZIPC_CK_CRC32, 0, n, d_src, slen.data(), d_dst, cap, false, dst_len, ck.data(), status, 0, plan, &inflated))
    return st;
  for (uint32_t i : inflated) {
    if (found) found[i] = ck[i];
    if (status[i] == ZIPC_OK && ck[i] != ms[i].crc32) status[i] = ZIPC_ERR_CHECKSUM;
  }
  std::vector<uint32_t> c1(stored.size());
  if (int st = stored_copy_crc(ctx, stored.size(), s1.data(), d1.data(), l1.data(), c1.data())) return st;
  for (size_t j = 0; j < stored.size(); j++) {
    const uint32_t i = stored[j];
    dst_len[i] = (size_t)l1[j];
    if (found) found[i] = c1[j];
    if (c1[j] != ms[i].crc32) status[i] = ZIPC_ERR_CHECKSUM;
  }
  return ZIPC_OK;
}

// Runs the encoder over n device-resident inputs.  Output of member i lands in a private slot
// (d_slot[i], capacity slot_cap[i]); the caller compacts.  Checksums are of the INPUT (crc_op); Adler-32 is folded
// per emitted block, which is what the reference's own zlib_decompress recomputes from the stream.
int deflate_run(zipc_b200_ctx *ctx, int level, int ck, int adler_mode, size_t n,
                const std::vector<const uint8_t *> &d_src, const size_t *src_len,
                const std::vector<uint8_t *> &d_slot, const std::vector<size_t> &slot_cap,
                size_t *out_len, uint32_t *checksum, int *status, const std::vector<uint32_t> *flags = nullptr,
                std::vector<uint32_t> *blocks_out = nullptr, std::vector<uint32_t> *nblocks_out = nullptr) {
  // blocks_out / nblocks_out (Adler-32 at a compressing level only): the source lengths of the blocks every input was emitted
  // as, input after input, and their number per input, INSTEAD of the checksums -- the caller folds them itself (the pieces of a
  // split member are folded as the one stream they form)
  if (!n) return ZIPC_OK;
  if (n > 0xFFFFFFF0ull) return ZIPC_ERR_INVALID_ARG;
  for (size_t i = 0; i < n; i++) if (src_len[i] > 0xFFFFFFFFull) return ZIPC_ERR_INVALID_ARG;
  std::vector<uint32_t> order(n);
  std::iota(order.begin(), order.end(), 0u);
  std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return src_len[a] > src_len[b]; });
  if (int st = ctx->h_desc.reserve(n * (sizeof(DeflateTask) + sizeof(CrcSeg)))) return st;
  if (int st = ctx->d_desc.reserve(n * sizeof(DeflateTask))) return st;
  if (int st = ctx->d_res.reserve(n * (sizeof(DeflateResult) + sizeof(uint32_t)))) return st;
  if (int st = ctx->h_res.reserve(n * (sizeof(DeflateResult) + sizeof(uint32_t)))) return st;
  DeflateTask *ht = ctx->h_desc.as<DeflateTask>();
  // Adler-32 is folded block by block over the encoder's own blocks (reference :1081-1086): the kernel reports
  // the source length of every block it emits
  const bool want_adler = checksum && ck == ZIPC_CK_ADLER32;
  const bool blocks_from_kernel = want_adler && level != ZIPC_LEVEL_NONE;
  std::vector<uint32_t> blk_off(n, 0);
  size_t blk_total = 0;
  if (blocks_from_kernel) {
    for (size_t i = 0; i < n; i++) { blk_off[i] = (uint32_t)blk_total; blk_total += deflate_max_blocks(src_len[i]); }
    if (blk_total > 0xFFFFFFF0ull) return ZIPC_ERR_INVALID_ARG;
    if (int st = ctx->d_blk.reserve(blk_total * sizeof(uint32_t) + 64)) return st;
  }
  uint32_t *d_blk = blocks_from_kernel ? ctx->d_blk.as<uint32_t>() : nullptr;
  for (size_t k = 0; k < n; k++) {
    uint32_t i = order[k];
    ht[k].src = d_src[i]; ht[k].src_len = src_len[i]; ht[k].dst = d_slot[i]; ht[k].dst_cap = slot_cap[i];
    ht[k].flags = flags ? (*flags)[i] : 0u; ht[k].blk_off = blk_off[i];
  }
  DeflateTask *dt = ctx->d_desc.as<DeflateTask>();
  DeflateResult *dr = ctx->d_res.as<DeflateResult>();
  // CRC-32 of the inputs FIRST: in a pipelined batch the kernels of the next groups take every SM the moment this group's
  // deflate kernel lets go of it, and a checksum kernel queued behind it would wait for all of them (measured: the
  // checksums of 16 groups piled up behind the last group's kernel, 7 ms)
  const bool want_crc = checksum && ck == ZIPC_CK_CRC32;
  uint32_t *dc = nullptr;
  if (want_crc) {
    if (int st = ctx->d_desc2.reserve(n * (sizeof(CrcSeg) + sizeof(uint32_t)))) return st;
    CrcSeg *hs = reinterpret_cast<CrcSeg *>(ht + n);
    for (size_t i = 0; i < n; i++) hs[i] = crc_seg(d_src[i], src_len[i]);
    CrcSeg *ds = ctx->d_desc2.as<CrcSeg>();
    dc = reinterpret_cast<uint32_t *>(ds + n);
    ZB_CUDA(ctx, cudaMemcpyAsync(ds, hs, n * sizeof(CrcSeg), cudaMemcpyHostToDevice, ctx->stream));
    if (int st = crc32_launch_segments(ctx, ds, (uint32_t)n, dc)) return st;
  }
  ZB_CUDA(ctx, cudaMemcpyAsync(dt, ht, n * sizeof(DeflateTask), cudaMemcpyHostToDevice, ctx->stream));
  UploadGate *gate = ctx->gate;
  const size_t ticket = ctx->gate_ticket;
  const bool ordered = gate && ticket < gate->done.size();
  if (ordered && ticket >= 2) {  // (see UploadGate)
    std::unique_lock<std::mutex> lk(gate->m);
    gate->cv.wait(lk, [&] { return gate->launched[ticket - 2] != 0; });
    lk.unlock();
    ZB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, gate->done[ticket - 2], 0));
  }
  const int launch_rc = deflate_launch(ctx, dt, (uint32_t)n, dr, level, d_blk, n ? src_len[order[0]] : 0);  // (order: longest first)
  if (ordered) {
    if (launch_rc == ZIPC_OK) cudaEventRecord(gate->done[ticket], ctx->stream);
    { std::lock_guard<std::mutex> lk(gate->m); gate->launched[ticket] = 1; }
    gate->cv.notify_all();
  }
  if (launch_rc) return launch_rc;
  DeflateResult *hr = ctx->h_res.as<DeflateResult>();
  ZB_CUDA(ctx, cudaMemcpyAsync(hr, dr, n * sizeof(DeflateResult), cudaMemcpyDeviceToHost, ctx->stream));
  uint32_t *hck = reinterpret_cast<uint32_t *>(hr + n);  // (pinned: a copy into the caller's pageable array would block every thread of a pipelined batch)
  if (want_crc) ZB_CUDA(ctx, cudaMemcpyAsync(hck, dc, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<uint32_t> h_blk;
  if (blocks_from_kernel) {
    h_blk.resize(blk_total);
    ZB_CUDA(ctx, cudaMemcpyAsync(h_blk.data(), d_blk, blk_total * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  }
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  pipe_mark(ctx, "kernel done");
  std::vector<uint32_t> nblk(n, 0);
  for (size_t k = 0; k < n; k++) {
    uint32_t i = order[k];
    status[i] = (int)hr[k].status;
    out_len[i] = (size_t)hr[k].out_len;
    nblk[i] = hr[k].status == ZIPC_OK ? hr[k].blocks : 0;
  }
  if (checksum) {
    if (ck == ZIPC_CK_CRC32) {
      for (size_t i = 0; i < n; i++) checksum[i] = hck[i] ^ 0xFFFFFFFFu;
    } else if (ck == ZIPC_CK_ADLER32) {
      // block lists per member, in member order
      std::vector<uint32_t> lens;
      if (blocks_from_kernel) {
        for (size_t i = 0; i < n; i++) lens.insert(lens.end(), h_blk.begin() + blk_off[i], h_blk.begin() + blk_off[i] + nblk[i]);
        if (blocks_out && nblocks_out) { *blocks_out = std::move(lens); *nblocks_out = nblk; return ZIPC_OK; }
      } else {  // level `None: stored blocks of kStoredBlock source bytes (reference :1106-1116)
        for (size_t i = 0; i < n; i++) {
          nblk[i] = 0;
          for (uint64_t o = 0; o < src_len[i]; o += kStoredBlock, nblk[i]++) lens.push_back((uint32_t)std::min<uint64_t>(kStoredBlock, src_len[i] - o));
        }
      }
      if (int st = adler32_blocked(ctx, d_src.data(), nblk.data(), lens.data(), n, adler_mode, checksum)) return st;
    } else {
      for (size_t i = 0; i < n; i++) checksum[i] = 0;
    }
  }
  return ZIPC_OK;
}

// Lays the n slots out in ctx->d_slots.
int make_slots(zipc_b200_ctx *ctx, size_t n, const size_t *src_len, std::vector<uint8_t *> &d_slot,
               std::vector<size_t> &slot_cap) {
  d_slot.resize(n); slot_cap.resize(n);
  size_t total = 0;
  std::vector<size_t> off(n);
  for (size_t i = 0; i < n; i++) { off[i] = total; slot_cap[i] = align_up(zipc_b200_deflate_bound(src_len[i]), 16); total += slot_cap[i]; }
  if (int st = ctx->d_slots.reserve(total + 64)) return st;
  for (size_t i = 0; i < n; i++) d_slot[i] = ctx->d_slots.as<uint8_t>() + off[i];
  return ZIPC_OK;
}

// Compacts slot outputs into ctx->d_out at the given offsets.
int compact(zipc_b200_ctx *ctx, size_t n, const std::vector<uint8_t *> &d_slot, const size_t *len,
            const std::vector<size_t> &off, size_t total) {
  if (int st = ctx->d_out.reserve(total + 64)) return st;
  if (int st = ctx->h_desc.reserve(n * sizeof(CopyDesc))) return st;
  if (int st = ctx->d_desc2.reserve(n * sizeof(CopyDesc))) return st;
  CopyDesc *h = ctx->h_desc.as<CopyDesc>();
  for (size_t i = 0; i < n; i++) { h[i].src = d_slot[i]; h[i].dst = ctx->d_out.as<uint8_t>() + off[i]; h[i].len = len[i]; }
  // A group of a pipelined batch compacts on a high-priority stream: its few CTAs then get the first SMs the running deflate
  // kernel (of a later group) gives up, ahead of the deflate kernels already queued behind that one.  (The host has seen
  // this group's results, so nothing on the context's stream is pending.)
  cudaStream_t s = ctx->stream;
  if (ctx->is_sub) {
    if (!ctx->hi_stream) {
      int lo = 0, hi = 0;
      ZB_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
      ZB_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->hi_stream, cudaStreamNonBlocking, hi));
    }
    s = ctx->hi_stream;
  }
  ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_desc2.p, h, n * sizeof(CopyDesc), cudaMemcpyHostToDevice, s));
  if (int st = gather_launch(ctx, ctx->d_desc2.as<CopyDesc>(), (uint32_t)n, s)) return st;
  if (s != ctx->stream) ZB_CUDA(ctx, stream_sync(ctx, s));
  return ZIPC_OK;
}

// ---- large members over several CTAs -------------------------------------------------------------------------------------
// A member of ZIPC_B200_SPLIT_MIN bytes or more (default 2 MiB, 320 KiB in a thin batch; 0 = never) is compressed as primed segments of 64 - 256 KiB, one
// CTA each: every segment but the last ends with a byte-aligning empty stored block, every segment but the first sees the
// 32 KiB of input before it, so the concatenation is ONE ordinary RFC 1951 stream, 5 bytes per segment larger than the
// member compressed by a single CTA -- which would have one SM to itself (~90 MB/s).  Adler-32 (zlib_compress,
// adler_32_and_deflate) is folded over the blocks of all pieces in stream order, as the reference's decoder will see them.
constexpr size_t kSplitSegment = 256u << 10, kSplitSegmentMin = 64u << 10;
struct Pieces {
  std::vector<uint32_t> member;          // piece -> member
  std::vector<uint8_t *> d_slot;         // piece -> where the kernel wrote it
  std::vector<size_t> len, rel;          // piece -> compressed length, offset inside its member's output
};
int deflate_members(zipc_b200_ctx *ctx, int level, int ck, int adler_mode, size_t n, const std::vector<const uint8_t *> &d_src,
                    const size_t *src_len, size_t *out_len, uint32_t *checksum, int *status, Pieces &pc) {
  // smallest member that is split: 2 MiB in a batch that fills the GPU with whole members anyway, 320 KiB in a thin one (fewer
  // members than two per SM: a 1.9 MiB member alone would sit on one SM for 21 ms).  ZIPC_B200_SPLIT_MIN, when set, is taken as
  // it is (read on every call, so that tests can vary it).
  const uint64_t split_min = [&]() -> uint64_t {
    const char *e = std::getenv("ZIPC_B200_SPLIT_MIN");
    if (e && *e) return std::strtoull(e, nullptr, 10);
    return !ctx->is_sub && n < 2 * (size_t)std::max(1, ctx->sm_count) ? (320ull << 10) : (2ull << 20);  // (a sub-context's batch is a part of a large one)
  }();
  const bool may_split = split_min && level != ZIPC_LEVEL_NONE;
  std::vector<const uint8_t *> e_src;
  std::vector<size_t> e_len;
  std::vector<uint32_t> e_flags;
  pc.member.clear();
  bool any_split = false;
  // The segment size follows the work: the large members' bytes over the SMs in whole waves (64 MiB on 148 SMs: 293 segments of
  // 224 KiB = two full waves instead of 256 of 256 KiB = one and three quarters), and never fewer segments than SMs while a
  // segment stays at 64 KiB or more (a 5 MiB member: 80 segments side by side, not 20).
  size_t seg_bytes = kSplitSegment;
  if (may_split) {
    uint64_t split_bytes = 0;
    for (size_t i = 0; i < n; i++) if (src_len[i] >= split_min) split_bytes += src_len[i];
    const uint64_t sms = (uint64_t)std::max(1, ctx->sm_count);
    const uint64_t waves = std::max<uint64_t>(1, (split_bytes + kSplitSegment * sms - 1) / (kSplitSegment * sms));
    const uint64_t even = (split_bytes + waves * sms - 1) / (waves * sms);
    seg_bytes = (size_t)std::min<uint64_t>(kSplitSegment, std::max<uint64_t>(kSplitSegmentMin, (even + 4095) & ~4095ull));
  }
  for (size_t i = 0; i < n; i++) {
    if (!may_split || src_len[i] < split_min) { e_src.push_back(d_src[i]); e_len.push_back(src_len[i]); e_flags.push_back(0u); pc.member.push_back((uint32_t)i); continue; }
    any_split = true;
    const size_t nseg = (src_len[i] + seg_bytes - 1) / seg_bytes;
    for (size_t k = 0; k < nseg; k++) {
      e_src.push_back(d_src[i] + k * seg_bytes);
      e_len.push_back(std::min(seg_bytes, src_len[i] - k * seg_bytes));
      e_flags.push_back((k + 1 < nseg ? kDeflateNotFinal : 0u) | (k ? (uint32_t)(32768 / kDeflatePrimeTile) << kDeflatePrimeShift : 0u));
      pc.member.push_back((uint32_t)i);
    }
  }
  const size_t m = e_src.size();
  std::vector<size_t> cap, e_out(m);
  std::vector<uint32_t> e_ck(m);
  std::vector<int> e_st(m);
  if (int st = make_slots(ctx, m, e_len.data(), pc.d_slot, cap)) return st;
  // Adler-32 of a split member: folded block by block over the blocks of ALL its pieces in stream order -- exactly what the
  // reference's zlib_decompress recomputes from the concatenated stream (the empty stored blocks between the pieces fold
  // nothing; zipc_deflate.ml:682-690, 1081-1086)
  const bool fold_here = any_split && checksum && ck == ZIPC_CK_ADLER32;
  std::vector<uint32_t> blk, nblk;
  if (int st = deflate_run(ctx, level, ck, adler_mode, m, e_src, e_len.data(), pc.d_slot, cap, e_out.data(), checksum ? e_ck.data() : nullptr,
                           e_st.data(), any_split ? &e_flags : nullptr, fold_here ? &blk : nullptr, fold_here ? &nblk : nullptr)) return st;
  pc.len = e_out;
  pc.rel.assign(m, 0);
  for (size_t i = 0; i < n; i++) { out_len[i] = 0; status[i] = ZIPC_OK; if (checksum) checksum[i] = 0; }
  for (size_t k = 0; k < m; k++) {
    const uint32_t i = pc.member[k];
    const bool first = k == 0 || pc.member[k - 1] != i;
    if (e_st[k] != ZIPC_OK && status[i] == ZIPC_OK) status[i] = e_st[k];
    pc.rel[k] = out_len[i];
    out_len[i] += e_out[k];
    if (checksum && !fold_here) checksum[i] = first ? e_ck[k] : (ck == ZIPC_CK_CRC32 ? zipc_b200_crc32_combine(checksum[i], e_ck[k], e_len[k]) : 0u);
  }
  if (fold_here) {  // (the pieces of a member follow each other, so do their block lists: per member, just their number)
    std::vector<uint32_t> member_blocks(n, 0);
    for (size_t k = 0; k < m; k++) member_blocks[pc.member[k]] += nblk[k];
    if (int st = adler32_blocked(ctx, d_src.data(), member_blocks.data(), blk.data(), n, adler_mode, checksum)) return st;
    for (size_t i = 0; i < n; i++) if (status[i] != ZIPC_OK) checksum[i] = 0;
  }
  for (size_t k = 0; k < m; k++)
    if (status[pc.member[k]] != ZIPC_OK) { pc.len[k] = 0; out_len[pc.member[k]] = 0; }
  return ZIPC_OK;
}
// the pieces to their places: member i's output starts at off[i] of ctx->d_out
int compact_pieces(zipc_b200_ctx *ctx, const Pieces &pc, const std::vector<size_t> &off, size_t total) {
  std::vector<size_t> poff(pc.member.size());
  for (size_t k = 0; k < poff.size(); k++) poff[k] = off[pc.member[k]] + pc.rel[k];
  return compact(ctx, poff.size(), pc.d_slot, pc.len.data(), poff, total);
}

// zlib framing of the members deflate_members compressed into pc (reference :1264-1277): 2 header bytes at to[i], the body's
// pieces behind them, the big-endian Adler-32 behind the body_len[i] bytes of body.  Header, pieces and trailer are placed
// by one device gather (one descriptor table, one launch) at any alignment of to[i]; a member whose to[i] is null is left out.
int place_zlib(zipc_b200_ctx *ctx, int level, size_t n, const Pieces &pc, const size_t *body_len, const uint32_t *adler,
               const std::vector<uint8_t *> &to) {
  const size_t np = pc.member.size();
  const unsigned cmf = 0x78, hdr = (cmf << 8) | ((unsigned)level << 6), flg = (hdr + 31 - hdr % 31) & 0xFF;
  if (int st = ctx->h_res.reserve(n * 8)) return st;
  if (int st = ctx->d_res.reserve(n * 8)) return st;
  if (int st = ctx->h_desc.reserve((2 * n + np) * sizeof(CopyDesc))) return st;
  if (int st = ctx->d_desc2.reserve((2 * n + np) * sizeof(CopyDesc))) return st;
  uint8_t *hb = ctx->h_res.as<uint8_t>();
  uint8_t *db = ctx->d_res.as<uint8_t>();
  CopyDesc *h = ctx->h_desc.as<CopyDesc>();
  size_t nd = 0;
  for (size_t i = 0; i < n; i++) {
    if (!to[i]) continue;
    hb[8 * i] = (uint8_t)cmf; hb[8 * i + 1] = (uint8_t)flg;
    hb[8 * i + 2] = (uint8_t)(adler[i] >> 24); hb[8 * i + 3] = (uint8_t)(adler[i] >> 16);
    hb[8 * i + 4] = (uint8_t)(adler[i] >> 8); hb[8 * i + 5] = (uint8_t)adler[i];
    h[nd++] = CopyDesc{db + 8 * i, to[i], 2};
    h[nd++] = CopyDesc{db + 8 * i + 2, to[i] + 2 + body_len[i], 4};
  }
  for (size_t k = 0; k < np; k++)
    if (to[pc.member[k]]) h[nd++] = CopyDesc{pc.d_slot[k], to[pc.member[k]] + 2 + pc.rel[k], pc.len[k]};
  ZB_CUDA(ctx, cudaMemcpyAsync(db, hb, n * 8, cudaMemcpyHostToDevice, ctx->stream));
  ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_desc2.p, h, nd * sizeof(CopyDesc), cudaMemcpyHostToDevice, ctx->stream));
  return gather_launch(ctx, ctx->d_desc2.as<CopyDesc>(), (uint32_t)nd);
}

// The paths of an archive's n members as Member.make keeps them (zipc.ml:244-255): backslashes become slashes.  Checked in
// member order: the path's length, then the size of a member that is deflated (compression NULL: every member; the encoder
// takes inputs below 4 GiB).
int archive_paths(size_t n, const char *const *paths, const uint32_t *path_len, const size_t *src_len, const int32_t *compression,
                  std::vector<std::string> &norm) {
  norm.resize(n);
  for (size_t i = 0; i < n; i++) {
    if (path_len[i] > 0xFFFF) return ZIPC_ERR_ZIP_PATH_LEN;
    if ((!compression || compression[i] == 8) && src_len[i] > 0xFFFFFFFFull) return ZIPC_ERR_ZIP_SIZE;
    norm[i].assign(paths[i], path_len[i]);
    for (char &c : norm[i]) if (c == '\\') c = '/';
  }
  return ZIPC_OK;
}
// File.make + Member.make over the n payloads (zipc.ml:138-143, 244-255): compression[i] (NULL: 8), clen[i] bytes of payload
// for src_len[i] bytes of data, CRC-32 crc[i]; mode / mtime may be NULL
void archive_members(size_t n, const std::vector<std::string> &norm, const int32_t *compression, const int32_t *mode,
                     const int64_t *mtime, const size_t *src_len, const size_t *clen, const uint32_t *crc,
                     std::vector<zipc_b200_member> &ms) {
  ms.resize(n);
  for (size_t i = 0; i < n; i++) {
    zipc_b200_member &m = ms[i];
    std::memset(&m, 0, sizeof m);
    m.path = norm[i].data(); m.path_len = (uint32_t)norm[i].size();
    m.mode = mode ? mode[i] : 0644;
    m.mtime = mtime ? std::max<int64_t>(mtime[i], 315532800) : 315532800;
    m.version_made_by = 0x314; m.version_needed = 20; m.gp_flags = 0x800;  // File.make defaults (zipc.ml:138-143)
    m.compression = compression ? compression[i] : 8;
    m.compressed_size = clen[i]; m.decompressed_size = src_len[i]; m.crc32 = crc[i];
  }
}

}  // namespace

int gather_launch(zipc_b200_ctx *ctx, const CopyDesc *d_descs, uint32_t n, cudaStream_t stream) {
  if (!n) return ZIPC_OK;
  uint32_t grid = std::min<uint32_t>(n, (uint32_t)ctx->sm_count * 8);
  gather_kernel<<<grid, 256, 0, stream ? stream : ctx->stream>>>(d_descs, n);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  return ZIPC_OK;
}

// One context's worth of zipc_b200_deflate_batch with a caller-defined layout of the outputs: `gap[i]` bytes (may be null)
// are left free in front of output i and every output's length is rounded up to `align` -- (nullptr, 16) is the public
// call's layout, (local file header sizes, 1) puts the payloads where they lie inside a ZIP archive.
int deflate_batch_layout(zipc_b200_ctx *ctx, int level, int ck, int adler_mode, size_t n, const void *const *src, const size_t *src_len,
                         void *dst, size_t dst_cap, size_t *dst_need, size_t *dst_off, size_t *dst_len, uint32_t *checksum, int *status,
                         const uint32_t *gap, size_t align) {
  DeviceGuard g(ctx->device);
  pipe_mark(ctx, "begin");
  std::vector<const uint8_t *> d_src;
  if (int st = upload_ranges(ctx, n, src, src_len, d_src)) return st;
  pipe_mark(ctx, "uploaded");
  Pieces pc;
  if (int st = deflate_members(ctx, level, ck, adler_mode, n, d_src, src_len, dst_len, checksum, status, pc)) return st;
  pipe_mark(ctx, "deflated");
  std::vector<size_t> off(n);
  size_t total = 0;
  for (size_t i = 0; i < n; i++) { off[i] = total + (gap ? gap[i] : 0); total = off[i] + align_up(dst_len[i], align); }
  if (int st = compact_pieces(ctx, pc, off, total)) return st;
  const int rc = finish_to_host(ctx, off, total, dst, dst_cap, dst_off, dst_need);
  pipe_mark(ctx, "compacted");
  return rc;
}

}  // namespace zb

using namespace zb;

extern "C" {

size_t zipc_b200_deflate_bound(size_t src_len) { return src_len + 6 * (src_len / 61440 + 2) + 16; }

int zipc_b200_deflate_batch(zipc_b200_ctx *ctx, int level, int ck, int adler_mode, size_t n, const void *const *src,
                            const size_t *src_len, void *dst, size_t dst_cap, size_t *dst_need, size_t *dst_off,
                            size_t *dst_len, uint32_t *checksum, int *status) {
  if (!ctx || level < 0 || level > 3 || ck < 0 || ck > 2 || (n && (!src || !src_len || !dst_off || !dst_len || !status)))
    return ZIPC_ERR_INVALID_ARG;
  if (dst_need) *dst_need = 0;
  if (!n) return ZIPC_OK;
  DeviceGuard g(ctx->device);
  if (zipc_b200_mctx *pipe = pipeline_for(ctx, n, src_len, dst)) {  // large batch: copies under the kernels
    const uint64_t l0 = pipeline_launches(pipe);
    const int rc = zipc_b200_multi_deflate_batch(pipe, level, ck, adler_mode, n, src, src_len, dst, dst_cap, dst_need, dst_off, dst_len, checksum, status);
    ctx->launches += pipeline_launches(pipe) - l0;
    if (rc != ZIPC_ERR_DST_TOO_SMALL) return rc;
  }
  return deflate_batch_layout(ctx, level, ck, adler_mode, n, src, src_len, dst, dst_cap, dst_need, dst_off, dst_len, checksum, status, nullptr, 16);
}

int zipc_b200_deflate_batch_dev(zipc_b200_ctx *ctx, int level, int ck, int adler_mode, size_t n, const void *d_src_v,
                                const size_t *src_off, const size_t *src_len, void *d_dst_v, const size_t *dst_off,
                                const size_t *dst_cap_each, size_t *dst_len, uint32_t *checksum, int *status) {
  if (!ctx || level < 0 || level > 3 || ck < 0 || ck > 2 ||
      (n && (!d_src_v || !src_off || !src_len || !d_dst_v || !dst_off || !dst_cap_each || !dst_len || !status)))
    return ZIPC_ERR_INVALID_ARG;
  if (!n) return ZIPC_OK;
  DeviceGuard g(ctx->device);
  const std::vector<uint8_t *> d_slot = slot_addrs(static_cast<uint8_t *>(d_dst_v), dst_off, n);
  for (uint8_t *p : d_slot) if ((uintptr_t)p & 3) return ZIPC_ERR_INVALID_ARG;  // output slots are written as 32-bit words
  return deflate_run(ctx, level, ck, adler_mode, n, slot_addrs(static_cast<const uint8_t *>(d_src_v), src_off, n), src_len, d_slot,
                     std::vector<size_t>(dst_cap_each, dst_cap_each + n), dst_len, checksum, status);
}

int zipc_b200_zlib_compress_batch(zipc_b200_ctx *ctx, int level, int adler_mode, size_t n, const void *const *src,
                                  const size_t *src_len, void *dst, size_t dst_cap, size_t *dst_need, size_t *dst_off,
                                  size_t *dst_len, uint32_t *adler, int *status) {
  if (!ctx || level < 0 || level > 3 || (n && (!src || !src_len || !dst_off || !dst_len || !status)))
    return ZIPC_ERR_INVALID_ARG;
  if (dst_need) *dst_need = 0;
  if (!n) return ZIPC_OK;
  DeviceGuard g(ctx->device);
  std::vector<const uint8_t *> d_src;
  if (int st = upload_ranges(ctx, n, src, src_len, d_src)) return st;
  std::vector<uint32_t> ad(n);
  Pieces pc;  // (a large payload is compressed as primed segments, one CTA each: several pieces per stream)
  if (int st = deflate_members(ctx, level, ZIPC_CK_ADLER32, adler_mode, n, d_src, src_len, dst_len, ad.data(), status, pc)) return st;
  // framed streams in ctx->d_out, so that fetch() sees complete streams
  std::vector<size_t> off(n), flen(n);
  size_t total = 0;
  for (size_t i = 0; i < n; i++) { off[i] = total; flen[i] = dst_len[i] + 6; total += align_up(flen[i], 16); }
  if (int st = ctx->d_out.reserve(total + 64)) return st;
  if (int st = place_zlib(ctx, level, n, pc, dst_len, ad.data(), slot_addrs(ctx->d_out.as<uint8_t>(), off.data(), n))) return st;
  for (size_t i = 0; i < n; i++) { dst_len[i] = flen[i]; if (adler) adler[i] = ad[i]; }
  return finish_to_host(ctx, off, total, dst, dst_cap, dst_off, dst_need);
}

int zipc_b200_zlib_compress_batch_dev(zipc_b200_ctx *ctx, int level, int adler_mode, size_t n, const void *d_src_v,
                                      const size_t *src_off, const size_t *src_len, void *d_dst_v, const size_t *dst_off,
                                      const size_t *dst_cap_each, size_t *dst_len, uint32_t *adler, int *status) {
  if (!ctx || level < 0 || level > 3 || (adler_mode != ZIPC_ADLER_REF_COMPAT && adler_mode != ZIPC_ADLER_RFC1950) ||
      (n && (!d_src_v || !src_off || !src_len || !d_dst_v || !dst_off || !dst_cap_each || !dst_len || !status)))
    return ZIPC_ERR_INVALID_ARG;
  if (!n) return ZIPC_OK;
  DeviceGuard g(ctx->device);
  std::vector<uint32_t> ad(n);
  Pieces pc;  // compressed into the library's slots as by zipc_b200_zlib_compress_batch: same pieces, same bytes
  if (int st = deflate_members(ctx, level, ZIPC_CK_ADLER32, adler_mode, n, slot_addrs(static_cast<const uint8_t *>(d_src_v), src_off, n),
                               src_len, dst_len, ad.data(), status, pc)) return st;
  // a stream goes to its slot only if all of it fits: a slot too small is not written at all
  std::vector<uint8_t *> to(n, nullptr);
  for (size_t i = 0; i < n; i++) {
    if (status[i] == ZIPC_OK && (dst_cap_each[i] < 6 || dst_len[i] > dst_cap_each[i] - 6)) status[i] = ZIPC_ERR_DST_TOO_SMALL;
    if (status[i] == ZIPC_OK) to[i] = static_cast<uint8_t *>(d_dst_v) + dst_off[i];
  }
  if (int st = place_zlib(ctx, level, n, pc, dst_len, ad.data(), to)) return st;
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));  // (the gather reads the pinned descriptor table: it must be through before the next call)
  for (size_t i = 0; i < n; i++) {
    dst_len[i] = to[i] ? dst_len[i] + 6 : 0;
    if (adler) adler[i] = to[i] ? ad[i] : 0u;
  }
  return ZIPC_OK;
}

// A member below the split threshold is one deflate stream of at most zipc_b200_deflate_bound(L) bytes.  A split member
// (deflate_members) is cut into nseg <= L / 65536 + 1 segments: every segment but the last has at least kSplitSegmentMin =
// 64 KiB.  The encoder closes a block every 61440 source bytes of a segment and never emits a block larger than its stored
// form (3 header bits, at most 7 padding bits, LEN / NLEN, the bytes: 42 bits over the source), and every segment but the
// last ends with an empty stored block (at most 42 bits).  A segment of l bytes has at most l / 61440 + 1 blocks, so all
// segments together have at most L / 61440 + nseg blocks and nseg - 1 empty stored blocks, and the body is at most
//   L + 6 (L / 61440 + 2 nseg) + 1  <=  L + 6 (L / 61440 + 2) + 12 (L / 65536) + 1  <=  deflate_bound(L) + 12 (L / 65536)
// bytes, 2 + 4 framing bytes around it.  (Level none is never split: stored blocks of 65534 bytes, within deflate_bound.)
size_t zipc_b200_zlib_bound(size_t src_len) { return zipc_b200_deflate_bound(src_len) + 12 * (src_len / kSplitSegmentMin) + 6; }

// Per member: its payload (a deflate body is a zlib stream without its 6 framing bytes), the local header with a ZIP64
// extra field (30 + 20 + path), the directory entry with the longest one (46 + 28 + path); then the ZIP64 end record, its
// locator and the EOCD.
size_t zipc_b200_zip_archive_bound(size_t n, const uint32_t *path_len, const size_t *src_len, const int32_t *compression) {
  if (n && (!path_len || !src_len)) return 0;
  size_t b = 56 + 20 + 22;
  for (size_t i = 0; i < n; i++)
    b += (compression && compression[i] == 0 ? src_len[i] : zipc_b200_zlib_bound(src_len[i]) - 6) + 30 + 20 + 46 + 28 + 2 * (size_t)path_len[i];
  return b;
}

// ---- segmented single stream -----------------------------------------------------------------------------
static int deflate_segments(zipc_b200_ctx *ctx, int level, const void *src, size_t len, size_t segment_size,
                            int last_piece, void *dst, size_t dst_cap, size_t *dst_len, uint64_t *index,
                            size_t index_cap_pairs, size_t *nseg_out, uint32_t *crc32, bool primed) {
  if (!ctx || level < 0 || level > 3 || (!src && len) || !dst_len || !nseg_out || segment_size < 4096 ||
      segment_size > 0x7FFFFFFFull)
    return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  const size_t nseg = len ? (len + segment_size - 1) / segment_size : 1;
  *nseg_out = nseg;
  if (index && index_cap_pairs < nseg + 1) return ZIPC_ERR_INVALID_ARG;
  // input to the device (one copy), segments are slices of it
  const uint8_t *d_base;
  if (int st = upload_buffer(ctx, src, len, &d_base)) return st;
  std::vector<const uint8_t *> d_src(nseg);
  std::vector<size_t> slen(nseg);
  std::vector<uint32_t> flags(nseg, kDeflateNotFinal);
  for (size_t i = 0; i < nseg; i++) { d_src[i] = d_base + i * segment_size; slen[i] = std::min(segment_size, len - i * segment_size); }
  if (last_piece) flags[nseg - 1] = 0;
  if (primed)  // every segment but the first sees the 32 KiB of input before it (whole tiles of it)
    for (size_t i = 1; i < nseg; i++) {
      const size_t before = std::min<size_t>(i * segment_size, 32768) / kDeflatePrimeTile;
      flags[i] |= (uint32_t)before << kDeflatePrimeShift;
    }
  std::vector<uint8_t *> d_slot;
  std::vector<size_t> cap, clen(nseg);
  std::vector<int> st_m(nseg);
  if (int st = make_slots(ctx, nseg, slen.data(), d_slot, cap)) return st;
  if (int st = deflate_run(ctx, level, ZIPC_CK_NONE, 0, nseg, d_src, slen.data(), d_slot, cap, clen.data(), nullptr, st_m.data(), &flags)) return st;
  for (size_t i = 0; i < nseg; i++) if (st_m[i]) return st_m[i];
  if (crc32)
    if (int st = crc32_to_host_word(ctx, d_base, len)) return st;
  // the pieces are byte aligned: concatenate without gaps
  std::vector<size_t> off(nseg);
  size_t total = 0;
  for (size_t i = 0; i < nseg; i++) { off[i] = total; total += clen[i]; }
  if (index) {
    for (size_t i = 0; i < nseg; i++) { index[2 * i] = off[i]; index[2 * i + 1] = (uint64_t)i * segment_size; }
    index[2 * nseg] = total; index[2 * nseg + 1] = len;
  }
  if (int st = compact(ctx, nseg, d_slot, clen.data(), off, total)) return st;
  const int rc = finish_to_host(ctx, off, total, dst, dst_cap, nullptr, dst_len);
  if (crc32 && (rc == ZIPC_OK || rc == ZIPC_ERR_DST_TOO_SMALL)) *crc32 = host_word_crc32(ctx);
  return rc;
}

int zipc_b200_deflate_segmented(zipc_b200_ctx *ctx, int level, const void *src, size_t len, size_t segment_size,
                                int last_piece, void *dst, size_t dst_cap, size_t *dst_len, uint64_t *index,
                                size_t index_cap_pairs, size_t *nseg_out, uint32_t *crc32) {
  return deflate_segments(ctx, level, src, len, segment_size, last_piece, dst, dst_cap, dst_len, index, index_cap_pairs, nseg_out, crc32, false);
}

int zipc_b200_deflate_primed(zipc_b200_ctx *ctx, int level, const void *src, size_t len, size_t segment_size,
                             int last_piece, void *dst, size_t dst_cap, size_t *dst_len, uint64_t *index,
                             size_t index_cap_pairs, size_t *nseg_out, uint32_t *crc32) {
  return deflate_segments(ctx, level, src, len, segment_size, last_piece, dst, dst_cap, dst_len, index, index_cap_pairs, nseg_out, crc32, true);
}

int zipc_b200_inflate_segmented(zipc_b200_ctx *ctx, const void *src, size_t len, const uint64_t *index, size_t nseg,
                                void *dst, size_t dst_cap, size_t *dst_len, uint32_t *crc32, int *status) {
  if (!ctx || (!src && len) || !index || !nseg || !dst_len || !status) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  const uint64_t ctotal = index[2 * nseg], utotal = index[2 * nseg + 1];
  if (ctotal > len) return ZIPC_ERR_INVALID_ARG;
  for (size_t i = 0; i < nseg; i++)
    if (index[2 * i] > index[2 * i + 2] || index[2 * i + 1] > index[2 * i + 3]) return ZIPC_ERR_INVALID_ARG;
  *dst_len = utotal;
  const uint8_t *d_base;
  if (int st = upload_buffer(ctx, src, len, &d_base)) return st;
  if (int st = ctx->d_out.reserve(utotal + 64)) return st;
  std::vector<const uint8_t *> d_src(nseg);
  std::vector<uint8_t *> d_dst(nseg);
  std::vector<size_t> clen(nseg), cap(nseg), ol(nseg);
  std::vector<int> st_m(nseg);
  for (size_t i = 0; i < nseg; i++) {
    d_src[i] = d_base + index[2 * i]; clen[i] = index[2 * i + 2] - index[2 * i];
    d_dst[i] = ctx->d_out.as<uint8_t>() + index[2 * i + 1]; cap[i] = index[2 * i + 3] - index[2 * i + 1];
  }
  if (int st = inflate_core(ctx, ZIPC_CK_NONE, 0, nseg, d_src, clen.data(), d_dst, cap, false, ol.data(), nullptr, st_m.data(), kInflateSegment)) return st;
  *status = ZIPC_OK;
  for (size_t i = 0; i < nseg; i++) {
    if (st_m[i]) { *status = st_m[i]; break; }
    if (ol[i] != cap[i]) { *status = ZIPC_ERR_CORRUPTED; break; }  // the index promised more bytes
  }
  if (crc32)
    if (int st = crc32_to_host_word(ctx, ctx->d_out.as<uint8_t>(), utotal)) return st;
  const int rc = finish_to_host(ctx, {}, utotal, dst, dst_cap, nullptr, nullptr);
  if (crc32 && (rc == ZIPC_OK || rc == ZIPC_ERR_DST_TOO_SMALL)) *crc32 = host_word_crc32(ctx);
  return rc;
}

// ---- archive layer ---------------------------------------------------------------------------------------
int zipc_b200_zip_extract_batch(zipc_b200_ctx *ctx, const zipc_b200_member *ms, size_t n, void *dst, size_t dst_cap,
                                size_t *dst_need, size_t *dst_off, size_t *dst_len, uint32_t *found, int *status) {
  if (!ctx || (n && (!ms || !dst_off || !dst_len || !status))) return ZIPC_ERR_INVALID_ARG;
  if (dst_need) *dst_need = 0;
  if (!n) return ZIPC_OK;
  DeviceGuard g(ctx->device);
  // the payloads and output slots of the members that are extracted (member_kind); the deflate ones may form download groups
  std::vector<const void *> src(n, nullptr);
  std::vector<size_t> slen(n, 0), cap(n, 0);
  std::vector<char> grouped(n, 0);
  bool all_deflate = true;   // (stored members are copied by a kernel that does not wait for a late half)
  for (size_t i = 0; i < n; i++) {
    const zipc_b200_member &m = ms[i];
    int kind_status;
    const int kind = member_kind(m, &kind_status);
    if (!kind) continue;
    if (m.compressed_size && !m.compressed_bytes) return ZIPC_ERR_INVALID_ARG;
    src[i] = m.compressed_bytes + m.start;
    slen[i] = (size_t)m.compressed_size;
    cap[i] = kind == 1 ? (size_t)m.compressed_size : (size_t)m.decompressed_size;
    grouped[i] = kind == 2;
    all_deflate &= kind != 1;
  }
  UploadSplit split;
  split.want = all_deflate && progressive_ok(ctx, n, cap.data(), slen.data(), grouped.data(), dst, dst_cap);
  std::vector<const uint8_t *> d_src;
  if (int st = upload_ranges(ctx, n, src.data(), slen.data(), d_src, &split)) return st;
  std::vector<size_t> off;
  size_t total = 0;
  DownloadPlan plan;
  if (int st = plan_arena(ctx, n, cap.data(), src.data(), slen.data(), grouped.data(), split, dst, dst_cap, off, total, plan)) return st;
  // whatever way this call ends, no progressive copy into the caller's arena outlives it
  struct CopyFence {
    zipc_b200_ctx *c;
    bool on;
    ~CopyFence() { if (on && c->copy_stream) cudaStreamSynchronize(c->copy_stream); }
  } fence{ctx, plan.ngroups != 0};
  if (int st = ctx->d_out.reserve(total + 64)) return st;
  if (int st = extract_members(ctx, ms, n, d_src, slot_addrs(ctx->d_out.as<uint8_t>(), off.data(), n), &plan, dst_len, found, status))
    return st;
  return finish_to_host(ctx, off, total, dst, dst_cap, dst_off, dst_need, &plan);
}

// The parser of zipc_b200_zip_parse_ex (host_util.cc) over an archive in device memory.  Copies, whatever the member count:
// the tail window the EOCD search needs, the ZIP64 end record if there is one, the central directory (unless the tail
// window holds it already), and the local header fields of all members through one kernel and one copy back.
int zipc_b200_zip_parse_dev(zipc_b200_ctx *ctx, const void *d_bytes, size_t len, unsigned flags, zipc_b200_member **members,
                            size_t *n_out) {
  if (!ctx || !members || !n_out || (!d_bytes && len)) return ZIPC_ERR_INVALID_ARG;
  *members = nullptr;
  *n_out = 0;
  if (len < 22) return ZIPC_ERR_ZIP_SHORT;
  DeviceGuard g(ctx->device);
  const uint8_t *d = static_cast<const uint8_t *>(d_bytes);
  const uint64_t tail_at = len > kZipTailWindow ? len - kZipTailWindow : 0;
  std::vector<uint8_t> tail(len - tail_at);
  if (int st = d2h(ctx, tail.data(), d + tail_at, tail.size())) return st;
  ZipEnd e;
  if (int st = zip_find_end(tail.data(), tail_at, len, flags, e)) return st;
  if (e.rec64 != ~0ull) {
    uint8_t rec[56];
    if (int st = d2h(ctx, rec, d + e.rec64, sizeof rec)) return st;
    if (int st = zip_read_end64(rec, len, e)) return st;
  }
  std::vector<uint8_t> cd_copy;  // (a directory inside the tail window is read from there)
  const uint8_t *cd;
  if (e.cd_start >= tail_at) {
    cd = tail.data() + (e.cd_start - tail_at);
  } else {
    cd_copy.resize((size_t)e.cd_size);
    if (int st = d2h(ctx, cd_copy.data(), d + e.cd_start, cd_copy.size())) return st;
    cd = cd_copy.data();
  }
  std::vector<zipc_b200_member> ms;
  std::vector<ZipLfh> lfh;
  const int cd_status = zip_walk_cd(cd, len, flags, e, ms, lfh);
  std::vector<uint32_t> idx;
  for (size_t k = 0; k < ms.size(); k++)
    if (!ms[k].is_dir && lfh[k].off + 30 <= len) idx.push_back((uint32_t)k);
  if (!idx.empty()) {
    const size_t m = idx.size();
    if (int st = ctx->h_res.reserve(m * sizeof(ZipLfh))) return st;
    if (int st = ctx->d_desc2.reserve(m * sizeof(ZipLfh))) return st;
    ZipLfh *hf = ctx->h_res.as<ZipLfh>(), *df = ctx->d_desc2.as<ZipLfh>();
    for (size_t j = 0; j < m; j++) hf[j] = lfh[idx[j]];
    ZB_CUDA(ctx, cudaMemcpyAsync(df, hf, m * sizeof(ZipLfh), cudaMemcpyHostToDevice, ctx->stream));
    zip_lfh_kernel<<<(unsigned)((m + 255) / 256), 256, 0, ctx->stream>>>(d, df, (uint32_t)m);
    ctx->launches++;
    ZB_CUDA(ctx, cudaGetLastError());
    ZB_CUDA(ctx, cudaMemcpyAsync(hf, df, m * sizeof(ZipLfh), cudaMemcpyDeviceToHost, ctx->stream));
    ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
    for (size_t j = 0; j < m; j++) lfh[idx[j]] = hf[j];
  }
  return zip_parse_finish(ms, lfh, cd_status, len, d, cd, e.cd_size, true, members, n_out);
}

// Zipc.File.to_binary_string over members whose payloads are in device memory, into the caller's device slots.  Deflate
// members go through the inflate core with CRC-32 (as zipc_b200_inflate_batch_dev), stored members through stored_copy_crc.
int zipc_b200_zip_extract_batch_dev(zipc_b200_ctx *ctx, const zipc_b200_member *ms, size_t n, void *d_dst_v, const size_t *dst_off,
                                    size_t *dst_len, uint32_t *found, int *status) {
  if (!ctx || (n && (!ms || !d_dst_v || !dst_off || !dst_len || !status))) return ZIPC_ERR_INVALID_ARG;
  if (!n) return ZIPC_OK;
  if (n > 0xFFFFFFF0ull) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  // every payload pointer must be device memory of this ctx's device: host members (zipc_b200_zip_parse_ex) passed here by
  // mistake are refused before anything runs.  One query per distinct pointer.
  std::vector<const uint8_t *> seen, d_src(n, nullptr);
  for (size_t i = 0; i < n; i++) {
    const zipc_b200_member &m = ms[i];
    int st_i;
    if (!member_kind(m, &st_i)) continue;
    d_src[i] = m.compressed_bytes + m.start;
    if (!m.compressed_bytes) {
      if (m.compressed_size) return ZIPC_ERR_INVALID_ARG;
      continue;
    }
    if (std::find(seen.begin(), seen.end(), m.compressed_bytes) != seen.end()) continue;
    if (!on_device(ctx, m.compressed_bytes)) return ZIPC_ERR_INVALID_ARG;
    seen.push_back(m.compressed_bytes);
  }
  ctx->epoch++;  // the caller's device bytes may have changed since the last call
  return extract_members(ctx, ms, n, d_src, slot_addrs(static_cast<uint8_t *>(d_dst_v), dst_off, n), nullptr, dst_len, found, status);
}

int zipc_b200_zip_deflate_archive(zipc_b200_ctx *ctx, int level, size_t n, const char *const *paths,
                                  const uint32_t *path_len, const void *const *src, const size_t *src_len,
                                  const int32_t *mode, const int64_t *mtime, const char *first, void *out,
                                  size_t out_cap, size_t *out_len) {
  return zipc_b200_zip_deflate_archive_ex(ctx, level, n, paths, path_len, src, src_len, mode, mtime, first, ZIPC_ZIP_REFERENCE, out, out_cap, out_len);
}

// flags: ZIPC_ZIP_* (include/zipc_b200.h).  With ZIP64 allowed more than 65,535 members and an archive of 4 GiB or more are
// written with ZIP64 records instead of being refused; the payloads are compressed and placed exactly as without the flag.
int zipc_b200_zip_deflate_archive_ex(zipc_b200_ctx *ctx, int level, size_t n, const char *const *paths,
                                     const uint32_t *path_len, const void *const *src, const size_t *src_len,
                                     const int32_t *mode, const int64_t *mtime, const char *first, unsigned flags, void *out,
                                     size_t out_cap, size_t *out_len) {
  if (!ctx || level < 0 || level > 3 || !out_len || (n && (!paths || !path_len || !src || !src_len)))
    return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  const bool zip64 = (flags & (ZIPC_ZIP_ALLOW_ZIP64 | ZIPC_ZIP_FORCE_ZIP64)) != 0;
  if (n > 0xFFFF && !zip64) return ZIPC_ERR_ZIP_COUNT;  // zipc.ml:574
  std::vector<std::string> norm;
  if (int st = archive_paths(n, paths, path_len, src_len, nullptr, norm)) return st;
  std::vector<size_t> clen(n);
  std::vector<uint32_t> crc(n);
  std::vector<int> st_m(n);
  auto fill_members = [&](std::vector<zipc_b200_member> &ms) {
    archive_members(n, norm, nullptr, mode, mtime, src_len, clen.data(), crc.data(), ms);
  };
  // A large archive whose members come in path order (the order Zipc.to_binary_string writes them in, none of them the
  // `first` member unless it is the first anyway): through the pipeline, every group's payloads copied straight to their
  // place in `out` while the later groups are compressed; the headers are written around them afterwards.
  if (out) {
    bool in_order = true;
    const char *f = first ? first : "mimetype";
    const size_t flen = std::strlen(f);
    for (size_t i = 0; i < n && in_order; i++) {
      if (i && !(norm[i - 1] < norm[i])) in_order = false;   // (bytewise, like String.compare; equal paths shadow each other)
      if (i && norm[i].size() == flen && std::memcmp(norm[i].data(), f, flen) == 0) in_order = false;
    }
    zipc_b200_mctx *pipe = in_order ? pipeline_for(ctx, n, src_len, out) : nullptr;
    if (pipe) {
      std::vector<uint32_t> gap(n);
      for (size_t i = 0; i < n; i++) gap[i] = 30u + (uint32_t)norm[i].size();
      std::vector<size_t> poff(n);
      size_t need = 0;
      const uint64_t l0 = pipeline_launches(pipe);
      const int rc = pipeline_deflate_gapped(pipe, level, n, src, src_len, gap.data(), out, out_cap, &need, poff.data(), clen.data(), crc.data(), st_m.data());
      ctx->launches += pipeline_launches(pipe) - l0;
      if (rc == ZIPC_OK) {
        for (size_t i = 0; i < n; i++) if (st_m[i]) return st_m[i];
        std::vector<zipc_b200_member> ms(n);
        fill_members(ms);
        std::vector<uint64_t> want(n, ~0ull);
        size_t total = 0;
        if (int st = zip_assemble_impl(ms.data(), n, first, nullptr, 0, &total, false, want.data(), flags)) return st;
        bool placed = true;
        for (size_t i = 0; i < n && placed; i++) placed = want[i] == poff[i];
        if (placed) return zip_assemble_impl(ms.data(), n, first, out, out_cap, out_len, false, nullptr, flags);
      } else if (rc != ZIPC_ERR_DST_TOO_SMALL) {
        return rc;
      }
      // (too small for the payloads, or not where the layout wants them: the plain path below reports / redoes it)
    }
  }
  std::vector<const uint8_t *> d_src;
  if (int st = upload_ranges(ctx, n, src, src_len, d_src)) return st;
  Pieces pc;
  if (int st = deflate_members(ctx, level, ZIPC_CK_CRC32, 0, n, d_src, src_len, clen.data(), crc.data(), st_m.data(), pc)) return st;
  for (size_t i = 0; i < n; i++) if (st_m[i]) return st_m[i];
  std::vector<zipc_b200_member> ms(n);
  fill_members(ms);
  // layout first, then the GPU gathers every payload to its archive offset, then headers on the host
  std::vector<uint64_t> poff(n, ~0ull);  // members shadowed by a later duplicate path keep ~0
  size_t total = 0;
  if (int st = zip_assemble_impl(ms.data(), n, first, nullptr, 0, &total, false, poff.data(), flags)) return st;
  *out_len = total;
  if (!out || out_cap < total) return ZIPC_ERR_DST_TOO_SMALL;
  std::vector<size_t> off(n);
  for (size_t i = 0; i < n; i++) off[i] = poff[i] != ~0ull ? (size_t)poff[i] : 0;
  for (size_t k = 0; k < pc.member.size(); k++) if (poff[pc.member[k]] == ~0ull) pc.len[k] = 0;  // shadowed by a later duplicate path
  if (int st = compact_pieces(ctx, pc, off, total)) return st;
  if (int st = d2h(ctx, out, ctx->d_out.p, total)) return st;
  return zip_assemble_impl(ms.data(), n, first, out, out_cap, out_len, false, nullptr, flags);
}

// The archive of zipc_b200_zip_deflate_archive_ex written into device memory from device payloads, stored members allowed.
// The deflate members are compressed as the host call compresses them, the layout is the host assembler's (make_layout), and
// the GPU places everything: deflate pieces by one gather, stored members by stored_copy_crc (copy and CRC-32 in one pass),
// headers and end records by zip_headers_kernel.
int zipc_b200_zip_deflate_archive_dev(zipc_b200_ctx *ctx, int level, size_t n, const char *const *paths, const uint32_t *path_len,
                                      const void *d_src_v, const size_t *src_off, const size_t *src_len, const int32_t *compression,
                                      const int32_t *mode, const int64_t *mtime, const char *first, unsigned flags,
                                      void *d_out_v, size_t out_cap, size_t *out_len) {
  if (!ctx || level < 0 || level > 3 || !out_len || !d_out_v || (n && (!paths || !path_len || !d_src_v || !src_off || !src_len)))
    return ZIPC_ERR_INVALID_ARG;
  if (n > 0xFFFFFFF0ull) return ZIPC_ERR_INVALID_ARG;
  for (size_t i = 0; compression && i < n; i++)
    if (compression[i] != 0 && compression[i] != 8) return ZIPC_ERR_INVALID_ARG;
  DeviceGuard g(ctx->device);
  if (!on_device(ctx, d_out_v) || (n && !on_device(ctx, d_src_v))) return ZIPC_ERR_INVALID_ARG;
  const bool zip64 = (flags & (ZIPC_ZIP_ALLOW_ZIP64 | ZIPC_ZIP_FORCE_ZIP64)) != 0;
  if (n > 0xFFFF && !zip64) return ZIPC_ERR_ZIP_COUNT;  // zipc.ml:574
  std::vector<std::string> norm;
  if (int st = archive_paths(n, paths, path_len, src_len, compression, norm)) return st;
  const uint8_t *base = static_cast<const uint8_t *>(d_src_v);
  uint8_t *out = static_cast<uint8_t *>(d_out_v);
  // 1. the deflate members, in member order, through the host call's path: the same pieces and bytes
  std::vector<uint32_t> defl;
  std::vector<const uint8_t *> d_src;
  std::vector<size_t> dlen;
  for (size_t i = 0; i < n; i++)
    if (!compression || compression[i] == 8) { defl.push_back((uint32_t)i); d_src.push_back(base + src_off[i]); dlen.push_back(src_len[i]); }
  const size_t nd = defl.size();
  std::vector<size_t> dclen(nd);
  std::vector<uint32_t> dcrc(nd);
  std::vector<int> dst_m(nd);
  Pieces pc;
  if (int st = deflate_members(ctx, level, ZIPC_CK_CRC32, 0, nd, d_src, dlen.data(), dclen.data(), dcrc.data(), dst_m.data(), pc)) return st;
  for (int s : dst_m) if (s) return s;
  // 2. the host call's layout; a stored member's payload is its data, its CRC-32 comes with the copy (3)
  std::vector<size_t> clen(src_len, src_len + n);
  std::vector<uint32_t> crc(n, 0);
  for (size_t k = 0; k < nd; k++) { clen[defl[k]] = dclen[k]; crc[defl[k]] = dcrc[k]; }
  std::vector<zipc_b200_member> ms;
  archive_members(n, norm, compression, mode, mtime, src_len, clen.data(), crc.data(), ms);
  Layout L;
  if (int st = make_layout(ms.data(), n, first, flags, L)) return st;
  *out_len = (size_t)L.total;
  if (out_cap < L.total) return ZIPC_ERR_DST_TOO_SMALL;
  std::vector<uint64_t> poff(n, ~0ull);  // members shadowed by a later duplicate path keep ~0 and are not written
  for (size_t j = 0; j < L.ord.size(); j++) poff[L.ord[j]] = L.lfh_at[j] + zip_lfh_size(ms[L.ord[j]].path_len, L.big[j]);
  // 3. payloads: the deflate pieces by one gather, then the stored members
  const size_t np = pc.member.size();
  if (int st = ctx->h_desc.reserve(np * sizeof(CopyDesc))) return st;
  if (int st = ctx->d_desc2.reserve(np * sizeof(CopyDesc))) return st;
  CopyDesc *hc = ctx->h_desc.as<CopyDesc>();
  size_t nc = 0;
  for (size_t k = 0; k < np; k++) {
    const uint64_t o = poff[defl[pc.member[k]]];
    if (o != ~0ull && pc.len[k]) hc[nc++] = CopyDesc{pc.d_slot[k], out + o + pc.rel[k], pc.len[k]};
  }
  if (nc) {
    ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_desc2.p, hc, nc * sizeof(CopyDesc), cudaMemcpyHostToDevice, ctx->stream));
    if (int st = gather_launch(ctx, ctx->d_desc2.as<CopyDesc>(), (uint32_t)nc)) return st;
    ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));  // (stored_copy_crc and the headers refill h_desc / d_desc2)
  }
  std::vector<uint32_t> stored;
  std::vector<const uint8_t *> s_src;
  std::vector<uint8_t *> s_dst;
  std::vector<uint64_t> s_len;
  for (size_t i = 0; compression && i < n; i++)
    if (compression[i] == 0 && poff[i] != ~0ull) { stored.push_back((uint32_t)i); s_src.push_back(base + src_off[i]); s_dst.push_back(out + poff[i]); s_len.push_back(src_len[i]); }
  std::vector<uint32_t> s_crc(stored.size());
  if (int st = stored_copy_crc(ctx, stored.size(), s_src.data(), s_dst.data(), s_len.data(), s_crc.data())) return st;  // (synchronises)
  for (size_t k = 0; k < stored.size(); k++) ms[stored[k]].crc32 = s_crc[k];
  // 4. headers and end records: one record per member and the names behind them, one upload, one kernel
  const size_t m = L.ord.size();
  size_t name_bytes = 0;
  for (size_t i : L.ord) name_bytes += ms[i].path_len;
  const size_t rec_bytes = m * sizeof(ZipHdr);
  if (int st = ctx->h_desc.reserve(rec_bytes + name_bytes)) return st;
  if (int st = ctx->d_desc2.reserve(rec_bytes + name_bytes)) return st;
  ZipHdr *hh = ctx->h_desc.as<ZipHdr>();
  char *hn = reinterpret_cast<char *>(hh + m);
  for (size_t j = 0, at = 0; j < m; j++) {
    const zipc_b200_member &mb = ms[L.ord[j]];
    hh[j] = zip_hdr(mb, L, j);
    hh[j].name = at;
    std::memcpy(hn + at, mb.path, mb.path_len);
    at += mb.path_len;
  }
  if (rec_bytes + name_bytes)
    ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_desc2.p, hh, rec_bytes + name_bytes, cudaMemcpyHostToDevice, ctx->stream));
  const ZipHdr *dh = ctx->d_desc2.as<ZipHdr>();
  zip_headers_kernel<<<(unsigned)((m + 1 + 255) / 256), 256, 0, ctx->stream>>>(dh, (uint32_t)m, reinterpret_cast<const char *>(dh + m),
                                                                             zip_tail(L), out);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  return ZIPC_OK;
}

}  // extern "C"
