// zip_api.cu -- deflate / zlib-compress / archive entry points of the C ABI (host orchestration) and the
// device gather that places the encoder's pieces (place_pieces: every compress call's output goes through it).
//
//   zipc_b200_deflate_batch        <- Zipc_deflate.deflate / crc_32_and_deflate / adler_32_and_deflate
//                                     (reference src/zipc_deflate.ml:1247-1259)
//   zipc_b200_zlib_compress_batch  <- Zipc_deflate.zlib_compress (:1262-1277); _dev: inputs and outputs in device memory
//   zipc_b200_zip_extract_batch    <- Zipc.File.to_binary_string over parsed members (src/zipc.ml:205-225); _dev: members
//                                     and outputs in device memory
//   zipc_b200_zip_parse_dev        <- Zipc.of_binary_string (src/zipc.ml:400-438) of an archive in device memory
//   zipc_b200_zip_deflate_archive  <- Zipc.File.deflate_of_binary_string + Zipc.to_binary_string
//                                     (src/zipc.ml:179-185, 570-588); _dev: payloads and archive in device memory.  Both
//                                     write through plan_archive + write_archive; the host call uploads before and
//                                     downloads after (a large batch in path order is pipelined instead)
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
// (d_slot[i], capacity slot_cap[i]); the caller places it (place_pieces).  Checksums are of the INPUT (crc_op); Adler-32 is folded
// per emitted block, which is what the reference's own zlib_decompress recomputes from the stream.
int deflate_run(zipc_b200_ctx *ctx, int level, int ck, int adler_mode, size_t n,
                const std::vector<const uint8_t *> &d_src, const size_t *src_len,
                const std::vector<uint8_t *> &d_slot, const std::vector<size_t> &slot_cap,
                size_t *out_len, uint32_t *checksum, int *status, const std::vector<uint32_t> *flags = nullptr,
                std::vector<uint64_t> *blocks_out = nullptr, std::vector<uint32_t> *nblocks_out = nullptr) {
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
      std::vector<uint64_t> lens;
      if (blocks_from_kernel) {
        for (size_t i = 0; i < n; i++) lens.insert(lens.end(), h_blk.begin() + blk_off[i], h_blk.begin() + blk_off[i] + nblk[i]);
        if (blocks_out && nblocks_out) { *blocks_out = std::move(lens); *nblocks_out = nblk; return ZIPC_OK; }
      } else {  // level `None: stored blocks of kStoredBlock source bytes (reference :1106-1116)
        for (size_t i = 0; i < n; i++) {
          nblk[i] = 0;
          for (uint64_t o = 0; o < src_len[i]; o += kStoredBlock, nblk[i]++) lens.push_back(std::min<uint64_t>(kStoredBlock, src_len[i] - o));
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
// The encoder inputs of one stream of len bytes at src cut into segments of seg bytes (one empty segment when len is 0),
// appended to e_src / e_len / e_flags; returns their number.  Every segment but the last ends with a byte-aligning empty stored
// block, the last one too unless last_final.  Primed, every segment but the first sees the (at most 32 KiB of) input before
// it, in whole tiles.
size_t cut_segments(const uint8_t *src, size_t len, size_t seg, bool primed, bool last_final, std::vector<const uint8_t *> &e_src,
                    std::vector<size_t> &e_len, std::vector<uint32_t> &e_flags) {
  const size_t nseg = len ? (len + seg - 1) / seg : 1;
  for (size_t k = 0; k < nseg; k++) {
    e_src.push_back(src + k * seg);
    e_len.push_back(std::min(seg, len - k * seg));
    uint32_t f = k + 1 < nseg || !last_final ? kDeflateNotFinal : 0u;
    if (primed && k) f |= (uint32_t)(std::min<size_t>(k * seg, 32768) / kDeflatePrimeTile) << kDeflatePrimeShift;
    e_flags.push_back(f);
  }
  return nseg;
}
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
    size_t nseg = 1;
    if (may_split && src_len[i] >= split_min) {
      any_split = true;
      nseg = cut_segments(d_src[i], src_len[i], seg_bytes, true, true, e_src, e_len, e_flags);
    } else {
      e_src.push_back(d_src[i]); e_len.push_back(src_len[i]); e_flags.push_back(0u);
    }
    pc.member.insert(pc.member.end(), nseg, (uint32_t)i);
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
  std::vector<uint64_t> blk;
  std::vector<uint32_t> nblk;
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
int gather_launch(zipc_b200_ctx *ctx, const CopyDesc *d_descs, uint32_t n, cudaStream_t stream) {
  uint32_t grid = std::min<uint32_t>(n, (uint32_t)ctx->sm_count * 8);
  gather_kernel<<<grid, 256, 0, stream>>>(d_descs, n);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  return ZIPC_OK;
}

// The pieces of pc to their places: piece k of member i = pc.member[k] goes to to[i] + pc.rel[k], at any alignment.  A member
// whose to[i] is null is left out (it failed, is shadowed, or its slot is too small).  With adler, each member is framed as a
// zlib stream of that level (reference :1264-1277): 2 header bytes at to[i], the body 2 bytes further, the big-endian adler[i]
// behind the body.  One descriptor table (framing bytes in front of it), one upload, one gather_kernel launch.  The copies are
// left queued on the context's stream (a wait here would cost every small call its time): the caller waits for that stream
// before the pinned table (ctx->h_desc) is refilled or the output is read.
int place_pieces(zipc_b200_ctx *ctx, const Pieces &pc, const std::vector<uint8_t *> &to, const uint32_t *adler = nullptr,
                 int level = 0) {
  const size_t n = to.size(), np = pc.member.size(), nf = adler ? n : 0;
  const size_t frame_bytes = 8 * nf, table_bytes = frame_bytes + (2 * nf + np) * sizeof(CopyDesc);
  if (int st = ctx->h_desc.reserve(table_bytes)) return st;
  if (int st = ctx->d_desc2.reserve(table_bytes)) return st;
  uint8_t *hb = ctx->h_desc.as<uint8_t>(), *db = ctx->d_desc2.as<uint8_t>();
  CopyDesc *h = reinterpret_cast<CopyDesc *>(hb + frame_bytes);
  size_t nd = 0;
  if (adler) {
    std::vector<size_t> body(n, 0);
    for (size_t k = 0; k < np; k++) body[pc.member[k]] += pc.len[k];
    const unsigned cmf = 0x78, hdr = (cmf << 8) | ((unsigned)level << 6), flg = (hdr + 31 - hdr % 31) & 0xFF;
    for (size_t i = 0; i < n; i++) {
      if (!to[i]) continue;
      uint8_t *f = hb + 8 * i;
      f[0] = (uint8_t)cmf; f[1] = (uint8_t)flg;
      f[2] = (uint8_t)(adler[i] >> 24); f[3] = (uint8_t)(adler[i] >> 16); f[4] = (uint8_t)(adler[i] >> 8); f[5] = (uint8_t)adler[i];
      h[nd++] = CopyDesc{db + 8 * i, to[i], 2};
      h[nd++] = CopyDesc{db + 8 * i + 2, to[i] + 2 + body[i], 4};
    }
  }
  const size_t skip = adler ? 2 : 0;
  for (size_t k = 0; k < np; k++)
    if (to[pc.member[k]] && pc.len[k]) h[nd++] = CopyDesc{pc.d_slot[k], to[pc.member[k]] + skip + pc.rel[k], pc.len[k]};
  if (!nd) return ZIPC_OK;
  // A group of a pipelined batch places its pieces on a high-priority stream: its few CTAs then get the first SMs the running
  // deflate kernel (of a later group) gives up, ahead of the deflate kernels already queued behind that one.  (The host has
  // seen this group's results, so nothing on the context's stream is pending.)
  cudaStream_t s = ctx->stream;
  if (ctx->is_sub) {
    if (!ctx->hi_stream) {
      int lo = 0, hi = 0;
      ZB_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
      ZB_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->hi_stream, cudaStreamNonBlocking, hi));
    }
    s = ctx->hi_stream;
  }
  ZB_CUDA(ctx, cudaMemcpyAsync(db, hb, frame_bytes + nd * sizeof(CopyDesc), cudaMemcpyHostToDevice, s));
  if (int st = gather_launch(ctx, reinterpret_cast<const CopyDesc *>(db + frame_bytes), (uint32_t)nd, s)) return st;
  if (s != ctx->stream) ZB_CUDA(ctx, stream_sync(ctx, s));
  return ZIPC_OK;
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

// An archive of n members whose data are at d_src[i] (device memory), planned: compressed, described, laid out.  pc's pieces
// name their archive member; poff: payload_offsets.
struct ArchivePlan {
  Pieces pc;
  std::vector<zipc_b200_member> ms;
  Layout L;
  std::vector<uint64_t> poff;
};
// The deflate members (compression NULL: every member) go through deflate_members with CRC-32, in member order.  Returns the
// first member's deflate status, then make_layout's; *out_len is set once the layout stands.  A stored member's CRC-32 comes
// with its copy (write_archive).
int plan_archive(zipc_b200_ctx *ctx, int level, size_t n, const std::vector<std::string> &norm, const std::vector<const uint8_t *> &d_src,
                 const size_t *src_len, const int32_t *compression, const int32_t *mode, const int64_t *mtime, const char *first,
                 unsigned flags, size_t *out_len, ArchivePlan &a) {
  std::vector<uint32_t> defl;
  std::vector<const uint8_t *> ds;
  std::vector<size_t> dlen;
  for (size_t i = 0; i < n; i++)
    if (!compression || compression[i] == 8) { defl.push_back((uint32_t)i); ds.push_back(d_src[i]); dlen.push_back(src_len[i]); }
  const size_t nd = defl.size();
  std::vector<size_t> dclen(nd);
  std::vector<uint32_t> dcrc(nd);
  std::vector<int> dst_m(nd);
  if (int st = deflate_members(ctx, level, ZIPC_CK_CRC32, 0, nd, ds, dlen.data(), dclen.data(), dcrc.data(), dst_m.data(), a.pc)) return st;
  for (int s : dst_m) if (s) return s;
  for (uint32_t &i : a.pc.member) i = defl[i];
  std::vector<size_t> clen(src_len, src_len + n);
  std::vector<uint32_t> crc(n, 0);
  for (size_t k = 0; k < nd; k++) { clen[defl[k]] = dclen[k]; crc[defl[k]] = dcrc[k]; }
  archive_members(n, norm, compression, mode, mtime, src_len, clen.data(), crc.data(), a.ms);
  if (int st = make_layout(a.ms.data(), n, first, flags, a.L)) return st;
  a.poff = payload_offsets(a.ms, a.L);
  *out_len = (size_t)a.L.total;
  return ZIPC_OK;
}
// The planned archive into device memory at out (a.L.total bytes): the deflate pieces by place_pieces, the stored members
// from d_src by stored_copy_crc (copy and CRC-32 in one pass), then the headers and end records by zip_headers_kernel from one
// record per member and the names behind them, one upload.  Shadowed members are not written.  The stream is through on return.
int write_archive(zipc_b200_ctx *ctx, ArchivePlan &a, const std::vector<const uint8_t *> &d_src, uint8_t *out) {
  const size_t n = a.ms.size();
  std::vector<uint8_t *> to(n, nullptr);
  std::vector<uint32_t> stored;
  std::vector<const uint8_t *> s_src;
  std::vector<uint8_t *> s_dst;
  std::vector<uint64_t> s_len;
  for (size_t i = 0; i < n; i++) {
    if (a.poff[i] == ~0ull) continue;
    if (a.ms[i].compression == 8) to[i] = out + a.poff[i];
    else { stored.push_back((uint32_t)i); s_src.push_back(d_src[i]); s_dst.push_back(out + a.poff[i]); s_len.push_back(a.ms[i].compressed_size); }
  }
  if (int st = place_pieces(ctx, a.pc, to)) return st;
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));  // (place_pieces)
  std::vector<uint32_t> s_crc(stored.size());
  if (int st = stored_copy_crc(ctx, stored.size(), s_src.data(), s_dst.data(), s_len.data(), s_crc.data())) return st;
  for (size_t k = 0; k < stored.size(); k++) a.ms[stored[k]].crc32 = s_crc[k];
  const Layout &L = a.L;
  const size_t m = L.ord.size();
  size_t name_bytes = 0;
  for (size_t i : L.ord) name_bytes += a.ms[i].path_len;
  const size_t rec_bytes = m * sizeof(ZipHdr);
  if (int st = ctx->h_desc.reserve(rec_bytes + name_bytes)) return st;
  if (int st = ctx->d_desc2.reserve(rec_bytes + name_bytes)) return st;
  ZipHdr *hh = ctx->h_desc.as<ZipHdr>();
  char *hn = reinterpret_cast<char *>(hh + m);
  for (size_t j = 0, at = 0; j < m; j++) {
    const zipc_b200_member &mb = a.ms[L.ord[j]];
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

}  // namespace

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
  if (int st = ctx->d_out.reserve(total + 64)) return st;
  if (int st = place_pieces(ctx, pc, slot_addrs(ctx->d_out.as<uint8_t>(), off.data(), n))) return st;
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
  if (int st = place_pieces(ctx, pc, slot_addrs(ctx->d_out.as<uint8_t>(), off.data(), n), ad.data(), level)) return st;
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
  if (int st = place_pieces(ctx, pc, to, ad.data(), level)) return st;
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));  // (place_pieces)
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
  std::vector<const uint8_t *> d_src;
  std::vector<size_t> slen, cap;
  std::vector<uint32_t> flags;
  cut_segments(d_base, len, segment_size, primed, last_piece != 0, d_src, slen, flags);
  Pieces pc;  // the pieces of one member, stream 0
  pc.member.assign(nseg, 0);
  pc.len.resize(nseg);
  std::vector<int> st_m(nseg);
  if (int st = make_slots(ctx, nseg, slen.data(), pc.d_slot, cap)) return st;
  if (int st = deflate_run(ctx, level, ZIPC_CK_NONE, 0, nseg, d_src, slen.data(), pc.d_slot, cap, pc.len.data(), nullptr, st_m.data(), &flags)) return st;
  for (size_t i = 0; i < nseg; i++) if (st_m[i]) return st_m[i];
  if (crc32)
    if (int st = crc32_to_host_word(ctx, d_base, len)) return st;
  // the pieces are byte aligned: concatenate without gaps
  pc.rel.resize(nseg);
  size_t total = 0;
  for (size_t i = 0; i < nseg; i++) { pc.rel[i] = total; total += pc.len[i]; }
  if (index) {
    for (size_t i = 0; i < nseg; i++) { index[2 * i] = pc.rel[i]; index[2 * i + 1] = (uint64_t)i * segment_size; }
    index[2 * nseg] = total; index[2 * nseg + 1] = len;
  }
  if (int st = ctx->d_out.reserve(total + 64)) return st;
  if (int st = place_pieces(ctx, pc, {ctx->d_out.as<uint8_t>()})) return st;
  const int rc = finish_to_host(ctx, {}, total, dst, dst_cap, nullptr, dst_len);
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
      std::vector<size_t> poff(n), clen(n);
      std::vector<uint32_t> crc(n);
      std::vector<int> st_m(n);
      size_t need = 0;
      const uint64_t l0 = pipeline_launches(pipe);
      const int rc = pipeline_deflate_gapped(pipe, level, n, src, src_len, gap.data(), out, out_cap, &need, poff.data(), clen.data(), crc.data(), st_m.data());
      ctx->launches += pipeline_launches(pipe) - l0;
      if (rc == ZIPC_OK) {
        for (size_t i = 0; i < n; i++) if (st_m[i]) return st_m[i];
        std::vector<zipc_b200_member> ms;
        archive_members(n, norm, nullptr, mode, mtime, src_len, clen.data(), crc.data(), ms);
        Layout L;
        if (int st = make_layout(ms.data(), n, first, flags, L)) return st;
        const std::vector<uint64_t> want = payload_offsets(ms, L);
        if (std::equal(want.begin(), want.end(), poff.begin())) return zip_assemble_impl(ms.data(), n, first, out, out_cap, out_len, false, flags);
      } else if (rc != ZIPC_ERR_DST_TOO_SMALL) {
        return rc;
      }
      // (too small for the payloads, or not where the layout wants them: the plain path below reports / redoes it)
    }
  }
  // the device call's steps between an upload and a download
  std::vector<const uint8_t *> d_src;
  if (int st = upload_ranges(ctx, n, src, src_len, d_src)) return st;
  ArchivePlan a;
  if (int st = plan_archive(ctx, level, n, norm, d_src, src_len, nullptr, mode, mtime, first, flags, out_len, a)) return st;
  if (!out || out_cap < a.L.total) return ZIPC_ERR_DST_TOO_SMALL;
  if (int st = ctx->d_out.reserve(a.L.total + 64)) return st;
  if (int st = write_archive(ctx, a, d_src, ctx->d_out.as<uint8_t>())) return st;
  return d2h(ctx, out, ctx->d_out.p, a.L.total);
}

// The archive of zipc_b200_zip_deflate_archive_ex written into device memory from device payloads, stored members allowed:
// plan_archive, then write_archive into the caller's buffer.  The deflate members are compressed as the host call compresses
// them, the layout is the host assembler's (make_layout), and the GPU places everything.
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
  const std::vector<const uint8_t *> d_src = slot_addrs(static_cast<const uint8_t *>(d_src_v), src_off, n);
  ArchivePlan a;
  if (int st = plan_archive(ctx, level, n, norm, d_src, src_len, compression, mode, mtime, first, flags, out_len, a)) return st;
  if (out_cap < a.L.total) return ZIPC_ERR_DST_TOO_SMALL;
  return write_archive(ctx, a, d_src, static_cast<uint8_t *>(d_out_v));
}

}  // extern "C"
