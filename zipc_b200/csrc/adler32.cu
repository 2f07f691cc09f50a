// adler32.cu -- Adler-32 at HBM bandwidth, in both the reference's flavour and RFC 1950's.
//
// Replaces Zipc_deflate.Adler_32.string / string_update (reference src/zipc_deflate.ml:166-206).
// The reference walks the buffer in 5552-byte chunks (first chunk = len mod 5552), keeps s1, s2
// as wrapping int32 and reduces them with the *signed* Int32.rem at each chunk end
// (zipc_deflate.ml:95,196).  That only differs from RFC 1950 when a chunk pushes s2 past 2^31.
//
// Device part (this file, bandwidth bound): one warp per chunk computes
//      A = sum b_i                  B = sum (n - i) * b_i          (i = 0..n-1, n <= 5552)
// with dp4a over coalesced 16-byte loads.  B < 2^32 always (255*5552*5553/2 = 3.93e9).
// Fold part (0.14 % of the bytes: 8 bytes per 5552): the chunk recurrence
//      s1' = rem(s1 + A)            s2' = rem(s2 + n*s1 + B)        (int32 wrap, then rem)
// is evaluated over the per-chunk (A, B) pairs; in REF_COMPAT mode it is order dependent (sign
// of the wrapped s2) and is therefore done as a scalar scan over the partials, in RFC1950 mode it
// is the same scan with unsigned arithmetic.
//
// Algorithmic bytes per launch: N.  Roofline: HBM.
#include "common.cuh"
#include "adler_core.cuh"

namespace zb {
namespace {

constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;
constexpr uint32_t kChunk = 5552;

// chunk c of a single buffer: c == 0 -> [0, first), else [first + (c-1)*5552, +5552)   (first may
// equal 5552 when len is a multiple of it; an empty first round is a no-op and is skipped)
__global__ void __launch_bounds__(kThreads)
adler_chunks_kernel(const uint8_t *__restrict__ src, uint32_t first, uint32_t nchunks, uint2 *__restrict__ ab) {
  const int lane = threadIdx.x & 31;
  for (uint32_t c = blockIdx.x * kWarps + (threadIdx.x >> 5); c < nchunks; c += gridDim.x * kWarps) {
    uint64_t off = c == 0 ? 0 : (uint64_t)first + (uint64_t)(c - 1) * kChunk;
    uint32_t n = c == 0 ? first : kChunk;
    uint32_t A, B;
    adler_range_warp<false>(src + off, n, lane, A, B);
    if (lane == 0) ab[c] = make_uint2(A, B);
  }
}

// arbitrary ranges (ptr, len <= 5552)
__global__ void __launch_bounds__(kThreads)
adler_ranges_kernel(const AdlerSeg *__restrict__ segs, uint32_t nseg, uint2 *__restrict__ ab) {
  const int lane = threadIdx.x & 31;
  for (uint32_t c = blockIdx.x * kWarps + (threadIdx.x >> 5); c < nseg; c += gridDim.x * kWarps) {
    uint32_t A, B;
    adler_range_warp<false>(segs[c].ptr, segs[c].len, lane, A, B);
    if (lane == 0) ab[c] = make_uint2(A, B);
  }
}


// ---- device-side fold of the per-chunk partial sums ----------------------------------------------------------
// s1 never wraps (s1 + A < 2^21), so s1 before chunk c is (1 + prefix sum of A) mod 65521: a scan.
// s2' = srem(wrap32(s2 + W)), W = n * s1_before + B < 2^32.  Writing s2 as (residue r, negative?):
//   M <= W < 2^31 - M   : no wrap whatever s2 is      -> r' = r + W,      result non-negative   ("L")
//   W >= 2^31 + M       : always wraps to a negative  -> r' = r + W - K,  result negative       ("H"), K = 2^32 mod M
//   W < M               : no wrap; stays non-negative if s2 was non-negative (a carry chain, resolved by a scan)
//   anything else       : depends on the exact s2 -> resolved serially, in order ("U"; ~4e-4 of chunks on random data)
// RFC 1950 mode is the same scan with every chunk treated as "L" and exact arithmetic.
constexpr int kFoldThreads = 1024;
constexpr int kFoldItems = 16;                        // consecutive chunks per thread -> 128-byte coalesced loads; fewer, larger tiles
constexpr int kFoldTile = kFoldThreads * kFoldItems;  // chunks per pass of the CTA
constexpr uint32_t kM = 65521u;
constexpr int kFoldSmem = kFoldTile * 7;

struct OpAddMod {
  __device__ __forceinline__ uint32_t operator()(uint32_t earlier, uint32_t later) const {
    uint32_t x = earlier + later;
    return x >= kM ? x - kM : x;
  }
};
// (g,p) in bits 1,0: g = "known non-negative afterwards", p = "sign passes through unchanged"
struct OpCarry {
  __device__ __forceinline__ uint32_t operator()(uint32_t earlier, uint32_t later) const {
    uint32_t g = (later >> 1) | (later & (earlier >> 1) & 1u);
    return (g & 1u) << 1 | (earlier & later & 1u);
  }
  static constexpr uint32_t identity = 1u;
};

// inclusive scan over the CTA (one value per thread); *total = reduction over all threads
template <typename Op>
__device__ __forceinline__ uint32_t block_scan(uint32_t v, uint32_t *scratch, uint32_t *total) {
  Op op;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x = op(t, x);
  }
  __syncthreads();  // scratch free again
  if (lane == 31) scratch[warp] = x;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = scratch[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w = op(t, w);
    }
    scratch[32 + lane] = w;
  }
  __syncthreads();
  *total = scratch[63];
  return warp ? op(scratch[32 + warp - 1], x) : x;
}

// One CTA per tile of kFoldTile chunks.  Everything that does not need the state before the tile runs in parallel over the
// tiles; what does is passed down a chain of tagged 64-bit words in global memory (tag = this launch's epoch, so nothing has
// to be cleared between calls):
//   chain_a[t] = byte-sum of tile t (mod M): every later tile adds up its predecessors' entries to know s1 at its start;
//   chain_s[t] = s2 after tile t (residue, sign): tile t + 1 waits for it only at the very end, for the handful of chunks
//                whose outcome depends on the exact s2 ("U"), which one thread walks through a dense list.
// Tiles are numbered in the order the CTAs start (a counter), so a tile only ever waits for tiles that are already running.
__device__ __forceinline__ uint64_t chain_wait(const uint64_t *p, uint32_t epoch) {
  uint64_t v;
  do { asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory"); } while ((uint32_t)(v >> 32) != epoch);
  return v;
}
__device__ __forceinline__ void chain_post(uint64_t *p, uint32_t epoch, uint32_t payload) {
  const uint64_t v = ((uint64_t)epoch << 32) | payload;
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(kFoldThreads, 1)
adler_fold_kernel(const uint2 *__restrict__ ab, uint32_t first, uint32_t nchunks, uint32_t epoch, unsigned int *__restrict__ counter,
                  uint64_t *__restrict__ chain_a, uint64_t *__restrict__ chain_s, uint32_t *__restrict__ out) {
  __shared__ uint32_t scratch[64];
  extern __shared__ __align__(16) uint8_t fold_smem[];  // kFoldSmem bytes: the tile's U chunks, in order: W, residue before, where the sign comes from
  uint32_t *uW = reinterpret_cast<uint32_t *>(fold_smem);
  uint16_t *uR = reinterpret_cast<uint16_t *>(fold_smem + kFoldTile * 4);
  uint8_t *uF = fold_smem + kFoldTile * 6;
  __shared__ uint8_t lastk[kFoldThreads];
  __shared__ uint32_t s_tile, s_nn, s_klast;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t K = (uint32_t)((1ull << 32) % kM);
  if (tid == 0) s_tile = atomicAdd(counter, 1u);
  __syncthreads();
  const uint32_t tile = s_tile, ntiles = gridDim.x;
  const uint32_t t0 = tile * kFoldTile, base = t0 + tid * kFoldItems;
  const int last = (int)min((uint32_t)kFoldTile, nchunks - t0) - 1;  // index of the tile's last chunk

  uint32_t A[kFoldItems], B[kFoldItems];
  if (base + kFoldItems <= nchunks) {
    const uint4 *p = reinterpret_cast<const uint4 *>(ab + base);  // 64-byte aligned: base is a multiple of 8
#pragma unroll
    for (int i = 0; i < kFoldItems / 2; i++) {
      uint4 u = p[i];
      A[2 * i] = u.x; B[2 * i] = u.y; A[2 * i + 1] = u.z; B[2 * i + 1] = u.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < kFoldItems; i++) {
      uint2 e = base + i < nchunks ? ab[base + i] : make_uint2(0u, 0u);
      A[i] = e.x; B[i] = e.y;
    }
  }
  // s1 before every chunk: the tile's own prefix sums, then the sums of the tiles before it
  uint32_t pa[kFoldItems], asum = 0;
#pragma unroll
  for (int i = 0; i < kFoldItems; i++) { pa[i] = asum; asum += A[i] % kM; }
  asum %= kM;
  uint32_t atot;
  const uint32_t ainc = block_scan<OpAddMod>(asum, scratch, &atot);
  if (tid == 0) chain_post(chain_a + tile, epoch, atot);
  uint32_t before = 0;
  for (uint32_t j = tid; j < tile; j += kFoldThreads) before = (before + (uint32_t)chain_wait(chain_a + j, epoch)) % kM;
  uint32_t s1_carry;
  block_scan<OpAddMod>(before, scratch, &s1_carry);
  s1_carry = (s1_carry + 1u) % kM;
  const uint32_t s1_thread = (s1_carry + ainc + kM - asum) % kM;
  // W, class
  uint32_t W[kFoldItems], k[kFoldItems], gp = OpCarry::identity;
#pragma unroll
  for (int i = 0; i < kFoldItems; i++) {
    uint32_t s1 = (s1_thread + pa[i]) % kM;
    uint32_t n = base + i == 0 ? first : 5552u;
    W[i] = n * s1 + B[i];  // < 2^32: 5552*65520 + 255*5552*5553/2
    uint32_t c;
    if (base + i >= nchunks) c = 4;                                    // past the end: identity
    else if (W[i] >= kM && W[i] < 0x80000000u - kM) c = 0;             // L
    else if (W[i] >= 0x80000000u + kM) c = 1;                          // H
    else if (W[i] < kM) c = 2;                                         // low W
    else c = 3;                                                        // U
    k[i] = c;
    if (c == 0) gp = 2u; else if (c == 1 || c == 3) gp = 0u;
  }
  uint32_t gtot;
  const uint32_t ginc = block_scan<OpCarry>(gp, scratch, &gtot);
  uint32_t gexc = __shfl_up_sync(0xffffffffu, ginc, 1);
  if (lane == 0) gexc = warp ? scratch[32 + warp - 1] : OpCarry::identity;
  // low-W chunks at the head of the tile (nothing before them fixes the sign) need the sign before the tile: the only
  // case in which the whole CTA waits for its predecessor (zero-filled data behind a negative state)
  bool open_head = (gexc & 3u) == 1u, needs = false;
#pragma unroll
  for (int i = 0; i < kFoldItems; i++) {
    if (k[i] == 2 && open_head) needs = true;
    if (k[i] != 2 && k[i] != 4) open_head = false;
  }
  uint32_t neg_in = 0, r_carry = 0;
  bool have_pred = tile == 0;
  if (__syncthreads_or(needs) && tile) {
    if (tid == 0) s_nn = (uint32_t)chain_wait(chain_s + tile - 1, epoch);
    __syncthreads();
    neg_in = s_nn >> 17; r_carry = s_nn & 0x1FFFFu; have_pred = true;
  }
  uint32_t nn_in = (gexc >> 1) | (gexc & (neg_in ^ 1u) & 1u);
  // resolve low-W chunks, deltas
  uint32_t pd[kFoldItems], dsum = 0, nu = 0;
#pragma unroll
  for (int i = 0; i < kFoldItems; i++) {
    if (k[i] == 2) k[i] = nn_in ? 0u : 3u;
    if (k[i] != 4) nn_in = k[i] == 0;
    nu += k[i] == 3;
    pd[i] = dsum;
    uint32_t w = W[i] % kM;
    dsum += k[i] == 0 ? w : k[i] == 1 ? (w + kM - K) % kM : 0u;
  }
  dsum %= kM;
  uint32_t dtot;
  const uint32_t dinc = block_scan<OpAddMod>(dsum, scratch, &dtot);
  const uint32_t r_thread = (dinc + kM - dsum) % kM;   // residue before the thread's chunks, without the tile's carry-in
  // the U chunks, in order
  lastk[tid] = (uint8_t)k[kFoldItems - 1];
  if (tid == last / kFoldItems) {
#pragma unroll
    for (int i = 0; i < kFoldItems; i++)
      if (i == last % kFoldItems) s_klast = k[i];
  }
  uint32_t nutot;
  {
    // (plain sums: at most kFoldTile)
    uint32_t x = nu;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += t; }
    __syncthreads();
    if (lane == 31) scratch[warp] = x;
    __syncthreads();
    if (warp == 0) {
      uint32_t w = scratch[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
      scratch[32 + lane] = w;
    }
    __syncthreads();
    nutot = scratch[63];
    uint32_t at = (warp ? scratch[32 + warp - 1] : 0u) + x - nu;
    if (nu) {
#pragma unroll
      for (int i = 0; i < kFoldItems; i++) {
        if (k[i] != 3) continue;
        const uint32_t kp = i ? k[i - 1] : tid ? (uint32_t)lastk[tid - 1] : 5u;
        uW[at] = W[i];
        uR[at] = (uint16_t)((r_thread + pd[i]) % kM);
        uF[at] = (uint8_t)(kp == 0 ? 0 : kp == 1 ? 1 : kp == 3 ? 2 : 3);   // sign before: +, -, the walk's own, the tile's carry-in
        at++;
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    if (!have_pred) {
      const uint32_t v = (uint32_t)chain_wait(chain_s + tile - 1, epoch);
      neg_in = v >> 17; r_carry = v & 0x1FFFFu;
    }
    bool neg = neg_in != 0;
    uint32_t c = 0;
    for (uint32_t e = 0; e < nutot; e++) {
      const uint32_t f = uF[e];
      if (f == 0) neg = false; else if (f == 1) neg = true; else if (f == 3) neg = neg_in != 0;
      const uint32_t rf = (uR[e] + r_carry) % kM, r = (rf + c) % kM;
      const long long v = (neg && r) ? (long long)r - kM : (long long)r;
      const long long X = v + (long long)uW[e];
      const long long Y = X >= (1ll << 31) ? X - (1ll << 32) : X;
      const uint32_t m = (uint32_t)(Y < 0 ? -Y : Y) % kM;  // |Y| < 2^31 + M
      neg = Y < 0;
      const uint32_t r2 = neg && m ? kM - m : m;
      c = (r2 + kM - rf) % kM;
    }
    // sign after the tile: the walk's if the last chunk was a U chunk, else what the last chunk's class says
    const uint32_t neg_out = s_klast == 3 ? (uint32_t)neg : (uint32_t)(s_klast == 1);
    const uint32_t r_out = (r_carry + dtot + c) % kM;
    if (tile + 1 < ntiles) chain_post(chain_s + tile, epoch, (neg_out << 17) | r_out);
    else {
      const uint32_t s1 = (s1_carry + atot) % kM;
      const uint32_t s2 = (neg_out && r_out) ? r_out - kM : r_out;
      *out = (s2 << 16) + s1;
      *counter = 0;
    }
  }
}
// ---- RFC 1950 mode: the chunk recurrence is a plain reduction ------------------------------------------------------------
// With exact arithmetic a run of chunks acts on (s1, s2) as s1' = s1 + A, s2' = s2 + N s1 + B  (N = bytes, A = byte sum,
// B = weighted sum), and two runs compose associatively: (N1, A1, B1) then (N2, A2, B2) = (N1 + N2, A1 + A2, B1 + B2 + N2 A1),
// all modulo 65521.  So the per-chunk pairs are reduced in order by a tree: thread (8 chunks) -> warp -> CTA -> the last CTA
// to finish combines the CTA results.  (The reference's signed remainder makes the same recurrence order dependent; that
// flavour keeps the scan of adler_fold_kernel.)
struct Seg { uint32_t n, a, b; };
__device__ __forceinline__ Seg seg_join(Seg l, Seg r) {
  Seg o;
  o.n = (l.n + r.n) % kM;
  o.a = (l.a + r.a) % kM;
  o.b = (uint32_t)(((uint64_t)l.b + r.b + (uint64_t)r.n * l.a) % kM);
  return o;
}
constexpr int kRedThreads = 1024, kRedItems = 8;
__global__ void __launch_bounds__(kRedThreads)
adler_reduce_rfc_kernel(const uint2 *__restrict__ ab, uint32_t first, uint32_t nchunks, Seg *__restrict__ cta_seg,
                        unsigned int *__restrict__ ticket, uint32_t *__restrict__ out) {
  __shared__ Seg warp_seg[32];
  __shared__ bool last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t base = (blockIdx.x * kRedThreads + tid) * kRedItems;
  Seg s{0, 0, 0};
#pragma unroll
  for (int i = 0; i < kRedItems; i++) {
    const uint32_t c = base + i;
    if (c < nchunks) {
      const uint2 e = ab[c];
      s = seg_join(s, Seg{(c == 0 ? first : kChunk) % kM, e.x % kM, e.y % kM});
    }
  }
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {  // ordered tree: lane l joins with lane l + o on its right
    Seg r;
    r.n = __shfl_down_sync(0xffffffffu, s.n, o); r.a = __shfl_down_sync(0xffffffffu, s.a, o); r.b = __shfl_down_sync(0xffffffffu, s.b, o);
    if ((lane & (2 * o - 1)) == 0) s = seg_join(s, r);
  }
  if (lane == 0) warp_seg[warp] = s;
  __syncthreads();
  if (warp == 0) {
    s = warp_seg[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      Seg r;
      r.n = __shfl_down_sync(0xffffffffu, s.n, o); r.a = __shfl_down_sync(0xffffffffu, s.a, o); r.b = __shfl_down_sync(0xffffffffu, s.b, o);
      if ((lane & (2 * o - 1)) == 0) s = seg_join(s, r);
    }
    if (lane == 0) {
      cta_seg[blockIdx.x] = s;
      __threadfence();
      last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
  }
  __syncthreads();
  if (last && tid == 0) {  // a few dozen CTA results, in order
    __threadfence();
    Seg t{0, 0, 0};
    for (uint32_t i = 0; i < gridDim.x; i++) t = seg_join(t, *(volatile Seg *)&cta_seg[i]);
    const uint32_t s1 = (1u + t.a) % kM, s2 = (t.n + t.b) % kM;  // from (s1, s2) = (1, 0)
    *out = (s2 << 16) + s1;
    *ticket = 0;
  }
}

}  // namespace

int adler32_launch_buffer(zipc_b200_ctx *ctx, const uint8_t *d_src, uint64_t len, int mode, uint32_t *h_out) {
  if (len == 0) { *h_out = 1; return ZIPC_OK; }
  uint32_t first = (uint32_t)(len % kChunk);
  if (first == 0) first = kChunk;
  uint64_t nchunks64 = 1 + (len - first) / kChunk;
  if (nchunks64 > 0xFFFFFFFFull) return ZIPC_ERR_INVALID_ARG;
  uint32_t nchunks = (uint32_t)nchunks64;
  if (int st = ctx->d_scratch2.reserve((size_t)nchunks * sizeof(uint2) + 64)) return st;
  uint2 *d_ab = ctx->d_scratch2.as<uint2>();
  uint32_t grid = (nchunks + kWarps - 1) / kWarps;
  uint32_t maxgrid = (uint32_t)ctx->sm_count * 4;
  if (grid > maxgrid) grid = maxgrid;
  {
    KernelTimer kt(ctx);
    adler_chunks_kernel<<<grid, kThreads, 0, ctx->stream>>>(d_src, first, nchunks, d_ab);
  }
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  // the result is one word: the last thread of the fold / reduction stores it straight into mapped host memory (a posted write
  // over PCIe) -- no copy operation, and no staging of a 4-byte copy into the caller's pageable word -- and the host reads it
  // once the stream is through
  if (int st = map_host_word(ctx)) return st;
  uint32_t *d_out = ctx->h_word;
  if (mode == ZIPC_ADLER_RFC1950) {
    // exact arithmetic: an ordered reduction over all SMs' worth of threads
    const uint32_t rgrid = (nchunks + kRedThreads * kRedItems - 1) / (kRedThreads * kRedItems);
    if (int st = ctx->d_adler.reserve(64 + (size_t)rgrid * sizeof(Seg))) return st;
    unsigned int *ticket = ctx->d_adler.as<unsigned int>();
    if (ctx->adler_ticket_at != (void *)ticket) { ZB_CUDA(ctx, cudaMemsetAsync(ticket, 0, sizeof(unsigned int), ctx->stream)); ctx->adler_ticket_at = ticket; }
    Seg *cta_seg = reinterpret_cast<Seg *>(ctx->d_adler.as<uint8_t>() + 64);
    adler_reduce_rfc_kernel<<<rgrid, kRedThreads, 0, ctx->stream>>>(d_ab, first, nchunks, cta_seg, ticket, d_out);
  } else {
    // the reference's flavour: one CTA per tile of chunks, the order-dependent part handed down a chain (no host round trip)
    const uint32_t ntiles = (nchunks + kFoldTile - 1) / kFoldTile;
    const size_t need = 64 + 2 * (size_t)ntiles * sizeof(uint64_t);
    if (need > ctx->d_adler_chain.cap) {  // tags of earlier launches must survive, fresh memory must read as "no tag"
      if (int st = ctx->d_adler_chain.reserve(2 * need)) return st;
      ZB_CUDA(ctx, cudaMemsetAsync(ctx->d_adler_chain.p, 0, ctx->d_adler_chain.cap, ctx->stream));
      ctx->adler_epoch = 0;
    }
    if (++ctx->adler_epoch == 0) {  // 2^32 launches later: start over
      ZB_CUDA(ctx, cudaMemsetAsync(ctx->d_adler_chain.p, 0, ctx->d_adler_chain.cap, ctx->stream));
      ctx->adler_epoch = 1;
    }
    unsigned int *counter = ctx->d_adler_chain.as<unsigned int>();
    uint64_t *chain_a = reinterpret_cast<uint64_t *>(ctx->d_adler_chain.as<uint8_t>() + 64), *chain_s = chain_a + ntiles;
    ZB_CUDA(ctx, cudaFuncSetAttribute(adler_fold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFoldSmem));  // per device
    adler_fold_kernel<<<ntiles, kFoldThreads, kFoldSmem, ctx->stream>>>(d_ab, first, nchunks, ctx->adler_epoch, counter, chain_a, chain_s, d_out);
  }
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  *h_out = *reinterpret_cast<volatile uint32_t *>(ctx->h_word);
  return ZIPC_OK;
}

int adler32_ranges(zipc_b200_ctx *ctx, const uint8_t *const *d_ptrs, const uint64_t *lens, size_t n, int mode,
                   uint32_t *h_out) {
  // chunk every range on the reference's grid (first chunk = len mod 5552)
  size_t total = 0;
  for (size_t i = 0; i < n; i++) total += lens[i] ? 1 + (lens[i] - 1) / kChunk : 0;
  if (total > 0xFFFFFFFFull) return ZIPC_ERR_INVALID_ARG;
  if (total == 0) { for (size_t i = 0; i < n; i++) h_out[i] = 1; return ZIPC_OK; }
  if (int st = ctx->h_desc.reserve(total * sizeof(AdlerSeg))) return st;
  if (int st = ctx->d_desc.reserve(total * sizeof(AdlerSeg))) return st;
  if (int st = ctx->d_scratch2.reserve(total * sizeof(uint2))) return st;
  if (int st = ctx->h_res.reserve(total * sizeof(uint2))) return st;
  AdlerSeg *h = ctx->h_desc.as<AdlerSeg>();
  size_t k = 0;
  for (size_t i = 0; i < n; i++) {
    uint64_t len = lens[i], off = 0;
    if (!len) continue;
    uint32_t first = (uint32_t)(len % kChunk);
    if (first == 0) first = kChunk;
    for (uint32_t m = first; off < len; off += m, m = kChunk) { h[k].ptr = d_ptrs[i] + off; h[k].len = m; h[k]._pad = 0; k++; }
  }
  ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_desc.p, h, total * sizeof(AdlerSeg), cudaMemcpyHostToDevice, ctx->stream));
  uint32_t grid = (uint32_t)((total + kWarps - 1) / kWarps);
  uint32_t maxgrid = (uint32_t)ctx->sm_count * 4;
  if (grid > maxgrid) grid = maxgrid;
  adler_ranges_kernel<<<grid, kThreads, 0, ctx->stream>>>(ctx->d_desc.as<AdlerSeg>(), (uint32_t)total, ctx->d_scratch2.as<uint2>());
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  uint2 *h_ab = ctx->h_res.as<uint2>();
  ZB_CUDA(ctx, cudaMemcpyAsync(h_ab, ctx->d_scratch2.p, total * sizeof(uint2), cudaMemcpyDeviceToHost, ctx->stream));
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  k = 0;
  for (size_t i = 0; i < n; i++) {
    uint32_t s1 = 1, s2 = 0;
    uint64_t len = lens[i], off = 0;
    if (len) {
      uint32_t first = (uint32_t)(len % kChunk);
      if (first == 0) first = kChunk;
      for (uint32_t m = first; off < len; off += m, m = kChunk, k++) adler_fold_step(s1, s2, m, h_ab[k].x, h_ab[k].y, mode);
    }
    h_out[i] = (s2 << 16) + s1;
  }
  return ZIPC_OK;
}

int adler32_blocked(zipc_b200_ctx *ctx, const uint8_t *const *d_ptrs, const uint32_t *nblk, const uint32_t *blk_len,
                    size_t n, int mode, uint32_t *h_out) {
  // every block is chunked on its own grid (first chunk = block length mod 5552), exactly what Adler_32.string_update
  // does when the reference calls it once per block with the packed state of the previous block
  size_t total = 0, nb = 0;
  for (size_t i = 0; i < n; i++)
    for (uint32_t b = 0; b < nblk[i]; b++, nb++) total += blk_len[nb] ? 1 + (blk_len[nb] - 1) / kChunk : 0;
  if (total > 0xFFFFFFFFull) return ZIPC_ERR_INVALID_ARG;
  if (total == 0) { for (size_t i = 0; i < n; i++) h_out[i] = 1; return ZIPC_OK; }
  if (int st = ctx->h_desc.reserve(total * sizeof(AdlerSeg))) return st;
  if (int st = ctx->d_desc.reserve(total * sizeof(AdlerSeg))) return st;
  if (int st = ctx->d_scratch2.reserve(total * sizeof(uint2))) return st;
  if (int st = ctx->h_res.reserve(total * sizeof(uint2))) return st;
  AdlerSeg *h = ctx->h_desc.as<AdlerSeg>();
  size_t k = 0;
  nb = 0;
  for (size_t i = 0; i < n; i++) {
    uint64_t off = 0;
    for (uint32_t b = 0; b < nblk[i]; b++, nb++) {
      const uint32_t len = blk_len[nb];
      if (!len) continue;
      uint32_t m = len % kChunk;
      if (m == 0) m = kChunk;
      for (uint32_t done = 0; done < len; done += m, m = kChunk) { h[k].ptr = d_ptrs[i] + off + done; h[k].len = m; h[k]._pad = 0; k++; }
      off += len;
    }
  }
  ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_desc.p, h, total * sizeof(AdlerSeg), cudaMemcpyHostToDevice, ctx->stream));
  uint32_t grid = (uint32_t)((total + kWarps - 1) / kWarps);
  uint32_t maxgrid = (uint32_t)ctx->sm_count * 4;
  if (grid > maxgrid) grid = maxgrid;
  adler_ranges_kernel<<<grid, kThreads, 0, ctx->stream>>>(ctx->d_desc.as<AdlerSeg>(), (uint32_t)total, ctx->d_scratch2.as<uint2>());
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  uint2 *h_ab = ctx->h_res.as<uint2>();
  ZB_CUDA(ctx, cudaMemcpyAsync(h_ab, ctx->d_scratch2.p, total * sizeof(uint2), cudaMemcpyDeviceToHost, ctx->stream));
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  k = 0;
  nb = 0;
  for (size_t i = 0; i < n; i++) {
    uint32_t state = 1;
    for (uint32_t b = 0; b < nblk[i]; b++, nb++) {
      const uint32_t len = blk_len[nb];
      if (!len) continue;
      uint32_t s1 = state & 0xFFFFu, s2 = state >> 16;  // the state is re-packed between blocks (zipc_deflate.ml:178,198)
      uint32_t m = len % kChunk;
      if (m == 0) m = kChunk;
      for (uint32_t done = 0; done < len; done += m, m = kChunk, k++) adler_fold_step(s1, s2, m, h_ab[k].x, h_ab[k].y, mode);
      state = (s2 << 16) + s1;
    }
    h_out[i] = state;
  }
  return ZIPC_OK;
}

}  // namespace zb
