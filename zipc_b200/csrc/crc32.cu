// crc32.cu -- CRC-32 (ZIP / ISO-HDLC, reflected 0xedb88320) at HBM bandwidth on sm_100a.
//
// Replaces Zipc_deflate.Crc_32.string / string_update (reference src/zipc_deflate.ml:106-164),
// which walks the buffer 4 bytes per step through one serial dependency.
//
// Decomposition (all integer, bit-exact by linearity of the CRC over GF(2)):
//   * The input is cut into segments (a ZIP member, or a tile of a large buffer).  One warp owns
//     one segment at a time.
//   * Inside a segment the 16-byte-aligned body is viewed as rows of 512 bytes = 32 lanes x 16 B.
//     Lane l reads its 16 bytes of every row with one coalesced LDG.128 and keeps FOUR running
//     states, one per 32-bit slot.  Each (lane, slot) column is therefore a sub-message whose words
//     are 512 bytes apart; its state is advanced with slice-by-4 tables that already contain the
//     508 zero bytes between consecutive words:  T'_k[b] = T_k[b] * x^(8*508) mod P.
//     That is 4 shared-memory lookups per 4 input bytes with no dependence between columns.
//   * The 4 x 256 strided tables are replicated once per lane ( [k/2][byte][k%2][lane] ), so a warp's 32
//     simultaneous lookups always hit 32 different banks: the LDS pipe runs conflict-free at one
//     lookup per lane per clock, and a lookup's address is one PRMT away from the data word.
//     128 KiB of shared memory, one 1024-thread CTA per SM.
//   * Each lane's last block is advanced with the ordinary tables, the four slots are merged
//     (3 x "append 4 zero bytes"), lanes are aligned to the end of the body by one GF(2)[x]
//     multiplication with x^(128*d), d in [0,31], and XOR-reduced over the warp.
//   * Large buffers: one tile per warp; tile states are merged by a small second kernel with a
//     Horner + tree scheme over x^(8*L) (crc32_combine_tiles).
//   * Stored ZIP members (stored_copy_crc_kernel): the same warp loop also writes every 16-byte word it
//     loaded to the member's output slot, so a payload is read once and written once (2N bytes) while
//     its CRC-32 is computed.  Members are cut into tiles of kStoredTile bytes, one warp each; every warp
//     advances its tile's state over the bytes of the member that follow the tile and XORs it into the
//     member's word.
//
// Algorithmic bytes per launch: N (every input byte is read exactly once, nothing is written
// but 4 bytes per segment).  Roofline: HBM.
#include "common.cuh"

namespace zb {

// ---------------------------------------------------------------------------------------------
// host-side GF(2) helpers
// ---------------------------------------------------------------------------------------------
static uint32_t g_x2n[64];
static bool g_x2n_ready = false;
static void x2n_init() {
  if (g_x2n_ready) return;
  uint32_t p = 0x40000000u;  // x^1
  for (int k = 0; k < 64; k++) { g_x2n[k] = p; p = gf_mul(p, p); }
  g_x2n_ready = true;
}
uint32_t gf_xpow8(uint64_t nbytes) {  // x^(8*nbytes) mod P
  x2n_init();
  uint32_t r = 0x80000000u;  // x^0
  // 8*nbytes = nbytes << 3: bit k of nbytes contributes x^(2^(k+3))
  for (int k = 0; nbytes; k++, nbytes >>= 1)
    if (nbytes & 1) r = gf_mul(r, g_x2n[(k + 3) & 63]);
  return r;
}

// Table block layout (uint32 words):
//   [0    .. 1023]  strided slice tables  TS[k][b] = T0[b] * x^(8*(k+508))
//   [1024 .. 2047]  ordinary slice tables T[k][b]  = T0[b] * x^(8*k)
//   [2048 .. 2079]  XP[m] = x^(128*m)   (advance a state by 16*m bytes)
//   [2080 .. 2143]  X2N[k] = x^(2^k)     (advance a state by any number of bytes: stored_copy_crc_kernel)
constexpr int kTabWords = 1024 + 1024 + 32 + 64;
constexpr int kStride = 512;

int crc_tables_upload(zipc_b200_ctx *ctx) {
  std::vector<uint32_t> t(kTabWords);
  uint32_t t0[256];
  for (uint32_t i = 0; i < 256; i++) {
    uint32_t c = i;
    for (int k = 0; k < 8; k++) c = (c & 1u) ? (kCrcPoly ^ (c >> 1)) : (c >> 1);
    t0[i] = c;
  }
  for (int k = 0; k < 4; k++) {
    uint32_t xs = gf_xpow8((uint64_t)k + kStride - 4), xo = gf_xpow8((uint64_t)k);
    for (int b = 0; b < 256; b++) {
      t[k * 256 + b] = gf_mul(t0[b], xs);
      t[1024 + k * 256 + b] = gf_mul(t0[b], xo);
    }
  }
  for (int m = 0; m < 32; m++) t[2048 + m] = gf_xpow8(16ull * m);
  x2n_init();
  for (int k = 0; k < 64; k++) t[2080 + k] = g_x2n[k];
  ZB_CUDA(ctx, cudaMalloc(&ctx->d_crc_tabs, kTabWords * sizeof(uint32_t)));
  ZB_CUDA(ctx, cudaMemcpyAsync(ctx->d_crc_tabs, t.data(), kTabWords * sizeof(uint32_t),
                               cudaMemcpyHostToDevice, ctx->stream));
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  return ZIPC_OK;
}

// ---------------------------------------------------------------------------------------------
// device code
// ---------------------------------------------------------------------------------------------
namespace {

constexpr int kThreads = 1024;
constexpr int kWarps = kThreads / 32;
constexpr int kRepWords = 4 * 256 * 32;
constexpr size_t kSmemBytes = (size_t)(kRepWords + 1024 + 32) * sizeof(uint32_t);

__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}

// One word through the lane-replicated strided tables.  Layout (bytes): table k, byte b, lane l at
//   (k >> 1) * 65536 + b * 256 + (k & 1) * 128 + l * 4
// so the variable part of an address is "b * 256 + l * 4": byte b of the word dropped into byte 1 of a register
// whose byte 0 already holds l * 4 -- ONE PRMT per lookup (the first two versions spent a shift or IMAD.HI plus a
// LOP3 per lookup and were bound by instruction issue, not by HBM).  The table/region offset rides in the LDS
// immediate.  A warp's 32 lookups still hit 32 different banks.
__device__ __forceinline__ uint32_t step_rep(const uint32_t *__restrict__ rep, uint32_t lane4, uint32_t u) {
  const char *t = reinterpret_cast<const char *>(rep);
  uint32_t i0 = __byte_perm(u, lane4, 0x5504);  // byte 0 of u -> T'_3
  uint32_t i1 = __byte_perm(u, lane4, 0x5514);  // byte 1      -> T'_2
  uint32_t i2 = __byte_perm(u, lane4, 0x5524);  // byte 2      -> T'_1
  uint32_t i3 = __byte_perm(u, lane4, 0x5534);  // byte 3      -> T'_0
  return *reinterpret_cast<const uint32_t *>(t + 65536 + 128 + i0) ^ *reinterpret_cast<const uint32_t *>(t + 65536 + i1) ^
         *reinterpret_cast<const uint32_t *>(t + 128 + i2) ^ *reinterpret_cast<const uint32_t *>(t + i3);
}
// one word through the ordinary slice-by-4 tables (state valid right after the word)
__device__ __forceinline__ uint32_t step_std(const uint32_t *__restrict__ st, uint32_t u) {
  return st[3 * 256 + (u & 0xffu)] ^ st[2 * 256 + ((u >> 8) & 0xffu)] ^
         st[1 * 256 + ((u >> 16) & 0xffu)] ^ st[u >> 24];
}
__device__ __forceinline__ uint32_t step_byte(const uint32_t *__restrict__ st, uint32_t c, uint32_t b) {
  return (c >> 8) ^ st[(c ^ b) & 0xffu];
}

// What crc_segment_warp does with the bytes it reads besides the CRC: nothing (NoStore), or write them to a destination
// (CopyStore).  Bytes outside the 16-byte-aligned body go through byte(); the body comes row by row through row(), called by
// the whole warp in row order, with valid = false for the lanes that have no block in the row.
struct NoStore {
  static constexpr bool kStores = false;
  static constexpr int kRows = 8;   // rows requested together by the main loop
  __device__ __forceinline__ void begin(uint32_t, uint64_t) {}
  __device__ __forceinline__ void byte(uint64_t, uint32_t) {}
  __device__ __forceinline__ void row(const uint4 &, uint64_t, int, bool) {}
};

__device__ __forceinline__ void st_v4(uint8_t *p, const uint4 &v) { *reinterpret_cast<uint4 *>(p) = v; }
// bytes [from, to) of v to p[from, to)
__device__ __forceinline__ void st_bytes(uint8_t *p, const uint4 &v, uint32_t from, uint32_t to) {
  for (uint32_t i = from; i < to; i++) {
    const uint32_t w = i < 4 ? v.x : i < 8 ? v.y : i < 12 ? v.z : v.w;
    p[i] = (uint8_t)(w >> (8 * (i & 3)));
  }
}

// The body's blocks land at dst + head + 16 b, i.e. at phase p of the destination's 16-byte words: aligned word b (at
// dbase + 16 b) holds the last p bytes of block b - 1 and the first 16 - p bytes of block b.  Lane l takes block b - 1 from
// lane l - 1 by shuffle, lane 0 from the previous row's lane 31 (the carry), and stores word b whole; word 0 and word nblk
// are the partial ends of the body.  Every store lies inside [dst, dst + len): no byte outside the slot is written.
struct CopyStore {
  static constexpr bool kStores = true;
  static constexpr int kRows = 4;   // (8 rows of loads in flight and the row being joined do not fit 64 registers)
  uint8_t *dst;       // destination of the segment's byte 0
  uint8_t *dbase;     // 16-byte aligned: dst + head - p
  uint64_t nblk;
  uint32_t p, q, sh;  // phase; the shift 16 - p as whole words (q) and bits (sh)
  uint4 carry;
  __device__ __forceinline__ explicit CopyStore(uint8_t *d) : dst(d) {}
  __device__ __forceinline__ void begin(uint32_t head, uint64_t nb) {
    p = (uint32_t)((uintptr_t)(dst + head) & 15);
    dbase = dst + head - p;
    nblk = nb;
    q = ((16 - p) >> 2) & 3;
    sh = ((16 - p) & 3) * 8;
    carry = make_uint4(0, 0, 0, 0);
  }
  __device__ __forceinline__ void byte(uint64_t i, uint32_t v) { dst[i] = (uint8_t)v; }
  // bytes 16 - p .. 15 of a, then bytes 0 .. 15 - p of b
  __device__ __forceinline__ uint4 join(const uint4 &a, const uint4 &b) const {
    uint32_t a0 = a.x, a1 = a.y, a2 = a.z, a3 = a.w, a4 = b.x, a5 = b.y, a6 = b.z, a7 = b.w;
    if (q & 2) { a0 = a2; a1 = a3; a2 = a4; a3 = a5; a4 = a6; a5 = a7; }
    if (q & 1) { a0 = a1; a1 = a2; a2 = a3; a3 = a4; a4 = a5; }
    return make_uint4(__funnelshift_r(a0, a1, sh), __funnelshift_r(a1, a2, sh), __funnelshift_r(a2, a3, sh),
                      __funnelshift_r(a3, a4, sh));
  }
  __device__ __forceinline__ void row(const uint4 &cur, uint64_t r, int lane, bool valid) {
    const int from = (lane + 31) & 31;
    uint4 prev = make_uint4(__shfl_sync(0xffffffffu, cur.x, from), __shfl_sync(0xffffffffu, cur.y, from),
                            __shfl_sync(0xffffffffu, cur.z, from), __shfl_sync(0xffffffffu, cur.w, from));
    const uint4 t = prev;
    if (lane == 0) prev = carry;
    carry = t;
    if (!valid) return;
    const uint64_t b = 32 * r + (uint64_t)lane;
    uint8_t *w = dbase + 16 * b;
    if (p == 0) { st_v4(w, cur); return; }
    const uint4 o = join(prev, cur);
    if (b) st_v4(w, o);
    else st_bytes(w, o, p, 16);
    if (b + 1 == nblk) st_bytes(w + 16, join(cur, cur), 0, p);
  }
};

// State after running seg.len bytes from seg.init; result valid in lane 0.  The sink sees every byte once (see NoStore).
template <class Sink>
__device__ uint32_t crc_segment_warp(const CrcSeg seg, int lane, const uint32_t *__restrict__ rep,
                                     const uint32_t *__restrict__ st, const uint32_t *__restrict__ xp, Sink &sink) {
  const uint8_t *ptr = seg.ptr;
  uint64_t len = seg.len;
  const uint32_t lane4 = (uint32_t)lane * 4u;
  if (len < 64) {  // tiny: one lane, bytewise
    uint32_t c = seg.init;
    if (lane == 0)
      for (uint32_t i = 0; i < (uint32_t)len; i++) { const uint32_t v = ptr[i]; c = step_byte(st, c, v); sink.byte(i, v); }
    return c;
  }
  uint32_t head = (uint32_t)((16 - ((uintptr_t)ptr & 15)) & 15);
  uint32_t c0 = 0, c1 = 0, c2 = 0, c3 = 0;
  if (lane == 0) {  // unaligned head, then the running state is folded into the first body word
    uint32_t c = seg.init;
    for (uint32_t i = 0; i < head; i++) { const uint32_t v = ptr[i]; c = step_byte(st, c, v); sink.byte(i, v); }
    c0 = c;
  }
  const uint8_t *body = ptr + head;
  uint64_t body_len = len - head;
  uint64_t nblk = body_len >> 4;           // full 16-byte blocks, >= 3
  uint32_t tail = (uint32_t)(body_len & 15);
  uint64_t rows = nblk >> 5;
  int k = (int)(nblk & 31);                // lanes < k own one more block
  const uint4 *p = reinterpret_cast<const uint4 *>(body) + lane;
  sink.begin(head, nblk);

  // rows [0, rows-1): nobody's last block -> strided tables for every lane
  // 8 rows (4 KiB per warp) are requested together, then consumed; with 32 warps per SM out of phase this keeps
  // enough loads in flight (a software-pipelined variant measured the same: the LDS pipe, ~75 % busy, is the
  // next limiter after HBM, not load latency).
  uint64_t R = rows > 0 ? rows - 1 : 0, r = 0;
  constexpr int G = Sink::kRows;
  for (; r + G <= R; r += G) {
    uint4 w[G];
#pragma unroll
    for (int j = 0; j < G; j++) w[j] = ldg_stream(p + 32 * (r + j));
#pragma unroll
    for (int j = 0; j < G; j++) {
      c0 = step_rep(rep, lane4, c0 ^ w[j].x);
      c1 = step_rep(rep, lane4, c1 ^ w[j].y);
      c2 = step_rep(rep, lane4, c2 ^ w[j].z);
      c3 = step_rep(rep, lane4, c3 ^ w[j].w);
      sink.row(w[j], r + j, lane, true);
    }
  }
  for (; r < R; r++) {
    uint4 w = ldg_stream(p + 32 * r);
    c0 = step_rep(rep, lane4, c0 ^ w.x);
    c1 = step_rep(rep, lane4, c1 ^ w.y);
    c2 = step_rep(rep, lane4, c2 ^ w.z);
    c3 = step_rep(rep, lane4, c3 ^ w.w);
    sink.row(w, r, lane, true);
  }
  bool has = false;
  if (rows >= 1) {  // row rows-1: last block of lanes >= k
    uint4 w = ldg_stream(p + 32 * (rows - 1));
    has = true;
    sink.row(w, rows - 1, lane, true);
    if (lane < k) {
      c0 = step_rep(rep, lane4, c0 ^ w.x); c1 = step_rep(rep, lane4, c1 ^ w.y);
      c2 = step_rep(rep, lane4, c2 ^ w.z); c3 = step_rep(rep, lane4, c3 ^ w.w);
    } else {
      c0 = step_std(st, c0 ^ w.x); c1 = step_std(st, c1 ^ w.y);
      c2 = step_std(st, c2 ^ w.z); c3 = step_std(st, c3 ^ w.w);
    }
  }
  if constexpr (Sink::kStores) {
    if (k) {  // partial row: last block of lanes < k (the whole warp takes part in the sink's shuffle)
      const uint4 w = lane < k ? ldg_stream(p + 32 * rows) : make_uint4(0, 0, 0, 0);
      sink.row(w, rows, lane, lane < k);
      if (lane < k) {
        has = true;
        c0 = step_std(st, c0 ^ w.x); c1 = step_std(st, c1 ^ w.y);
        c2 = step_std(st, c2 ^ w.z); c3 = step_std(st, c3 ^ w.w);
      }
    }
  } else if (lane < k) {  // partial row: last block of lanes < k
    uint4 w = ldg_stream(p + 32 * rows);
    has = true;
    c0 = step_std(st, c0 ^ w.x); c1 = step_std(st, c1 ^ w.y);
    c2 = step_std(st, c2 ^ w.z); c3 = step_std(st, c3 ^ w.w);
  }
  // merge the four slots: state valid at the end of this lane's last block
  uint32_t s = step_std(st, step_std(st, step_std(st, c0) ^ c1) ^ c2) ^ c3;
  // align to the end of the last full block of the body: advance by 16*d bytes
  uint64_t nrows_l = rows + (lane < k ? 1 : 0);
  if (has) {
    uint32_t d = (uint32_t)(nblk - 1 - (uint64_t)lane - 32 * (nrows_l - 1));
    if (d) s = gf_mul(s, xp[d]);
  } else {
    s = 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s ^= __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) {
    const uint8_t *t = body + (nblk << 4);
    for (uint32_t i = 0; i < tail; i++) { const uint32_t v = t[i]; s = step_byte(st, s, v); sink.byte(head + (nblk << 4) + i, v); }
  }
  return s;
}

__device__ __forceinline__ void load_tables(const uint32_t *__restrict__ g_tabs, uint32_t *smem) {
  // replicate the strided tables per lane: word (k>>1)*16384 + b*64 + (k&1)*32 + lane  <-  TS[k][b].
  // Thread t fetches TS entry t once; each warp then broadcasts its 32 entries by shuffle and stores them
  // 32 lanes wide (conflict-free), instead of 32 dependent global loads per thread.
  {
    const int t = threadIdx.x, lane = t & 31;
    const uint32_t v = g_tabs[t];  // blockDim.x == 1024 == number of TS entries
#pragma unroll 8
    for (int e = 0; e < 32; e++) {
      int idx = (t & ~31) + e, k = idx >> 8, b = idx & 255;
      smem[(k >> 1) * 16384 + b * 64 + (k & 1) * 32 + lane] = __shfl_sync(0xffffffffu, v, e);
    }
  }
  for (int i = threadIdx.x; i < 1024 + 32; i += blockDim.x) smem[kRepWords + i] = g_tabs[1024 + i];
  __syncthreads();
}

// Independent segments pulled from a queue, one warp each.
__global__ void __launch_bounds__(kThreads, 1)
crc32_segments_kernel(const CrcSeg *__restrict__ segs, uint32_t nseg, const uint32_t *__restrict__ g_tabs,
                      uint32_t *__restrict__ states, unsigned int *__restrict__ queue) {
  extern __shared__ __align__(16) uint32_t smem[];
  load_tables(g_tabs, smem);
  const int lane = threadIdx.x & 31;
  const uint32_t *rep = smem, *st = smem + kRepWords, *xp = st + 1024;
  for (;;) {
    unsigned int s = 0;
    if (lane == 0) s = atomicAdd(queue, 1u);
    s = __shfl_sync(0xffffffffu, s, 0);
    if (s >= nseg) break;
    NoStore none;
    uint32_t c = crc_segment_warp(segs[s], lane, rep, st, xp, none);
    if (lane == 0) states[s] = c;
  }
}

// One large buffer cut into uniform tiles of `tile` bytes (multiple of 512); warp w of the grid
// owns tile w.  Tile 0 starts from the CRC init value, the others from 0.
__global__ void __launch_bounds__(kThreads, 1)
crc32_tiles_kernel(const uint8_t *__restrict__ src, uint64_t len, uint64_t tile, uint32_t ntiles,
                   const uint32_t *__restrict__ g_tabs, uint32_t *__restrict__ states) {
  extern __shared__ __align__(16) uint32_t smem[];
  load_tables(g_tabs, smem);
  const int lane = threadIdx.x & 31;
  const uint32_t *rep = smem, *st = smem + kRepWords, *xp = st + 1024;
  for (uint32_t t = blockIdx.x * kWarps + (threadIdx.x >> 5); t < ntiles; t += gridDim.x * kWarps) {
    CrcSeg seg;
    uint64_t off = (uint64_t)t * tile;
    seg.ptr = src + off;
    seg.len = len - off < tile ? len - off : tile;
    seg.init = t == 0 ? 0xFFFFFFFFu : 0u;
    NoStore none;
    uint32_t c = crc_segment_warp(seg, lane, rep, st, xp, none);
    if (lane == 0) states[t] = c;
  }
}

// total = sum_t state[t] * x^(8 * bytes after tile t).  Tiles 0..F-1 are full (L bytes), tile F is
// the last one (last_len bytes, may be L).  xl = x^(8*last_len); xg[0] = x^(8L), xg[1] = x^(8LG),
// xg[2+l] = x^(8LG 2^l).  One CTA of 1024 threads.
constexpr int kCombThreads = 1024;
struct CombConsts { uint32_t xg[12]; };
__global__ void __launch_bounds__(kCombThreads, 1)
crc32_combine_tiles_kernel(const uint32_t *__restrict__ states, uint32_t F, uint32_t G, uint32_t xl,
                           const CombConsts cc, uint32_t *__restrict__ out) {
  __shared__ uint32_t v[kCombThreads];
  const uint32_t *xg = cc.xg;
  const uint32_t q = threadIdx.x;
  // u[j] = state[F-1-j]; thread q: sum_{i<G} u[qG+i] X^i by Horner from the high end
  uint32_t acc = 0;
  const uint32_t X = xg[0];
  for (int i = (int)G - 1; i >= 0; i--) {
    uint32_t j = q * G + (uint32_t)i;
    uint32_t s = j < F ? states[F - 1 - j] : 0u;
    acc = gf_mul(acc, X) ^ s;
  }
  v[q] = acc;
  __syncthreads();
  // tree: v[m] = v[2m] ^ v[2m+1] * Y_l
  int lvl = 0;
  for (uint32_t n = kCombThreads; n > 1; n >>= 1, lvl++) {
    uint32_t a = 0;
    if (q < n / 2) a = v[2 * q] ^ gf_mul(v[2 * q + 1], xg[1 + lvl]);
    __syncthreads();
    if (q < n / 2) v[q] = a;
    __syncthreads();
  }
  if (q == 0) *out = (gf_mul(v[0], xl) ^ states[F]) ^ 0xFFFFFFFFu;
}

// Stored members: tile t of the launch copies tiles[t].len bytes from src to dst and XORs its state, advanced over the
// tiles[t].after bytes of its member that follow it, into acc[tiles[t].member] (zeroed before the launch).  A member's first
// tile starts from the CRC init value, so acc ends as the member's state before the final XOR.  Tiles pulled from a queue.
constexpr size_t kCopySmemBytes = kSmemBytes + 64 * sizeof(uint32_t);
__global__ void __launch_bounds__(kThreads, 1)
stored_copy_crc_kernel(const StoredTile *__restrict__ tiles, uint32_t ntiles, const uint32_t *__restrict__ g_tabs,
                       uint32_t *__restrict__ acc, unsigned int *__restrict__ queue) {
  extern __shared__ __align__(16) uint32_t smem[];
  if (threadIdx.x < 64) smem[kRepWords + 1024 + 32 + threadIdx.x] = g_tabs[2080 + threadIdx.x];  // (load_tables syncs)
  load_tables(g_tabs, smem);
  const int lane = threadIdx.x & 31;
  const uint32_t *rep = smem, *st = smem + kRepWords, *xp = st + 1024, *x2n = xp + 32;
  for (;;) {
    unsigned int t = 0;
    if (lane == 0) t = atomicAdd(queue, 1u);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= ntiles) break;
    const StoredTile d = tiles[t];
    CopyStore sink(d.dst);
    uint32_t c = crc_segment_warp(CrcSeg{d.src, d.len, d.init, 0}, lane, rep, st, xp, sink);
    if (d.after) {  // times x^(8 after): bit i of `after` contributes x^(2^(i+3)); lane l takes bits l and l + 32
      uint32_t f = (d.after >> lane) & 1 ? x2n[lane + 3] : 0x80000000u;
      if (d.after >> 32 && lane < 29 && (d.after >> (lane + 32)) & 1) f = gf_mul(f, x2n[lane + 35]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) f = gf_mul(f, __shfl_xor_sync(0xffffffffu, f, o));
      c = gf_mul(c, f);
    }
    if (lane == 0) atomicXor(acc + d.member, c);
  }
}

unsigned long long g_attr_devs = 0;  // bit d: attributes set on device d (function attributes are per device)
int ensure_attrs(zipc_b200_ctx *ctx) {
  if (g_attr_devs >> (ctx->device & 63) & 1ull) return ZIPC_OK;
  ZB_CUDA(ctx, cudaFuncSetAttribute(crc32_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)kSmemBytes));
  ZB_CUDA(ctx, cudaFuncSetAttribute(crc32_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)kSmemBytes));
  ZB_CUDA(ctx, cudaFuncSetAttribute(stored_copy_crc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)kCopySmemBytes));
  g_attr_devs |= 1ull << (ctx->device & 63);
  return ZIPC_OK;
}

}  // namespace

int crc32_launch_segments(zipc_b200_ctx *ctx, const CrcSeg *d_segs, uint32_t nseg, uint32_t *d_states) {
  if (nseg == 0) return ZIPC_OK;
  if (int st = ensure_attrs(ctx)) return st;
  if (int st = ctx->d_small.reserve(256)) return st;
  unsigned int *queue = ctx->d_small.as<unsigned int>();
  ZB_CUDA(ctx, cudaMemsetAsync(queue, 0, sizeof(unsigned int), ctx->stream));
  uint32_t grid = (nseg + kWarps - 1) / kWarps;
  if (grid > (uint32_t)ctx->sm_count) grid = (uint32_t)ctx->sm_count;
  crc32_segments_kernel<<<grid, kThreads, kSmemBytes, ctx->stream>>>(d_segs, nseg, ctx->d_crc_tabs, d_states, queue);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  return ZIPC_OK;
}

int crc32_launch_buffer(zipc_b200_ctx *ctx, const uint8_t *d_src, uint64_t len, uint32_t *d_crc) {
  if (int st = ensure_attrs(ctx)) return st;
  const uint32_t max_tiles = (uint32_t)ctx->sm_count * kWarps;
  // tile length: multiple of 512, at least 4 KiB so tiny buffers do not fan out pointlessly
  uint64_t tile = (len + max_tiles - 1) / max_tiles;
  if (tile < 4096) tile = 4096;
  if (const char *e = getenv("ZIPC_B200_CRC_TILE")) { uint64_t v = strtoull(e, nullptr, 10); if (v >= 4096 && v < tile) tile = v; }  // tuning knob
  tile = (tile + 511) & ~511ull;
  uint32_t ntiles = len ? (uint32_t)((len + tile - 1) / tile) : 1;
  uint32_t F = ntiles - 1;
  uint64_t last_len = len - (uint64_t)F * tile;
  // combine constants
  uint32_t G = (F + kCombThreads - 1) / kCombThreads;
  if (G == 0) G = 1;
  CombConsts cc;
  cc.xg[0] = gf_xpow8(tile);
  cc.xg[1] = gf_xpow8(tile * G);
  for (int l = 1; l < 11; l++) cc.xg[1 + l] = gf_mul(cc.xg[l], cc.xg[l]);
  if (int st = ctx->d_scratch2.reserve((size_t)(ntiles + 1) * sizeof(uint32_t))) return st;
  uint32_t *d_states = ctx->d_scratch2.as<uint32_t>();
  uint32_t grid = (ntiles + kWarps - 1) / kWarps;
  if (grid > (uint32_t)ctx->sm_count) grid = (uint32_t)ctx->sm_count;
  {
    KernelTimer kt(ctx);
    crc32_tiles_kernel<<<grid, kThreads, kSmemBytes, ctx->stream>>>(d_src, len, tile, ntiles, ctx->d_crc_tabs, d_states);
  }
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  crc32_combine_tiles_kernel<<<1, kCombThreads, 0, ctx->stream>>>(d_states, F, G, gf_xpow8(last_len), cc, d_crc);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  return ZIPC_OK;
}

int stored_copy_crc(zipc_b200_ctx *ctx, size_t n, const uint8_t *const *src, uint8_t *const *dst, const uint64_t *len,
                    uint32_t *crc) {
  if (!n) return ZIPC_OK;
  if (n > 0xFFFFFFF0ull) return ZIPC_ERR_INVALID_ARG;
  size_t ntiles = 0;
  for (size_t i = 0; i < n; i++) ntiles += len[i] ? (len[i] + kStoredTile - 1) / kStoredTile : 1;
  if (ntiles > 0xFFFFFFF0ull) return ZIPC_ERR_INVALID_ARG;
  if (int st = ensure_attrs(ctx)) return st;
  const size_t tile_bytes = ntiles * sizeof(StoredTile);
  if (int st = ctx->h_desc.reserve(tile_bytes + n * sizeof(uint32_t))) return st;
  if (int st = ctx->d_desc2.reserve(tile_bytes + n * sizeof(uint32_t))) return st;
  if (int st = ctx->d_small.reserve(256)) return st;
  StoredTile *ht = ctx->h_desc.as<StoredTile>();
  size_t t = 0;
  for (size_t i = 0; i < n; i++) {  // (a zero-length member is one empty tile: its word ends as the init value)
    uint64_t off = 0;
    do {
      const uint64_t l = len[i] - off < kStoredTile ? len[i] - off : kStoredTile;
      ht[t++] = StoredTile{src[i] + off, dst[i] + off, l, len[i] - off - l, (uint32_t)i, off ? 0u : 0xFFFFFFFFu};
      off += l;
    } while (off < len[i]);
  }
  StoredTile *dt = ctx->d_desc2.as<StoredTile>();
  uint32_t *d_acc = reinterpret_cast<uint32_t *>(ctx->d_desc2.as<uint8_t>() + tile_bytes);
  unsigned int *queue = ctx->d_small.as<unsigned int>();
  ZB_CUDA(ctx, cudaMemcpyAsync(dt, ht, tile_bytes, cudaMemcpyHostToDevice, ctx->stream));
  ZB_CUDA(ctx, cudaMemsetAsync(d_acc, 0, n * sizeof(uint32_t), ctx->stream));
  ZB_CUDA(ctx, cudaMemsetAsync(queue, 0, sizeof(unsigned int), ctx->stream));
  uint32_t grid = (uint32_t)((ntiles + kWarps - 1) / kWarps);
  if (grid > (uint32_t)ctx->sm_count) grid = (uint32_t)ctx->sm_count;
  {
    KernelTimer kt(ctx);
    stored_copy_crc_kernel<<<grid, kThreads, kCopySmemBytes, ctx->stream>>>(dt, (uint32_t)ntiles, ctx->d_crc_tabs, d_acc, queue);
  }
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  uint32_t *h_acc = reinterpret_cast<uint32_t *>(ctx->h_desc.as<uint8_t>() + tile_bytes);
  ZB_CUDA(ctx, cudaMemcpyAsync(h_acc, d_acc, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  ZB_CUDA(ctx, stream_sync(ctx, ctx->stream));
  for (size_t i = 0; i < n; i++) crc[i] = h_acc[i] ^ 0xFFFFFFFFu;
  return ZIPC_OK;
}

}  // namespace zb
