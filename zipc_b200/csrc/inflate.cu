// inflate.cu -- batched DEFLATE decoder for sm_100a: one *warp* per stream, speculative token decoding.
//
// Replaces the decode side of the reference (src/zipc_deflate.ml:532-718): read_bits (:564-579),
// the bit-at-a-time read_symbol (:584-591), read_block_symbols (:593-616), the three block readers
// (:618-680) and the driver inflate_and_crc (:692-709).  Results are bit-exact, including which of
// the two errors ("Corrupted data stream" / "Expected decompression size exceeded") a bad stream
// yields: checks are evaluated in the reference's order, token by token.
//
// Design (why it is not a translation):
//   * Huffman decoding is serial per stream: a token's position is known only after the previous token
//     is decoded.  The first version ran one decoder state machine per lane (8 per warp); its profile
//     showed the SM waiting on that dependent chain (~2000 clk per token and stream, 55 % issue
//     utilisation, a 256 KiB member bounding the whole batch).  This version breaks the chain:
//       - D1 (speculate): the warp looks at a window of 32*NB bits.  Lane l decodes, for each of its NB
//         bit offsets, the complete token that WOULD start there (literal, or length + distance with
//         their extra bits: two table lookups, branch free, NB independent chains per lane) and posts
//         (token, bit length) in shared memory.
//       - D2 (walk): every lane follows the chain start -> start + bits -> ... through that table: 32
//         straight-line steps of four instructions, no exit tests (a candidate that stops the walk counts
//         as zero bits; a ballot finds the first repeated address).  Up to 32 tokens per round.
//       - checks (distance, size, input overrun) run in parallel, one token per lane; the first failing
//         token cuts the round and decides the error, as the serial reference would.
//   * E (copy): the round's literal bytes and match bytes whose source precedes the round are flattened
//     over the 32 lanes (byte b of the round's independent bytes -> lane b % 32); matches that read
//     bytes of the same round follow in order.  Back-references read the stream's own earlier output
//     from global memory through L2 (ld.global.cg), at most 32 KiB back.
//   * Compressed input is staged in a 512-byte ring per warp, refilled by the copy engine one refill ahead
//     (cp.async.bulk of 128 bytes against a per-warp mbarrier; guarded loads for the last words of a stream).
//   * Lookup tables: 2^LB literal/length entries (16 bit) and 2^DB distance entries (32 bit) per warp in
//     shared memory; longer codes (rare) take the canonical walk.  The fixed-Huffman tables are built
//     once per CTA; dynamic tables are built cooperatively by the warp.
//   * 32 warps per CTA, one CTA per SM, streams handed out through a global queue (longest first; in download
//     order when the batch's arena is copied out progressively, api.cu plan_arena).
//   * One LARGE stream (no index): find_starts_kernel + this kernel in SPEC mode (16-bit symbols with window
//     markers) + win_*_kernel / resolve_kernel; orchestrated by api.cu par_speculate / par_resolve.
//
// Algorithmic bytes: C + U per stream (compressed read + uncompressed written).  The kernel is
// issue/latency bound (bit parsing), not HBM bound: see DESIGN.md.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "adler_core.cuh"

namespace zb {
namespace {

#ifndef ZB_INFLATE_LB
#define ZB_INFLATE_LB 11
#endif
constexpr int LB = ZB_INFLATE_LB;       // literal/length table bits
#ifndef ZB_INFLATE_DB
#define ZB_INFLATE_DB 8
#endif
constexpr int DB = ZB_INFLATE_DB;        // distance table bits (>= 7: the area also hosts the 128-entry code-length table)
#ifndef ZB_INFLATE_NB
#define ZB_INFLATE_NB 10
#endif
constexpr int NB = ZB_INFLATE_NB;        // candidate bit offsets per lane: lane l owns offsets l, l + 32, ...
constexpr int WBITS = 32 * NB;  // speculation window
#ifndef ZB_INFLATE_WARPS
#define ZB_INFLATE_WARPS 32
#endif
constexpr int WARPS = ZB_INFLATE_WARPS;    // warps per CTA (one CTA per SM)
constexpr int THREADS = WARPS * 32;
constexpr int ROUND_TOKENS = 32;  // one token per lane
// Refills of the compressed-input ring: ZB_INFLATE_BULK = 1 asks the copy engine (cp.async.bulk, 128 bytes per refill, completion
// on a per-warp mbarrier) instead of one coalesced load per lane kept in a register until it is needed.
#ifndef ZB_INFLATE_BULK
#define ZB_INFLATE_BULK 1
#endif
// the bulk copies carry an L2 evict_first policy: the compressed bytes are read once, the L2 lines are wanted for the streams'
// 32 KiB histories (C3, ncu: DRAM reads 4.48 -> 4.34 GB per launch, kernel 13.55 -> 13.51 ms; profiles/r02_inflate_evict_first.txt)
#ifndef ZB_INFLATE_IN_EVICT_FIRST
#define ZB_INFLATE_IN_EVICT_FIRST 1
#endif
#ifndef ZB_INFLATE_SPEC_PER_CTA
#define ZB_INFLATE_SPEC_PER_CTA 4
#endif
constexpr int kRingWords = ZB_INFLATE_BULK ? 128 : 64;
constexpr uint32_t kRingMask = kRingWords - 1;
constexpr int SYMS_PER_SLOT = 320;     // sorted symbols: 288 litlen + 32 dist

// Table entries are laid out for the speculative pass (D1), whose only question is "how many bits, or stop":
// lit entry  (16 bit): [7:0] candidate byte, [15:8] literal byte | length symbol - 257
//     candidate byte: literal -> code length;  length symbol -> kCbIsLen | (code length + the length's extra bits);
//                     end of block -> kCbStop | code length;  kCbInvalid / kCbLong (both >= kCbSlow)
// dist entry (32 bit): [7:0] code length + extra bits, or kDbInvalid / kDbLong (then the sum with any length part is
//                      >= kCbSlow);  [11:8] code length;  [26:12] distance base
constexpr uint32_t kCbIsLen = 0x40u, kCbStop = 0x80u, kCbSlow = 0xC0u, kCbInvalid = 0xFEu, kCbLong = 0xFFu;
constexpr uint16_t kLitInvalid = (uint16_t)kCbInvalid, kLitLong = (uint16_t)kCbLong;
constexpr uint32_t kDbInvalid = 0xC0u, kDbLong = 0xC1u;   // + (<= 20 bits of the length part) stays below 0x100
constexpr uint32_t kDistInvalid = kDbInvalid, kDistLong = kDbLong;
struct __align__(16) WarpTabs {
  uint16_t lit[1 << LB];
  uint32_t dist[1 << DB];
  uint16_t lit_cnt[16];
  uint16_t dist_cnt[16];
};
struct __align__(16) WarpScratch {
  uint8_t len[320];
  uint32_t cnt[16];
  uint16_t next[16];
  uint16_t symoff[16];
  int err;
};
// candidate table entry (8 bit): bits the token starting at this offset occupies (1..48);
//                                kCbStop | code length (< kCbSlow): end of block;  >= kCbSlow: not decodable through
//                                the tables (long or invalid code).  Bit 7 set = the walk stops here.
// per-stream values that are read a few times per round at most live in shared memory, not in registers
// (the kernel runs many warps per SM: 64..80 registers per thread)
struct WarpState {
  const uint32_t *srcw;    // word-aligned base of the input (at or before the first stream byte)
  const uint8_t *src;
  uint64_t src_len, out_cap;
  uint64_t ad_from;        // output offset up to which the Adler-32 is accounted
  uint64_t limit;          // first input bit past the stream, counted from srcw
  uint32_t nwords;         // words that may be read
  uint32_t skew;           // bits between srcw and the stream start (0, 8, 16, 24)
  uint32_t nblk;           // speculative chunks: non-empty blocks decoded so far
};
struct __align__(16) WarpWork {
  WarpState st;
  union {
    uint8_t cand[WBITS + 64];  // by bit offset from the round's start; the 64 bytes behind the window say "stop"
    WarpScratch build;    // table construction never overlaps a decoding round
  };
  uint16_t tokq[ROUND_TOKENS + 2];  // candidate addresses of the round's tokens, in order, then where the walk ended
  uint32_t slow_tx[ROUND_TOKENS];   // slow path tokens: the token ...
  uint16_t slow_end[ROUND_TOKENS];  // ... and the bit offset where it ends
  alignas(16) uint32_t ring[kRingWords];  // compressed input: words [w0, w0 + 64) of the stream (+ the segment on its way, bulk variant)
  alignas(8) uint64_t ldbar;              // bulk variant: mbarrier of the warp's refills
  uint8_t cidx[32];       // E1: lane holding the r-th independent token
};

constexpr size_t kSmemBytes = sizeof(WarpTabs) * (WARPS + 1) + sizeof(WarpWork) * WARPS + 64 + 128 + 64;
static_assert(kSmemBytes <= 227 * 1024, "one CTA of 32 warps per SM: tables + work areas must fit the opt-in shared memory");

enum : uint32_t { S_IDLE = 0, S_HDR = 1, S_DATA = 2, S_STORED = 3, S_FINISH = 4, S_EXIT = 5 };

__constant__ uint16_t c_len_tab[29] = {  // base | extra << 9   (RFC 1951 3.2.5; reference :245-255)
    3 | 0 << 9,   4 | 0 << 9,   5 | 0 << 9,   6 | 0 << 9,   7 | 0 << 9,   8 | 0 << 9,   9 | 0 << 9,   10 | 0 << 9,
    11 | 1 << 9,  13 | 1 << 9,  15 | 1 << 9,  17 | 1 << 9,  19 | 2 << 9,  23 | 2 << 9,  27 | 2 << 9,  31 | 2 << 9,
    35 | 3 << 9,  43 | 3 << 9,  51 | 3 << 9,  59 | 3 << 9,  67 | 4 << 9,  83 | 4 << 9,  99 | 4 << 9,  115 | 4 << 9,
    131 | 5 << 9, 163 | 5 << 9, 195 | 5 << 9, 227 | 5 << 9, 258 | 0 << 9};
__constant__ uint32_t c_dist_tab[30] = {  // base | extra << 16   (reference :277-288)
    1 | 0 << 16,     2 | 0 << 16,     3 | 0 << 16,      4 | 0 << 16,      5 | 1 << 16,      7 | 1 << 16,
    9 | 2 << 16,     13 | 2 << 16,    17 | 3 << 16,     25 | 3 << 16,     33 | 4 << 16,     49 | 4 << 16,
    65 | 5 << 16,    97 | 5 << 16,    129 | 6 << 16,    193 | 6 << 16,    257 | 7 << 16,    385 | 7 << 16,
    513 | 8 << 16,   769 | 8 << 16,   1025 | 9 << 16,   1537 | 9 << 16,   2049 | 10 << 16,  3073 | 10 << 16,
    4097 | 11 << 16, 6145 | 11 << 16, 8193 | 12 << 16,  12289 | 12 << 16, 16385 | 13 << 16, 24577 | 13 << 16};
__constant__ uint8_t c_clen_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// ---- compressed input: a 64-word ring per warp, all state warp-uniform -----------------------------------------
struct Input {
  uint32_t w0;             // ring holds words [w0, w0 + 64), w0 % 32 == 0
#if ZB_INFLATE_BULK
  uint32_t ph;             // bit 0: parity of the mbarrier phase the next refill completes; bit 1: a refill is on its way
#else
  uint32_t pre;            // word w0 + 64 + lane, requested one refill ahead
#endif
  uint64_t P;              // read position in bits from st.srcw
  __device__ __forceinline__ uint32_t load(const WarpState &st, uint32_t k) const {
    uint32_t w = 0;
    if (k < st.nwords) asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(w) : "l"(st.srcw + k));
    return w;
  }
#if ZB_INFLATE_BULK
  // words [k, k + 32) into their ring slots: by the copy engine when all of them exist (the source is 16-byte aligned by
  // construction of srcw), else by guarded loads (the last words of a stream)
  __device__ __forceinline__ void request(WarpWork &wk, uint32_t k, int lane) {
    if (k + 32u <= wk.st.nwords) {
      if (lane == 0) {
        const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&wk.ldbar);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%1], %0;" ::"r"(128u), "r"(bar) : "memory");
#if ZB_INFLATE_IN_EVICT_FIRST
        // the compressed bytes are read once: they are the first to leave L2, which the streams' 32 KiB histories need
        uint64_t pol;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                     ::"r"((uint32_t)__cvta_generic_to_shared(&wk.ring[k & kRingMask])), "l"(wk.st.srcw + k), "r"(128u), "r"(bar), "l"(pol) : "memory");
#else
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"((uint32_t)__cvta_generic_to_shared(&wk.ring[k & kRingMask])), "l"(wk.st.srcw + k), "r"(128u), "r"(bar) : "memory");
#endif
      }
      ph |= 2u;
    } else {
      wk.ring[(k & kRingMask) + lane] = load(wk.st, k + lane);
    }
  }
  __device__ __forceinline__ void settle(WarpWork &wk) {  // the refill on its way, if any, has arrived (every lane sees it)
    if (ph & 2u) {
      const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&wk.ldbar);
      uint32_t ok = 0;
      for (uint32_t spins = 0; !ok && spins < (1u << 26); spins++)
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(bar), "r"(ph & 1u) : "memory");
      ph = (ph & 1u) ^ 1u;
    }
    __syncwarp();  // nobody opens the next phase before everybody has seen this one complete
  }
  __device__ __forceinline__ void seek_bits(WarpWork &wk, uint64_t bitpos, int lane) {
    settle(wk);
    P = bitpos;
    w0 = (uint32_t)(bitpos >> 5) & ~31u;
    const uint32_t x = load(wk.st, w0 + lane), y = load(wk.st, w0 + 32 + lane);
    wk.ring[(w0 & kRingMask) + lane] = x;
    wk.ring[((w0 + 32u) & kRingMask) + lane] = y;
    __syncwarp();
    request(wk, w0 + 64, lane);
    __syncwarp();
  }
#else
  __device__ __forceinline__ void seek_bits(WarpWork &wk, uint64_t bitpos, int lane) {
    P = bitpos;
    w0 = (uint32_t)(bitpos >> 5) & ~31u;
    __syncwarp();
    const uint32_t x = load(wk.st, w0 + lane), y = load(wk.st, w0 + 32 + lane);
    wk.ring[(w0 & 32u) + lane] = x;          // slot of word k is k & 63
    wk.ring[((w0 & 32u) ^ 32u) + lane] = y;
    pre = load(wk.st, w0 + 64 + lane);
    __syncwarp();
  }
#endif
  // st.src / st.src_len are set: derive the rest (lane 0 writes) and fill the ring
  __device__ __forceinline__ void open(WarpWork &wk, int lane) {
    if (lane == 0) {
      const uint32_t a = (uint32_t)((uintptr_t)wk.st.src & (ZB_INFLATE_BULK ? 15 : 3));
      wk.st.srcw = reinterpret_cast<const uint32_t *>(wk.st.src - a);
      wk.st.nwords = (uint32_t)((a + wk.st.src_len + 3) >> 2);
      wk.st.skew = 8 * a;
      wk.st.limit = (uint64_t)(8 * a) + 8 * wk.st.src_len;
    }
    __syncwarp();
    seek_bits(wk, wk.st.skew, lane);
  }
  // afterwards words [P >> 5, (P >> 5) + 32] are in the ring
  __device__ __forceinline__ void ensure(WarpWork &wk, int lane) {
    while ((uint32_t)(P >> 5) >= w0 + 32) {
#if ZB_INFLATE_BULK
      settle(wk);            // words [w0 + 64, w0 + 96) are there
      w0 += 32;
      request(wk, w0 + 64, lane);
      __syncwarp();
#else
      __syncwarp();
      wk.ring[(w0 & 32u) + lane] = pre;
      w0 += 32;
      pre = load(wk.st, w0 + 64 + lane);
      __syncwarp();
#endif
    }
  }
  __device__ __forceinline__ uint32_t peek32(const WarpWork &wk) const {  // the next 32 bits (uniform: broadcast reads)
    uint32_t k = (uint32_t)(P >> 5);
    return __funnelshift_r(wk.ring[k & kRingMask], wk.ring[(k + 1) & kRingMask], (uint32_t)P & 31u);
  }
  __device__ __forceinline__ static uint32_t peek32_at(const WarpWork &wk, uint64_t pos) {
    uint32_t k = (uint32_t)(pos >> 5);
    return __funnelshift_r(wk.ring[k & kRingMask], wk.ring[(k + 1) & kRingMask], (uint32_t)pos & 31u);
  }
  __device__ __forceinline__ uint32_t get(WarpWork &wk, uint32_t n, int lane) {  // n <= 16
    ensure(wk, lane);
    uint32_t v = peek32(wk) & ((1u << n) - 1u);
    P += n;
    return v;
  }
  __device__ __forceinline__ uint64_t consumed(const WarpWork &wk) const { return P - wk.st.skew; }   // stream bits read
  __device__ __forceinline__ bool overrun(const WarpWork &wk) const { return P > wk.st.limit; }
};

#if ZB_INFLATE_BULK
__device__ __forceinline__ void input_bar_init(WarpWork &wk, int lane) {
  if (lane == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(&wk.ldbar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
}
#else
__device__ __forceinline__ void input_bar_init(WarpWork &, int) {}
#endif

// ---- canonical walk for codes longer than the table (the reference's read_symbol, :584-591) --------
// Returns the symbol and its length, or -1 (the reference would run off counts.(16)).
__device__ __forceinline__ int canon_decode(uint32_t bits, const uint16_t *cnt, const uint16_t *syms, uint32_t &len_out) {
  int base = 0, offs = 0;
  for (int len = 1; len <= 15; len++) {
    offs = 2 * offs + (int)(bits & 1u);
    bits >>= 1;
    int count = cnt[len];
    if (offs < count) { len_out = (uint32_t)len; return syms[base + offs]; }
    base += count;
    offs -= count;
  }
  len_out = 15;
  return -1;
}

// ---- table construction (warp cooperative) -------------------------------------------------------------
// Builds one canonical decoder from ws.len[first .. first+n) into lut (2^bits entries), cnt[16] and the
// sorted symbol list syms (global).  Follows Huffman.init_decoder (reference :355-391) for what is accepted:
// over-subscribed -> corrupt; incomplete -> corrupt unless empty or a single code of length 1.
// max_valid_sym: symbols above it decode to "corrupt" (286/287 and 30/31 of the fixed codes).
template <bool IS_DIST>
__device__ void build_decoder_warp(WarpScratch &ws, int first, int n, int bits, void *lut_v, uint16_t *cnt,
                                   uint16_t *syms, const uint16_t *s_len_tab, const uint32_t *s_dist_tab, int lane) {
  uint16_t *lut16 = reinterpret_cast<uint16_t *>(lut_v);
  uint32_t *lut32 = reinterpret_cast<uint32_t *>(lut_v);
  if (lane < 16) ws.cnt[lane] = 0;
  __syncwarp();
  for (int i = lane; i < n; i += 32) {
    int l = ws.len[first + i];
    if (l) atomicAdd(&ws.cnt[l], 1u);
  }
  {  // clear the table: 0 = invalid
    const int words = IS_DIST ? (1 << bits) : (1 << bits) / 2;
    for (int i = lane; i < words; i += 32) lut32[i] = IS_DIST ? kDistInvalid : (uint32_t)kLitInvalid * 0x10001u;
  }
  __syncwarp();
  if (lane == 0) {
    int available = 1, num_codes = 0, code = 0, bad = 0;
    for (int l = 0; l < 16; l++) {
      int used = l ? (int)ws.cnt[l] : 0;
      if (used > available) bad = 1;                      // over-subscribed (:371)
      available = 2 * (available - used);
      ws.symoff[l] = (uint16_t)num_codes;                 // start of the length class in syms[]
      num_codes += used;
      int prev_used = l > 1 ? (int)ws.cnt[l - 1] : 0;     // canonical first code (RFC 1951 3.2.2)
      code = l ? (code + prev_used) << 1 : 0;
      ws.next[l] = (uint16_t)code;
      cnt[l] = (uint16_t)used;
    }
    if ((num_codes > 1 && available > 0) || (num_codes == 1 && ws.cnt[1] != 1)) bad = 1;  // (:377-378)
    if (bad) ws.err = 1;
    else {
      uint16_t off[16];
      for (int l = 0; l < 16; l++) off[l] = ws.symoff[l];
      int max_sym = -1;
      for (int i = 0; i < n; i++) {                       // symbols sorted by (length, symbol)
        int l = ws.len[first + i];
        if (!l) continue;
        max_sym = i;
        syms[off[l]++] = (uint16_t)i;
      }
      if (num_codes == 1) { cnt[1] = 2; syms[1] = (uint16_t)(max_sym + 1); }  // padding (:389-390)
    }
  }
  __syncwarp();
  if (ws.err) return;
  // Sorted position j of length class l carries code next[l] + (j - symoff[l]); codes are stored
  // bit-reversed because the stream delivers them most significant bit first.
  int total = 0;
  for (int l = 1; l < 16; l++) total += (int)ws.cnt[l];
  for (int j = lane; j < total; j += 32) {
    int l = 15;
    for (int t = 1; t < 15; t++)
      if (j < (int)ws.symoff[t + 1]) { l = t; break; }
    int sym = syms[j];
    uint32_t code = (uint32_t)ws.next[l] + (uint32_t)(j - (int)ws.symoff[l]);
    uint32_t rev = __brev(code) >> (32 - l);
    if (l <= bits) {
      if (IS_DIST) {
        uint32_t e = kDistInvalid;                        // 30, 31 never occur in valid data (:608)
        if (sym <= 29) { uint32_t dt = s_dist_tab[sym]; e = ((dt & 0xFFFFu) << 12) | ((uint32_t)l << 8) | ((uint32_t)l + (dt >> 16)); }
        for (uint32_t k = rev; k < (1u << bits); k += (1u << l)) lut32[k] = e;
      } else {
        uint16_t e = kLitInvalid;                         // 286, 287 never occur in valid data (:598)
        if (sym < 256) e = (uint16_t)((sym << 8) | l);
        else if (sym == 256) e = (uint16_t)(kCbStop | l);
        else if (sym <= 285) { uint32_t lt = s_len_tab[sym - 257]; e = (uint16_t)(((sym - 257) << 8) | kCbIsLen | (l + (lt >> 9))); }
        for (uint32_t k = rev; k < (1u << bits); k += (1u << l)) lut16[k] = e;
      }
    } else {
      if (IS_DIST) lut32[rev & ((1u << bits) - 1u)] = kDistLong;
      else lut16[rev & ((1u << bits) - 1u)] = kLitLong;
    }
  }
  __syncwarp();
}

// ---- one token through the canonical walk (codes longer than the tables), all lanes alike --------------------------
// pos: bit position of the token (the ring covers at least 1024 bits from the round's start).
// Returns 0 = token (tx, bits set), 1 = end of block (bits set), 2 = corrupt.
__device__ __noinline__ uint32_t slow_token(const WarpWork &wk, const WarpTabs &T, const uint16_t *syms,
                                            const uint16_t *s_len_tab, const uint32_t *s_dist_tab, uint64_t pos,
                                            uint32_t &tx, uint32_t &bits) {
  uint32_t w = Input::peek32_at(wk, pos);
  const uint32_t e = T.lit[w & ((1u << LB) - 1u)];
  int sym = -1;          // literal/length symbol
  uint32_t used = 0;     // bits of its code
  const uint32_t cb = e & 0xFFu;
  if (!(cb & kCbStop)) {
    const uint32_t p = cb & 31u;
    if (cb & kCbIsLen) { sym = 257 + (int)(e >> 8); used = p - (s_len_tab[e >> 8] >> 9); }
    else { sym = (int)(e >> 8); used = p; }
  } else if (cb == kCbLong) {
    sym = canon_decode(w, T.lit_cnt, syms, used);
    if (sym > 285) sym = -1;
  } else if (cb < kCbSlow) {
    sym = 256; used = cb & 31u;
  }  // kCbInvalid: sym stays -1
  bits = used;
  if (sym < 0) return 2;
  if (sym == 256) return 1;
  if (sym < 256) { tx = (uint32_t)sym; return 0; }
  const uint32_t lt = s_len_tab[sym - 257];
  const uint32_t ebits = lt >> 9;
  w = Input::peek32_at(wk, pos + used);
  const uint32_t mlen = (lt & 0x1FFu) + (w & ((1u << ebits) - 1u));
  used += ebits;
  w = Input::peek32_at(wk, pos + used);
  const uint32_t e2 = T.dist[w & ((1u << DB) - 1u)];
  uint32_t dist;
  if ((e2 & 0xFFu) < kDbInvalid) {
    const uint32_t dl = (e2 >> 8) & 15u, dtot = e2 & 0xFFu;
    dist = (e2 >> 12) + ((w >> dl) & ~(0xFFFFFFFFu << (dtot - dl)));
    used += dtot;
  } else {
    uint32_t dl = 0;
    int dsym = e2 == kDistLong ? canon_decode(w, T.dist_cnt, syms + 288, dl) : -1;
    if (dsym < 0 || dsym > 29) { bits = used; return 2; }
    used += dl;
    w = Input::peek32_at(wk, pos + used);
    const uint32_t dt = s_dist_tab[dsym];
    dist = (dt & 0xFFFFu) + (w & ((1u << (dt >> 16)) - 1u));
    used += dt >> 16;
  }
  tx = (mlen << 16) | dist;
  bits = used;
  return 0;
}

// ---- dynamic block header (reference :623-669): HLIT / HDIST / HCLEN, the code length code, the run-length coded lengths,
// then both decoders.  Called right after the three block-type bits; every lane parses the header redundantly (uniform
// control flow, broadcast reads of the ring).  Returns true if the header is not acceptable to the reference's decoder.
__device__ bool read_dynamic_header(Input &in, WarpWork &wk, WarpTabs &mine, uint16_t *my_syms, const uint16_t *s_len_tab,
                                    const uint32_t *s_dist_tab, int lane) {
  WarpScratch &ws = wk.build;
  // every lane parses the header redundantly (uniform control flow, broadcast reads of the ring)
  uint32_t hlit = 257 + in.get(wk, 5, lane);
  uint32_t hdist = 1 + in.get(wk, 5, lane);
  uint32_t hclen = 4 + in.get(wk, 4, lane);
  bool bad = hlit > 286 || hdist > 30;
  // code length code lengths, 3 bits per symbol, packed by symbol
  uint64_t clc = 0;
  for (uint32_t i = 0; i < hclen; i++) clc |= (uint64_t)in.get(wk, 3, lane) << (3 * c_clen_order[i]);
  if (in.overrun(wk)) bad = true;
  // code-length decoder (7-bit table in the distance area, 8-bit entries: len << 5 | sym)
  uint8_t *cl_lut = reinterpret_cast<uint8_t *>(mine.dist);
  uint64_t next = 0;  // next code per length, 8 bits each
  if (!bad) {
    uint64_t cnt5 = 0;  // codes per length, 5 bits each (max 19)
    int max_sym = -1;
    for (int s = 0; s < 19; s++) {
      uint32_t l = (uint32_t)(clc >> (3 * s)) & 7u;
      if (l) { cnt5 += 1ull << (5 * l); max_sym = s; }
    }
    int available = 1, num_codes = 0, code = 0;
    for (int l = 0; l < 8; l++) {
      int used = l ? (int)((cnt5 >> (5 * l)) & 31u) : 0;
      if (used > available) bad = true;
      available = 2 * (available - used);
      num_codes += used;
      int prev_used = l > 1 ? (int)((cnt5 >> (5 * (l - 1))) & 31u) : 0;
      code = l ? (code + prev_used) << 1 : 0;
      next |= (uint64_t)(code & 0xff) << (8 * l);
    }
    if ((num_codes > 1 && available > 0) || (num_codes == 1 && ((cnt5 >> 5) & 31u) != 1) || max_sym == -1)
      bad = true;
  }
  if (!bad) {
    __syncwarp();
    reinterpret_cast<uint32_t *>(cl_lut)[lane] = 0;
    __syncwarp();
    if (lane == 0) {
      for (int s = 0; s < 19; s++) {
        uint32_t l = (uint32_t)(clc >> (3 * s)) & 7u;
        if (!l) continue;
        uint32_t code = (uint32_t)(next >> (8 * l)) & 0xffu;
        next += 1ull << (8 * l);
        uint32_t rev = __brev(code) >> (32 - l);
        for (uint32_t k = rev; k < 128; k += (1u << l)) cl_lut[k] = (uint8_t)((l << 5) | s);
      }
    }
    __syncwarp();
    // decode hlit + hdist code lengths straight into the build scratch
    uint32_t num = 0, total = hlit + hdist, prev = 0;
    while (num < total && !bad) {
      in.ensure(wk, lane);
      uint32_t w = in.peek32(wk);
      uint32_t e = cl_lut[w & 127u];
      if (!e) { bad = true; break; }
      uint32_t used = e >> 5;
      uint32_t sym = e & 31u, rep = 1, val = sym;
      if (sym == 16) {
        if (num == 0) { bad = true; break; }
        rep = 3 + ((w >> used) & 3u); used += 2; val = prev;
      } else if (sym == 17) { rep = 3 + ((w >> used) & 7u); used += 3; val = 0; }
      else if (sym == 18) { rep = 11 + ((w >> used) & 127u); used += 7; val = 0; }
      in.P += used;
      if (rep > total - num) { bad = true; break; }
      if (lane == 0)
        for (uint32_t r = 0; r < rep; r++) ws.len[num + r] = (uint8_t)val;
      num += rep;
      prev = val;
    }
    if (in.overrun(wk)) bad = true;
    __syncwarp();
    if (!bad) {
      for (uint32_t i = total + lane; i < 320; i += 32) ws.len[i] = 0;
      if (lane == 0) ws.err = 0;
      __syncwarp();
      if (ws.len[256] == 0) bad = true;  // no end-of-block code (:662)
      __syncwarp();
      if (!bad) build_decoder_warp<false>(ws, 0, (int)hlit, LB, mine.lit, mine.lit_cnt, my_syms, s_len_tab, s_dist_tab, lane);
      __syncwarp();
      if (!bad && !ws.err) build_decoder_warp<true>(ws, (int)hlit, (int)hdist, DB, mine.dist, mine.dist_cnt, my_syms + 288, s_len_tab, s_dist_tab, lane);
      __syncwarp();
      if (ws.err) bad = true;
    }
  }
  return bad;
}

// ---- the kernel ------------------------------------------------------------------------------------------
// SPEC: speculative decoding of one chunk of a large stream (intra-stream parallel inflate).  The chunk starts at a block
// header somewhere inside the stream, so the 32 KiB of output that precede it are unknown: the output is 16-bit symbols, a
// byte or 0x8000 | w = "byte w of that unknown window" (copies of such symbols simply carry them along), resolved later by
// resolve_kernel.  Decoding stops at the first block boundary at or after the task's stop_bit.
template <bool COUNT_ONLY, bool SPEC>
__global__ void __launch_bounds__(THREADS, 1)
inflate_kernel(const InflateTask *__restrict__ tasks, uint32_t ntasks, InflateResult *__restrict__ results,
               unsigned int *__restrict__ queue, uint16_t *__restrict__ g_syms, int adler_mode,
               unsigned int *__restrict__ group_count, uint32_t *__restrict__ group_flag,
               const uint32_t *__restrict__ upload_flag, uint32_t upload_serial, uint64_t *__restrict__ block_lens) {
  // adler_mode: -1 = no checksum in this kernel, else ZIPC_ADLER_* (fused per-block Adler-32 of the output)
  // group_count / group_flag (may be null): streams left in each download group; the warp that finishes a group's last
  // stream raises the group's flag (mapped host memory), and the host starts copying that range of the arena
  // block_lens (SPEC, may be null): kSpecBlocks entries per task, the output lengths of the chunk's non-empty blocks (64 bits:
  // one block may output 4 GiB or more)
  // upload_flag / upload_serial: a stream whose flags name part p >= 1 of a split upload is opened only once *upload_flag has
  // reached upload_serial + p (its bytes travel on another stream while this kernel already works on the first part)
  extern __shared__ __align__(16) uint8_t smem_raw[];
  WarpTabs *tabs = reinterpret_cast<WarpTabs *>(smem_raw);                  // [WARPS] + fixed
  WarpTabs &fixed = tabs[WARPS];
  WarpWork *works = reinterpret_cast<WarpWork *>(tabs + WARPS + 1);
  uint16_t *s_len_tab = reinterpret_cast<uint16_t *>(works + WARPS);
  uint32_t *s_dist_tab = reinterpret_cast<uint32_t *>(s_len_tab + 32);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpTabs &mine = tabs[warp];
  WarpWork &wk = works[warp];
  WarpScratch &ws = wk.build;
  const uint32_t slot = blockIdx.x * WARPS + warp;
  uint16_t *my_syms = g_syms + (size_t)slot * SYMS_PER_SLOT;
  uint16_t *fixed_syms = g_syms + (size_t)(gridDim.x * WARPS + blockIdx.x) * SYMS_PER_SLOT;
  const uint32_t lt_mask = (1u << lane) - 1u;

  if (threadIdx.x < 29) s_len_tab[threadIdx.x] = c_len_tab[threadIdx.x];
  if (threadIdx.x < 30) s_dist_tab[threadIdx.x] = c_dist_tab[threadIdx.x];
  __syncthreads();
  // fixed-Huffman decoders, once per CTA (reference :334-349)
  if (warp == 0) {
    for (int i = lane; i < 320; i += 32) {
      uint8_t l = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
      ws.len[i] = l;
    }
    if (lane == 0) ws.err = 0;
    __syncwarp();
    build_decoder_warp<false>(ws, 0, 288, LB, fixed.lit, fixed.lit_cnt, fixed_syms, s_len_tab, s_dist_tab, lane);
    build_decoder_warp<true>(ws, 288, 32, DB, fixed.dist, fixed.dist_cnt, fixed_syms + 288, s_len_tab, s_dist_tab, lane);
  }
  __syncthreads();

  // decoder state: identical in all lanes of the warp (no broadcasts needed, branches are uniform)
  uint32_t state = S_IDLE, task = 0, status = ZIPC_OK;
  Input in{};
  input_bar_init(wk, lane);
  WarpState &st = wk.st;
  uint8_t *dst = nullptr;
  uint64_t out_pos = 0;
  bool final_blk = false, first_task = true, segment = false, use_fixed = false;
  uint32_t stored_len = 0;
  uint64_t stored_at = 0;     // stream offset of the stored block's bytes
  uint32_t ad_state = 1;      // running Adler-32 (reference :558, :682-690)
  bool ad_pending = false;    // a block just ended: fold [st.ad_from, out_pos)
  uint64_t stop_bit = ~0ull;  // SPEC: finish at the first block boundary at or after this stream bit
  typedef typename std::conditional<SPEC, uint16_t, uint8_t>::type elem_t;  // what one output symbol is

  for (;;) {
    // ---- A: pull work -----------------------------------------------------------------------------------
    if (state == S_IDLE) {
      // first task: interleaved over the CTAs so the longest streams (sorted first) spread over all SMs;
      // afterwards from the shared queue, which starts behind the statically assigned ones
      if (first_task) { task = (uint32_t)warp * gridDim.x + blockIdx.x; first_task = false; }
      else {
        if (lane == 0) task = atomicAdd(queue, 1u);
        task = __shfl_sync(0xffffffffu, task, 0);
      }
      if (task >= ntasks) {
#if ZB_INFLATE_BULK
        in.settle(wk);  // no copy may land in this CTA's shared memory after it is gone
#endif
        break;
      }
      const InflateTask t = tasks[task];
      if (!COUNT_ONLY && !SPEC && ((t.flags >> kInflatePartShift) & kInflatePartMask) && upload_flag) {
        const uint32_t need = upload_serial + ((t.flags >> kInflatePartShift) & kInflatePartMask);
        // (bounded: if that copy failed the host reports it; the warp then decodes whatever is there and the call fails anyway)
        uint32_t seen = 0;
        for (uint32_t spins = 0; spins < (1u << 24); spins++) {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(upload_flag) : "memory");
          if ((int32_t)(seen - need) >= 0) break;
          __nanosleep(256);
        }
      }
      __syncwarp();
      if (lane == 0) { st.src = t.src; st.src_len = t.src_len; st.out_cap = t.dst_cap; st.ad_from = 0; st.nblk = 0; }
      dst = t.dst; segment = (t.flags & kInflateSegment) != 0;
      out_pos = 0; status = ZIPC_OK; final_blk = false;
      ad_state = 1; ad_pending = false;
      in.open(wk, lane);
      if (SPEC) { in.seek_bits(wk, (uint64_t)st.skew + t.start_bit, lane); stop_bit = t.stop_bit; }
      state = S_HDR;
    }

    // ---- B: block header (reference :692-702, :623-661, :671-677) ------------------------------------------
    if (state == S_HDR && segment && in.consumed(wk) == st.src_len * 8) {
      state = S_FINISH;  // a segment ends at the block boundary where its input ends (byte aligned by construction)
    }
    if (state == S_HDR) {
      uint32_t h = in.get(wk, 3, lane);
      final_blk = h & 1u;
      uint32_t type = h >> 1;
      if (in.overrun(wk)) { status = ZIPC_ERR_CORRUPTED; state = S_FINISH; }
      else if (type == 0) {
        in.P += (8u - ((uint32_t)in.consumed(wk) & 7u)) & 7u;  // to the byte boundary
        uint32_t length = in.get(wk, 16, lane), inv = in.get(wk, 16, lane);
        uint64_t pos = in.consumed(wk) >> 3;
        if (in.overrun(wk) || length != ((~inv) & 0xFFFFu) || st.src_len - pos < length) {
          status = ZIPC_ERR_CORRUPTED; state = S_FINISH;
        } else if (out_pos + length > st.out_cap) {
          status = ZIPC_ERR_SIZE_EXCEEDED; state = S_FINISH;
        } else {
          stored_len = length;
          stored_at = pos;
          in.seek_bits(wk, (uint64_t)st.skew + 8 * (pos + length), lane);
          state = S_STORED;
        }
      } else if (type == 1) {
        use_fixed = true;
        state = S_DATA;
      } else if (type == 2) {
        const bool bad = read_dynamic_header(in, wk, mine, my_syms, s_len_tab, s_dist_tab, lane);
        if (bad) { status = ZIPC_ERR_CORRUPTED; state = S_FINISH; }
        else {
          use_fixed = false;
          state = S_DATA;
        }
      } else {
        status = ZIPC_ERR_CORRUPTED; state = S_FINISH;
      }
    }

    // ---- D: one round of up to 32 tokens (reference :593-616) ---------------------------------------------------
    if (state == S_DATA) {
      const WarpTabs &T = use_fixed ? fixed : mine;
      const uint16_t *lit_lut = T.lit;
      const uint32_t *dist_lut = T.dist;
      uint32_t n = 0, rel = 0;                 // tokens and bytes of this round (uniform)
      uint32_t tx = 0, trel = 0, tend = 0;     // lane i: token i, its output offset in the round, its end in the input
      const uint64_t P0 = in.P;
      uint32_t stop = 0;                       // 1 = end of block, 3 = undecodable token (corrupt stream)
      uint32_t eob_bits = 0;
      uint32_t slowmask = 0;                   // bit k: token k went through the slow path
      in.ensure(wk, lane);
      // D1: how many bits would a token starting at bit P + lane + 32 j occupy?  Straight-line code: both table
      // lookups are made for every candidate (NB independent chains per lane); values are decoded later, and only
      // for the offsets that turn out to be real token starts.
      {
        const uint32_t sh = ((uint32_t)in.P & 31u) + lane;
        const uint32_t wi = (uint32_t)(in.P >> 5) + (sh >> 5);
        const uint32_t s = sh & 31u;
        const uint32_t dist_sa = (uint32_t)__cvta_generic_to_shared(dist_lut);
        uint32_t a[NB + 2];
#pragma unroll
        for (int t = 0; t < NB + 2; t++) a[t] = wk.ring[(wi + t) & kRingMask];
#pragma unroll
        for (int j = 0; j < NB; j++) {
          const uint32_t lo = __funnelshift_r(a[j], a[j + 1], s), hi = __funnelshift_r(a[j + 1], a[j + 2], s);
          const uint32_t e = lit_lut[lo & ((1u << LB) - 1u)];
          const uint32_t p = e & 31u;
          const uint32_t d32 = __funnelshift_r(lo, hi, p);
          uint32_t e2;  // volatile: keeps the load out of a branch
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(e2) : "r"(dist_sa + 4u * (d32 & ((1u << DB) - 1u))));
          // length symbol (and not a stop entry): bits of the whole token, >= kCbSlow if the distance part is not
          // decodable;  anything else: the candidate byte as stored in the table
          const uint32_t c = (e & 0xC0u) == kCbIsLen ? p + (e2 & 0xFFu) : e;
          wk.cand[j * 32 + lane] = (uint8_t)c;
        }
        if (lane < 16) reinterpret_cast<uint32_t *>(wk.cand + WBITS)[lane] = 0xFEFEFEFEu;  // (table building reuses the area)
      }
      __syncwarp();
      // D2: follow the chain of real tokens through the candidates.  All lanes walk alike, 32 steps, straight line:
      // load the candidate, note its address as token k, add the bits it occupies.  A candidate with bit 7 set (end
      // of block, a code the tables do not hold, the padding behind the window) counts as zero bits, so the walk
      // stays where it stopped and the tokens from there on repeat one address: token k is real iff entry k + 1
      // differs from entry k.  4 instructions per step, no branch (the loop with its exit tests carried 10).
      {
        const uint32_t cand_sa = (uint32_t)__cvta_generic_to_shared(wk.cand);
        const uint32_t tokq_sa = (uint32_t)__cvta_generic_to_shared(wk.tokq);
        uint32_t ca = cand_sa;
        // the queue keeps the low 16 bits of a token's candidate address: offset = (entry - cand_sa) mod 2^16
        asm volatile(
            "{\n"
            ".reg .s32 c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+0], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+2], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+4], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+6], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+8], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+10], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+12], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+14], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+16], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+18], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+20], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+22], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+24], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+26], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+28], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+30], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+32], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+34], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+36], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+38], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+40], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+42], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+44], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+46], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+48], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+50], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+52], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+54], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+56], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+58], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+60], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
              "  ld.shared.s8 c, [%0];\n  st.shared.u16 [%1+62], %0;\n  max.s32 c, c, 0;\n  add.u32 %0, %0, c;\n"
            "  st.shared.u16 [%1+64], %0;\n"
            "}\n"
            : "+r"(ca)
            : "r"(tokq_sa)
            : "memory");
        __syncwarp();
        const uint32_t q0 = wk.tokq[lane], q1 = wk.tokq[lane + 1];
        const uint32_t stuck = __ballot_sync(0xffffffffu, q0 == q1);
        n = stuck ? (uint32_t)(__ffs((int)stuck) - 1) : (uint32_t)ROUND_TOKENS;
        uint32_t o = (ca - cand_sa) & 0xFFFFu;   // where the walk stands: behind the last real token
        if (n < (uint32_t)ROUND_TOKENS && o < (uint32_t)WBITS) {
          const uint32_t c = wk.cand[o];
          if (c < kCbSlow) { stop = 1; eob_bits = c & 31u; }
          else {
            // long or invalid code: this one token goes through the canonical walk and ends the round
            uint32_t stx = 0, sbits = 0;
            const uint32_t r = slow_token(wk, T, g_syms + (size_t)(use_fixed ? gridDim.x * WARPS + blockIdx.x : slot) * SYMS_PER_SLOT, s_len_tab, s_dist_tab, P0 + o, stx, sbits);
            if (r) { stop = r == 1 ? 1u : 3u; eob_bits = sbits; }
            else {
              wk.slow_tx[n] = stx;
              wk.slow_end[n] = (uint16_t)(o + sbits);
              slowmask = 1u << n;
              o += sbits;
              n++;
            }
          }
        }
        in.P += o;
      }
      __syncwarp();
      // lane i decodes token i (table entries are known to be plain ones); output offsets by a scan over the lengths
      {
        uint32_t tlen = 0;
        const uint32_t oq = (wk.tokq[lane] - (uint32_t)__cvta_generic_to_shared(wk.cand)) & 0xFFFFu;
        if ((slowmask >> lane) & 1u) {
          tx = wk.slow_tx[lane];
          tlen = (tx >> 16) ? tx >> 16 : 1u;
          tend = wk.slow_end[lane];
        } else if (lane < (int)n) {
          const uint32_t o = oq;
          const uint64_t pb = P0 + o;
          const uint32_t k = (uint32_t)(pb >> 5), sb = (uint32_t)pb & 31u;
          const uint32_t w0 = wk.ring[k & kRingMask], w1 = wk.ring[(k + 1) & kRingMask], w2 = wk.ring[(k + 2) & kRingMask];
          const uint32_t lo = __funnelshift_r(w0, w1, sb), hi = __funnelshift_r(w1, w2, sb);
          const uint32_t e = lit_lut[lo & ((1u << LB) - 1u)];
          const uint32_t p = e & 31u;
          if (e & kCbIsLen) {
            const uint32_t lt = s_len_tab[e >> 8];
            const uint32_t ebits = lt >> 9;
            const uint32_t mlen = (lt & 0x1FFu) + ((lo >> (p - ebits)) & ~(0xFFFFFFFFu << ebits));
            const uint32_t d32 = __funnelshift_r(lo, hi, p);
            const uint32_t e2 = dist_lut[d32 & ((1u << DB) - 1u)];
            const uint32_t dl = (e2 >> 8) & 15u, dtot = e2 & 0xFFu;
            const uint32_t dist = (e2 >> 12) + ((d32 >> dl) & ~(0xFFFFFFFFu << (dtot - dl)));
            tx = (mlen << 16) | dist;
            tlen = mlen;
            tend = o + p + dtot;
          } else {
            tx = e >> 8;
            tlen = 1;
            tend = o + p;
          }
        }
        uint32_t inc = tlen;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          uint32_t v = __shfl_up_sync(0xffffffffu, inc, d);
          if (lane >= d) inc += v;
        }
        trel = inc - tlen;
        rel = __shfl_sync(0xffffffffu, inc, 31);
      }
      __syncwarp();  // cand / tokq are rewritten by the next round

      // checks, one token per lane, in the reference's order: input overrun / distance -> corrupted, then size
      if (state == S_DATA) {
        const bool have = lane < (int)n;
        const uint32_t mlen = tx >> 16, mdist = tx & 0xFFFFu;
        const uint32_t tlen = mlen ? mlen : 1u;
        const uint32_t hist0 = out_pos < 32768 ? (uint32_t)out_pos : 32768u;
        const uint64_t room64 = st.out_cap - out_pos;
        const uint32_t room0 = room64 > 0x7FFFFFFFull ? 0x7FFFFFFFu : (uint32_t)room64;
        // (SPEC: a distance may reach into the unknown window before the chunk; the format caps it at 32768)
        const bool corrupt = have && ((!SPEC && mlen && mdist > min(hist0 + trel, 32768u)) || P0 + tend > st.limit);
        const bool exceed = have && trel + tlen > room0;
        const uint32_t fm = __ballot_sync(0xffffffffu, corrupt || exceed);
        if (fm) {
          const int f = __ffs((int)fm) - 1;
          n = (uint32_t)f;
          rel = __shfl_sync(0xffffffffu, trel, f);
          status = __shfl_sync(0xffffffffu, (int)corrupt, f) ? ZIPC_ERR_CORRUPTED : ZIPC_ERR_SIZE_EXCEEDED;
          state = S_FINISH;
          stop = 0;
        }
      }
      if (stop == 3 && state == S_DATA) { status = ZIPC_ERR_CORRUPTED; state = S_FINISH; }
      if (stop == 1 && state == S_DATA) {  // end of block
        in.P += eob_bits;
        if (in.overrun(wk)) { status = ZIPC_ERR_CORRUPTED; state = S_FINISH; }
        else {
          state = final_blk ? S_FINISH : S_HDR; ad_pending = true;
          if (SPEC && in.consumed(wk) >= stop_bit) state = S_FINISH;
        }
      }

      // ---- E: execute the round's tokens -------------------------------------------------------------------
      if (!COUNT_ONLY && n) {
        const bool have = lane < (int)n;
        const uint32_t mlen = have ? tx >> 16 : 0u, mdist = tx & 0xFFFFu;
        const uint32_t tlen = have ? (mlen ? mlen : 1u) : 0u;
        // a match is independent of this round when all of its source bytes precede the round
        const bool dep = mlen && mdist < trel + min(mdist, mlen);
        elem_t *const obase = reinterpret_cast<elem_t *>(dst) + out_pos;
        // element q of a match whose output starts at round offset orel: from the output `odist` elements back (overlapping
        // matches repeat their first odist elements), or -- SPEC only -- from the unknown window before the chunk
        auto fetch = [&](uint32_t orel, uint32_t olen, uint32_t odist, uint32_t q) -> uint32_t {
          const uint32_t qq = odist < olen ? q % odist : q;
          unsigned int v;
          if (SPEC) {
            const int64_t sidx = (int64_t)(out_pos + orel + qq) - (int64_t)odist;
            if (sidx < 0) return 0x8000u | (uint32_t)(32768 + sidx);
            asm volatile("ld.global.cg.u16 %0, [%1];" : "=r"(v) : "l"(reinterpret_cast<const uint16_t *>(dst) + sidx) : "memory");
          } else {
            asm volatile("ld.global.cg.u8 %0, [%1];" : "=r"(v) : "l"(dst + out_pos + orel + qq - odist) : "memory");
          }
          return v;
        };
        // E1: literals go straight out, one lane each (no loads involved)
        if (have && !mlen) obase[trel] = (elem_t)tx;
        // independent matches: their bytes flattened over the lanes
        const uint32_t li = (dep || !mlen) ? 0u : tlen;
        uint32_t incI = li;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          uint32_t v = __shfl_up_sync(0xffffffffu, incI, o);
          if (lane >= o) incI += v;
        }
        const uint32_t totalI = __shfl_sync(0xffffffffu, incI, 31);
        const uint32_t bI = __ballot_sync(0xffffffffu, li != 0);
        if (li) wk.cidx[__popc(bI & lt_mask)] = (uint8_t)lane;
        __syncwarp();
        const uint32_t istart = incI - li;
        uint32_t rbase = 0;  // independent tokens that end before the current window
        constexpr int kPasses = 4;  // loads of up to 128 bytes are in flight before the first store
        for (uint32_t base = 0; base < totalI; base += 32 * kPasses) {
          uint32_t val[kPasses];
          elem_t *dq[kPasses];
#pragma unroll
          for (int u = 0; u < kPasses; u++) {
            const uint32_t wb = base + 32 * u;
            if (wb >= totalI) { dq[u] = nullptr; val[u] = 0; continue; }   // (uniform) nothing left for this pass
            const uint32_t b = wb + lane;
            const bool act = b < totalI;
            const uint32_t endrel = incI - wb;   // end of my token relative to the window
            const uint32_t M = __reduce_or_sync(0xffffffffu, (li && (endrel - 1u) < 32u) ? 1u << (endrel - 1u) : 0u);
            const uint32_t r = rbase + __popc(M & lt_mask);
            rbase += __popc(M);
            const int own = act ? (int)wk.cidx[r] : 0;
            const uint32_t ox = __shfl_sync(0xffffffffu, tx, own);
            const uint32_t orel = __shfl_sync(0xffffffffu, trel, own);
            const uint32_t q = b - __shfl_sync(0xffffffffu, istart, own);
            const uint32_t olen = ox >> 16, odist = ox & 0xFFFFu;
            dq[u] = act ? obase + orel + q : nullptr;
            val[u] = ox & 0xFFu;
            if (act && olen) val[u] = fetch(orel, olen, odist, q);
          }
#pragma unroll
          for (int u = 0; u < kPasses; u++)
            if (dq[u]) *dq[u] = (elem_t)val[u];
        }
        __syncwarp();
        // E2: matches that read bytes produced in this round, in token order
        uint32_t dm = __ballot_sync(0xffffffffu, dep);
        while (dm) {
          const int t = __ffs((int)dm) - 1;
          dm &= dm - 1;
          const uint32_t ox = __shfl_sync(0xffffffffu, tx, t);
          const uint32_t orel = __shfl_sync(0xffffffffu, trel, t);
          const uint32_t olen = ox >> 16, odist = ox & 0xFFFFu;
          for (uint32_t q = lane; q < olen; q += 32) obase[orel + q] = (elem_t)fetch(orel, olen, odist, q);
          __syncwarp();
        }
      }
      out_pos += rel;
    }

    // ---- stored block: one coalesced copy from the input (reference :678-680) ------------------------------------
    if (state == S_STORED) {
      if (!COUNT_ONLY) {
        elem_t *dp = reinterpret_cast<elem_t *>(dst) + out_pos;
        const uint8_t *sp = st.src + stored_at;
        for (uint32_t i = lane; i < stored_len; i += 32) dp[i] = sp[i];
        __syncwarp();
      }
      out_pos += stored_len;
      state = final_blk ? S_FINISH : S_HDR;
      if (SPEC && in.consumed(wk) >= stop_bit) state = S_FINISH;
      ad_pending = true;
    }

    // ---- G: checksum of the block that just ended (reference inflated_block_crc, :682-690) ---------------------
    // Adler-32 restarts its 5552-byte chunk grid at every block and, as written in the reference, reduces
    // with a signed remainder, so it has to be folded block by block to stay bit-exact.
    if (ad_pending) {
      if (SPEC && block_lens) {
        // speculative chunk: the output length of every non-empty block goes to the chunk's list: the host folds the Adler-32
        // of a large zlib stream over these blocks
        if (lane == 0) {
          const uint64_t blen = out_pos - st.ad_from;
          if (blen) {
            if (st.nblk < kSpecBlocks) block_lens[(size_t)task * kSpecBlocks + st.nblk] = blen;
            st.nblk++;
            st.ad_from = out_pos;
          }
        }
        __syncwarp();
      }
      if (!COUNT_ONLY && !SPEC && adler_mode >= 0) {
        __syncwarp();
        ad_state = adler_update_warp<true>(ad_state, dst + st.ad_from, out_pos - st.ad_from, adler_mode, lane);
        ad_state = __shfl_sync(0xffffffffu, ad_state, 0);
        __syncwarp();
        if (lane == 0) st.ad_from = out_pos;
        __syncwarp();
      }
      ad_pending = false;
    }

    // ---- F: report -------------------------------------------------------------------------------------------
    if (state == S_FINISH) {
      if (lane == 0) {
        InflateResult r;
        r.out_len = status == ZIPC_OK ? out_pos : 0;
        r.status = status;
        r._pad = status == ZIPC_OK ? ad_state : 0;  // fused Adler-32 of the output (when requested)
        r.end_bit = in.consumed(wk);
        r.final_seen = final_blk ? 1u : 0u;
        r._pad2 = SPEC ? st.nblk : 0u;              // (speculative chunks) non-empty blocks decoded: their lengths are in the chunk's list
        if (SPEC && block_lens && st.nblk > kSpecBlocks && status == ZIPC_OK) { r.status = ZIPC_ERR_DST_TOO_SMALL; r.out_len = 0; }  // list full: not this way
        results[task] = r;
      }
      if (!COUNT_ONLY && !SPEC && group_count) {
        __threadfence();   // every lane: my bytes of this stream are out
        __syncwarp();
        if (lane == 0 && atomicSub(&group_count[tasks[task].group], 1u) == 1u) {
          __threadfence_system();
          *reinterpret_cast<volatile uint32_t *>(&group_flag[tasks[task].group]) = 1u;
        }
      }
      state = S_IDLE;
    }
  }
}

// ---- intra-stream parallel inflate: where do blocks start? -----------------------------------------------------------------
// A deflate stream has no index, but a dynamic-Huffman block header is so constrained (HLIT / HDIST ranges, a complete
// code-length code, run-length coded lengths that fit exactly, an end-of-block code, complete literal/length and distance
// codes) that scanning for a bit position where a valid one starts finds real block starts with next to no false positives
// (the approach of pugz / rapidgzip).  One warp per chunk k >= 1 scans [8 k chunk_bytes, 8 (k + 1) chunk_bytes): the lanes
// test 32 consecutive bit offsets with a cheap filter (block type, HLIT, HDIST, Kraft sum of the code-length code); offsets
// that pass are validated by the decoder's own header reader, in order, and the first valid one is reported.  A wrong
// guess is caught later: the chunk before it must END exactly there, or the caller falls back to serial decoding.
// Stored and fixed blocks are not looked for (their headers say too little); the previous chunk just runs through them.
constexpr uint32_t kFindSplit = 4;
__global__ void __launch_bounds__(THREADS, 1)
find_starts_kernel(const uint8_t *__restrict__ src, uint64_t src_len, uint64_t first_bit, uint64_t chunk_bytes, uint32_t nchunks,
                   uint64_t *__restrict__ found, uint16_t *__restrict__ g_syms) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  WarpTabs *tabs = reinterpret_cast<WarpTabs *>(smem_raw);
  WarpWork *works = reinterpret_cast<WarpWork *>(tabs + WARPS + 1);
  uint16_t *s_len_tab = reinterpret_cast<uint16_t *>(works + WARPS);
  uint32_t *s_dist_tab = reinterpret_cast<uint32_t *>(s_len_tab + 32);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // Kraft weight (in 1/128) of three 3-bit code lengths at once: the fixed-Huffman slot of the table area is unused here
  uint8_t *kraft3 = reinterpret_cast<uint8_t *>(&tabs[WARPS]);
  if (threadIdx.x < 29) s_len_tab[threadIdx.x] = c_len_tab[threadIdx.x];
  if (threadIdx.x < 30) s_dist_tab[threadIdx.x] = c_dist_tab[threadIdx.x];
  if (threadIdx.x < 512) {
    uint32_t w = 0;
    for (int f = 0; f < 3; f++) { const uint32_t l = (threadIdx.x >> (3 * f)) & 7u; w += l ? 128u >> l : 0u; }
    kraft3[threadIdx.x] = (uint8_t)w;   // <= 3 * 64
  }
  __syncthreads();
  WarpTabs &mine = tabs[warp];
  WarpWork &wk = works[warp];
  uint16_t *my_syms = g_syms + (size_t)(blockIdx.x * WARPS + warp) * SYMS_PER_SLOT;
  Input in{};
  input_bar_init(wk, lane);
  // kFindSplit warps share a nominal chunk (a quarter of its bit offsets each); the earliest hit wins (atomicMin: `found` starts as ~0)
  for (uint32_t u = kFindSplit + blockIdx.x * WARPS + warp; u < nchunks * kFindSplit; u += gridDim.x * WARPS) {
    const uint32_t k = u / kFindSplit, part = u % kFindSplit;
    __syncwarp();
    if (lane == 0) { wk.st.src = src; wk.st.src_len = src_len; wk.st.out_cap = 0; wk.st.ad_from = 0; }
    in.open(wk, lane);
    const uint64_t skew = wk.st.skew, limit = wk.st.limit;
    const uint64_t span = (8 * chunk_bytes / kFindSplit + 31) & ~31ull;
    const uint64_t cbeg = skew + first_bit + 8 * (uint64_t)k * chunk_bytes;   // (the nominal chunks are laid from first_bit on)
    const uint64_t beg = cbeg + part * span;
    uint64_t end = part + 1 == kFindSplit ? cbeg + 8 * chunk_bytes : beg + span;
    if (end > limit) end = limit;
    uint64_t hit = ~0ull;
    in.seek_bits(wk, beg, lane);
    for (uint64_t base = beg; base < end && hit == ~0ull; base += 32) {
      if ((uint32_t)(base >> 5) < in.w0) in.seek_bits(wk, base, lane);  // a header parse moved the ring on
      in.P = base;
      in.ensure(wk, lane);
      // cheap filter at offset base + lane: 17 bits of block header + up to 19 three-bit code-length code lengths
      const uint64_t pos = base + lane;
      bool ok = pos < end && pos + 17 + 57 <= limit;
      const uint32_t w0 = Input::peek32_at(wk, pos), w1 = Input::peek32_at(wk, pos + 32), w2 = Input::peek32_at(wk, pos + 64);
      ok = ok && (w0 & 7u) == 4u;                                        // BFINAL 0, BTYPE 2
      ok = ok && ((w0 >> 3) & 31u) <= 29u && ((w0 >> 8) & 31u) <= 29u;   // HLIT <= 286, HDIST <= 30
      if (ok) {
        const uint32_t hclen = 4 + ((w0 >> 13) & 15u);
        unsigned long long cl = (unsigned long long)(w0 >> 17) | ((unsigned long long)w1 << 15) | ((unsigned long long)w2 << 47);
        cl &= ~0ull >> (64 - 3 * hclen);                                 // the lengths that are there (12 .. 57 bits)
        uint32_t kraft = 0;
#pragma unroll
        for (int g = 0; g < 7; g++) kraft += kraft3[(uint32_t)(cl >> (9 * g)) & 511u];
        ok = kraft == 128u;                                              // a complete code over the code lengths
      }
      uint32_t surv = __ballot_sync(0xffffffffu, ok);
      while (surv) {  // full validation by the decoder's own header reader, in stream order
        const int l = __ffs((int)surv) - 1;
        surv &= surv - 1;
        const uint64_t cand = base + l;
        if ((uint32_t)(cand >> 5) < in.w0) in.seek_bits(wk, cand, lane);
        const uint32_t hlit = 257u + ((Input::peek32_at(wk, cand) >> 3) & 31u);
        in.P = cand + 3;
        if (read_dynamic_header(in, wk, mine, my_syms, s_len_tab, s_dist_tab, lane)) continue;
        // A header that checks out can still be an accident of the bits inside a block: nearly all such accidents are
        // degenerate codes (two symbols of one bit, ...).  A start is only worth something if it is certain, a missed one
        // costs nothing but parallelism (the chunk before it decodes on through it): ask for a code of some substance.
        uint32_t coded = 0;
        for (uint32_t i = lane; i < hlit; i += 32) coded += wk.build.len[i] != 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) coded += __shfl_xor_sync(0xffffffffu, coded, o);
        if (coded >= 12u) { hit = cand; break; }
      }
    }
    if (lane == 0 && hit != ~0ull) atomicMin(reinterpret_cast<unsigned long long *>(&found[k]), (unsigned long long)(hit - skew));
  }
#if ZB_INFLATE_BULK
  in.settle(wk);
#endif
}

// ---- resolve the speculative symbols ------------------------------------------------------------------------------------------
// Chunk k turns the 32 KiB before it (window k) into the 32 KiB after it (window k + 1): entry j of that map is a byte, or
// "entry w of window k".  Such maps compose associatively, so the windows of all chunks come out of a parallel prefix over
// the chunks (log2(chunks) rounds of pointer doubling, every round all chunks at once) instead of a walk chunk by chunk.
// map[k][j], 16 bits each; after the last round map[k] IS window k + 1 (a marker left over would refer to bytes before the
// stream: corrupt).
__global__ void __launch_bounds__(256)
win_init_kernel(const uint16_t *__restrict__ spec, const uint64_t *__restrict__ spec_off, const uint64_t *__restrict__ len,
                uint16_t *__restrict__ map) {
  const uint32_t k = blockIdx.y;
  const uint64_t n = len[k];
  const uint16_t *s = spec + spec_off[k];
  uint16_t *m = map + (size_t)k * 32768;
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < 32768; j += gridDim.x * blockDim.x)
    m[j] = n >= 32768 ? s[n - 32768 + j] : (j < 32768 - n ? (uint16_t)(0x8000u | (j + (uint32_t)n)) : s[j - (32768 - (uint32_t)n)]);
}
__global__ void __launch_bounds__(256)
win_round_kernel(const uint16_t *__restrict__ in, uint16_t *__restrict__ out, uint32_t stride) {
  const uint32_t k = blockIdx.y;
  const uint16_t *m = in + (size_t)k * 32768;
  const uint16_t *prev = k >= stride ? in + (size_t)(k - stride) * 32768 : nullptr;
  uint16_t *o = out + (size_t)k * 32768;
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < 32768; j += gridDim.x * blockDim.x) {
    uint16_t v = m[j];
    if ((v & 0x8000u) && prev) v = prev[v & 0x7FFFu];
    o[j] = v;
  }
}

// every symbol of every chunk to its byte (blockIdx.y = chunk); window k = map[k - 1]
__global__ void __launch_bounds__(256)
resolve_kernel(const uint16_t *__restrict__ spec, const uint64_t *__restrict__ spec_off, const uint64_t *__restrict__ out_off,
               const uint64_t *__restrict__ len, const uint16_t *__restrict__ map, uint8_t *__restrict__ dst, uint32_t *__restrict__ bad) {
  const uint32_t k = blockIdx.y;
  const uint64_t n = len[k];
  const uint16_t *s = spec + spec_off[k];
  const uint16_t *W = k ? map + (size_t)(k - 1) * 32768 : nullptr;
  uint8_t *o = dst + out_off[k];
  for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t v = s[e];
    if (v & 0x8000u) {
      v = W ? W[v & 0x7FFFu] : 0x8000u;
      if (v & 0x8000u) { *bad = 1; v = 0; }   // a reference to bytes before the stream
    }
    o[e] = (uint8_t)v;
  }
}

unsigned long long g_attr_devs = 0;  // bit d: attributes set on device d (function attributes are per device)

}  // namespace

int inflate_launch(zipc_b200_ctx *ctx, const InflateTask *d_tasks, uint32_t n, InflateResult *d_results,
                   bool count_only, int adler_mode, unsigned int *d_group_count, uint32_t *group_flag, const uint32_t *d_upflag,
                   uint32_t upload_serial) {
  if (n == 0) return ZIPC_OK;
  if (!(g_attr_devs >> (ctx->device & 63) & 1ull)) {
    ZB_CUDA(ctx, cudaFuncSetAttribute(inflate_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    ZB_CUDA(ctx, cudaFuncSetAttribute(inflate_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    ZB_CUDA(ctx, cudaFuncSetAttribute(inflate_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    ZB_CUDA(ctx, cudaFuncSetAttribute(find_starts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    g_attr_devs |= 1ull << (ctx->device & 63);
  }
  // one warp per stream.  A small batch takes only as many CTAs as it fills with streams (32 per CTA), so that the kernels of
  // other groups of a pipelined batch -- other streams of the same device -- find free SMs next to it
  uint32_t grid = (uint32_t)ctx->sm_count;
  if (n < 8u * grid) { if (grid > n) grid = n; }                        // few streams: spread them, a stream alone on an SM runs faster
  else if (grid > (n + WARPS - 1) / WARPS) grid = (n + WARPS - 1) / WARPS;
  size_t sym_bytes = (size_t)(grid * WARPS + grid) * SYMS_PER_SLOT * sizeof(uint16_t);
  if (int st = ctx->d_scratch.reserve(sym_bytes + 256 + 4096)) return st;
  unsigned int *queue = reinterpret_cast<unsigned int *>(ctx->d_scratch.as<uint8_t>() + sym_bytes);
  {
    unsigned int start = grid * WARPS;  // tasks [0, start) are assigned statically
    ZB_CUDA(ctx, cudaMemcpyAsync(queue, &start, sizeof start, cudaMemcpyHostToDevice, ctx->stream));
  }
  KernelTimer kt(ctx);
  if (count_only)
    inflate_kernel<true, false><<<grid, THREADS, kSmemBytes, ctx->stream>>>(d_tasks, n, d_results, queue, ctx->d_scratch.as<uint16_t>(), -1, nullptr, nullptr, nullptr, 0, nullptr);
  else
    inflate_kernel<false, false><<<grid, THREADS, kSmemBytes, ctx->stream>>>(d_tasks, n, d_results, queue, ctx->d_scratch.as<uint16_t>(), adler_mode,
                                                                            d_group_count, group_flag, d_upflag, upload_serial, nullptr);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  return ZIPC_OK;
}

int inflate_find_starts(zipc_b200_ctx *ctx, const uint8_t *d_src, uint64_t src_len, uint64_t first_bit, uint64_t chunk_bytes,
                        uint32_t nchunks, uint64_t *d_found) {
  if (!(g_attr_devs >> (ctx->device & 63) & 1ull)) {
    ZB_CUDA(ctx, cudaFuncSetAttribute(inflate_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    ZB_CUDA(ctx, cudaFuncSetAttribute(inflate_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    ZB_CUDA(ctx, cudaFuncSetAttribute(inflate_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    ZB_CUDA(ctx, cudaFuncSetAttribute(find_starts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    g_attr_devs |= 1ull << (ctx->device & 63);
  }
  uint32_t grid = (nchunks * kFindSplit + WARPS - 1) / WARPS;
  if (grid > (uint32_t)ctx->sm_count) grid = (uint32_t)ctx->sm_count;
  if (grid == 0) grid = 1;
  size_t sym_bytes = (size_t)(grid * WARPS + grid) * SYMS_PER_SLOT * sizeof(uint16_t);
  if (int st = ctx->d_scratch.reserve(sym_bytes + 256 + 4096)) return st;
  ZB_CUDA(ctx, cudaMemsetAsync(d_found, 0xFF, (size_t)nchunks * sizeof(uint64_t), ctx->stream));
  find_starts_kernel<<<grid, THREADS, kSmemBytes, ctx->stream>>>(d_src, src_len, first_bit, chunk_bytes, nchunks, d_found, ctx->d_scratch.as<uint16_t>());
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  return ZIPC_OK;
}

int inflate_launch_spec(zipc_b200_ctx *ctx, const InflateTask *d_tasks, uint32_t n, InflateResult *d_results, uint64_t *d_block_lists) {
  if (n == 0) return ZIPC_OK;
  // Spread the chunks: a chunk is one block of the stream on one warp, and the call waits for the slowest of them -- a warp with
  // few neighbours on its SM decodes nearly twice as fast as one of 32 (35 against 16-20 MB/s).  About four chunks per CTA, over
  // this context's share of the SMs (all of them, or 1 / lanes when several large streams are decoded at a time).
  const uint32_t sms = ctx->sm_share ? ctx->sm_share : (uint32_t)ctx->sm_count;
  uint32_t grid = std::max(1u, (n + ZB_INFLATE_SPEC_PER_CTA - 1) / ZB_INFLATE_SPEC_PER_CTA);
  if (grid > sms) grid = sms;
  size_t sym_bytes = (size_t)(grid * WARPS + grid) * SYMS_PER_SLOT * sizeof(uint16_t);
  if (int st = ctx->d_scratch.reserve(sym_bytes + 256 + 4096)) return st;
  unsigned int *queue = reinterpret_cast<unsigned int *>(ctx->d_scratch.as<uint8_t>() + sym_bytes);
  unsigned int start = grid * WARPS;  // tasks [0, start) are assigned statically
  ZB_CUDA(ctx, cudaMemcpyAsync(queue, &start, sizeof start, cudaMemcpyHostToDevice, ctx->stream));
  KernelTimer kt(ctx);
  inflate_kernel<false, true><<<grid, THREADS, kSmemBytes, ctx->stream>>>(d_tasks, n, d_results, queue, ctx->d_scratch.as<uint16_t>(), -1, nullptr, nullptr, nullptr, 0, d_block_lists);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  return ZIPC_OK;
}

int inflate_resolve(zipc_b200_ctx *ctx, const uint16_t *d_spec, const uint64_t *d_spec_off, const uint64_t *d_out_off,
                    const uint64_t *d_len, uint32_t nchunks, uint8_t *d_windows, uint8_t *d_dst, uint32_t *d_bad) {
  if (!nchunks) return ZIPC_OK;
  // d_windows: two map arrays of nchunks * 32768 16-bit entries (ping-pong of the doubling rounds)
  uint16_t *a = reinterpret_cast<uint16_t *>(d_windows), *b = a + (size_t)nchunks * 32768;
  const dim3 wgrid(8, nchunks);
  win_init_kernel<<<wgrid, 256, 0, ctx->stream>>>(d_spec, d_spec_off, d_len, a);
  ctx->launches++;
  for (uint32_t stride = 1; stride < nchunks; stride <<= 1) {
    win_round_kernel<<<wgrid, 256, 0, ctx->stream>>>(a, b, stride);
    ctx->launches++;
    std::swap(a, b);
  }
  dim3 grid((unsigned)std::max(1, ctx->sm_count * 8 / (int)std::min<uint32_t>(nchunks, 64u)), nchunks);
  resolve_kernel<<<grid, 256, 0, ctx->stream>>>(d_spec, d_spec_off, d_out_off, d_len, a, d_dst, d_bad);
  ctx->launches++;
  ZB_CUDA(ctx, cudaGetLastError());
  return ZIPC_OK;
}

}  // namespace zb
