// deflate_core.h -- the per-thread building blocks of the encoder, written __host__ __device__ so the
// same code runs in the sm_100a kernel (deflate.cu) and in the host-side model used by the tests to
// cross-check the kernel's token stream (tools/deflate_model.cc -- test scaffolding, not product).
//
// What this restates of the reference (src/zipc_deflate.ml), and what it deliberately does not:
//   * same hash (4 bytes * 0x9E3779B1, :1145-1148), same minimum match 4 / maximum 258 / window 32768
//     (:1141-1143), same one-step lazy rule (:1224-1241), same exact bit costs for the stored / fixed /
//     dynamic choice (:1045-1104) -- without the reference's never-cleared codelen_sym_freqs.
//   * different on purpose: the search is two-phase.  EVERY position gets a shallow walk of its exact hash
//     chain (1-2 candidates, all positions in parallel); a first lazy parse over those lengths tells which
//     positions a parse visits at all (about 30 % of them), and only these -- plus the positions a match taken
//     there would land on, transitively -- continue their walk to the level's full depth, which is where the
//     reference spends its chain budget too (it searches only where its serial parse lands, :1219-1241).  The
//     final parse then runs over the improved lengths.  Huffman lengths come from the in-place
//     minimum-redundancy algorithm on sorted frequencies plus a Kraft repair (the reference rebuilds with
//     halved frequency caps, :404-473), blocks are cut every 30 tiles of 2048 bytes.
//     The streams are valid RFC 1951 and round-trip through the reference's inflate; they are not
//     byte-identical to the reference's (DESIGN.md).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ZHD __host__ __device__ __forceinline__
#else
#define ZHD inline
#endif

namespace zb {
namespace dfl {

constexpr int kWindow = 32768;
constexpr int kMinMatch = 4;
constexpr int kMaxMatch = 258;
constexpr int kTile = 2048;            // positions matched / parsed per step
constexpr int kTilesPerBlock = 30;     // 61440 source bytes per deflate block (+ <= 257 of overhang, or one byte less when the
                                       // lazy parse decides the token at a block's last position only in the next tile)
constexpr int kHashBits = 14;
constexpr int kRing = 65536;           // input ring in shared memory (power of two)
constexpr int kNumLit = 286, kNumDist = 30, kNumClen = 19;

struct LevelParams {
  int shallow;      // chain steps every position gets
  int shallow_nice; // ... and the length at which that walk stops early
  int depth;        // total chain steps of a position the parse visits (the reference: max_chain 4 / 128 / 4096, :754-764)
  int nice;         // length at which the deep walk stops early
  int rounds;       // parse -> deepen rounds before the final parse
  int hops;         // the deep walks also cover the positions matches would land on, this many landings away
};
ZHD LevelParams level_params(int level) {
  LevelParams p;
  // fast, default: the whole chain budget at every position, no deep walks (the walks of ALL positions run in lock step,
  // which is what a SIMT machine is good at; measured, DESIGN.md).  best: shallow everywhere, deep where a parse goes.
  if (level <= 1) { p.shallow = 4; p.shallow_nice = 32; p.depth = 4; p.nice = 32; p.rounds = 0; p.hops = 0; }
  else if (level == 2) { p.shallow = 12; p.shallow_nice = 128; p.depth = 12; p.nice = 128; p.rounds = 0; p.hops = 0; }
  else { p.shallow = 2; p.shallow_nice = 32; p.depth = 1024; p.nice = 258; p.rounds = 2; p.hops = 2; }
#ifdef ZB_FORCE_HOPS
  p.hops = ZB_FORCE_HOPS;
#endif
#ifdef ZB_DEFAULT_DEPTH  // tuning builds of the host model: chain budget / nice length of level default
  if (level == 2) { p.shallow = p.depth = ZB_DEFAULT_DEPTH; p.shallow_nice = p.nice = ZB_DEFAULT_NICE; }
#endif
  return p;
}

ZHD uint32_t hash4(uint32_t v) { return (v * 0x9E3779B1u) >> (32 - kHashBits); }

// ---- format tables (RFC 1951 3.2.5) ------------------------------------------------------------------
ZHD uint32_t len_sym_of(uint32_t len, uint32_t &extra_bits, uint32_t &extra_val) {
  // symbol 257.. for a match length 3..258
  if (len == 258) { extra_bits = 0; extra_val = 0; return 285; }
  uint32_t l = len - 3;
  if (l < 8) { extra_bits = 0; extra_val = 0; return 257 + l; }
  uint32_t hb = 31 - (uint32_t)
#if defined(__CUDA_ARCH__)
      __clz(l);
#else
      __builtin_clz(l);
#endif
  extra_bits = hb - 2;
  uint32_t idx = (l >> extra_bits) & 3u;
  extra_val = l & ((1u << extra_bits) - 1u);
  return 257 + 4 * extra_bits + 4 + idx;
}
ZHD uint32_t dist_sym_of(uint32_t dist, uint32_t &extra_bits, uint32_t &extra_val) {
  uint32_t d = dist - 1;
  if (d < 4) { extra_bits = 0; extra_val = 0; return d; }
  uint32_t hb = 31 - (uint32_t)
#if defined(__CUDA_ARCH__)
      __clz(d);
#else
      __builtin_clz(d);
#endif
  extra_bits = hb - 1;
  extra_val = d & ((1u << extra_bits) - 1u);
  return 2 * hb + ((d >> extra_bits) & 1u);
}
ZHD uint32_t len_extra_bits_of_sym(uint32_t sym) {  // sym 257..285
  if (sym < 265 || sym == 285) return 0;
  return (sym - 261) >> 2;
}
ZHD uint32_t dist_extra_bits_of_sym(uint32_t sym) { return sym < 4 ? 0 : (sym >> 1) - 1; }
ZHD uint32_t fixed_lit_len(uint32_t sym) { return sym < 144 ? 8 : sym < 256 ? 9 : sym < 280 ? 7 : 8; }

// ---- tokens -------------------------------------------------------------------------------------------
// literal: byte value (dist field 0); match: dist << 9 | len   (the reference's packing, :766-776)
ZHD uint32_t tok_lit(uint32_t b) { return b; }
ZHD uint32_t tok_match(uint32_t len, uint32_t dist) { return (dist << 9) | len; }

// ---- match search --------------------------------------------------------------------------------------
// Ring: input bytes at (pos & 0xFFFF); prev: chain links by (pos & 0x7FFF), 16-bit positions.
template <class Ring>
ZHD uint32_t ring_load32(const Ring &ring, uint32_t pos) {
  uint32_t i = pos & (kRing - 1);
  uint32_t a = i >> 2, s = (i & 3u) * 8u;
  uint32_t lo = ring.word(a), hi = ring.word((a + 1) & (kRing / 4 - 1));
#if defined(__CUDA_ARCH__)
  return __funnelshift_r(lo, hi, s);
#else
  return s ? (lo >> s) | (hi << (32 - s)) : lo;
#endif
}

// 8 bytes at pos as two little-endian words
template <class Ring>
ZHD void ring_load64(const Ring &ring, uint32_t pos, uint32_t &w0, uint32_t &w1) {
  uint32_t i = pos & (kRing - 1);
  uint32_t a = i >> 2, s = (i & 3u) * 8u;
  uint32_t x0 = ring.word(a), x1 = ring.word((a + 1) & (kRing / 4 - 1)), x2 = ring.word((a + 2) & (kRing / 4 - 1));
#if defined(__CUDA_ARCH__)
  w0 = __funnelshift_r(x0, x1, s);
  w1 = __funnelshift_r(x1, x2, s);
#else
  w0 = s ? (x0 >> s) | (x1 << (32 - s)) : x0;
  w1 = s ? (x1 >> s) | (x2 << (32 - s)) : x1;
#endif
}

template <class Ring>
ZHD uint32_t ring_load8(const Ring &ring, uint32_t pos) {
  return ring.byte(pos & (kRing - 1));
}

// The chain walk of one position as a resumable state machine, so that a GPU lane can interleave the
// walks of its positions (a warp then waits for the slowest lane's TOTAL work, not for the slowest lane
// of every position) while the host model simply runs it to completion.
struct MatchState {
  uint32_t p, max_len, best, best_dist, last_dist, reach, c;
  uint32_t pw0, pw1;   // the 8 bytes at p
  uint32_t chk;        // the byte at p + best: a candidate can only beat `best` if it matches there
  int steps;
  bool done;
  bool more;           // the walk stopped only because its step budget ran out: it can be resumed
};

template <class Ring>
ZHD void match_begin(MatchState &m, const Ring &ring, uint32_t p, uint32_t n, uint32_t first_cand, int depth) {
  m.p = p;
  m.max_len = n - p < (uint32_t)kMaxMatch ? n - p : (uint32_t)kMaxMatch;
  m.best = kMinMatch - 1; m.best_dist = 0; m.last_dist = 0;
  m.reach = p < (uint32_t)kWindow ? p : (uint32_t)kWindow;
  m.c = first_cand;
  ring_load64(ring, p, m.pw0, m.pw1);
  m.chk = (m.pw0 >> 24) & 0xFFu;  // byte at p + 3
  m.steps = depth;
  m.done = depth <= 0;
  m.more = false;
}

// What a walk leaves behind for a later continuation, in 16 bits: the last candidate it evaluated (the chain goes on
// from that candidate's link), or the position itself when there is nothing to continue.
ZHD uint32_t match_resume_token(const MatchState &m) { return (m.more ? m.p - m.last_dist : m.p) & 0xFFFFu; }

// Continues the walk of position p from (len, dist, token) as left by an earlier walk; false if there is nothing to do.
// `trim`: chain links of candidates below this absolute position are not followed.  The deep walks of a tile run
// while the next tile is being inserted into the chains, which overwrites the links of the positions 32 KiB
// before it; stopping there keeps every walk independent of that timing (the candidates themselves are still
// compared: the input ring holds them).
template <class Ring, class Prev>
ZHD bool match_resume(MatchState &m, const Ring &ring, const Prev &prev, uint32_t p, uint32_t n, uint32_t len, uint32_t dist,
                      uint32_t token, int steps, uint32_t trim) {
  const uint32_t last = (p - token) & 0xFFFFu;
  if (last == 0 || steps <= 0 || p - last < trim) return false;
  m.p = p;
  m.max_len = n - p < (uint32_t)kMaxMatch ? n - p : (uint32_t)kMaxMatch;
  m.best = len >= (uint32_t)kMinMatch ? len : kMinMatch - 1;
  m.best_dist = len >= (uint32_t)kMinMatch ? dist : 0;
  if (m.best >= m.max_len) return false;
  m.last_dist = last;
  m.reach = p < (uint32_t)kWindow ? p : (uint32_t)kWindow;
  m.c = prev.link(p - last);
  ring_load64(ring, p, m.pw0, m.pw1);
  m.chk = ring_load8(ring, p + m.best);
  m.steps = steps;
  m.done = false;
  m.more = false;
  return true;
}

// Length of the match between position p (whose first 8 bytes are pw0, pw1) and the candidate position cp, at most max_len.
template <class Ring>
ZHD uint32_t match_compare(const Ring &ring, uint32_t p, uint32_t cp, uint32_t pw0, uint32_t pw1, uint32_t max_len) {
  uint32_t len;
  // candidates of one chain nearly always share the first 4 bytes (same hash), so both words are fetched at
  // once: 3 aligned loads for 8 bytes instead of 2 + 2
  uint32_t w0, w1;
  ring_load64(ring, cp, w0, w1);
  uint32_t x = w0 ^ pw0;
  if (x) len = (uint32_t)
#if defined(__CUDA_ARCH__)
      (__ffs((int)x) - 1) >> 3;
#else
      __builtin_ctz(x) >> 3;
#endif
  else {
    x = w1 ^ pw1;
    if (x) len = 4 + ((uint32_t)
#if defined(__CUDA_ARCH__)
        (__ffs((int)x) - 1) >> 3);
#else
        __builtin_ctz(x) >> 3);
#endif
    else {
      len = 8;
      while (len < max_len) {
        x = ring_load32(ring, cp + len) ^ ring_load32(ring, p + len);
        if (x) {
#if defined(__CUDA_ARCH__)
          len += (uint32_t)(__ffs((int)x) - 1) >> 3;
#else
          len += (uint32_t)__builtin_ctz(x) >> 3;
#endif
          break;
        }
        len += 4;
      }
    }
  }
  return len > max_len ? max_len : len;
}

// Evaluates one candidate of the chain.
template <class Ring, class Prev>
ZHD void match_step(MatchState &m, const Ring &ring, const Prev &prev, int nice) {
  uint32_t dist = (m.p - m.c) & 0xFFFFu;
  if (dist == 0 || dist > m.reach || dist <= m.last_dist) { m.done = true; return; }  // empty / out of window / stale
  m.last_dist = dist;
  uint32_t cp = m.p - dist;
  if (m.best < m.max_len && ring_load8(ring, cp + m.best) == m.chk) {
    const uint32_t len = match_compare(ring, m.p, cp, m.pw0, m.pw1, m.max_len);
    if (len > m.best) {
      m.best = len; m.best_dist = dist;
      if (len >= (uint32_t)nice || len == m.max_len) { m.done = true; return; }
      m.chk = ring_load8(ring, m.p + len);
    }
  }
  m.c = prev.link(cp);
  if (--m.steps <= 0) { m.done = true; m.more = true; }
}

// after a step of a deep walk: do not follow the link of a candidate below `trim` (see match_resume)
ZHD void match_trim(MatchState &m, uint32_t trim) {
  if (!m.done && m.p - m.last_dist < trim) { m.done = true; m.more = false; }
}

// Longest match for absolute position p (p + 4 <= n).  Returns len (0 if < 4) and sets dist.
// first_cand is the chain head as it was just before p was inserted.
template <class Ring, class Prev>
ZHD uint32_t find_match(const Ring &ring, const Prev &prev, uint32_t p, uint32_t n, uint32_t first_cand,
                        int depth, int nice, uint32_t &dist_out) {
  MatchState m;
  match_begin(m, ring, p, n, first_cand, depth);
  while (!m.done) match_step(m, ring, prev, nice);
  dist_out = m.best_dist;
  return m.best >= (uint32_t)kMinMatch ? m.best : 0;
}

// ---- lazy parse as a successor function ------------------------------------------------------------------
// Node (p, kind): kind 0 = "at p, nothing pending", kind 1 = "at p, match of p-1 pending".
// mlen_p = match length found at p (0 when p is beyond the last searchable position),
// mlen_prev = match length found at p-1 (only read for kind 1).  Returns the next node's position and
// kind; *emit is 0 (nothing), 1 (literal at p), 2 (literal at p-1), 3 (match at p-1).
ZHD uint32_t lazy_next(uint32_t p, uint32_t kind, uint32_t mlen_p, uint32_t mlen_prev, uint32_t &next_kind,
                       uint32_t &emit) {
  if (kind == 0) {
    if (mlen_p >= (uint32_t)kMinMatch) { next_kind = 1; emit = 0; return p + 1; }
    next_kind = 0; emit = 1; return p + 1;
  }
  if (mlen_p > mlen_prev) { next_kind = 1; emit = 2; return p + 1; }
  next_kind = 0; emit = 3; return p - 1 + mlen_prev;
}

// ---- Huffman code lengths -----------------------------------------------------------------------------
// In-place minimum redundancy lengths (Moffat & Katajainen) for m >= 2 frequencies sorted ascending in A.
// On return A[i] is the code length of the i-th least frequent symbol.
ZHD void min_redundancy_lengths(uint32_t *A, int m) {
  A[0] += A[1];
  int root = 0, leaf = 2, next;
  for (next = 1; next < m - 1; next++) {
    if (leaf >= m || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = (uint32_t)next; }
    else A[next] = A[leaf++];
    if (leaf >= m || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = (uint32_t)next; }
    else A[next] += A[leaf++];
  }
  A[m - 2] = 0;
  for (next = m - 3; next >= 0; next--) A[next] = A[A[next]] + 1;
  int avbl = 1, used = 0, dpth = 0;
  root = m - 2; next = m - 1;
  while (avbl > 0) {
    while (root >= 0 && (int)A[root] == dpth) { used++; root--; }
    while (avbl > used) { A[next--] = (uint32_t)dpth; avbl--; }
    avbl = 2 * used; dpth++; used = 0;
  }
}

// keys: (freq << 9 | sym) for the used symbols, sorted ascending, m of them.  Writes len[sym] for all
// nsym symbols (0 for unused), limited to max_bits.  scratch: m words.
ZHD void huff_lengths_from_sorted(const uint32_t *keys, int m, int nsym, int max_bits, uint8_t *len,
                                  uint32_t *scratch) {
  for (int s = 0; s < nsym; s++) len[s] = 0;
  if (m == 0) return;
  if (m == 1) { len[keys[0] & 0x1FFu] = 1; return; }
  for (int i = 0; i < m; i++) scratch[i] = keys[i] >> 9;
  min_redundancy_lengths(scratch, m);
  // Limit to max_bits keeping the code COMPLETE (the reference's decoder rejects incomplete codes,
  // :377-378): clamp, lengthen the least frequent codes until the Kraft sum fits, then hand the slack
  // back by shortening codes, most frequent first (increments are powers of two, so this lands on 1).
  uint32_t kraft = 0, one = 1u << max_bits;
  for (int i = 0; i < m; i++) {
    if ((int)scratch[i] > max_bits) scratch[i] = (uint32_t)max_bits;
    kraft += one >> scratch[i];
  }
  for (int i = 0; kraft > one && i < m; i++)
    while ((int)scratch[i] < max_bits && kraft > one) { scratch[i]++; kraft -= one >> scratch[i]; }
  for (int i = m - 1; kraft < one && i >= 0; i--)
    while (scratch[i] > 1 && kraft + (one >> scratch[i]) <= one) { kraft += one >> scratch[i]; scratch[i]--; }
  if (kraft != one) {  // cannot happen for deflate-sized alphabets; keep a complete code regardless
    int L = 1;
    while ((1 << L) < m) L++;
    int shorter = (1 << L) - m;  // this many codes of length L-1, the rest of length L
    for (int i = 0; i < m; i++) scratch[i] = (uint32_t)(i >= m - shorter ? L - 1 : L);
  }
  for (int i = 0; i < m; i++) len[keys[i] & 0x1FFu] = (uint8_t)scratch[i];
}

// canonical codes (RFC 1951 3.2.2), stored bit-reversed, packed code | len << 16
ZHD void canonical_codes(const uint8_t *len, int nsym, uint32_t *code) {
  uint32_t count[16], next[16];
  for (int i = 0; i < 16; i++) count[i] = 0;
  for (int s = 0; s < nsym; s++) count[len[s]]++;
  count[0] = 0;
  uint32_t c = 0;
  next[0] = 0;
  for (int l = 1; l < 16; l++) { c = (c + count[l - 1]) << 1; next[l] = c; }
  for (int s = 0; s < nsym; s++) {
    uint32_t l = len[s];
    if (!l) { code[s] = 0; continue; }
    uint32_t v = next[l]++, r = 0;
    for (uint32_t b = 0; b < l; b++) r |= ((v >> b) & 1u) << (l - 1 - b);
    code[s] = r | (l << 16);
  }
}

// ---- serial bit writer into a byte buffer (block headers) ----------------------------------------------------
struct BitSink {
  uint8_t *out;
  uint64_t acc;
  uint32_t nacc;
  uint32_t pos;  // bytes written
  ZHD void put(uint32_t v, uint32_t n) {
    acc |= (uint64_t)v << nacc;
    nacc += n;
    while (nacc >= 8) { out[pos++] = (uint8_t)acc; acc >>= 8; nacc -= 8; }
  }
  ZHD uint32_t bits() const { return pos * 8 + nacc; }
  ZHD void flush() { if (nacc) { out[pos++] = (uint8_t)acc; acc = 0; nacc = 0; } }
};

// Run-length encodes the hlit + hdist code lengths into code-length symbols (RFC 1951 3.2.7).
// syms[k] = sym | extra << 8.  Returns the count; freq[19] receives the symbol frequencies.
ZHD int rle_code_lengths(const uint8_t *lens, int n, uint16_t *syms, uint32_t *freq) {
  for (int i = 0; i < kNumClen; i++) freq[i] = 0;
  int k = 0, i = 0;
  while (i < n) {
    uint8_t v = lens[i];
    int run = 1;
    while (i + run < n && lens[i + run] == v) run++;
    if (v == 0) {
      int r = run;
      while (r >= 11) { int t = r > 138 ? 138 : r; syms[k++] = (uint16_t)(18 | ((t - 11) << 8)); freq[18]++; r -= t; }
      if (r >= 3) { syms[k++] = (uint16_t)(17 | ((r - 3) << 8)); freq[17]++; r = 0; }
      while (r-- > 0) { syms[k++] = 0; freq[0]++; }
    } else {
      syms[k++] = v; freq[v]++;
      int r = run - 1;
      while (r >= 3) { int t = r > 6 ? 6 : r; syms[k++] = (uint16_t)(16 | ((t - 3) << 8)); freq[16]++; r -= t; }
      while (r-- > 0) { syms[k++] = v; freq[v]++; }
    }
    i += run;
  }
  return k;
}

}  // namespace dfl
}  // namespace zb
