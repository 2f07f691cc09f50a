// deflate_model.cc -- host-side model of the GPU encoder's algorithm (TEST SCAFFOLDING, not product).
// It drives the same __host__ __device__ building blocks (zipc_b200/csrc/deflate_core.h) serially, so
// its output must equal the kernel's byte for byte; tests use it to localise kernel bugs and to measure
// the compression ratio of the algorithm without a GPU.   Build: tools/build_model.sh
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../zipc_b200/csrc/deflate_core.h"

using namespace zb::dfl;

namespace {
struct Ring {
  std::vector<uint32_t> w;
  Ring() : w(kRing / 4, 0) {}
  uint32_t word(uint32_t a) const { return w[a]; }
  uint32_t byte(uint32_t i) const { return reinterpret_cast<const uint8_t *>(w.data())[i]; }
  void put(uint32_t pos, uint8_t b) {
    uint32_t i = pos & (kRing - 1);
    reinterpret_cast<uint8_t *>(w.data())[i] = b;
  }
};
struct Prev {
  std::vector<uint16_t> l;
  Prev() : l(kWindow, 0) {}
  uint32_t link(uint32_t pos) const { return l[pos & (kWindow - 1)]; }
};

struct Block {
  std::vector<uint32_t> toks;
  uint32_t fl[kNumLit], fd[kNumDist];
  uint64_t src_start = 0, src_len = 0;
  void reset(uint64_t start) { toks.clear(); memset(fl, 0, sizeof fl); memset(fd, 0, sizeof fd); src_start = start; src_len = 0; }
};

void lengths_for(const uint32_t *freq, int nsym, int max_bits, uint8_t *len) {
  std::vector<uint32_t> keys, scratch;
  for (int s = 0; s < nsym; s++) if (freq[s]) keys.push_back((freq[s] << 9) | (uint32_t)s);
  std::sort(keys.begin(), keys.end());
  scratch.resize(keys.size() + 1);
  huff_lengths_from_sorted(keys.data(), (int)keys.size(), nsym, max_bits, len, scratch.data());
}

void finalize_block(Block &b, const uint8_t *src, bool final, BitSink &out) {
  b.fl[256] += 1;
  uint8_t ll[kNumLit + kNumDist + 2], cl[kNumClen];
  lengths_for(b.fl, kNumLit, 15, ll);
  int hlit = kNumLit;
  while (hlit > 257 && ll[hlit - 1] == 0) hlit--;
  uint8_t dl[kNumDist];
  lengths_for(b.fd, kNumDist, 15, dl);
  int hdist = kNumDist;
  while (hdist > 1 && dl[hdist - 1] == 0) hdist--;
  uint8_t both[kNumLit + kNumDist];
  for (int i = 0; i < hlit; i++) both[i] = ll[i];
  for (int i = 0; i < hdist; i++) both[hlit + i] = dl[i];
  uint16_t rsyms[kNumLit + kNumDist];
  uint32_t cfreq[kNumClen];
  int nr = rle_code_lengths(both, hlit + hdist, rsyms, cfreq);
  lengths_for(cfreq, kNumClen, 7, cl);
  static const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
  int hclen = 19;
  while (hclen > 4 && cl[order[hclen - 1]] == 0) hclen--;
  // exact costs (reference :1045-1079)
  uint64_t sym_dyn = 0, sym_fix = 0;
  for (int s = 0; s < kNumLit; s++) {
    uint32_t eb = s >= 257 ? len_extra_bits_of_sym((uint32_t)s) : 0;
    sym_dyn += (uint64_t)b.fl[s] * (ll[s] + eb);
    sym_fix += (uint64_t)b.fl[s] * (fixed_lit_len((uint32_t)s) + eb);
  }
  for (int s = 0; s < kNumDist; s++) {
    uint32_t eb = dist_extra_bits_of_sym((uint32_t)s);
    sym_dyn += (uint64_t)b.fd[s] * (dl[s] + eb);
    sym_fix += (uint64_t)b.fd[s] * (5 + eb);
  }
  uint64_t hdr_dyn = 3 + 5 + 5 + 4 + 3 * (uint64_t)hclen;
  for (int s = 0; s < kNumClen; s++) hdr_dyn += (uint64_t)cfreq[s] * (cl[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0));
  uint64_t dlen = hdr_dyn + sym_dyn, flen = 3 + sym_fix;
  uint64_t nlen = 3 + ((8 - ((out.bits() + 3) & 7)) & 7) + 32 + 8 * b.src_len;
  uint32_t lcode[kNumLit], dcode[kNumDist], ccode[kNumClen];
  if (nlen <= dlen && nlen <= flen) {
    out.put(final ? 1 : 0, 3);
    out.put(0, (8 - (out.bits() & 7)) & 7);
    out.put((uint32_t)b.src_len, 16);
    out.put((uint32_t)(~b.src_len) & 0xFFFF, 16);
    for (uint64_t i = 0; i < b.src_len; i++) out.put(src[b.src_start + i], 8);
    return;
  }
  if (flen <= dlen) {
    uint8_t fl8[288], fd8[32];
    for (int s = 0; s < 288; s++) fl8[s] = (uint8_t)fixed_lit_len((uint32_t)s);
    for (int s = 0; s < 32; s++) fd8[s] = 5;
    uint32_t fl_code[288], fd_code[32];
    canonical_codes(fl8, 288, fl_code);
    canonical_codes(fd8, 32, fd_code);
    memcpy(lcode, fl_code, sizeof lcode);
    memcpy(dcode, fd_code, sizeof dcode);
    out.put(final ? 3 : 2, 3);
  } else {
    canonical_codes(ll, kNumLit, lcode);
    canonical_codes(dl, kNumDist, dcode);
    canonical_codes(cl, kNumClen, ccode);
    out.put(final ? 5 : 4, 3);
    out.put((uint32_t)(hlit - 257), 5);
    out.put((uint32_t)(hdist - 1), 5);
    out.put((uint32_t)(hclen - 4), 4);
    for (int i = 0; i < hclen; i++) out.put(cl[order[i]], 3);
    for (int i = 0; i < nr; i++) {
      uint32_t s = rsyms[i] & 0xFF, ex = rsyms[i] >> 8;
      out.put(ccode[s] & 0xFFFF, ccode[s] >> 16);
      if (s == 16) out.put(ex, 2);
      else if (s == 17) out.put(ex, 3);
      else if (s == 18) out.put(ex, 7);
    }
  }
  for (uint32_t t : b.toks) {
    uint32_t dist = t >> 9, len = t & 0x1FF;
    if (!dist) { out.put(lcode[len] & 0xFFFF, lcode[len] >> 16); continue; }
    uint32_t eb, ev, s = len_sym_of(len, eb, ev);
    out.put(lcode[s] & 0xFFFF, lcode[s] >> 16);
    out.put(ev, eb);
    s = dist_sym_of(dist, eb, ev);
    out.put(dcode[s] & 0xFFFF, dcode[s] >> 16);
    out.put(ev, eb);
  }
  out.put(lcode[256] & 0xFFFF, lcode[256] >> 16);
}
}  // namespace

extern "C" {
// returns 0; *out is malloc'ed.
// Order of the phases per tile t, as in the kernel (it matters: chain links of positions 32 KiB back are overwritten
// by the insertion of the next tile, so that happens after the deep walks of this one): rounds of { P0(t) parse,
// D(t) deep walks }, P1(t) final parse, I(t+1) insertion, S(t+1) shallow walks.
// One segment of a larger stream, as encode_member (deflate.cu) writes it: src[0, prime) is the input right before the
// segment (a multiple of the tile), hashed and inserted into the chains but not searched, parsed or emitted; the parse
// starts at `prime` with nothing pending and blocks count tiles from there.  A not_final segment keeps BFINAL off and ends
// with a byte-aligning empty stored block.  prime = 0, not_final = 0 is a whole member (zipc_model_deflate).
int zipc_model_deflate_ex(int level, const uint8_t *src, uint64_t n64, uint64_t prime64, int not_final, uint8_t **out_p,
                          uint64_t *out_len) {
  const uint32_t n = (uint32_t)n64, prime = (uint32_t)prime64;
  if (prime % kTile || prime > n || (prime && prime == n)) return 1;
  LevelParams lp = level_params(level);
  Ring ring;
  Prev prev;
  std::vector<uint16_t> head(1u << kHashBits, 0);
  // per tile (two generations: t and t + 1): first candidate / resume token, match length and distance
  std::vector<uint16_t> tok[2], mlen[2], mdist[2];
  for (int g = 0; g < 2; g++) { tok[g].assign(kTile, 0); mlen[g].assign(kTile + 1, 0); mdist[g].assign(kTile + 1, 0); }
  std::vector<uint8_t> obuf((size_t)n + n / 8 + 1024);
  BitSink sink{obuf.data(), 0, 0, 0};
  Block blk;
  blk.reset(prime);
  uint32_t pos = prime, kind = 0, loaded = 0;
  int tiles_in_block = 0;

  auto insert = [&](uint32_t ts, int g) {
    uint32_t te = std::min(ts + (uint32_t)kTile, n), want = std::min(n, te + (uint32_t)kTile);
    for (; loaded < want; loaded++) ring.put(loaded, src[loaded]);
    for (uint32_t p = ts; p < te; p++) {
      if (p + 4 > n) { tok[g][p - ts] = 0; continue; }
      uint32_t h = hash4(ring_load32(ring, p));
      tok[g][p - ts] = head[h];
      prev.l[p & (kWindow - 1)] = head[h];
      head[h] = (uint16_t)p;
    }
  };
  auto shallow = [&](uint32_t ts, int g, uint32_t carry_len, uint32_t carry_dist) {
    uint32_t te = std::min(ts + (uint32_t)kTile, n);
    mlen[g][0] = (uint16_t)carry_len; mdist[g][0] = (uint16_t)carry_dist;  // slot 0 holds position ts-1, slot 1+i holds ts+i
    for (uint32_t p = ts; p < te; p++) {
      uint32_t i = p - ts, l = 0, d = 0, rt = p & 0xFFFFu;
      if (p + 4 <= n && p >= prime) {
        MatchState m;
        match_begin(m, ring, p, n, tok[g][i], lp.shallow);
        while (!m.done) match_step(m, ring, prev, lp.shallow_nice);
        l = m.best >= (uint32_t)kMinMatch ? m.best : 0; d = m.best_dist; rt = match_resume_token(m);
      }
      mlen[g][1 + i] = (uint16_t)l; mdist[g][1 + i] = (uint16_t)d; tok[g][i] = (uint16_t)rt;
    }
  };

  if (n) { insert(0, 0); shallow(0, 0, 0, 0); }
  int g = 0;
  for (uint32_t ts = 0; ts < n; ts += kTile, g ^= 1) {
    const uint32_t te = std::min(ts + (uint32_t)kTile, n);
    std::vector<uint16_t> &ML = mlen[g], &MD = mdist[g], &TK = tok[g];
    if (te <= prime) {  // a priming tile: nothing is parsed or emitted
      insert(te, g ^ 1); shallow(te, g ^ 1, 0, 0);
      continue;
    }
    // D: visited positions continue their chain walk to the full depth; so do the positions a match taken there would land on
    // and their lazy look-ahead (inside this tile), up to lp.hops landings away (breadth first).  A position is deepened at
    // most once.
    std::vector<uint8_t> claimed(kTile, 0);
    // links of candidates that the insertion of tile t + 1 overwrites are not followed (the kernel inserts concurrently)
    const uint32_t te1 = std::min(te + (uint32_t)kTile, n);
    const uint32_t trim = (te < n && te1 > (uint32_t)kWindow) ? te1 - (uint32_t)kWindow : 0u;
    for (int round = 0; round < lp.rounds; round++) {
      // P0: which positions would a lazy parse over the current lengths visit?  Guessed paths, not stitched together: from
      // the start of every 64-position sub-range (nothing pending), each followed to the end of its own sub-range.  Paths
      // through the node graph merge after a few tokens, and the landings below cover the stretch before they do.  (The
      // guess does not depend on where the real parse enters the tile, so it can be made before the previous tile is done.)
      std::vector<uint32_t> todo;
      std::vector<int> hop;  // how many landings away from a visited position
      auto walk = [&](uint32_t q, uint32_t k, uint32_t end) {
        while (q < end) {
          uint32_t nk, em;
          if (q + 4 <= n && !claimed[q - ts]) { todo.push_back(q); hop.push_back(0); }
          q = lazy_next(q, k, ML[1 + q - ts], ML[q - ts], nk, em);
          k = nk;
        }
      };
      for (uint32_t r = ts; r < te; r += 64) {
        walk(r, 0, std::min(te, r + 64));
      }
      for (size_t ti = 0; ti < todo.size(); ti++) {
        const uint32_t p = todo[ti], i = p - ts;
        if (claimed[i]) continue;
        claimed[i] = 1;
        MatchState m;
        if (match_resume(m, ring, prev, p, n, ML[1 + i], MD[1 + i], TK[i], lp.depth - lp.shallow, trim)) {
          while (!m.done) { match_step(m, ring, prev, lp.nice); match_trim(m, trim); }
          if (m.best >= (uint32_t)kMinMatch) { ML[1 + i] = (uint16_t)m.best; MD[1 + i] = (uint16_t)m.best_dist; }
        }
        if (ML[1 + i] >= (uint32_t)kMinMatch && hop[ti] < lp.hops)
          for (uint32_t q = p + ML[1 + i], k = 0; k < 2; k++, q++)
            if (q < te && q + 4 <= n && !claimed[q - ts]) { todo.push_back(q); hop.push_back(hop[ti] + 1); }
      }
    }
    // P1: the final parse
    while (pos < te) {
      uint32_t nk, em;
      uint32_t ml = ML[1 + pos - ts], mp = ML[pos - ts];
      uint32_t np = lazy_next(pos, kind, ml, mp, nk, em);
      if (em == 1) { uint8_t b = src[pos]; blk.toks.push_back(tok_lit(b)); blk.fl[b]++; blk.src_len += 1; }
      else if (em == 2) { uint8_t b = src[pos - 1]; blk.toks.push_back(tok_lit(b)); blk.fl[b]++; blk.src_len += 1; }
      else if (em == 3) {
        uint32_t d = MD[pos - ts], eb, ev;
        blk.toks.push_back(tok_match(mp, d));
        blk.fl[len_sym_of(mp, eb, ev)]++; blk.fd[dist_sym_of(d, eb, ev)]++;
        blk.src_len += mp;
      }
      pos = np; kind = nk;
    }
    if (te < n) { insert(te, g ^ 1); shallow(te, g ^ 1, ML[te - ts], MD[te - ts]); }  // slot 0 carries position te-1
    tiles_in_block++;
    bool last = te == n;
    if (tiles_in_block == kTilesPerBlock || last) {
      uint64_t next_start = blk.src_start + blk.src_len;
      finalize_block(blk, src, last && !not_final, sink);
      blk.reset(next_start);
      tiles_in_block = 0;
    }
  }
  if (n == 0) finalize_block(blk, src, !not_final, sink);
  if (not_final) {  // 000, pad to the byte, LEN 0, NLEN ffff
    sink.put(0, 3);
    sink.put(0, (8 - (sink.bits() & 7)) & 7);
    sink.put(0, 16);
    sink.put(0xFFFFu, 16);
  }
  sink.flush();
  uint8_t *o = (uint8_t *)malloc(sink.pos ? sink.pos : 1);
  memcpy(o, obuf.data(), sink.pos);
  *out_p = o; *out_len = sink.pos;
  return 0;
}
int zipc_model_deflate(int level, const uint8_t *src, uint64_t n64, uint8_t **out_p, uint64_t *out_len) {
  return zipc_model_deflate_ex(level, src, n64, 0, 0, out_p, out_len);
}
// The encoder's code length builder on its own: freq[nsym] (each < 2^23) -> out[nsym], at most max_bits.
void zipc_model_huff_lengths(const uint32_t *freq, int nsym, int max_bits, uint8_t *out) { lengths_for(freq, nsym, max_bits, out); }
void zipc_model_free(void *p) { free(p); }
}
