"""An independent reader of the encoder's deflate streams: it decodes a raw RFC 1951 stream block by block and checks every
choice the encoder documents (deflate_core.h header comment, finalize_block / encode_member in deflate.cu) against a plain
Python restatement.  It shares no code with the encoder, its host model or the oracle.

What the encoder promises, and what is checked here:
  * the stream decodes to the input;
  * segments: a segment of a larger stream ends with a non-final empty stored block (000, zero pad, 0000 ffff), which the
    encoder writes nowhere else; BFINAL only on the last block of the last segment; the pad bits of the last byte are zero;
  * blocks: counted from the first byte a segment emits, block k holds exactly the tokens that start in
    [61440 k, 61440 (k + 1)) -- a match may hang over the end by at most 257 bytes; only the last block is shorter.  One
    exception, from the lazy parse: a token at the last position of a block's last tile that is only decided at the next
    tile's first position (a literal or a match pending there) opens the next block, which then starts one byte early;
  * tokens: matches of 4 to 258 bytes, distances of at most 32768 that never reach before the segment start minus its prime;
  * stored blocks: LEN is the block's source length, NLEN its complement, zero pad bits;
  * dynamic headers: HLIT / HDIST trimmed to the last used symbol (at least 257 / 1), the shortest HCLEN (at least 4), a
    nonzero length exactly for the used symbols, code lengths run-length coded by the greedy rule of rle_code_lengths;
  * code lengths: exactly what the documented builder gives on the block's own token frequencies (the minimum-redundancy
    lengths of Moffat and Katajainen on (freq, sym) sorted ascending, clamped to the limit, the least frequent codes
    lengthened until the Kraft sum fits, then the most frequent shortened first), limits 15 / 15 / 7; and, independently of
    that builder: complete codes, the Huffman optimum whenever a Huffman code fits the limit, never below the optimum
    length-limited code (package-merge);
  * block type: the cheapest of the exact stored / fixed / dynamic costs, ties going to stored, then fixed.  A stored block
    does not carry its tokens; its alternatives are costed when the tokens are forced (no 4-byte string of the block occurs
    earlier within reach, so the encoder can only have had literals).

check() raises CheckError (with the rule's name in .rule) on the first violation and otherwise returns a Report: one
BlockReport per block with its type, source range, tokens, the three costs, the depth of the unconstrained code per
alphabet and how far the header's lengths are above the optimum length-limited code."""
from __future__ import annotations

import heapq
from dataclasses import dataclass, field

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CLEN_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
CLEN_EXTRA = [0] * 16 + [2, 3, 7]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
NUM_LIT, NUM_DIST, NUM_CLEN = 286, 30, 19
LIMITS = {"lit": 15, "dist": 15, "clen": 7}
BLOCK_SRC = 61440          # 30 tiles of 2048 bytes
MAX_OVERHANG = 257
WINDOW = 32768

STORED, FIXED, DYNAMIC = "stored", "fixed", "dynamic"


class CheckError(AssertionError):
    def __init__(self, rule, message):
        super().__init__(f"[{rule}] {message}")
        self.rule = rule


def _fail(rule, message):
    raise CheckError(rule, message)


# ---- code lengths: the documented builder, and the references it is held to ---------------------------------------------
def encoder_lengths(freq, limit):
    """The encoder's documented builder, restated: minimum-redundancy lengths on (freq, sym) sorted ascending, clamp to
    `limit`, lengthen the least frequent codes until the Kraft sum fits, shorten the most frequent first while it stays <= 1.
    One used symbol gets one code of length 1."""
    lens = [0] * len(freq)
    keys = sorted((f, s) for s, f in enumerate(freq) if f)
    m = len(keys)
    if m == 0:
        return lens
    if m == 1:
        lens[keys[0][1]] = 1
        return lens
    depth = _two_queue_depths([f for f, _ in keys])
    one = 1 << limit
    depth = [min(d, limit) for d in depth]
    kraft = sum(one >> d for d in depth)
    for i in range(m):
        while kraft > one and depth[i] < limit:
            depth[i] += 1
            kraft -= one >> depth[i]
    for i in range(m - 1, -1, -1):
        while kraft < one and depth[i] > 1 and kraft + (one >> depth[i]) <= one:
            kraft += one >> depth[i]
            depth[i] -= 1
    if kraft != one:
        L = (m - 1).bit_length()
        shorter = (1 << L) - m
        depth = [L - 1 if i >= m - shorter else L for i in range(m)]
    for (_, s), d in zip(keys, depth):
        lens[s] = d
    return lens


def _two_queue_depths(w):
    """Huffman code lengths for weights w (sorted ascending, >= 2 of them) by the two-queue method: the two lightest of the
    next leaf and the next internal node are merged, a tie going to the leaf.  Leaf depths are handed out shallowest first to
    the heaviest leaves (which is what the in-place algorithm of Moffat and Katajainen computes)."""
    m = len(w)
    nodes = []         # internal nodes in creation order: weight, parent index, leaf children
    leaf = root = 0
    for _ in range(m - 1):
        kids = []
        weight = 0
        for _ in range(2):
            if leaf < m and (root >= len(nodes) or not nodes[root][0] < w[leaf]):
                weight += w[leaf]
                leaf += 1
                kids.append(None)
            else:
                weight += nodes[root][0]
                kids.append(root)
                root += 1
        idx = len(nodes)
        nodes.append([weight, None, sum(k is None for k in kids)])
        for k in kids:
            if k is not None:
                nodes[k][1] = idx
    depth = [0] * len(nodes)
    count = {}
    for i in range(len(nodes) - 1, -1, -1):
        if nodes[i][1] is not None:
            depth[i] = depth[nodes[i][1]] + 1
        if nodes[i][2]:
            count[depth[i] + 1] = count.get(depth[i] + 1, 0) + nodes[i][2]
    out = []
    for d in sorted(count):
        out += [d] * count[d]
    return out[::-1]   # ascending weight -> deepest first


def huffman_cost_depth(freq):
    """(cost, depth) of an optimal unconstrained code (heapq; ties merge the shallower subtree first, which gives the
    smallest depth any optimal code has)"""
    h = [(f, 0, i) for i, f in enumerate(f for f in freq if f)]
    if len(h) <= 1:
        return sum(f for f, _, _ in h), len(h)
    heapq.heapify(h)
    cost, k = 0, len(h)
    while len(h) > 1:
        a, b = heapq.heappop(h), heapq.heappop(h)
        cost += a[0] + b[0]
        heapq.heappush(h, (a[0] + b[0], max(a[1], b[1]) + 1, k))
        k += 1
    return cost, h[0][1]


def package_merge_cost(freq, limit):
    """cost of the optimal code with no length above `limit` (package-merge; the cost is the weight of the first 2n - 2
    items of the last list)"""
    leaves = sorted(f for f in freq if f)
    n = len(leaves)
    if n <= 1:
        return sum(leaves)
    assert n <= (1 << limit)
    cur = leaves
    for _ in range(limit - 1):
        cur = sorted(leaves + [cur[i] + cur[i + 1] for i in range(0, len(cur) - 1, 2)])
    return sum(cur[:2 * n - 2])


def kraft_ok(lens):
    """complete (Kraft sum 1), or the lone code of length 1, or no code at all"""
    used = [l for l in lens if l]
    if len(used) <= 1:
        return used in ([], [1])
    return sum(1 << (15 - l) for l in used) == 1 << 15


def greedy_rle(lens):
    """rle_code_lengths' rule: a run of zeros takes 18 (11-138) while it can, then 17 (3-10), then single zeros; a run of a
    length takes the length once, then 16 (3-6 repeats) while it can, then single lengths.  [(sym, extra)]"""
    out, i, n = [], 0, len(lens)
    while i < n:
        v, j = lens[i], i
        while j < n and lens[j] == v:
            j += 1
        r = j - i
        if v == 0:
            while r >= 11:
                t = min(r, 138)
                out.append((18, t - 11))
                r -= t
            if r >= 3:
                out.append((17, r - 3))
                r = 0
            out += [(0, 0)] * r
        else:
            out.append((v, 0))
            r -= 1
            while r >= 3:
                t = min(r, 6)
                out.append((16, t - 3))
                r -= t
            out += [(v, 0)] * r
        i = j
    return out


def _table(lens, what):
    """decoding table over the next max(lens) bits (LSB first): sym << 4 | length, -1 where no code starts"""
    maxlen = max(lens) if any(lens) else 1
    tab = [-1] * (1 << maxlen)
    counts = [0] * 16
    for l in lens:
        counts[l] += 1
    counts[0] = 0
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + counts[b - 1]) << 1
        nxt[b] = code
    for s, l in enumerate(lens):
        if l:
            c = nxt[l]
            nxt[l] += 1
            if c >> l:
                _fail("invalid", f"over-subscribed {what} code")
            r = int(format(c, f"0{l}b")[::-1], 2)
            tab[r::1 << l] = [(s << 4) | l] * (1 << (maxlen - l))
    return tab, maxlen


_FIXED_TABLES = None


def _fixed_tables():
    global _FIXED_TABLES
    if _FIXED_TABLES is None:
        _FIXED_TABLES = (_table(FIXED_LIT, "fixed literal/length"), _table([5] * 32, "fixed distance"))
    return _FIXED_TABLES


# ---- reports ------------------------------------------------------------------------------------------------------------
@dataclass
class BlockReport:
    type: str
    final: bool
    bit_start: int                 # where the block header starts in the stream
    segment: int
    index: int                     # block number inside its segment
    src_start: int                 # absolute position in the input
    src_len: int
    matches: list = field(default_factory=list)   # (source position, length, distance)
    literals: int = 0
    tokens_known: bool = True      # False for a stored block whose tokens are not forced
    freq_l: list | None = None     # token frequencies, end-of-block included
    freq_d: list | None = None
    hlit: int = 0
    hdist: int = 0
    hclen: int = 0
    lit_lengths: list | None = None
    dist_lengths: list | None = None
    clen_lengths: list | None = None   # by code-length symbol
    rle: list | None = None
    costs: dict = field(default_factory=dict)    # stored / fixed / dynamic, in bits (None when not known)
    depth: dict = field(default_factory=dict)    # lit / dist / clen: depth of the unconstrained optimal code
    gap: dict = field(default_factory=dict)      # lit / dist / clen: header cost - optimum length-limited cost, in bits
    huff_cost: dict = field(default_factory=dict)  # lit / dist / clen: cost of the unconstrained optimal code


@dataclass
class Report:
    blocks: list
    segments: list                 # (src_start, src_end, byte_start, byte_end), byte_end past the empty stored block
    bits: int

    @property
    def matches(self):
        return [m for b in self.blocks for m in b.matches]

    def of_type(self, t):
        return [b for b in self.blocks if b.type == t]


# ---- costs ----------------------------------------------------------------------------------------------------------------
def _sym_costs(freq_l, freq_d, ll, dl):
    c = 0
    for s, f in enumerate(freq_l):
        if f:
            c += f * (ll[s] + (LEN_EXTRA[s - 257] if s >= 257 else 0))
    for s, f in enumerate(freq_d):
        if f:
            c += f * (dl[s] + DIST_EXTRA[s])
    return c


def _expected_header(freq_l, freq_d):
    """the dynamic header the encoder builds for these token frequencies: (ll, dl, hlit, hdist, rle, cl, hclen, bits)"""
    ll = encoder_lengths(freq_l, 15)
    dl = encoder_lengths(freq_d, 15)
    hlit = max(257, max((s + 1 for s in range(NUM_LIT) if ll[s]), default=0))
    hdist = max(1, max((s + 1 for s in range(NUM_DIST) if dl[s]), default=0))
    rle = greedy_rle(ll[:hlit] + dl[:hdist])
    cfreq = [0] * NUM_CLEN
    for s, _ in rle:
        cfreq[s] += 1
    cl = encoder_lengths(cfreq, 7)
    hclen = max(4, max((i + 1 for i in range(NUM_CLEN) if cl[CLEN_ORDER[i]]), default=0))
    bits = 3 + 5 + 5 + 4 + 3 * hclen + sum(cl[s] + CLEN_EXTRA[s] for s, _ in rle)
    return ll, dl, hlit, hdist, rle, cl, hclen, bits


def block_costs(freq_l, freq_d, src_len, bit_start):
    """exact bits of the three block types for these tokens (end of block included in freq_l), the block starting at bit_start"""
    pad = (8 - ((bit_start + 3) & 7)) & 7
    fixed = 3 + _sym_costs(freq_l, freq_d, FIXED_LIT, [5] * NUM_DIST)
    ll, dl, *_, hbits = _expected_header(freq_l, freq_d)
    return {STORED: 3 + pad + 32 + 8 * src_len, FIXED: fixed, DYNAMIC: hbits + _sym_costs(freq_l, freq_d, ll, dl)}


def _cheapest(costs):
    return min((STORED, FIXED, DYNAMIC), key=lambda t: (costs[t], (STORED, FIXED, DYNAMIC).index(t)))


def _literal_only(data, start, end, floor, seg_end):
    """True if no 4-byte string starting in [start, end) (and ending by seg_end) occurs at an earlier position within the
    window and not before `floor`: the encoder can then only have emitted literals there"""
    last = {}
    mv = memoryview(data)
    stop = min(end, seg_end - 3)
    for q in range(max(floor, start - WINDOW), stop):
        k = bytes(mv[q:q + 4])
        if q >= start:
            p = last.get(k)
            if p is not None and q - p <= WINDOW:
                return False
        last[k] = q
    return True


# ---- the reader -------------------------------------------------------------------------------------------------------
def check(stream: bytes, data: bytes, primes=None, final: bool = True) -> Report:
    """Decodes `stream` (raw deflate) and checks it against the input `data` and the encoder's rules.  primes[k]: how many
    bytes before the start of segment k its matches may reach (default 0 for every segment).  final: the stream is a whole
    member (its last block has BFINAL); otherwise it is a non-final piece, which ends with an empty stored block."""
    stream = bytes(stream)
    data = bytes(data)
    nbits_total = 8 * len(stream)
    acc = nacc = ip = 0
    out = bytearray()
    blocks, segments = [], []
    seg = 0
    seg_src = 0          # where the current segment starts in the input
    seg_byte = 0
    seg_blocks = []      # blocks of the current segment

    def prime_of(k):
        return 0 if primes is None else (primes[k] if k < len(primes) else 0)

    floor = seg_src - prime_of(0)   # matches may not reach before this position
    saw_final = False
    while True:
        # ---- block header
        bitpos = 8 * ip - nacc
        if bitpos + 3 > nbits_total:
            _fail("segment_end" if not final else "bfinal", f"stream ends at bit {bitpos} without a final block")
        if nacc < 48:
            acc |= int.from_bytes(stream[ip:ip + 6], "little") << nacc
            ip += 6
            nacc += 48
        bfinal, btype = acc & 1, (acc >> 1) & 3
        acc >>= 3
        nacc -= 3
        blk_start = len(out)
        rel = blk_start - seg_src
        k = len(seg_blocks)
        br = BlockReport(type="", final=bool(bfinal), bit_start=bitpos, segment=seg, index=k, src_start=blk_start, src_len=0)
        if btype == 3:
            _fail("invalid", f"block type 3 at bit {bitpos}")
        if btype == 0:
            br.type = STORED
            pad = nacc & 7
            if acc & ((1 << pad) - 1):
                _fail("pad", f"nonzero pad bits in the stored block header at bit {bitpos}")
            acc >>= pad
            nacc -= pad
            # drop the look-ahead back to the byte boundary
            ip -= nacc >> 3
            acc = nacc = 0
            if ip + 4 > len(stream):
                _fail("invalid", "stream ends inside a stored block header")
            ln = stream[ip] | stream[ip + 1] << 8
            nln = stream[ip + 2] | stream[ip + 3] << 8
            if nln != (~ln) & 0xFFFF:
                _fail("stored_len", f"NLEN {nln:#x} is not the complement of LEN {ln:#x} at bit {bitpos}")
            ip += 4
            if ip + ln > len(stream):
                _fail("invalid", "stream ends inside a stored block")
            out += stream[ip:ip + ln]
            ip += ln
            br.src_len = ln
            if ln == 0 and not bfinal:
                # the end of a segment
                if any(b.type == STORED and b.src_len == 0 and not b.final for b in seg_blocks):
                    _fail("segment_end", "two empty stored blocks in one segment")
                _check_segment(seg_blocks, seg_src, blk_start)
                segments.append((seg_src, blk_start, seg_byte, ip))
                blocks += seg_blocks
                seg += 1
                seg_src, seg_byte, seg_blocks = blk_start, ip, []
                floor = seg_src - prime_of(seg)
                if not final and ip == len(stream):
                    break
                continue
            if ln == 0:
                _fail("segment_end", f"an empty final stored block at bit {bitpos}")
            br.tokens_known = False
        else:
            if btype == 1:
                br.type = FIXED
                (lt, lmax), (dt, dmax) = _fixed_tables()
            else:
                br.type = DYNAMIC
                if nacc < 48:
                    acc |= int.from_bytes(stream[ip:ip + 6], "little") << nacc
                    ip += 6
                    nacc += 48
                hlit, hdist, hclen = (acc & 31) + 257, ((acc >> 5) & 31) + 1, ((acc >> 10) & 15) + 4
                acc >>= 14
                nacc -= 14
                cl = [0] * NUM_CLEN
                for i in range(hclen):
                    if nacc < 8:
                        acc |= int.from_bytes(stream[ip:ip + 6], "little") << nacc
                        ip += 6
                        nacc += 48
                    cl[CLEN_ORDER[i]] = acc & 7
                    acc >>= 3
                    nacc -= 3
                if hlit > NUM_LIT or hdist > NUM_DIST:
                    _fail("invalid", f"HLIT {hlit} / HDIST {hdist} out of range at bit {bitpos}")
                ct, cmax = _table(cl, "code-length")
                cmask = (1 << cmax) - 1
                lens, rle = [], []
                while len(lens) < hlit + hdist:
                    if nacc < 24:
                        acc |= int.from_bytes(stream[ip:ip + 6], "little") << nacc
                        ip += 6
                        nacc += 48
                    e = ct[acc & cmask]
                    if e < 0:
                        _fail("invalid", "undecodable code-length symbol")
                    s, l = e >> 4, e & 15
                    acc >>= l
                    nacc -= l
                    ex = 0
                    if s >= 16:
                        ex = acc & ((1 << CLEN_EXTRA[s]) - 1)
                        acc >>= CLEN_EXTRA[s]
                        nacc -= CLEN_EXTRA[s]
                    rle.append((s, ex))
                    if s < 16:
                        lens.append(s)
                    elif s == 16:
                        if not lens:
                            _fail("invalid", "code-length symbol 16 with nothing to repeat")
                        lens += [lens[-1]] * (3 + ex)
                    else:
                        lens += [0] * ((3 if s == 17 else 11) + ex)
                if len(lens) > hlit + hdist:
                    _fail("invalid", "code lengths run past HLIT + HDIST")
                br.hlit, br.hdist, br.hclen, br.rle, br.clen_lengths = hlit, hdist, hclen, rle, cl
                br.lit_lengths = lens[:hlit] + [0] * (NUM_LIT - hlit)
                br.dist_lengths = lens[hlit:] + [0] * (NUM_DIST - hdist)
                if not br.lit_lengths[256]:
                    _fail("invalid", "no end-of-block code")
                lt, lmax = _table(br.lit_lengths, "literal/length")
                dt, dmax = _table(br.dist_lengths, "distance")
            # ---- tokens
            lmask, dmask = (1 << lmax) - 1, (1 << dmax) - 1
            fl, fd = [0] * NUM_LIT, [0] * NUM_DIST
            matches = br.matches
            tile_lo, tile_hi = seg_src + BLOCK_SRC * k - (k > 0), seg_src + BLOCK_SRC * (k + 1)
            nlit = 0
            while True:
                if nacc < 48:
                    acc |= int.from_bytes(stream[ip:ip + 6], "little") << nacc
                    ip += 6
                    nacc += 48
                e = lt[acc & lmask]
                if e < 0:
                    _fail("invalid", f"undecodable literal/length code near bit {8 * ip - nacc}")
                s = e >> 4
                l = e & 15
                acc >>= l
                nacc -= l
                if s < 256:
                    p = len(out)
                    if not tile_lo <= p < tile_hi:
                        _fail("boundary", f"segment {seg} block {k}: a token at {p - seg_src} outside "
                                          f"[{BLOCK_SRC * k}, {BLOCK_SRC * (k + 1)})")
                    out.append(s)
                    fl[s] += 1
                    nlit += 1
                    continue
                if s == 256:
                    fl[256] += 1
                    break
                if s > 285:
                    _fail("invalid", f"literal/length symbol {s}")
                eb = LEN_EXTRA[s - 257]
                length = LEN_BASE[s - 257] + (acc & ((1 << eb) - 1))
                acc >>= eb
                nacc -= eb
                e = dt[acc & dmask]
                if e < 0:
                    _fail("invalid", "undecodable distance code")
                ds = e >> 4
                acc >>= e & 15
                nacc -= e & 15
                if ds >= NUM_DIST:
                    _fail("invalid", f"distance symbol {ds}")
                eb = DIST_EXTRA[ds]
                dist = DIST_BASE[ds] + (acc & ((1 << eb) - 1))
                acc >>= eb
                nacc -= eb
                p = len(out)
                fl[s] += 1
                fd[ds] += 1
                if not tile_lo <= p < tile_hi:
                    _fail("boundary", f"segment {seg} block {k}: a match at {p - seg_src} outside "
                                      f"[{BLOCK_SRC * k}, {BLOCK_SRC * (k + 1)})")
                if length < 4:
                    _fail("match_length", f"a match of {length} bytes at {p}")
                if dist > WINDOW:
                    _fail("distance", f"distance {dist} at {p}")
                if dist > p - floor:
                    _fail("reach", f"distance {dist} at {p} reaches before {floor} (segment {seg} starts at {seg_src})")
                if dist >= length:
                    out += out[p - dist:p - dist + length]
                else:
                    chunk = out[p - dist:]
                    out += (chunk * (length // dist + 1))[:length]
                matches.append((p, length, dist))
            br.literals = nlit
            br.freq_l, br.freq_d = fl, fd
            br.src_len = len(out) - blk_start
        if 8 * ip - nacc > nbits_total:
            _fail("invalid", "stream ends inside a block")
        if out[blk_start:] != data[blk_start:len(out)]:
            i = next(i for i in range(blk_start, len(out)) if i >= len(data) or out[i] != data[i])
            _fail("decoded", f"decoded bytes differ from the input at {i}")
        seg_blocks.append(br)
        if bfinal:
            saw_final = True
            if not final:
                _fail("bfinal", f"BFINAL on a block of a non-final piece at bit {bitpos}")
            _check_segment(seg_blocks, seg_src, len(out))
            segments.append((seg_src, len(out), seg_byte, None))
            blocks += seg_blocks
            break
    end_bit = 8 * ip - nacc
    if saw_final:
        used = (end_bit + 7) // 8
        if used != len(stream):
            _fail("trailing", f"{len(stream) - used} bytes after the final block")
        if end_bit & 7 and stream[-1] >> (end_bit & 7):
            _fail("pad", "nonzero pad bits in the last byte")
        segments[-1] = segments[-1][:3] + (used,)
    if len(out) != len(data):
        _fail("decoded", f"{len(out)} bytes decoded, {len(data)} expected")
    seg_ends = {s[0]: s[1] for s in segments}
    for b in blocks:
        _check_block(b, data, seg_ends, prime_of)
    return Report(blocks=blocks, segments=segments, bits=end_bit)


def _check_segment(seg_blocks, seg_src, seg_end):
    """block k of a segment covers [61440 k + overhang, 61440 (k + 1) + overhang'): an overhang of at most 257 bytes, or
    -1 where the lazy parse decided the token at the tile's last position only at the next tile"""
    if not seg_blocks:
        _fail("segment_end", f"an empty segment at {seg_src}")
    for b in seg_blocks:
        lo = seg_src + BLOCK_SRC * b.index
        if not lo - (b.index > 0) <= b.src_start <= lo + MAX_OVERHANG:
            _fail("boundary", f"block {b.index} of the segment at {seg_src} starts at {b.src_start - seg_src}")
        end = b.src_start + b.src_len
        last = b is seg_blocks[-1]
        if not last and not lo + BLOCK_SRC - 1 <= end <= lo + BLOCK_SRC + MAX_OVERHANG:
            _fail("boundary", f"block {b.index} of the segment at {seg_src} ends at {end - seg_src}: only the last may be short")
        if last and end - lo > BLOCK_SRC + MAX_OVERHANG:
            _fail("boundary", f"the last block of the segment at {seg_src} holds {end - lo} bytes")
    if seg_blocks[-1].src_start + seg_blocks[-1].src_len != seg_end:
        _fail("boundary", "blocks do not cover the segment")


def _check_block(b, data, seg_ends, prime_of):
    if b.type == STORED:
        seg_start = max(s for s in seg_ends if s <= b.src_start)
        floor = seg_start - prime_of(b.segment)
        if _literal_only(data, b.src_start, b.src_start + b.src_len, floor, seg_ends[seg_start]):
            b.tokens_known = True
            fl = [0] * NUM_LIT
            for v in data[b.src_start:b.src_start + b.src_len]:
                fl[v] += 1
            fl[256] += 1
            b.freq_l, b.freq_d, b.literals = fl, [0] * NUM_DIST, b.src_len
        else:
            b.costs = {STORED: 3 + ((8 - ((b.bit_start + 3) & 7)) & 7) + 32 + 8 * b.src_len, FIXED: None, DYNAMIC: None}
            return
    fl, fd = b.freq_l, b.freq_d
    ll, dl, hlit, hdist, rle, cl, hclen, _ = _expected_header(fl, fd)
    cfreq = [0] * NUM_CLEN
    for s, _ in rle:
        cfreq[s] += 1
    for name, f in (("lit", fl), ("dist", fd), ("clen", cfreq)):
        b.huff_cost[name], b.depth[name] = huffman_cost_depth(f)
    if b.type == DYNAMIC:
        # header fields
        if b.hlit != hlit:
            _fail("hlit", f"HLIT {b.hlit}, the last used literal/length symbol gives {hlit} (block at bit {b.bit_start})")
        if b.hdist != hdist:
            _fail("hdist", f"HDIST {b.hdist}, the last used distance symbol gives {hdist} (block at bit {b.bit_start})")
        for what, f, lens in (("literal/length", fl, b.lit_lengths), ("distance", fd, b.dist_lengths)):
            bad = [s for s in range(len(f)) if bool(f[s]) != bool(lens[s])]
            if bad:
                _fail("used_lengths", f"{what} symbols {bad[:8]}: a length exactly for the used symbols (block at bit {b.bit_start})")
        if b.rle != greedy_rle(b.lit_lengths[:b.hlit] + b.dist_lengths[:b.hdist]):
            _fail("rle", f"code lengths not run-length coded by the greedy rule (block at bit {b.bit_start})")
        bcf = [0] * NUM_CLEN
        for s, _ in b.rle:
            bcf[s] += 1
        bad = [s for s in range(NUM_CLEN) if bool(bcf[s]) != bool(b.clen_lengths[s])]
        if bad:
            _fail("used_lengths", f"code-length symbols {bad}: a length exactly for the used symbols (block at bit {b.bit_start})")
        want_hclen = max(4, max((i + 1 for i in range(NUM_CLEN) if b.clen_lengths[CLEN_ORDER[i]]), default=0))
        if b.hclen != want_hclen:
            _fail("hclen", f"HCLEN {b.hclen}, the last nonzero code-length-code length gives {want_hclen}")
        # the code lengths: complete, optimal where a Huffman code fits, never below package-merge, then exactly the builder's
        for name, f, lens in (("lit", fl, b.lit_lengths), ("dist", fd, b.dist_lengths), ("clen", bcf, b.clen_lengths)):
            if not kraft_ok(lens):
                _fail("incomplete", f"{name} code is not complete (block at bit {b.bit_start})")
            if max(lens) > LIMITS[name]:
                _fail("limit", f"{name} code longer than {LIMITS[name]} bits")
            cost = sum(x * y for x, y in zip(f, lens))
            hc, hd = huffman_cost_depth(f)
            if sum(1 for x in f if x) >= 2:
                if hd <= LIMITS[name] and cost != hc:
                    _fail("suboptimal", f"{name} code costs {cost} bits, a Huffman code within the limit {hc} "
                                        f"(block at bit {b.bit_start})")
                pm = package_merge_cost(f, LIMITS[name])
                if cost < pm:
                    _fail("invalid", f"{name} code below the length-limited optimum: not a prefix code")
                b.gap[name] = cost - pm
            else:
                b.gap[name] = 0
        for name, got, want in (("literal/length", b.lit_lengths, ll), ("distance", b.dist_lengths, dl),
                                ("code-length", b.clen_lengths, cl)):
            if list(got) != list(want):
                diff = [s for s in range(len(want)) if got[s] != want[s]]
                _fail("lengths", f"{name} lengths differ from the documented builder at symbols {diff[:8]} "
                                 f"(block at bit {b.bit_start})")
    b.costs = block_costs(fl, fd, b.src_len, b.bit_start)
    want = _cheapest(b.costs)
    if b.type != want:
        _fail("block_type", f"a {b.type} block at bit {b.bit_start} where {want} is cheapest: {b.costs}")
