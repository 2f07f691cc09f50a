"""A deflate stream writer for tests (RFC 1951), and a catalogue of streams that sit on the edges of the reference decoder's
acceptance rules (oracle/zipc_oracle.c: hdec_init, inf_block_symbols, inf_dynamic_block, inf_stored_block).

The writer derives nothing and checks nothing: block headers take explicit HLIT / HDIST / HCLEN, code-length-code lengths
and code-length symbols, so that invalid streams can be written as easily as valid ones.  Bits go out LSB first, Huffman
codes MSB first (RFC 1951 3.1.1).  Alongside the bits it keeps `out`, the bytes a decoder produces up to the point where the
stream stops being valid (the whole output for a valid stream).

Plain Python, no GPU: the CPU tests decode every catalogue stream with the oracle and with Python's zlib."""
from __future__ import annotations

from dataclasses import dataclass

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CLEN_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
CLEN_EXTRA = {16: 2, 17: 3, 18: 7}
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32


def canonical(lengths):
    """RFC 1951 3.2.2: {symbol: (code, length)} for every non-zero length.  Over-subscribed lengths give codes that do not
    fit their length; they are masked, which is as good as any bits for a stream the decoder must refuse."""
    counts = [0] * 16
    for n in lengths:
        counts[n] += 1
    counts[0] = 0
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + counts[b - 1]) << 1
        nxt[b] = code
    out = {}
    for s, n in enumerate(lengths):
        if n:
            out[s] = (nxt[n] & ((1 << n) - 1), n)
            nxt[n] += 1
    return out


def complete_lengths(symbols, size):
    """lengths (a list of `size`) of a complete code over `symbols`: the shortest ones first, no two lengths more than one
    apart; a lone symbol gets one code of length 1"""
    symbols = list(symbols)
    k = len(symbols)
    lengths = [0] * size
    if k == 1:
        lengths[symbols[0]] = 1
        return lengths
    d = (k - 1).bit_length()
    short = (1 << d) - k
    for i, s in enumerate(symbols):
        lengths[s] = d - 1 if i < short else d
    return lengths


def chain_lengths(symbols, size):
    """lengths of a complete code that is a chain: symbols[0] has length 1, symbols[1] length 2, ... symbols[13] length 14,
    symbols[14] and symbols[15] length 15"""
    assert len(symbols) == 16
    lengths = [0] * size
    for i, s in enumerate(symbols):
        lengths[s] = min(i + 1, 15)
    return lengths


def plain_symbols(lengths):
    """code-length symbols that spell the lengths one by one (no 16 / 17 / 18)"""
    return [(n, 0) for n in lengths]


def rle_symbols(lengths):
    """code-length symbols as an encoder would write them: 17 / 18 for runs of zeros, 16 for runs of the previous length
    (runs cross the HLIT / HDIST boundary when the lengths are given as one list)"""
    out, i = [], 0
    while i < len(lengths):
        v, j = lengths[i], i
        while j < len(lengths) and lengths[j] == v:
            j += 1
        run = j - i
        if v == 0 and run >= 3:
            r = min(run, 138)
            out.append((18, r - 11) if r >= 11 else (17, r - 3))
            i += r
            continue
        out.append((v, 0))
        i += 1
        run -= 1
        while run >= 3:
            r = min(run, 6)
            out.append((16, r - 3))
            i += r
            run -= r
    return out


def clen_code_for(symbols):
    """(hclen, code-length-code lengths in transmission order) of a complete code over the code-length symbols used"""
    used = sorted({s for s, _ in symbols})
    by_sym = complete_lengths(used, 19)
    hclen = max(4, max(CLEN_ORDER.index(s) for s in used) + 1)
    return hclen, [by_sym[s] for s in CLEN_ORDER[:hclen]]


class Writer:
    def __init__(self):
        self.buf = bytearray()
        self.acc = 0        # bits not yet in buf (fewer than 8)
        self.nacc = 0
        self.out = bytearray()
        self.lit = self.dist = None

    # ---- bits
    @property
    def nbits(self):
        return 8 * len(self.buf) + self.nacc

    def bits(self, value, count):
        """count bits of value, least significant first"""
        assert 0 <= value < (1 << count) or count == 0
        self.acc |= value << self.nacc
        self.nacc += count
        while self.nacc >= 8:
            self.buf.append(self.acc & 0xFF)
            self.acc >>= 8
            self.nacc -= 8

    def code(self, code, length):
        """a Huffman code, most significant bit first"""
        self.bits(int(format(code, f"0{length}b")[::-1], 2) if length else 0, length)

    def pad_byte(self, fill=0):
        """up to the next byte boundary with fill bits (0 or 1)"""
        while self.nacc:
            self.bits(fill, 1)

    def raw(self, data):
        assert self.nacc == 0
        self.buf += data

    def finish(self):
        """the stream, the last byte padded with zero bits"""
        return bytes(self.buf) + (bytes([self.acc]) if self.nacc else b"")

    # ---- block headers
    def header(self, final, btype):
        self.bits(int(final), 1)
        self.bits(btype, 2)

    def stored(self, data, final=False, length=None, nlen=None, fill=0):
        """stored block: header, fill bits to the byte boundary, LEN, NLEN (default: ~LEN), the payload"""
        self.header(final, 0)
        self.pad_byte(fill)
        length = len(data) if length is None else length
        nlen = (~length) & 0xFFFF if nlen is None else nlen
        self.raw(bytes([length & 0xFF, length >> 8, nlen & 0xFF, nlen >> 8]))
        self.raw(data)
        self.out += data

    def fixed(self, final=False):
        self.header(final, 1)
        self.use(FIXED_LIT, FIXED_DIST)

    def use(self, lit_lengths, dist_lengths):
        """the codes the tokens of this block are written with (kept bit-reversed, ready for bits())"""
        rev = lambda codes: {s: (int(format(c, f"0{n}b")[::-1], 2), n) for s, (c, n) in codes.items()}
        self.lit, self.dist = rev(canonical(lit_lengths)), rev(canonical(dist_lengths))

    def dynamic_header(self, final, hlit, hdist, hclen, clen_lengths, symbols):
        """dynamic block header exactly as given: HLIT (257..288), HDIST (1..32), HCLEN (4..19), the first hclen code-length-
        code lengths (transmission order), then each (symbol, extra bits) of the code lengths"""
        self.header(final, 2)
        self.bits(hlit - 257, 5)
        self.bits(hdist - 1, 5)
        self.bits(hclen - 4, 4)
        by_sym = [0] * 19
        for i in range(hclen):
            self.bits(clen_lengths[i], 3)
            by_sym[CLEN_ORDER[i]] = clen_lengths[i]
        codes = canonical(by_sym)
        for s, extra in symbols:
            self.code(*codes[s])
            if s in CLEN_EXTRA:
                self.bits(extra, CLEN_EXTRA[s])

    def dynamic(self, final, lit_lengths, dist_lengths, symbols=None, hclen=None):
        """a dynamic header for the given lengths (HLIT / HDIST their counts), spelled with `symbols` (default: rle_symbols)
        and a complete code-length code over the symbols used; the block's tokens use these codes"""
        if symbols is None:
            symbols = rle_symbols(list(lit_lengths) + list(dist_lengths))
        h, cl = clen_code_for(symbols)
        if hclen is not None:
            cl, h = cl + [0] * (hclen - h), hclen
        self.dynamic_header(final, len(lit_lengths), len(dist_lengths), h, cl, symbols)
        self.use(lit_lengths, dist_lengths)

    # ---- tokens
    def sym(self, s):
        """a literal/length symbol; one the code has no code for writes nothing (the stream is invalid by then)"""
        if s in self.lit:
            self.bits(*self.lit[s])

    def literal(self, b):
        self.sym(b)
        self.out.append(b)

    def literals(self, data):
        for b in data:
            self.literal(b)

    def match(self, length, dist, lsym=None, lextra=None, dsym=None, dextra=None):
        """a (length, distance) pair; the symbols and extra bits are derived unless given (length 258 is 285 by default, or
        lsym=284, lextra=31).  A distance code that has no codes writes nothing for the distance."""
        if lsym is None:
            lsym = max(i for i in range(29) if LEN_BASE[i] <= length and (i < 28 or length == 258)) + 257
            if length == 258:
                lsym = 285
        if lextra is None:
            lextra = length - LEN_BASE[lsym - 257]
        if dsym is None:
            dsym = max(i for i in range(30) if DIST_BASE[i] <= dist)
        if dextra is None:
            dextra = dist - DIST_BASE[dsym]
        self.sym(lsym)
        self.bits(lextra, LEN_EXTRA[lsym - 257] if lsym <= 285 else 0)
        if self.dist:
            self.bits(*self.dist[dsym])
            self.bits(dextra, DIST_EXTRA[dsym] if dsym < 30 else 0)
        if dist <= len(self.out):
            start = len(self.out) - dist
            if dist >= length:
                self.out += self.out[start:start + length]
            else:
                for _ in range(length):
                    self.out.append(self.out[-dist])

    def eob(self):
        self.sym(256)

    def fill_to_phase(self, phase, b8, b9, before=0):
        """literals b8 (8-bit code) and b9 (9-bit code) until the stream is `before` bits short of bit phase `phase`"""
        while (self.nbits + before) % 8 != phase:
            self.literal(b9)
        self.literal(b8)


# ==== the catalogue ========================================================================================================
@dataclass
class Case:
    name: str
    stream: bytes
    out: bytes          # what the stream decodes to, or (invalid) what it produces before the error
    valid: bool


TEXT = b"the quick brown fox jumps over the lazy dog; " * 8
ALL_LIT = list(range(286))
FF = 0xFF


def _lit_lengths(n=286, drop=(), extra=()):
    syms = [s for s in range(min(n, 286)) if s not in drop] + list(extra)
    return complete_lengths(syms, n)


def _dist_lengths(n=30, drop=()):
    return complete_lengths([s for s in range(min(n, 30)) if s not in drop], n)


def _text_block(w, final, data=TEXT, lit=None, dist=None, symbols=None, hclen=None):
    w.dynamic(final, lit or _lit_lengths(), dist or _dist_lengths(), symbols, hclen)
    w.literals(data[:50])
    w.match(200, 45)
    w.literals(b"end")
    w.eob()


def _one(name, build, valid=True):
    w = Writer()
    build(w)
    return Case(name, w.finish(), bytes(w.out), valid)


def header_cases():
    cs = []
    for hlit, ok in ((286, True), (287, False), (288, False)):
        cs.append(_one(f"hlit_{hlit}", lambda w, h=hlit: _text_block(w, True, lit=_lit_lengths(h)), ok))
    for hdist, ok in ((30, True), (31, False), (32, False)):
        cs.append(_one(f"hdist_{hdist}", lambda w, h=hdist: _text_block(w, True, dist=_dist_lengths(h)), ok))

    def hclen4(w):   # only 16, 17, 18 and 0 can be spelled: every length is 0, so there is no end-of-block code
        w.dynamic_header(True, 257, 1, 4, [1, 0, 2, 2], [(18, 127), (18, 109)])
    cs.append(_one("hclen_4_all_lengths_zero", hclen4, False))

    def hclen5(w):   # 16, 17, 18, 0, 8: 255 literals and end-of-block at length 8, no distance code: a literal-only block
        lit = [8] * 256 + [8]
        lit[7] = 0
        dist = [0]
        syms = [(8, 0)] * 7 + [(0, 0)] + [(8, 0)] * 249 + [(0, 0)]
        w.dynamic_header(True, 257, 1, 5, [0, 0, 0, 1, 1], syms)
        w.use(lit, dist)
        w.literals(TEXT[:60])
        w.eob()
    cs.append(_one("hclen_5_literal_only", hclen5))
    cs.append(_one("hclen_19", lambda w: _text_block(w, True, hclen=19)))
    return cs


def clen_code_cases():
    lit, dist = _lit_lengths(), _dist_lengths()
    syms = plain_symbols(lit + dist)
    used = sorted({s for s, _ in syms})

    def with_clen(by_sym_lengths, symbols=syms, lit_l=lit):
        def build(w):
            hclen = max(4, max(CLEN_ORDER.index(s) for s in range(19) if by_sym_lengths[s]) + 1) if any(by_sym_lengths) else 19
            w.dynamic_header(True, len(lit_l), 30, hclen, [by_sym_lengths[s] for s in CLEN_ORDER[:hclen]], symbols)
            w.use(lit_l, dist)
            w.literals(TEXT[:30])
            w.eob()
        return build
    cs = [_one("clen_complete", with_clen(complete_lengths(used, 19)))]
    over = complete_lengths(used, 19)
    over[used[0]] = 1
    over[used[1]] = 1
    cs.append(_one("clen_oversubscribed", with_clen(over), False))
    inc = complete_lengths(used + [15], 19)   # a code for 15, which is never used: drop it and the code is incomplete
    inc[15] = 0
    cs.append(_one("clen_incomplete", with_clen(inc), False))
    # a single code of length 1 (accepted by the code-length decoder): every length is 9, which leaves the literal/length code
    # of 257 codes incomplete
    one9 = [0] * 19
    one9[9] = 1
    cs.append(_one("clen_single_length_1", with_clen(one9, [(9, 0)] * (257 + 30), [9] * 257), False))
    # the same single code, followed by a 1 bit: the symbol after the code's only one
    def single_then_one(w):
        w.dynamic_header(True, 257, 1, 7, [0, 0, 0, 0, 0, 0, 1], [])
        w.bits(1, 1)
    cs.append(_one("clen_single_length_1_then_bit_1", single_then_one, False))
    two = [0] * 19
    two[8] = 2
    cs.append(_one("clen_single_length_2", with_clen(two, [(8, 0)] * 287, [8] * 257), False))
    cs.append(_one("clen_no_code", lambda w: (w.dynamic_header(True, 257, 1, 19, [0] * 19, []), w.bits(0, 16)), False))
    return cs


def rle_cases():
    cs = []
    lit, dist = _lit_lengths(), _dist_lengths()

    def explicit(name, lit_l, dist_l, symbols, ok, hlit=None, hdist=None):
        def build(w):
            h, cl = clen_code_for(symbols)
            w.dynamic_header(True, hlit or len(lit_l), hdist or len(dist_l), h, cl, symbols)
            w.use(lit_l, dist_l)
            w.literals(TEXT[:50])
            w.match(10, 45)
            w.eob()
        cs.append(_one(name, build, ok))
    explicit("rle_16_first", lit, dist, [(16, 0)] + plain_symbols(lit[3:] + dist), False)
    # 16 as the first distance length: copies the last literal/length length (5) over the first three distance lengths
    lit16 = [8] * 211 + [9] * 74 + [5]
    dist16 = complete_lengths([3, 4] + list(range(3)) + list(range(5, 30)), 30)
    assert lit16[285] == dist16[0] == dist16[1] == dist16[2] == 5
    explicit("rle_16_first_distance_length", lit16, dist16, plain_symbols(lit16) + [(16, 0)] + plain_symbols(dist16[3:]), True)
    # zero runs across the boundary: literal/length 270..285 unused and distance 0..4 unused (an 18 of 21), or literal/length
    # 283..285 and distance 0..3 (a 17 of 7)
    for name, nl, nd, sym in (("rle_18_across_boundary", 16, 5, (18, 10)), ("rle_17_across_boundary", 3, 4, (17, 4))):
        ll = _lit_lengths(drop=range(286 - nl, 286))
        dl = _dist_lengths(drop=range(nd))
        explicit(name, ll, dl, plain_symbols(ll[:286 - nl]) + [sym] + plain_symbols(dl[nd:]), True)
    # a run that fills the lengths exactly vs one that overruns by one: the last 12 distance lengths are 0
    dl = _dist_lengths(drop=range(18, 30))
    head = plain_symbols(lit + dl[:18])
    explicit("rle_18_fills_exactly", lit, dl, head + [(18, 1)], True)
    explicit("rle_18_overruns_by_one", lit, dl, head + [(18, 2)], False)
    # the same with 16 over the last three distance lengths (all 5): a repeat of 3, or of 4
    dl16 = complete_lengths(range(30), 30)
    assert dl16[26:] == [5] * 4
    explicit("rle_16_fills_exactly", lit, dl16, plain_symbols(lit + dl16[:27]) + [(16, 0)], True)
    explicit("rle_16_overruns_by_one", lit, dl16, plain_symbols(lit + dl16[:27]) + [(16, 1)], False)
    # no end-of-block code
    nl = _lit_lengths(drop=(256,))
    explicit("rle_no_end_of_block", nl, dist, rle_symbols(nl + dist), False)
    return cs


def litlen_code_cases():
    cs = []
    over = _lit_lengths()
    over[5] = 1
    cs.append(_one("lit_oversubscribed", lambda w: _text_block(w, True, lit=over), False))
    inc = _lit_lengths()
    inc[1] = 0
    cs.append(_one("lit_incomplete", lambda w: _text_block(w, True, lit=inc), False))

    def eob_only(bit):
        def build(w):
            lit = [0] * 256 + [1]
            w.dynamic(True, lit, [0])
            w.bits(bit, 1)
        return build
    cs.append(_one("lit_only_end_of_block", eob_only(0)))
    cs.append(_one("lit_only_end_of_block_bit_1", eob_only(1), False))
    return cs


def dist_code_cases():
    cs = []
    lit = _lit_lengths()

    def block(dist_l, tokens, pad=0):
        def build(w):
            w.dynamic(True, lit, dist_l)
            tokens(w)
            w.eob()
            w.bits(pad, 16)
        return build
    cs.append(_one("dist_empty_literal_only", block([0], lambda w: w.literals(TEXT[:90]))))
    cs.append(_one("dist_empty_with_length", block([0], lambda w: (w.literals(TEXT[:20]), w.match(10, 5))), False))
    cs.append(_one("dist_empty_with_length_ones", block([0], lambda w: (w.literals(TEXT[:20]), w.match(10, 5)), 0xFFFF), False))
    one = [0, 0, 0, 1]
    cs.append(_one("dist_single_code_bit_0", block(one, lambda w: (w.literals(TEXT[:20]), w.match(30, 4)))))

    def bit1(w):
        w.literals(TEXT[:20])
        w.sym(270)           # length 23 .. 26: 2 extra bits
        w.bits(0, 2)
        w.bits(1, 1)         # the distance code's only code is 0
    cs.append(_one("dist_single_code_bit_1", block(one, bit1), False))
    cs.append(_one("dist_single_code_length_2", block([0, 0, 0, 2], lambda w: w.literals(TEXT[:20])), False))
    return cs


# A literal/length code and a distance code that are chains: every length 1 .. 15 occurs.  'h' has 8 bits and 'i' 9 (the
# padding that sets a token's bit phase), 'j' .. 'n' 10 .. 14, end-of-block and 284 have 15.
LONG_LIT_SYMS = [ord(c) for c in "abcdefghijklmn"] + [284, 256]
LONG_DIST_SYMS = list(range(14)) + [28, 29]


def long_code_cases():
    cs = []
    lit = chain_lengths(LONG_LIT_SYMS, 286)
    dist = chain_lengths(LONG_DIST_SYMS, 30)
    assert [lit[c] for c in b"hijklmn"] == [8, 9, 10, 11, 12, 13, 14] and lit[284] == lit[256] == 15 and dist[29] == 15

    def codes(w):   # every code of every length, each distance symbol at its largest distance
        w.stored(bytes(range(256)) * 128)
        w.dynamic(True, lit, dist)
        w.literals(b"abcdefghijklmn" * 3)
        for d in LONG_DIST_SYMS:
            w.match(227 + d, DIST_BASE[d] + (1 << DIST_EXTRA[d]) - 1, lsym=284)
        w.eob()
    cs.append(_one("long_codes_every_length", codes))

    def tokens48(w):
        """4096 tokens (284 with 31 extra, distance 29 with 8191 extra: 48 bits) one every 105 bits: token starts cover every
        residue mod 4096 bits, so every bit phase across each 128-byte refill and the 512-byte ring"""
        w.stored(bytes((i * 7 + (i >> 8)) & 0xFF for i in range(32768)))
        w.dynamic(True, lit, dist)
        for _ in range(4096):
            w.match(258, 32768, lsym=284, lextra=31, dsym=29, dextra=8191)
            w.literals(b"ihhhhhh")
        w.eob()
    cs.append(_one("long_codes_48_bit_tokens", tokens48))

    def eob15_end(w):   # the stream ends on the last bit of a 15-bit end-of-block code
        w.dynamic(True, lit, dist)
        w.literals(b"abc")
        w.fill_to_phase(0, ord("h"), ord("i"), before=15)
        w.eob()
        assert w.nacc == 0
    cs.append(_one("long_codes_end_of_block_15_bits_last_bit", eob15_end))
    return cs


def fixed_cases():
    cs = []

    def sym_block(s, dsym=None):
        def build(w):
            w.fixed(True)
            w.literals(b"abc")
            if dsym is None:
                w.sym(s)
            else:
                w.match(3, 1, dsym=dsym, dextra=0)
            w.bits(0, 16)
        return build
    for s in (286, 287):
        cs.append(_one(f"fixed_litlen_{s}", sym_block(s), False))
    for d in (30, 31):
        cs.append(_one(f"fixed_dist_{d}", sym_block(None, d), False))

    def len258(w):
        w.fixed(True)
        w.literals(b"xyz")
        w.match(258, 3)                              # 285
        w.match(258, 3, lsym=284, lextra=31)         # 284 + 31
        w.eob()
    cs.append(_one("fixed_length_258_both_ways", len258))

    def d32768(w):
        w.fixed(False)
        w.literals(bytes((i * 13) & 0xFF for i in range(300)))
        for _ in range(127):
            w.match(258, 300)
        w.eob()
        w.fixed(True)
        w.match(258, 32768)
        w.match(3, 32768)
        w.eob()
    cs.append(_one("fixed_distance_32768", d32768))
    return cs


def distance_cases():
    cs = []
    for extra, ok in ((0, True), (1, False)):
        def first(w, e=extra):
            w.fixed(True)
            w.literals(b"abc")
            w.match(5, 3 + e)
            w.eob()
        cs.append(_one(f"dist_first_match_{'equal' if ok else 'plus_1'}", first, ok))

        def after_stored(w, e=extra):
            w.stored(TEXT[:100])
            w.fixed(True)
            w.match(7, 100 + e)
            w.eob()
        cs.append(_one(f"dist_after_stored_{'equal' if ok else 'plus_1'}", after_stored, ok))

        def second_block(w, e=extra):
            w.fixed(False)
            w.literals(TEXT[:50])
            w.eob()
            w.dynamic(True, _lit_lengths(), _dist_lengths())
            w.match(20, 50 + e)
            w.eob()
        cs.append(_one(f"dist_second_block_{'equal' if ok else 'plus_1'}", second_block, ok))
    return cs


def _shift(w, phase):
    """a non-final fixed block that leaves the stream at bit phase `phase` for the next block header"""
    w.fixed(False)
    w.fill_to_phase(phase, ord("a"), 0xE9, before=7)
    w.eob()


def stored_cases():
    cs = []
    cs.append(_one("stored_len_0", lambda w: w.stored(b"", True)))
    big = bytes((i * 31 + (i >> 9)) & 0xFF for i in range(65535))
    cs.append(_one("stored_len_65535", lambda w: w.stored(big, True)))
    for bit in (0, 15):
        cs.append(_one(f"stored_nlen_bit_{bit}", lambda w, b=bit: w.stored(TEXT[:20], True, nlen=((~20) & 0xFFFF) ^ (1 << b)), False))
    for cut in (0, 1, 2, 3):
        def cut_header(w, c=cut):
            w.fixed(False)
            w.literals(b"ab")
            w.eob()
            w.header(True, 0)
            w.pad_byte()
            w.raw(bytes([20, 0, 0xEB, 0xFF])[:c])
        cs.append(_one(f"stored_header_cut_{cut}", cut_header, False))
    cs.append(_one("stored_payload_short", lambda w: (w.stored(TEXT[:99], True, length=100)), False))
    for phase in range(8):
        def at_phase(w, p=phase):
            _shift(w, p)
            w.stored(TEXT[:33], True, fill=1)
        cs.append(_one(f"stored_header_phase_{phase}", at_phase))

    def refills(w):
        for k, n in enumerate((1, 127, 128, 129, 255, 256, 257, 300, 511, 512, 513, 1000, 0, 2000)):
            _shift(w, k % 8)
            w.stored(bytes((i * 11 + k) & 0xFF for i in range(n)), fill=k & 1)
        w.fixed(True)
        w.match(258, 1000)
        w.eob()
    cs.append(_one("stored_payloads_across_refills", refills))
    return cs


def end_cases():
    cs = []
    cs.append(_one("end_block_type_3", lambda w: (w.stored(b"abc"), w.header(True, 3), w.bits(0, 16)), False))

    def no_final(w):
        w.fixed(False)
        w.literals(TEXT[:40])
        w.eob()
    cs.append(_one("end_no_final_block", no_final, False))
    cs.append(_one("end_no_final_block_stored", lambda w: w.stored(TEXT[:40]), False))

    def trailing(w):
        w.fixed(True)
        w.literals(TEXT[:40])
        w.eob()
        w.pad_byte(1)
        w.raw(b"\x03\xff trailing bytes")
    cs.append(_one("end_bytes_after_final_block", trailing))

    def last_bit(w):
        w.fixed(True)
        w.literals(TEXT[:41])
        w.fill_to_phase(0, ord("a"), 0xE9, before=7)
        w.eob()
        assert w.nacc == 0
    cs.append(_one("end_on_last_bit_of_end_of_block", last_bit))
    return cs


ADLER_LENGTHS = (0, 1, 5551, 5552, 5553, 11104)


def _ff_tokens(w, n):
    if n:
        w.literal(FF)
    left = max(n - 1, 0)
    while left >= 3:
        k = min(258, left)
        if 0 < left - k < 3:
            k -= 3
        w.match(k, 1)
        left -= k
    w.literals(b"\xff" * left)


def _ff_block(w, kind, n, final):
    if kind == "stored":
        w.stored(b"\xff" * n, final)
        return
    if kind == "fixed":
        w.fixed(final)
    else:
        w.dynamic(final, _lit_lengths(), _dist_lengths())
    _ff_tokens(w, n)
    w.eob()


def adler_cases():
    cs = []
    for kind in ("stored", "fixed", "dynamic"):
        for n in ADLER_LENGTHS:
            cs.append(_one(f"adler_{kind}_{n}", lambda w, k=kind, m=n: _ff_block(w, k, m, True)))

        def all_lengths(w, k=kind):
            for i, m in enumerate(ADLER_LENGTHS):
                _ff_block(w, k, m, i == len(ADLER_LENGTHS) - 1)
        cs.append(_one(f"adler_{kind}_all_lengths", all_lengths))

    def mixed(w):
        kinds = ("stored", "fixed", "dynamic")
        for i, m in enumerate(ADLER_LENGTHS * 2):
            _ff_block(w, kinds[i % 3], m, i == 2 * len(ADLER_LENGTHS) - 1)
    cs.append(_one("adler_mixed_kinds", mixed))
    return cs


def all_cases():
    cs = (header_cases() + clen_code_cases() + rle_cases() + litlen_code_cases() + dist_code_cases() + long_code_cases()
          + fixed_cases() + distance_cases() + stored_cases() + end_cases() + adler_cases())
    assert len({c.name for c in cs}) == len(cs)
    return cs
