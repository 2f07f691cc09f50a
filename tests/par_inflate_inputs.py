"""Large raw deflate streams, built with tests/deflate_writer.py, that each put one rule of the many-warp inflate (DESIGN.md
§4.6) to work: chunk counts around powers of two, chunks whose output is thinner than a window, the finder's substance rule,
blocks the finder does not look for, false starts and re-cuts up to the 16-pass limit, a final block in mid-buffer, the
block-length list of a chunk, its symbol budget, and a match before the start of the stream.

Every input is laid out on the grid of nominal chunks of CHUNK bytes (ZIPC_B200_PAR_CHUNK) and is at least PAR_MIN bytes long
(ZIPC_B200_PAR_MIN).  `intent` states, on the plan of tests/par_inflate_model.py, what the input was built to reach; the CPU
test fails, naming the input, when a change of the builders makes it drift."""
from __future__ import annotations

import random
from dataclasses import dataclass
from typing import Callable

import deflate_writer as dw
import par_inflate_model as pm

CHUNK = 4096
PAR_MIN = 20000
U = 8 * CHUNK            # bits per nominal chunk

# CODE_X: literals 0 .. 252 of 8 bits; 253 .. 255, end-of-block, 284 (lengths 227 .. 257) and 285 (258) of 9 bits; all 30
# distances (0 and 1 of 4 bits, the others of 5).  Any bit count of 63 or more is a whole number of 8- and 9-bit literals,
# and every 8 stream bits whose code value is at most 252 are one literal: bits can be spelled.
LIT_X = dw.complete_lengths(list(range(257)) + [284, 285], 286)
DIST_X = dw.complete_lengths(range(30), 30)
LIT_CHAIN = dw.chain_lengths(dw.LONG_LIT_SYMS, 286)        # 'a' of 1 bit ... 'n' of 14, 284 and end-of-block of 15
DIST_CHAIN = dw.chain_lengths(dw.LONG_DIST_SYMS, 30)


def _text(seed, n):
    rng = random.Random(seed)
    words = [bytes(rng.choice(b"etaoinshrdlucmfwypvbgkqjxz") for _ in range(rng.randrange(2, 9))) for _ in range(400)]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(words) + b" "
    return bytes(out[:n])


class Stream:
    """a Writer with the block builders of this file"""

    def __init__(self, seed, high=False):
        self.w = dw.Writer()
        self.rng = random.Random(seed)
        self.high = high        # literals 128 .. 252 (mean byte ~190: the signed-remainder quirk of the reference's Adler-32)
        self.block_out = 0      # output where the current block began
        self.prev_out = 0       # output where the block before it began

    def lit8(self):
        return self.rng.randrange(128, 253) if self.high else self.rng.choice(b"etaoinshrdlu cmfwypvbgkqjxz.,")

    def begin(self, lit=LIT_X, dist=DIST_X, final=False):
        self.w.dynamic(final, lit, dist)
        self.prev_out, self.block_out = self.block_out, len(self.w.out)

    def far_matches(self, length=240, edge=True):
        """matches at distances 32768 and 32767 and, with CODE_X, to the first byte of the previous block and one either side"""
        w = self.w
        for d in (32768, 32767, 0, 1, -1) if edge and self.prev_out < self.block_out else (32768, 32767):
            if d < 2:
                d += len(w.out) - self.prev_out
            if 1 <= d <= min(len(w.out), 32768):
                w.match(length, d)

    def fill_x(self, bits):
        """CODE_X literals of exactly `bits` bits (>= 63)"""
        b = bits % 8
        a = (bits - 9 * b) // 8
        assert a >= 0, bits
        return [self.lit8() for _ in range(a)] + [253] * b

    def fill_chain(self, bits):
        """LIT_CHAIN literals of exactly `bits` bits: 'b' .. 'n' (2 .. 14 bits) at random, then 'a' (1 bit)"""
        out = []
        while bits > 14:
            k = self.rng.randrange(1, 14)
            out.append(ord("a") + k)
            bits -= k + 1
        return out + [ord("a")] * bits

    def end_at(self, end_bit, out_len=None, chain=False, dist=1):
        """fill the current block so that it ends (after its end-of-block code) on bit end_bit, with exactly out_len bytes of
        output when given: matches of 227 .. 257 bytes at distance `dist` (all of one cost), then literals"""
        w = self.w
        eob = 15 if chain else 9
        fill = self.fill_chain if chain else self.fill_x
        if out_len is None:
            lits, lens = fill(end_bit - eob - w.nbits), []
        else:
            probe = dw.Writer()
            probe.out = bytearray(max(dist, 1))
            probe.use(LIT_CHAIN if chain else LIT_X, DIST_CHAIN if chain else DIST_X)
            probe.match(240, dist, lsym=284)
            cost = probe.nbits
            for k in range(0, 100000):
                room = end_bit - eob - w.nbits - k * cost
                assert room >= 0, "no room for the output asked"
                lits = fill(room)
                need = out_len - (len(w.out) - self.block_out) - len(lits)
                if 227 * k <= need <= 257 * k:
                    lens = [need // k + (i < need % k) for i in range(k)] if k else []
                    break
        for n in lens:
            w.match(n, dist, lsym=284)
        w.literals(bytes(lits))
        w.eob()
        assert w.nbits == end_bit, (w.nbits, end_bit)
        if out_len is not None:
            assert len(w.out) - self.block_out == out_len

    def final(self):
        self.w.fixed(True)
        self.w.literals(b"end")
        self.w.eob()

    def finish(self):
        return self.w.finish(), bytes(self.w.out)


@dataclass
class Input:
    name: str
    stream: bytes
    out: bytes
    intent: Callable      # intent(plan, walk) -> None, or the reason the plan is not what the input was built for
    what: str


def _want(cond, why):
    return None if cond else why


def chunk_count(k):
    """one findable dynamic block in each of k - 1 nominal chunks (and block 0 at bit 0): k accepted chunks, ceil(log2 k)
    pointer-doubling rounds.  Every block opens with far matches (32768, 32767, the previous block's first byte and one
    either side) and holds ~4 KiB of output, less than a window: every window is made of many predecessors."""
    n = max(k, 5)
    at = sorted({round(j * n / k) for j in range(1, k)})
    s = Stream(100 + k)
    for j in range(len(at) + 1):
        s.begin()
        s.far_matches()
        end = at[j] * U + 2000 + 37 * j if j < len(at) else n * U - 300
        s.end_at(end)
    s.final()
    st, out = s.finish()
    return Input(f"chunks_{k}", st, out,
                 lambda p, w: _want(p.outcome == "parallel" and len(p.passes) == 1 and len(p.chunks) == k,
                                    f"wants 1 pass of {k} chunks"),
                 f"{k} accepted chunks")


def thin_windows():
    """15-bit codes over 4 KiB chunks: ~2.3 KiB of output per chunk, matches at 32768 and 32767 (copies through more than
    16 predecessors); a chunk of zero output (a findable block holding only its end-of-block code, across a nominal
    boundary); chunks of exactly 32767, 32768 and 32769 bytes"""
    s = Stream(7)
    n = 44
    exact = {20: 32767, 24: 32768, 28: 32769}
    for c in range(n):
        if c == 11:     # the empty block: the only start in nominal chunk 11, it ends in 12 where the next block begins
            s.begin(LIT_X, DIST_X)
            s.w.eob()
            continue
        s.begin(LIT_CHAIN, DIST_CHAIN)
        if len(s.w.out) >= 32768:
            s.w.match(258, 32768, lsym=284, lextra=31, dsym=29, dextra=8191)
            s.w.match(257, 32767, lsym=284)
        end = (c + 1) * U + 1500 if c + 1 < n else n * U - 300
        if c == 10:
            end = 12 * U - 40       # (over nominal chunk 11, up to the empty block 40 bits before its end)
        s.end_at(end, exact.get(c), chain=True)
    s.final()
    st, out = s.finish()

    def intent(p, w):
        lens = [c.out_len for c in p.chunks]
        return _want(p.outcome == "parallel" and len(p.passes) == 1 and 0 in lens and
                     {32767, 32768, 32769} <= set(lens) and sorted(lens)[len(lens) // 2] < 32768,
                     "wants 1 pass with chunks of 0, 32767, 32768 and 32769 bytes, most thinner than a window")
    return Input("thin_windows", st, out, intent, "chunks of 0, ~2.3 Ki, 32767, 32768, 32769 bytes")


def substance():
    """a true dynamic start with 11 coded literal/length symbols (not found: the chunk before runs through it) and one with
    12 (found)"""
    s = Stream(11)
    marks = {}
    for c in range(8):
        if c in (3, 5):
            coded = 11 if c == 3 else 12
            syms = [ord(x) for x in "etaoinshrdlucm"[:coded - 2]] + [256, 284]
            marks[coded] = s.w.nbits
            s.begin(dw.complete_lengths(syms, 286), [1])
            s.w.match(240, 1, lsym=284)
            while s.w.nbits < (c + 1) * U + 1000 - 16:
                s.w.literal(syms[s.rng.randrange(coded - 2)])
            s.w.eob()
            continue
        s.begin()
        s.end_at((c + 1) * U + 1000 + 11 * c)
    s.final()
    st, out = s.finish()

    def intent(p, w):
        starts = {c.start for c in p.chunks}
        return _want(p.outcome == "parallel" and marks[11] not in starts and marks[12] in starts,
                     "wants the 12-symbol start found and the 11-symbol one run through")
    return Input("substance_11_12", st, out, intent, "coded 11 (not found) / 12 (found)")


def unsearched(first):
    """stored and fixed blocks the finder does not look for: a first block that is stored or fixed, a stored block over
    several nominal chunks, empty stored blocks (sync-flush markers) and fixed blocks between dynamic ones"""
    s = Stream(21 if first == "stored" else 22)
    text = _text(5, 20000)
    if first == "stored":
        s.w.stored(text[:3000])
    else:
        s.w.fixed()
        s.w.literals(text[:1500])
        s.w.eob()
    for c in range(1, 12):
        s.begin()
        s.far_matches()
        s.end_at(s.w.nbits + U + 1000 + 5 * c)
        if c == 3:
            s.w.stored(text[3000:15000])            # 12000 bytes: over three nominal chunks
        elif c in (5, 6):
            s.w.stored(b"")
            s.w.stored(b"")                          # (sync-flush markers)
        elif c in (8, 9):
            s.w.fixed()
            s.w.literals(text[15000:15400 + 100 * c])
            s.w.eob()
    s.final()
    st, out = s.finish()
    kinds = {b.start: b.btype for b in pm.walk(st).blocks}

    def intent(p, w):
        return _want(p.outcome == "parallel" and len(p.chunks) >= 6 and all(kinds.get(c.start, 2) == 2 for c in p.chunks[1:]),
                     "wants a parallel plan whose chunks (after the first) all begin at dynamic blocks")
    return Input(f"unsearched_first_{first}", st, out, intent, f"first block {first}, stored / fixed / sync-flush blocks")


def _spell(bits):
    """CODE_X literals whose codes are exactly `bits` (then zero bits up to the end of the last code), or None: the parse of
    the bits by the code meets the end-of-block or a length code"""
    table, maxlen = pm._code_table(LIT_X)
    bits = bits + [0] * 9
    out, i = [], 0
    while i < len(bits) - 9:
        sym, n = table[sum(b << j for j, b in enumerate(bits[i:i + maxlen]))]
        if sym > 255:
            return None
        out.append(sym)
        i += n
    return out


def _header_bits(nlit, ndist):
    """the bits of a valid non-final dynamic header: complete codes over nlit literal/length and ndist distance symbols"""
    h = dw.Writer()
    h.dynamic(False, dw.complete_lengths(range(nlit), 286), dw.complete_lengths(range(ndist), 30))
    v = int.from_bytes(h.finish(), "little")
    return [(v >> i) & 1 for i in range(h.nbits)]


def recuts(r, high=False):
    """r false starts: in each of the first r blocks a valid dynamic header spelled in CODE_X literals ~700 bits ahead of the
    next true start, in the same nominal chunk on the grid of every pass.  Blocks are 1.5 nominal chunks long, so each pass
    accepts one chunk and re-cuts from a true start that is not a byte boundary; r = 16 uses up the passes."""
    s = Stream(300 + r, high)
    nblocks = max(r + 1, 4) + 1
    for i in range(nblocks):
        s.begin()
        s.far_matches()
        end = (3 * (i + 1) * U) // 2 + 2 * i + 1     # (odd: the re-cuts start off byte boundaries)
        if i < r:
            target = end - 700
            lead = s.fill_x(target - 9 * 0 - s.w.nbits)   # literals up to the false header's first bit
            s.w.literals(bytes(lead))
            assert s.w.nbits == target
            # the header, behind `phase` zero bits, parsed into literals of CODE_X (a header whose bits parse into a code
            # that is not a literal is passed over)
            vals = next(v for nlit in range(286, 200, -1) for ndist in (30, 29, 28) for phase in range(1, 8)
                        if (target + phase) % 8 and (v := _spell([0] * phase + _header_bits(nlit, ndist))) is not None)
            s.w.literals(bytes(vals))
            s.end_at(end)
        else:
            s.end_at(end if i + 1 < nblocks else (3 * nblocks * U) // 2 - 200)
    s.final()
    st, out = s.finish()
    if r < 16:
        return Input(f"recuts_{r}" + ("_adler_quirk" if high else ""), st, out,
                     lambda p, w: _want(p.outcome == "parallel" and p.recuts == r and len(p.passes) == r + 1 and
                                        all(q.first_bit % 8 for q in p.passes[1:]),
                                        f"wants {r} re-cuts from bits that are not byte boundaries, then the final block"),
                     f"{r} false starts")
    return Input(f"recuts_{r}", st, out, lambda p, w: _want(p.outcome == "passes_used_up" and len(p.passes) == 16,
                                                            "wants the 16 passes used up"), f"{r} false starts")


def final_mid_buffer():
    """a final block followed by a whole second stream, whose block starts the finder reports: the output stops at the final
    block, decoded in parallel"""
    a = chunk_count(4)
    b = chunk_count(9)
    lead = len(pm.walk(a.stream).blocks)
    return Input("final_mid_buffer", a.stream + b.stream, a.out,
                 lambda p, w: _want(p.outcome == "parallel" and len(w.blocks) == lead and
                                    any(f > 8 * len(a.stream) for q in p.passes for f in q.starts),
                                    "wants the second stream's starts found and the output to stop at the first's final block"),
                 "final block, then a second stream")


def block_list(nonempty):
    """one chunk of `nonempty` non-empty blocks -- its dynamic block and fixed blocks of one literal -- plus empty fixed
    and stored blocks that do not count, between two findable starts"""
    s = Stream(400 + nonempty)
    for c in range(8):
        s.begin()
        s.far_matches()
        if c == 3:
            s.w.literals(b"list")
            s.w.eob()
            for j in range(nonempty - 2):   # (with the dynamic blocks before and after them)
                s.w.fixed()
                s.w.literal(s.lit8())
                s.w.eob()
                if j % 50 == 7:
                    s.w.fixed()
                    s.w.eob()
                    s.w.stored(b"")
            s.begin()
        s.end_at((c + 1) * U + 3000 + 7 * c)
    s.final()
    st, out = s.finish()
    if nonempty <= pm.SPEC_BLOCKS:
        return Input(f"block_list_{nonempty}", st, out,
                     lambda p, w: _want(p.outcome == "parallel" and max(c.blocks for c in p.chunks) == nonempty,
                                        f"wants a parallel plan with a chunk of {nonempty} non-empty blocks"),
                     f"{nonempty} non-empty blocks in a chunk")
    return Input(f"block_list_{nonempty}", st, out,
                 lambda p, w: _want(p.outcome == "block_list" and len(p.passes) == 2, "wants the list to overflow on a re-cut"),
                 f"{nonempty} non-empty blocks in a chunk")


def symbol_budget(extra):
    """chunk 0 (block 0, up to the start found in nominal chunk 1) outputs exactly 24 bytes + 65536 symbols + extra"""
    s = Stream(500 + extra)
    end = U + 3000
    s.begin()
    s.w.literal(ord("x"))
    s.end_at(end, 24 * ((end + 7) // 8) + 65536 + extra, dist=1)
    for c in range(1, 6):
        s.begin()
        s.far_matches()
        s.end_at((c + 1) * U + 3000 if c < 5 else 6 * U - 300)
    s.final()
    st, out = s.finish()
    if extra == 0:
        return Input("symbol_budget_exact", st, out,
                     lambda p, w: _want(p.outcome == "parallel" and p.chunks[0].out_len == 24 * ((end + 7) // 8) + 65536,
                                        "wants chunk 0 at its symbol budget, accepted"), "chunk 0 at 24 x bytes + 65536")
    return Input("symbol_budget_plus_1", st, out,
                 lambda p, w: _want(p.outcome == "symbol_budget" and len(p.passes) == 1, "wants chunk 0 one symbol over"),
                 "chunk 0 one symbol over its budget")


def match_before_start():
    """a stored block of 10000 bytes, then a dynamic block with a match 20000 back: the speculation accepts it, the resolve
    does not"""
    s = Stream(600)
    s.w.stored(_text(6, 10000))
    s.begin()
    s.w.literals(b"reach")
    s.w.match(240, 20000)
    s.end_at(s.w.nbits + U)
    for c in range(4):
        s.begin()
        s.end_at(s.w.nbits + U)
    s.final()
    st, _ = s.finish()
    return Input("match_before_start", st, b"",
                 lambda p, w: _want(p.outcome == "match_before_start", "wants a plan that only the resolve refuses"),
                 "a match before the start of the stream")


def all_inputs():
    out = [chunk_count(k) for k in (2, 3, 4, 5, 8, 9, 16, 17, 32, 33)]
    out += [thin_windows(), substance(), unsearched("stored"), unsearched("fixed")]
    out += [recuts(1), recuts(2, high=True), recuts(15), recuts(16), final_mid_buffer()]
    out += [block_list(256), block_list(257), symbol_budget(0), symbol_budget(1), match_before_start()]
    return out
