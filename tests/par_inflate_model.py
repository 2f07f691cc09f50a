"""A plain restatement of the plan of the many-warp inflate of one large stream (DESIGN.md §4.6; api.cu par_speculate /
par_resolve / inflate_core, inflate.cu find_starts_kernel).  It shares no code with the library, the oracle or the writer.

- walk(stream): every block of a raw deflate stream -- start bit, type, BFINAL, output length, end bit -- decoded the way
  the reference decoder reads it (zipc_deflate.ml:593-709), and whether a match reaches before the start of the stream.
- Finder: find_starts_kernel.  A candidate at bit p needs BFINAL 0, BTYPE 2, HLIT <= 29, HDIST <= 29, p + 74 <= the stream's
  bits and a complete code-length code (a numpy filter over every offset), then a header that read_dynamic_header accepts
  with at least 12 coded literal/length symbols (plain Python, for the few offsets that pass the filter).  Nominal chunks
  of chunk_bytes are laid from the pass's first bit; chunk 0 is not scanned; the earliest hit of a nominal chunk counts.
- plan(stream, chunk_bytes): the passes of par_speculate with their chunks, and the outcome: "parallel" or the named
  fallback that sends the stream to the one-warp decoder.
- calls(plan, cap): what counters 1 to 4 of the context (Context.parallel_counters) move by in one inflate call."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

CLEN_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]

SPEC_BLOCKS = 256      # kSpecBlocks: non-empty block lengths a speculative chunk reports
MAX_PASSES = 16
FIND_TAIL = 74         # 17 header bits + 19 code-length code lengths: the filter reads that far


class Corrupt(Exception):
    pass


class Bits:
    """LSB-first bit reader over bytes; reading past the end gives zero bits and is caught by the caller's bound check"""

    def __init__(self, data: bytes):
        self.data = bytes(data) + bytes(16)
        self.nbits = 8 * len(data)

    def peek(self, pos, n):
        b = pos >> 3
        return (int.from_bytes(self.data[b:b + 8], "little") >> (pos & 7)) & ((1 << n) - 1)


def _code_table(lengths):
    """decoder over `lengths` as the reference builds it (zipc_deflate.ml:355-391): over-subscribed -> corrupt; incomplete
    -> corrupt unless there is no code, or exactly one code of length 1.  -> (table indexed by the next maxlen stream bits,
    maxlen); an entry is (symbol, length) or None"""
    count = [0] * 16
    for n in lengths:
        count[n] += 1
    count[0] = 0
    left = 1
    for n in range(1, 16):
        left = 2 * left - count[n]
        if left < 0:
            raise Corrupt("over-subscribed code")
    ncodes = sum(count)
    if ncodes == 0:
        return [], 0
    if (ncodes > 1 and left > 0) or (ncodes == 1 and count[1] != 1):
        raise Corrupt("incomplete code")
    maxlen = max(n for n in lengths if n)
    table = [None] * (1 << maxlen)
    code, nxt = 0, [0] * 16
    for n in range(1, 16):
        code = (code + count[n - 1]) << 1
        nxt[n] = code
    for s, n in enumerate(lengths):
        if not n:
            continue
        c = nxt[n]
        nxt[n] += 1
        rev = int(format(c, f"0{n}b")[::-1], 2)
        for k in range(rev, 1 << maxlen, 1 << n):
            table[k] = (s, n)
    return table, maxlen


def _decode(bits, pos, table, maxlen):
    e = table[bits.peek(pos, maxlen)] if maxlen else None
    if e is None:
        raise Corrupt("no code")
    return e


def read_dynamic_header(bits, pos):
    """the header after the 3 block-type bits at `pos` (reference :623-669).  -> (bit after it, literal/length lengths,
    distance lengths); Corrupt if the reference refuses it or it runs past the stream's end"""
    hlit = 257 + bits.peek(pos, 5)
    hdist = 1 + bits.peek(pos + 5, 5)
    hclen = 4 + bits.peek(pos + 10, 4)
    pos += 14
    if hlit > 286 or hdist > 30:
        raise Corrupt("HLIT / HDIST")
    cl = [0] * 19
    for i in range(hclen):
        cl[CLEN_ORDER[i]] = bits.peek(pos, 3)
        pos += 3
    if pos > bits.nbits:
        raise Corrupt("overrun")
    if not any(cl):
        raise Corrupt("empty code-length code")
    table, maxlen = _code_table(cl)
    lengths, prev = [], 0
    while len(lengths) < hlit + hdist:
        sym, n = _decode(bits, pos, table, maxlen)
        pos += n
        if sym < 16:
            rep, val = 1, sym
        elif sym == 16:
            if not lengths:
                raise Corrupt("repeat of nothing")
            rep, val = 3 + bits.peek(pos, 2), prev
            pos += 2
        elif sym == 17:
            rep, val = 3 + bits.peek(pos, 3), 0
            pos += 3
        else:
            rep, val = 11 + bits.peek(pos, 7), 0
            pos += 7
        if rep > hlit + hdist - len(lengths):
            raise Corrupt("lengths overrun")
        lengths += [val] * rep
        prev = val
    if pos > bits.nbits:
        raise Corrupt("overrun")
    lit, dist = lengths[:hlit], lengths[hlit:]
    if lit[256] == 0:
        raise Corrupt("no end-of-block code")
    _code_table(lit)
    _code_table(dist)
    return pos, lit, dist


FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32


@dataclass
class Block:
    start: int          # bit of the block header
    btype: int
    final: bool
    out_len: int
    end: int            # bit after the block (its end-of-block code, or its stored bytes)
    reaches_before_start: bool = False


@dataclass
class Walk:
    blocks: list
    out: bytes
    error: str | None     # the stream stops being valid at the end of the last block listed (None: a final block ends it)
    error_bit: int = 0


def walk(stream: bytes) -> Walk:
    """every block of the stream up to the final one (bytes after it are not read), or up to the first error.  A match that
    reaches before the start of the stream is flagged on its block and its bytes are taken as zeros: the speculative decode
    does not look at distances, the resolve does."""
    bits = Bits(stream)
    out = bytearray()
    blocks = []
    pos = 0
    fixed = (_code_table(FIXED_LIT), _code_table(FIXED_DIST))
    while True:
        start, out0, far = pos, len(out), False
        try:
            if pos + 3 > bits.nbits:
                raise Corrupt("overrun")
            h = bits.peek(pos, 3)
            final, btype = bool(h & 1), h >> 1
            pos += 3
            if btype == 0:
                pos = (pos + 7) & ~7
                length, nlen = bits.peek(pos, 16), bits.peek(pos + 16, 16)
                pos += 32
                if pos > bits.nbits or length != (~nlen & 0xFFFF) or pos + 8 * length > bits.nbits:
                    raise Corrupt("stored block")
                out += stream[pos >> 3:(pos >> 3) + length]
                pos += 8 * length
            elif btype == 3:
                raise Corrupt("block type 3")
            else:
                if btype == 1:
                    (lt, lm), (dt, dm) = fixed
                else:
                    pos, lit, dist = read_dynamic_header(bits, pos)
                    (lt, lm), (dt, dm) = _code_table(lit), _code_table(dist)
                while True:
                    sym, n = _decode(bits, pos, lt, lm)
                    pos += n
                    if sym < 256:
                        out.append(sym)
                    elif sym == 256:
                        break
                    else:
                        if sym > 285:
                            raise Corrupt("length symbol")
                        ln = LEN_BASE[sym - 257] + bits.peek(pos, LEN_EXTRA[sym - 257])
                        pos += LEN_EXTRA[sym - 257]
                        ds, n = _decode(bits, pos, dt, dm)
                        pos += n
                        if ds > 29:
                            raise Corrupt("distance symbol")
                        d = DIST_BASE[ds] + bits.peek(pos, DIST_EXTRA[ds])
                        pos += DIST_EXTRA[ds]
                        if d > len(out):
                            far = True
                            out += bytes(ln)
                        elif d >= ln:
                            out += out[len(out) - d:len(out) - d + ln]
                        else:
                            for _ in range(ln):
                                out.append(out[-d])
                    if pos > bits.nbits:
                        raise Corrupt("overrun")
            if pos > bits.nbits:
                raise Corrupt("overrun")
        except Corrupt as e:
            del out[out0:]
            return Walk(blocks, bytes(out), str(e), start)
        blocks.append(Block(start, btype, final, len(out) - out0, pos, far))
        if final:
            return Walk(blocks, bytes(out), None)


# ---- the finder ----------------------------------------------------------------------------------------------------------
_KRAFT = np.array([0] + [128 >> n for n in range(1, 8)], dtype=np.int32)


def valid_starts(stream: bytes, coded_min: int = 12) -> np.ndarray:
    """every bit offset where find_starts_kernel accepts a block start, ascending"""
    nbits = 8 * len(stream)
    n = nbits - FIND_TAIL + 1
    if n <= 0:
        return np.zeros(0, dtype=np.int64)
    b = np.unpackbits(np.frombuffer(bytes(stream), dtype=np.uint8), bitorder="little").astype(np.int32)

    def field(at, width):
        v = np.zeros(n, dtype=np.int32)
        for i in range(width):
            v |= b[at + i:at + i + n] << i
        return v
    ok = (field(0, 3) == 4) & (field(3, 5) <= 29) & (field(8, 5) <= 29)
    hclen = 4 + field(13, 4)
    kraft = np.zeros(n, dtype=np.int32)
    for i in range(19):
        kraft += np.where(i < hclen, _KRAFT[field(17 + 3 * i, 3)], 0)
    ok &= kraft == 128
    bits = Bits(stream)
    hits = []
    for p in np.flatnonzero(ok):
        try:
            _, lit, _ = read_dynamic_header(bits, int(p) + 3)
        except Corrupt:
            continue
        if sum(1 for x in lit if x) >= coded_min:
            hits.append(int(p))
    return np.array(hits, dtype=np.int64)


def find_starts(hits: np.ndarray, nbits: int, first_bit: int, chunk_bytes: int, nchunks: int):
    """found[k] for nominal chunks k = 1 .. nchunks - 1 laid from first_bit (None: no hit)"""
    found = [None]
    for k in range(1, nchunks):
        lo = first_bit + 8 * k * chunk_bytes
        hi = min(lo + 8 * chunk_bytes, nbits)
        i = int(np.searchsorted(hits, lo))
        found.append(int(hits[i]) if i < len(hits) and hits[i] < hi else None)
    return found


# ---- the plan ------------------------------------------------------------------------------------------------------------
@dataclass
class Chunk:
    start: int
    end: int
    out_len: int
    blocks: int         # non-empty blocks


@dataclass
class Pass:
    first_bit: int
    starts: list        # the chunk starts of the pass (first_bit and the found starts)
    accepted: list      # Chunk of every chunk the pass accepted
    stop: str           # why the chain ended: "final", "recut" (a chunk ended past the next found start), "failed <why>"


@dataclass
class Plan:
    # "parallel", or the fallback: "no_start" (none in the first pass), "chunk0_corrupt" (chunk 0 of a pass fails to decode),
    # "block_list" (over 256 non-empty blocks), "symbol_budget" (over 24 bytes + 65536 symbols), "match_before_start"
    # (refused by the resolve), "passes_used_up", "ran_off_end", "too_few_chunks" (under 4 nominal chunks), "symbol_room"
    # (a re-cut needs more symbols than the first pass set aside), "not_tried"; an output over the cap is the call's (calls())
    outcome: str
    passes: list = field(default_factory=list)
    total: int = 0
    tried: bool = True  # False: the stream is not sent to the many-warp decoder at all

    @property
    def chunks(self):
        return [c for p in self.passes for c in p.accepted]

    @property
    def recuts(self):
        return sum(p.stop == "recut" for p in self.passes)

    @property
    def cached(self):
        """the speculation reached the final block: the plan is kept for the real pass of the same call"""
        return self.outcome in ("parallel", "match_before_start")

    def describe(self):
        return "%s: %d pass(es), %d chunk(s), %d re-cut(s), output %d" % (self.outcome, len(self.passes), len(self.chunks),
                                                                      self.recuts, self.total)


def _chunk(w: Walk, start, stop, cap):
    """the speculative decode of one chunk that starts at the true block boundary `start`, up to the first block boundary at
    or after `stop` or the final block: (Chunk, it ends on the final block, None) or (None, False, why)"""
    i = next(j for j, b in enumerate(w.blocks + [None]) if b is None or b.start == start)
    out = nblk = 0
    while True:
        if i == len(w.blocks):
            return None, False, "corrupt"
        b = w.blocks[i]
        out += b.out_len
        if out > cap:
            return None, False, "symbol_budget"
        nblk += b.out_len > 0
        if b.final or b.end >= stop:
            break
        i += 1
    if nblk > SPEC_BLOCKS:
        return None, False, "block_list"
    return Chunk(start, b.end, out, nblk), b.final, None


def plan(stream: bytes, chunk_bytes: int = 8192, par_min: int | None = None, w: Walk | None = None,
         hits: np.ndarray | None = None) -> Plan:
    """par_speculate and the acceptance of inflate_core for one stream, with ZIPC_B200_PAR_CHUNK = chunk_bytes and
    ZIPC_B200_PAR_MIN = par_min (None: the size rule of par_select for a batch of this one stream)"""
    L = len(stream)
    cb = max(4096, chunk_bytes)
    if par_min is None:
        tried = L >= 65536   # (alone in its batch, a stream of 64 KiB or more costs less on the many-warp decoder)
    else:
        tried = par_min != 0 and L >= par_min
    if not tried:
        return Plan("not_tried", tried=False)
    w = w if w is not None else walk(stream)
    hits = hits if hits is not None else valid_starts(stream)
    nbits = 8 * L
    nch0 = -(-L // cb)
    if nch0 < 4:
        return Plan("too_few_chunks")
    passes = []
    from_bit = spec_used = spec_cap = 0
    for p in range(MAX_PASSES):
        nch = min(nch0, -(-(nbits - from_bit) // (8 * cb)))
        starts = [from_bit]
        if nch >= 2:
            for f in find_starts(hits, nbits, from_bit, cb, nch)[1:]:
                if f is not None and f > starts[-1]:
                    starts.append(f)
        m = len(starts)
        if p == 0 and m < 2:
            passes.append(Pass(from_bit, starts, [], "failed no start"))
            return Plan("no_start", passes)
        capv, need = [], spec_used
        for k in range(m):
            stop = starts[k + 1] if k + 1 < m else nbits
            capv.append((24 * ((stop - starts[k] + 7) // 8) + 65536 + 7) & ~7)
            need += capv[-1]
        if p == 0:
            spec_cap = need + need // 8 + (8 << 20)
            if spec_cap > (6 << 30):
                passes.append(Pass(from_bit, starts, [], "failed symbol room"))
                return Plan("symbol_room", passes)
        elif need > spec_cap:
            passes.append(Pass(from_bit, starts, [], "failed symbol room"))
            return Plan("symbol_room", passes)
        acc, stop_why, final = [], None, False
        for k in range(m):
            c, final, why = _chunk(w, starts[k], starts[k + 1] if k + 1 < m else float("inf"), capv[k])
            if c is None:
                stop_why = "failed " + why
                break
            acc.append(c)
            if final:
                stop_why = "final"
                break
            if k + 1 == m or c.end != starts[k + 1]:
                stop_why = "recut"
                break
        passes.append(Pass(from_bit, starts, acc, stop_why))
        if not acc:
            why = stop_why.split()[1]
            return Plan("chunk0_corrupt" if why == "corrupt" else why, passes)
        if final:
            total = sum(c.out_len for q in passes for c in q.accepted)
            reach = any(b.reaches_before_start for b in w.blocks)
            return Plan("match_before_start" if reach else "parallel", passes, total)
        from_bit = acc[-1].end
        spec_used += sum(capv[:len(acc)])   # (spec_off[used - 1] + capv[used - 1])
        if from_bit >= nbits:
            return Plan("ran_off_end", passes)
    return Plan("passes_used_up", passes)


@dataclass
class Counts:
    streams: int = 0
    fallbacks: int = 0
    passes: int = 0
    chunks: int = 0

    def tuple(self):
        return (self.streams, self.fallbacks, self.passes, self.chunks)


def _one(pl: Plan, cap, count_only, cache_hit, c: Counts):
    """inflate_core's `one` for a stream: -> it was decoded by many warps"""
    if not cache_hit:
        c.passes += len(pl.passes)
    ok = pl.cached
    if ok and cap is not None and pl.total > cap:
        ok = False
    if ok and not count_only:
        c.chunks += len(pl.chunks)
        ok = pl.outcome == "parallel"
    if ok:
        c.streams += 1
    else:
        c.fallbacks += 1
    return ok


def calls(pl: Plan, cap) -> Counts:
    """what counters 1 to 4 move by in one inflate call of this stream with output cap `cap` (None: the call sizes the output
    first with a count-only pass, and a plan that reaches the final block there serves the real pass)"""
    c = Counts()
    if not pl.tried:
        return c
    if cap is not None:
        _one(pl, cap, False, False, c)
        return c
    ok = _one(pl, None, True, False, c)
    _one(pl, pl.total if ok else 0, False, pl.cached, c)
    return c
