"""Deflate streams whose output passes 4 GiB and is known without decoding them, for the inflate tests past 2^32
(test_gpu_inflate_past_4gib.py); test_big_output_inputs_cpu.py holds every builder to its properties.

Every stream outputs a 32,768-byte random prefix P, tiled: out[i] = P[i mod 32768].  P comes first (one stored block),
every later match is (length, 32768), and every later literal is the byte such a match would have copied.  So the expected
bytes, CRC-32 and Adler-32 of a stream follow from P and its total length alone.

- expand(total): P, then ONE fixed-Huffman block of (258, 32768) matches (26 bits each, so 4 of them are a 13-byte period);
  a last shorter match or one or two literals set the exact total.  ~80-fold expansion and no dynamic header: the finder
  of the many-warp decoder has nothing to find, so this stream is always decoded by one warp, in one block.
- spread(total): P, then dynamic-Huffman blocks of 4096 output bytes each, every one with its own header of 12 or more
  coded symbols, ~27-fold expansion: under the symbol budget of a nominal 8 KiB chunk (24 bytes + 65536 symbols, 32-fold)
  and, over the whole stream, under the 6 GiB symbols the many-warp decoder sets aside.  It is decoded by many warps.
- big_block(total): P, four small dynamic blocks, ONE dynamic block of total - 65536 bytes of mostly literals at ~20-fold
  expansion (under 24), then three small dynamic blocks and a small final one.  The many-warp decoder takes the large block
  as one chunk, and its output length needs more than 32 bits.

A stream is written once with its repeated unit twice (Writer of deflate_writer.py), and the unit is then tiled as whole
bytes: a unit is a whole number of bytes long and outputs a multiple of 32,768 bytes, so its bits do not depend on where
it sits.  Plain Python and numpy, no GPU."""
from __future__ import annotations

import zlib
from dataclasses import dataclass

import numpy as np

from deflate_writer import LEN_BASE, Writer, complete_lengths

PERIOD = 32768
P_SEED = 4_294_967_296 + 7
TWO32 = 1 << 32
SMALL_OUT = 4096            # output bytes of a small dynamic block (divides PERIOD)
SMALL_LITS = 64             # literals in a small block (the rest are matches): sets its expansion
BIG_MATCHES = 122           # matches of 258 per 32 KiB period of the large block of big_block; the rest are literals
# lengths of the full-size streams: the output crosses 2^32 by one byte; the output puts matches in
# [2^32, 2^32 + 32768) and ends at an odd offset past 2^32 + 65536
LEN_JUST_OVER = TWO32 + 1
LEN_LONG = TWO32 + 65536 + 4097


def prefix() -> bytes:
    return np.random.default_rng(P_SEED).integers(0, 256, PERIOD, dtype=np.uint8).tobytes()


def expected(total: int, start: int = 0, length: int | None = None) -> np.ndarray:
    """out[start:start + length] of any stream of this file"""
    length = total - start if length is None else length
    p = np.frombuffer(prefix(), dtype=np.uint8)
    reps = -(-(start % PERIOD + length) // PERIOD)
    return np.tile(p, reps)[start % PERIOD:start % PERIOD + length]


def expected_crc32(total: int, piece: int = 64 << 20) -> int:
    """zlib.crc32 of the output, over host slices of `piece` bytes (a multiple of PERIOD)"""
    crc, p = 0, np.tile(np.frombuffer(prefix(), dtype=np.uint8), piece // PERIOD)
    for off in range(0, total, piece):
        crc = zlib.crc32(p[:min(piece, total - off)], crc)
    return crc


@dataclass
class BlockRec:
    bit: int            # where the block header starts (in the written copy: head, unit twice, tail)
    out: int            # output position of the block's first byte in the FULL stream
    btype: int


@dataclass
class Big:
    name: str
    total: int
    copies: int         # units in the full stream
    head: bytes         # stream = head + mid * (copies - 1) + last
    mid: bytes
    last: bytes
    head_bits: int      # bits before the first unit
    unit_bits: int
    unit_out: int
    blocks: list        # BlockRec of the written copy (head, unit 1, unit 2, tail)
    matches: list       # (bit, output position in the full stream, length) of every match of the written copy

    @property
    def nbytes(self) -> int:
        return len(self.head) + len(self.mid) * (self.copies - 1) + len(self.last)

    def stream(self) -> bytes:
        return b"".join([self.head, self.mid * (self.copies - 1), self.last])

    def block_table(self):
        """(start bit, output start, BTYPE) of every block of the full stream, numpy arrays; output lengths follow from the
        next block's output start and self.total"""
        h, U = self.head_bits, self.unit_bits
        parts = []
        head = [b for b in self.blocks if b.bit < h]
        unit = [b for b in self.blocks if h <= b.bit < h + U]
        tail = [b for b in self.blocks if b.bit >= h + 2 * U]
        shift = (self.copies - 2) * U
        parts.append(np.array([(b.bit, b.out, b.btype) for b in head], dtype=np.int64).reshape(-1, 3))
        if unit:
            u = np.array([(b.bit, b.out, b.btype) for b in unit], dtype=np.int64)
            i = np.arange(self.copies, dtype=np.int64)[:, None]
            parts.append(np.stack([u[:, 0] + i * U, u[:, 1] + i * self.unit_out,
                                   np.broadcast_to(u[:, 2], (self.copies, len(u)))], axis=2).reshape(-1, 3))
        parts.append(np.array([(b.bit + shift, b.out, b.btype) for b in tail], dtype=np.int64).reshape(-1, 3))
        t = np.concatenate(parts)
        return t[:, 0], t[:, 1], t[:, 2]

    def match_bytes(self, lo: int, hi: int) -> int:
        """how many output bytes of [lo, hi) of the full stream matches copy (the unit's matches at every copy)"""
        h, U = self.head_bits, self.unit_bits
        n = 0
        for bit, out, ln in self.matches:
            if h <= bit < h + U:
                i = np.arange(self.copies, dtype=np.int64)
                s = out + i * self.unit_out
                n += int(np.clip(np.minimum(s + ln, hi) - np.maximum(s, lo), 0, None).sum())
            elif bit < h or bit >= h + 2 * U:
                n += max(0, min(out + ln, hi) - max(out, lo))
        return n

    def block_lengths(self) -> np.ndarray:
        _, out, _ = self.block_table()
        return np.diff(np.append(out, self.total))


class _W(Writer):
    """a Writer that records its blocks, with literals given their values in the FULL stream (pos + shift)"""

    def __init__(self):
        super().__init__()
        self.recs = []
        self.mrecs = []
        self.full = 0       # output position in the full stream

    def block(self, btype):
        self.recs.append(BlockRec(self.nbits, self.full, btype))

    def lit_at(self, p):
        self.literal(p[self.full % PERIOD])
        self.full += 1

    def match258(self, length):
        self.mrecs.append((self.nbits, self.full, length))
        self.match(length, PERIOD)
        self.full += length


def _tokens(w: _W, p: bytes, length: int, nlits: int):
    """`length` output bytes: nlits literals, then matches of 258, then a shorter match or one or two literals"""
    nlits = min(nlits, length)
    for _ in range(nlits):
        w.lit_at(p)
    left = length - nlits
    while left >= 258:
        w.match258(258)
        left -= 258
    if left >= 3:
        w.match258(left)
    else:
        for _ in range(left):
            w.lit_at(p)


def _len_sym(n):
    """the length symbol of a match of 3 <= n < 258"""
    return 257 + max(i for i in range(28) if LEN_BASE[i] <= n)


def _dynamic(w: _W, p: bytes, length: int, nlits: int, final: bool):
    """a dynamic block of `length` output bytes written by _tokens, with a complete literal/length code over the symbols it
    uses and a distance code of symbols 28 and 29 (one distance symbol alone would be an incomplete code)"""
    pos = w.full
    syms = {p[(pos + k) % PERIOD] for k in range(min(nlits, length))} | {256, 285}
    r = (length - min(nlits, length)) % 258
    if r >= 3:
        syms.add(_len_sym(r))
    elif r:
        syms |= {p[(pos + length - k - 1) % PERIOD] for k in range(r)}
    assert final or len(syms) >= 12    # (the finder takes headers of 12 coded symbols or more)
    syms = sorted(syms)
    w.block(2)
    w.dynamic(final, complete_lengths(syms, 286), complete_lengths([28, 29], 30))
    _tokens(w, p, length, nlits)
    w.eob()


def _finish(name, total, w: _W, h, u1, u2, copies, unit_out):
    assert u1 - h == u2 - u1 and (u1 - h) % 8 == 0
    s2 = w.finish()
    ub = (u1 - h) // 8
    a = h // 8 + ub
    return Big(name, total, copies, s2[:a], s2[a:a + ub], s2[a + ub:], h, u1 - h, unit_out, w.recs, w.mrecs)


def _units(write_group, w: _W):
    """groups written until they fill whole bytes: (bits before, bits after one unit, after two, groups per unit)"""
    h = w.nbits
    g = 0
    while True:
        write_group()
        g += 1
        if (w.nbits - h) % 8 == 0:
            break
    u1 = w.nbits
    for _ in range(g):
        write_group()
    return h, u1, w.nbits, g


def _head(w: _W, p: bytes):
    w.block(0)
    w.stored(p)
    w.full = PERIOD


def expand(total: int) -> Big:
    p = prefix()
    q, r = divmod(total - PERIOD, 258)
    assert q >= 8
    w = _W()
    _head(w, p)
    w.block(1)
    w.fixed(final=True)

    def group():
        for _ in range(4):
            w.match258(258)
    h, u1, u2, g = _units(group, w)   # 4 tokens = 104 bits = 13 bytes
    per = 4 * g
    copies = q // per
    assert copies >= 2
    w.full = PERIOD + copies * per * 258
    for _ in range(q - copies * per):
        w.match258(258)
    if r >= 3:
        w.match258(r)
    else:
        for _ in range(r):
            w.lit_at(p)
    w.eob()
    assert w.full == total
    # (the unit outputs 4 g 258 bytes, not a multiple of PERIOD: matches carry no literal values, so its bits do not
    # depend on where it sits either; the literals after the units are written at their positions in the full stream)
    return _finish("expand", total, w, h, u1, u2, copies, per * 258)


def spread(total: int) -> Big:
    p = prefix()
    K, r = divmod(total - PERIOD, SMALL_OUT)
    nblocks = K + (r > 0)
    w = _W()
    _head(w, p)

    def group():
        for _ in range(PERIOD // SMALL_OUT):
            _dynamic(w, p, SMALL_OUT, SMALL_LITS, False)
    h, u1, u2, g = _units(group, w)
    per = g * PERIOD // SMALL_OUT            # blocks per unit
    copies = (nblocks - 1) // per
    assert copies >= 2
    w.full = PERIOD + copies * per * SMALL_OUT
    for k in range(copies * per, nblocks):
        n = SMALL_OUT if k < K else r
        _dynamic(w, p, n, SMALL_LITS, k == nblocks - 1)
    assert w.full == total
    return _finish("spread", total, w, h, u1, u2, copies, g * PERIOD)


def big_block(total: int) -> Big:
    p = prefix()
    big_out = total - PERIOD - 8 * SMALL_OUT
    J, rem = divmod(big_out, PERIOD)
    nlits = PERIOD - 258 * BIG_MATCHES
    w = _W()
    _head(w, p)
    for _ in range(4):
        _dynamic(w, p, SMALL_OUT, SMALL_LITS, False)
    w.block(2)
    w.dynamic(False, complete_lengths(list(range(256)) + list(range(257, 286)) + [256], 286), complete_lengths([28, 29], 30))

    def period():
        _tokens(w, p, PERIOD, nlits)
    h, u1, u2, g = _units(period, w)
    copies = J // g
    assert copies >= 2
    w.full = PERIOD + 4 * SMALL_OUT + copies * g * PERIOD
    for _ in range(J - copies * g):
        period()
    _tokens(w, p, rem, nlits)
    w.eob()
    for k in range(4):
        _dynamic(w, p, SMALL_OUT, SMALL_LITS, k == 3)
    assert w.full == total
    return _finish("big_block", total, w, h, u1, u2, copies, g * PERIOD)


BUILDERS = {"expand": expand, "spread": spread, "big_block": big_block}


def small_total(name: str) -> int:
    """a total of a few MiB for the same construction (the repeat count cut), odd, at no multiple of a unit"""
    return {"expand": PERIOD + 3 * (1 << 20) + 1, "spread": PERIOD + 4 * (1 << 20) + 4095,
            "big_block": 65536 + 3 * (1 << 20) + 4097}[name]


def zlib_wrap(raw: bytes, adler: int) -> bytes:
    """a zlib stream (RFC 1950) around a raw deflate stream, with the given trailer"""
    return b"\x78\x9c" + raw + adler.to_bytes(4, "big")


def chunk_plan(big: Big, chunk_bytes: int = 8192):
    """The first pass of par_speculate over the full stream, without decoding it, for a stream whose only finder hits are
    its dynamic block starts (test_big_output_inputs_cpu.py checks that on the small stream of the same construction):
    -> (chunk start bits, chunk output lengths, chunk compressed bytes, symbols set aside: spec_cap).  The chunks chain up,
    because every hit is a true block start."""
    import par_inflate_model as pm
    bits, outs, btype = big.block_table()
    nbits = 8 * big.nbytes
    nch = -(-big.nbytes // chunk_bytes)
    hits = bits[(btype == 2) & (np.arange(len(bits)) < len(bits) - 1)]   # (the finder never takes a final block)
    lo = 8 * chunk_bytes * np.arange(1, nch, dtype=np.int64)
    i = np.searchsorted(hits, lo)
    ok = i < len(hits)
    f = np.where(ok, hits[np.minimum(i, len(hits) - 1)], -1)
    ok &= f < np.minimum(lo + 8 * chunk_bytes, nbits)
    starts = np.unique(np.concatenate([[0], f[ok]]))
    stops = np.append(starts[1:], nbits)
    nbytes = (stops - starts + 7) // 8
    cap = (24 * nbytes + 65536 + 7) & ~7
    need = int(cap.sum())
    out_at = outs[np.searchsorted(bits, starts)]
    out_len = np.diff(np.append(out_at, big.total))
    assert pm.SPEC_BLOCKS == 256
    return starts, out_len, nbytes, need + need // 8 + (8 << 20)


def adler32_blocks(big: Big, mode: str) -> int:
    """The Adler-32 of the output folded block by block as the reference does (zipc_deflate.ml:682-690): every non-empty
    block on its own 5552-byte chunk grid, the state packed and unpacked in between; mode "ref" is the reference's signed
    remainder (checksum_inputs.step), "rfc" exact RFC 1950 arithmetic (then it is zlib.adler32 of the output).  The sums of
    a chunk depend only on its offset mod 32768 and its length, so they are computed once per pair."""
    import checksum_inputs as ci
    p2 = np.tile(np.frombuffer(prefix(), dtype=np.uint8), 2).astype(np.float64)
    w = np.arange(ci.CHUNK, 0, -1, dtype=np.float64)
    sums = {}

    def ab(pos, n):
        key = (pos % PERIOD, n)
        if key not in sums:
            v = p2[key[0]:key[0] + n]
            sums[key] = (int(v.sum()), int(v @ w[ci.CHUNK - n:]))
        return sums[key]
    _, outs, _ = big.block_table()
    state = 1
    for s, n in zip(outs.tolist(), big.block_lengths().tolist()):
        if not n:
            continue
        s1, s2 = state & 0xFFFF, state >> 16
        first = n % ci.CHUNK or ci.CHUNK
        pos, m = s, first
        while pos < s + n:
            a, b = ab(pos, m)
            if mode == "ref":
                s1, s2, _ = ci.step(s1, s2, m, a, b)
            else:
                s1, s2 = (s1 + a) % ci.M, (s2 + m * s1 + b) % ci.M
            pos += m
            m = ci.CHUNK
        state = ci.pack(s1, s2)
    return state


ZIP_NAME = b"big.bin"


def zip64_archive(raw: bytes, total: int, crc: int) -> tuple[bytes, int]:
    """A ZIP archive of one deflated member (raw deflate stream `raw`, `total` bytes out, CRC-32 `crc`), ZIP64 as APPNOTE
    4.5.3 has it: both sizes 0xFFFFFFFF in the local header and the directory entry, the real ones in a ZIP64 extra field
    (id 1: size, then compressed size).  -> (archive, offset of the member's data)"""
    import struct
    extra = struct.pack("<HHQQ", 1, 16, total, len(raw))
    lfh = struct.pack("<IHHHHHIIIHH", 0x04034B50, 45, 0, 8, 0, 0x21, crc, 0xFFFFFFFF, 0xFFFFFFFF, len(ZIP_NAME),
                      len(extra)) + ZIP_NAME + extra
    cd = struct.pack("<IHHHHHHIIIHHHHHII", 0x02014B50, 45, 45, 0, 8, 0, 0x21, crc, 0xFFFFFFFF, 0xFFFFFFFF, len(ZIP_NAME),
                     len(extra), 0, 0, 0, 0, 0) + ZIP_NAME + extra
    cd_at = len(lfh) + len(raw)
    eocd = struct.pack("<IHHHHIIH", 0x06054B50, 0, 0, 1, 1, len(cd), cd_at, 0)
    return b"".join([lfh, raw, cd, eocd]), len(lfh)
