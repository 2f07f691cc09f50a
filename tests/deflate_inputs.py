"""Inputs built to reach particular rules of the encoder (deflate_core.h, finalize_block in deflate.cu), each with a test of
whether a checked stream of it does reach that rule.

corpus() -> {name: Input}; Input.reached(data, report) takes deflate_checker's report of a stream of the input (see
test_deflate_checker_cpu.py, which holds every entry to its target on the host model's output, so that an entry which
quietly stops reaching its rule fails there).  Seeded, plain Python and numpy, no GPU."""
from __future__ import annotations

import random
from dataclasses import dataclass
from typing import Callable

import numpy as np

BLOCK = 61440
LIMIT_DEPTH = 15
CLEN_LIMIT_DEPTH = 7


@dataclass
class Input:
    name: str
    data: bytes
    target: str                                   # the rule, in words
    reached: Callable                             # (data, report) -> bool


def hash4(v):
    """the encoder's hash of 4 little-endian bytes (deflate_core.h), restated for building inputs"""
    return ((v * 0x9E3779B1) & 0xFFFFFFFF) >> 18


def _fresh(rng, n):
    """n random bytes with bit 7 set: 4-byte strings of them occur nowhere else in these inputs"""
    return bytes(b | 0x80 for b in rng.randbytes(n))


_WORDS = None


def _filler(rng, n):
    """n bytes of lowercase words and spaces (compressible: blocks of it are dynamic, their tokens in the stream)"""
    global _WORDS
    if _WORDS is None:
        r = random.Random(7)
        _WORDS = ["".join(r.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(r.randrange(2, 9))) for _ in range(300)]
    out = []
    k = 0
    while k < n:
        w = rng.choice(_WORDS) + " "
        out.append(w)
        k += len(w)
    return "".join(out).encode()[:n]


def no_repeat(n, k, rng, weights=None):
    """n bytes over the alphabet [0, k) (optionally weighted) in which no 4-byte string occurs twice: the encoder can only
    emit literals for them"""
    seen, out = set(), bytearray()
    syms = list(range(k))
    while len(out) < n:
        for _ in range(64):
            b = rng.choices(syms, weights)[0] if weights else rng.randrange(k)
            if len(out) < 3 or bytes(out[-3:]) + bytes([b]) not in seen:
                break
        else:
            raise ValueError("alphabet too small for a string without repeats")
        if len(out) >= 3:
            seen.add(bytes(out[-3:]) + bytes([b]))
        out.append(b)
    return bytes(out)


# ---- targets (on the checker's report) ------------------------------------------------------------------------------
def _dyn(report):
    return [b for b in report.blocks if b.type == "dynamic"]


def _literal_only_dynamic(data, r):
    return any(b.hdist == 1 and b.dist_lengths[0] == 0 and not b.matches for b in _dyn(r))


def _single_distance_symbol(data, r):
    return any(sum(1 for x in b.dist_lengths if x) == 1 and max(b.dist_lengths) == 1 for b in _dyn(r))


def _depth_over(alphabet, limit):
    return lambda data, r: any(b.depth.get(alphabet, 0) > limit for b in r.blocks if b.tokens_known)


def _match_at(pos, dist, length=None):
    def f(data, r):
        return any(p == pos and d == dist and (length is None or l == length) for p, l, d in r.matches)
    return f


def _match_over(pos, dist):
    """a match at distance `dist` covers position pos (it may start a byte early, where the bytes before agree too)"""
    return lambda data, r: any(d == dist and p <= pos < p + l for p, l, d in r.matches)


def _no_match_in(lo, hi):
    return lambda data, r: not any(lo <= p < hi for p, _, _ in r.matches)


# ---- builders -----------------------------------------------------------------------------------------------------------
def literal_only(rng):
    """a skewed alphabet of 40 symbols, no 4-byte string twice: a dynamic block of literals only, HDIST = 1 with the one
    distance length 0"""
    w = [1.0 / (1 + i) for i in range(40)]
    return no_repeat(20000, 40, rng, w)


def periodic(period, n, rng):
    unit = bytes(rng.sample(range(256), period)) if period else b""
    return (unit * (n // period + 1))[:n] if period else bytes(n)


def fibonacci_lengths(levels=18, k=64, seed=1):
    """matches whose length symbols have Fibonacci counts (the most frequent the shortest length), each copying the 3 random
    literals (of k values) before it at distance 3: an unconstrained literal/length code deeper than 15 in the first block.
    (The literals' share of the alphabet decides how deep the chain of length symbols ends up; seed and k were picked by
    running the host model.)"""
    rng = random.Random(seed)
    fib = [1, 1]
    while len(fib) < levels:
        fib.append(fib[-1] + fib[-2])
    lengths = [4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67][:levels]
    toks = [L for L, c in zip(lengths, fib[::-1]) for _ in range(c)]
    rng.shuffle(toks)
    out = bytearray()
    for L in toks:
        out += bytes(rng.randrange(k) for _ in range(3))
        for _ in range(L):
            out.append(out[-3])
        nxt = rng.randrange(k)          # breaks the period: the match is exactly L long
        while nxt == out[-3]:
            nxt = rng.randrange(k)
        out.append(nxt)
    return bytes(out)


def fibonacci_distances(rng, levels=17):
    """matches of 4 bytes whose distance symbols have Fibonacci counts (the most frequent the nearest code), each copying the
    fresh random bytes just before it: an unconstrained distance code deeper than 15"""
    fib = [1, 1]
    while len(fib) < levels:
        fib.append(fib[-1] + fib[-2])
    # the most frequent codes are the nearest ones whose 4-byte strings stay unique (distance 1 and 2 repeat one or two
    # random bytes, which recur all over the input: they get the smallest counts)
    base = [3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 2, 1, 257, 385, 513][:levels]
    toks = [d for d, c in zip(base, fib[::-1]) for _ in range(c)]
    rng.shuffle(toks)
    out = bytearray()
    for d in toks:
        fresh = bytearray(rng.randbytes(d))
        out += fresh
        src = len(out) - d
        for i in range(4):
            out.append(out[src + i])
        # the byte after the match differs from the one after its source: the match is exactly 4 long
        nxt = rng.randrange(256)
        while nxt == out[src + 4]:
            nxt = rng.randrange(256)
        out.append(nxt)
    return bytes(out)


# (seed, total weight per byte of input); whether the result reaches the target is asserted on the host model's output
CLEN_SEARCH = (3, 11)


def clen_deep(rng):
    """literals only, their frequencies chosen so that neighbouring byte values get alternating code lengths with
    Fibonacci-like counts per length: the code-length alphabet then has no runs to fold and a skewed histogram"""
    seed, scale = CLEN_SEARCH
    r = random.Random(seed)
    # lengths 5..13 with counts 1, 1, 2, 3, 5, 8, 13, ... assigned to byte values in an interleaved order
    counts = {}
    fib = [1, 1, 2, 3, 5, 8, 13, 21, 34, 55, 89]
    lens = list(range(4, 15))
    r.shuffle(lens)
    for L, c in zip(lens, fib):
        counts[L] = c
    vals = [L for L, c in counts.items() for _ in range(c)]
    r.shuffle(vals)
    vals = vals[:256]
    weights = [2.0 ** (15 - L) for L in vals]
    n = min(60000, int(sum(weights) / scale))
    return no_repeat(n, len(vals), rng, weights)


def stored_near_tie(rng):
    """8000 literals over 251 byte values, none of their 4-byte strings repeated: as the first block of a member the dynamic
    block is 3 bits cheaper than the stored one (whose header pads 5 bits): a stored cost without the pad picks stored"""
    return no_repeat(8000, 251, random.Random(6))


def _stored_within_pad(data, r):
    b = r.blocks[0]
    pad = (8 - ((b.bit_start + 3) & 7)) & 7
    return b.tokens_known and b.type == "dynamic" and 0 < b.costs["stored"] - b.costs["dynamic"] <= pad


def window_edge(rng, gap):
    """a unique 300-byte chunk, then fresh bytes, then the chunk again `gap` bytes after the first copy"""
    lead = _filler(rng, 5000)
    chunk = _fresh(rng, 300)
    return lead + chunk + _filler(rng, gap - 300) + chunk + _filler(rng, 3000), len(lead) + gap


def window_edge_primed(rng, gap, seg=65536):
    """the same pair, the second copy 100 bytes into the second segment of `seg` bytes: the first copy lies in its prime"""
    at = seg + 100
    pre = _filler(rng, at - gap)
    chunk = _fresh(rng, 300)
    body = _filler(rng, gap - 300)
    return pre + chunk + body + chunk + _filler(rng, 40000), at


def stale_heads(rng):
    """a 4-byte string, 70000 zeros (whose only 4-byte string hashes elsewhere), then the string again and fresh bytes: the
    16-bit chain head of its hash is more than 65536 positions old when it comes back"""
    q = b"\x11\x22\x33\x44\x55\x66\x77\x88"
    assert hash4(int.from_bytes(q[:4], "little")) != hash4(0)
    return q + bytes(70000) + q + _filler(rng, 5000) + q


def _stale_reached(data, r):
    a = np.frombuffer(data, dtype=np.uint8).astype(np.uint32)
    v = a[:-3] | a[1:-2] << 8 | a[2:-1] << 16 | a[3:] << 24
    h = ((v.astype(np.uint64) * 0x9E3779B1) & 0xFFFFFFFF) >> 18
    last = {}
    for p in range(len(h)):
        k = int(h[p])
        if k in last and p - last[k] > 65536:
            return True
        last[k] = p
    return False


def collisions(rng, count=2400):
    """many distinct 4-byte values with one hash, each followed by a fresh byte, then some of them again from far back in the
    chain: chains longer than every level's budget (4 / 12 / 1024 steps)"""
    g = np.random.default_rng(rng.randrange(1 << 30))
    want = None
    vals = []
    while len(vals) < count:
        v = g.integers(0, 1 << 32, size=1 << 22, dtype=np.uint64)
        h = ((v * 0x9E3779B1) & 0xFFFFFFFF) >> 18
        if want is None:
            want = int(h[0])
        vals += [int(x) for x in np.unique(v[h == want])]
    vals = vals[:count]
    body = b"".join(x.to_bytes(4, "little") + bytes([rng.randrange(256)]) for x in vals)
    again = b"".join(vals[i].to_bytes(4, "little") + vals[i + 1].to_bytes(4, "little") for i in (0, 5, 100, 900, 1300, 2000, 2390))
    return body + _fresh(rng, 100) + again + _fresh(rng, 100)


def _chain_over(budget):
    def f(data, r):
        a = np.frombuffer(data, dtype=np.uint8).astype(np.uint32)
        v = a[:-3] | a[1:-2] << 8 | a[2:-1] << 16 | a[3:] << 24
        h = ((v.astype(np.uint64) * 0x9E3779B1) & 0xFFFFFFFF) >> 18
        _, counts = np.unique(h, return_counts=True)
        return counts.max() > budget
    return f


def match_edges(rng):
    """{name: (data, reached)}: matches of exactly 258 and 259 bytes, matches ending at n and n - 1"""
    r = _fresh(rng, 400)
    out = {}
    for L in (258, 259):
        d = r[:L] + _filler(rng, 1000) + r[:L] + b"\x00" + _filler(rng, 100)
        out[f"match{L}"] = (d, _match_at(L + 1000, L + 1000, 258))
    d = r[:300] + _filler(rng, 700)
    out["match_ends_at_n"] = (d + r[:300], lambda data, rep: max(p + l for p, l, _ in rep.matches) == len(data))
    out["match_ends_at_n_1"] = (d + r[:300] + b"\xff", lambda data, rep: max(p + l for p, l, _ in rep.matches) == len(data) - 1)
    return out


def overhang(rng, start):
    """fresh bytes with a 300-byte chunk repeated at `start` (the last position of tile 29 is 61439)"""
    chunk = _fresh(rng, 300)
    head = _filler(rng, start - 20000) + chunk + _filler(rng, 20000 - 300)
    return head + chunk + _filler(rng, 2000)


def lazy_chain(rng, m=200):
    """chunks X[i : 2 i + 4] for i < m, then X: at X + i the match is i + 4 long and the one at X + i + 1 is longer, so the
    lazy parse defers a literal at every step over m positions (the stitched warp parse of a tile)"""
    while True:   # no two different 4-byte strings of X share a hash (a colliding chain would end the walks early)
        x = _fresh(rng, 2 * m + 8)
        grams = {x[i:i + 4] for i in range(len(x) - 3)}
        if len({hash4(int.from_bytes(g, "little")) for g in grams}) == len(grams):
            break
    pre = bytearray()
    for i in range(m + 1):
        pre += x[i:2 * i + 4] + _filler(rng, 2)     # (lowercase: it ends every match against a chunk)
    return bytes(pre) + x + _filler(rng, 500), len(pre), m


def _lazy_reached(start, run):
    """no match starts in the first `run` positions of X and one starts right after: literals deferred over `run` positions"""
    return lambda data, r: not any(start <= p < start + run for p, _, _ in r.matches) and \
        any(p == start + run for p, _, _ in r.matches)


def realistic(rng):
    g = np.random.default_rng(rng.randrange(1 << 30))
    f32 = g.standard_normal(60000).astype(np.float32)
    bf16 = (f32.view(np.uint32) >> 16).astype(np.uint16)
    text = bytes(b | 0x80 for b in (b"the quick brown fox jumps over the lazy dog " * 3000))
    return {"float32": f32.tobytes(), "bfloat16": bf16.tobytes(), "text_bit7": text}


def corpus():
    rng = random.Random(1951)
    c = {}

    def add(name, data, target, reached):
        c[name] = Input(name, data, target, reached)

    add("literal_only", literal_only(rng), "a dynamic block of literals only: HDIST 1, one zero length", _literal_only_dynamic)
    add("zeros", bytes(100000), "one distance symbol (distance 1)", _single_distance_symbol)
    add("period2", periodic(2, 100000, rng), "one distance symbol (distance 2)", _single_distance_symbol)
    add("period3", periodic(3, 100000, rng), "one distance symbol (distance 3)", _single_distance_symbol)
    add("fib_lengths", fibonacci_lengths(), "unconstrained literal/length depth > 15", _depth_over("lit", LIMIT_DEPTH))
    add("fib_distances", fibonacci_distances(rng), "unconstrained distance depth > 15", _depth_over("dist", LIMIT_DEPTH))
    add("clen_deep", clen_deep(rng), "unconstrained code-length depth > 7", _depth_over("clen", CLEN_LIMIT_DEPTH))
    add("stored_tie", stored_near_tie(rng), "dynamic cheaper than stored by less than the stored header's pad",
        _stored_within_pad)
    d, at = window_edge(rng, 32768)
    add("window_32768", d, "a match at distance exactly 32768", _match_over(at, 32768))
    d, at = window_edge(rng, 32769)
    add("window_32769", d, "the same chunk at 32769: literals", _no_match_in(at - 1, at + 300))
    add("stale_heads", stale_heads(rng), "a chain head more than 65536 positions old", _stale_reached)
    add("collisions", collisions(rng), "a hash chain longer than level best's 1024 steps", _chain_over(1024))
    for name, (d, f) in match_edges(rng).items():
        add(name, d, name.replace("_", " "), f)
    for k in range(1, 9):
        add(f"tiny{k}", (b"abcabcab" if k % 2 else bytes(8))[:k], "a member of 1 to 8 bytes", lambda data, r: True)
    add("overhang", overhang(rng, BLOCK - 2), "a 258-byte match from the last decided position of tile 29: the next "
        "block starts 256 bytes into the overhang", lambda data, r: any(b.index == 1 and b.src_start == BLOCK + 256
                                                                        for b in r.blocks))
    add("deferred", overhang(rng, BLOCK - 1), "a match at the last position of tile 29, decided at tile 30: the next block "
        "starts one byte early", lambda data, r: any(b.index == 1 and b.src_start == BLOCK - 1 for b in r.blocks))
    d, start, m = lazy_chain(rng)
    add("lazy_chain", d, f"a literal deferred at {m} positions in a row", _lazy_reached(start, m))
    for name, d in realistic(rng).items():
        add(name, d, "realistic binary", lambda data, r: True)
    return c


def primed_corpus():
    """inputs for primed segments of 64 KiB: the window edge across the segment start"""
    rng = random.Random(1952)
    c = {}
    d, at = window_edge_primed(rng, 32768)
    c["primed_window_32768"] = Input("primed_window_32768", d, "a match at distance 32768 into the prime",
                                     _match_over(at, 32768))
    d, at = window_edge_primed(rng, 32769)
    c["primed_window_32769"] = Input("primed_window_32769", d, "the same at 32769: literals", _no_match_in(at - 1, at + 300))
    return c
