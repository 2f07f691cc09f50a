"""The chain walk of levels fast and default restated twice in plain Python, and inputs aimed at each rule of it.

serial_walk is match_begin + match_step + match_resume_token of deflate_core.h, which the kernel's shallow_batches runs:
one candidate after the other, a running best, the one-byte filter, the early stop.  pair_walk is the walk taken apart as
tools/experiments/deflate_walk_pairs.cu.txt runs it (measured slower, DESIGN.md section 4.4 (g)): list the candidates first
(the same stops: dist 0, out of reach, stale), compare every one of them without a running best, then pick the winner with
one max over keys.  Both return (len, dist, resume token) per position; the CPU test holds them equal, the GPU test holds the
kernel to the host model on the same inputs.  Seeded, no GPU."""
from __future__ import annotations

import random

import deflate_inputs as di

TILE = 2048
WINDOW = 32768
MAX_MATCH = 258
MIN_MATCH = 4
LEVELS = {"fast": (4, 32), "default": (12, 128)}      # (chain steps, nice length): level_params of deflate_core.h


def hash4(d, p):
    return di.hash4(int.from_bytes(d[p:p + 4], "little"))


def chains(d):
    """per tile, after its positions are in the chains: (ts, te, prev, first); prev holds 16-bit links by p mod 32768 and
    first[i] is the chain head position ts + i saw (its first candidate), as the front end's insertion leaves them"""
    n = len(d)
    head = [0] * (1 << 14)
    prev = [0] * WINDOW
    for ts in range(0, n, TILE):
        te = min(ts + TILE, n)
        first = [0] * (te - ts)
        for p in range(ts, te):
            if p + 4 > n:
                continue
            h = hash4(d, p)
            first[p - ts] = prev[p & (WINDOW - 1)] = head[h]
            head[h] = p & 0xFFFF
        yield ts, te, prev, first


def match_len(d, p, cp, max_len):
    n = 0
    while n < max_len and d[cp + n] == d[p + n]:
        n += 1
    return n


def serial_walk(d, prev, p, c, steps, nice):
    max_len = min(len(d) - p, MAX_MATCH)
    best, best_dist, last, reach, more = MIN_MATCH - 1, 0, 0, min(p, WINDOW), False
    while True:
        dist = (p - c) & 0xFFFF
        if dist == 0 or dist > reach or dist <= last:
            break
        last = dist
        cp = p - dist
        if best < max_len and d[cp + best] == d[p + best]:
            n = match_len(d, p, cp, max_len)
            if n > best:
                best, best_dist = n, dist
                if n >= nice or n == max_len:
                    break
        c = prev[cp & (WINDOW - 1)]
        steps -= 1
        if steps <= 0:
            more = True
            break
    return (best if best >= MIN_MATCH else 0), best_dist, ((p - last) if more else p) & 0xFFFF


def candidates(d, prev, p, c, steps):
    """the distances of p's candidates in chain order, at most `steps`, up to the first empty, out-of-reach or stale one"""
    reach, last, out = min(p, WINDOW), 0, []
    while len(out) < steps:
        dist = (p - c) & 0xFFFF
        if not last < dist <= reach:
            break
        out.append(dist)
        last = dist
        c = prev[(p - dist) & (WINDOW - 1)]
    return out


def pair_walk(d, prev, p, c, steps, nice):
    dists = candidates(d, prev, p, c, steps)
    max_len = min(len(d) - p, MAX_MATCH)
    win = 0
    for k, dist in enumerate(dists):
        n = match_len(d, p, p - dist, max_len)
        # a stop (len >= nice or len == max_len) beats everything, the first stop most; otherwise the longest, the first of them
        key = (0x8000 | (15 - k) << 9 | n) if (n >= nice or n == max_len) else (n << 4 | (15 - k))
        win = max(win, key << 16 | dist)
    key = win >> 16
    stop = key & 0x8000
    n = key & 0x1FF if stop else key >> 4
    token = (p - dists[steps - 1]) & 0xFFFF if (not stop and len(dists) == steps) else p & 0xFFFF
    return (n, win & 0xFFFF, token) if n >= MIN_MATCH else (0, 0, token)


def walks(d, level, walk, prime=0):
    """{p: (len, dist, token)} for every searched position: p >= prime (positions below only prime the window), p + 4 <= n"""
    steps, nice = LEVELS[level]
    out = {}
    for ts, te, prev, first in chains(d):
        for p in range(max(ts, prime), min(te, len(d) - 3)):
            out[p] = walk(d, prev, p, first[p - ts], steps, nice)
    return out


def walk_details(d, level, prime=0):
    """{p: [(dist, len), ...]} every candidate of every searched position with its match length (for the reach tests)"""
    steps, _ = LEVELS[level]
    out = {}
    for ts, te, prev, first in chains(d):
        for p in range(max(ts, prime), min(te, len(d) - 3)):
            ml = min(len(d) - p, MAX_MATCH)
            out[p] = [(x, match_len(d, p, p - x, ml)) for x in candidates(d, prev, p, first[p - ts], steps)]
    return out


# ---- inputs -----------------------------------------------------------------------------------------------------------------
def same_hash_runs(rng):
    """a repeated 4-gram and a run of zeros: every position of a tile on one chain, far more than 12 of them"""
    return di._filler(rng, 3000) + b"wxyz" * 700 + di._filler(rng, 1500) + bytes(3000) + di._filler(rng, 800)


def tile_crossings(rng):
    """for o = 0 .. 12, a fresh 4-gram seen 14 times before a tile boundary and o + 1 times right after it: the last copy's
    chain has o candidates inside its tile, then continues below it.  Every copy is followed by its own bytes, so the lengths
    of the candidates differ (and some tie)"""
    out = bytearray(di._filler(rng, 4096))
    for o in range(13):
        x = di._fresh(rng, 4)
        ext = [di._fresh(rng, 12) for _ in range(4)]
        boundary = (len(out) // TILE + 2) * TILE
        before = b"".join(x + ext[i % 4][:1 + i % 9] + b" " for i in range(14))
        out += di._filler(rng, boundary - len(out) - len(before)) + before
        assert len(out) == boundary
        out += b"".join(x + ext[(i + 1) % 4][:2 + i % 7] + b" " for i in range(o + 1))
    return bytes(out + di._filler(rng, 3000))


def nice_stop(rng):
    """a copy of 130 bytes near the last one and a copy of 300 bytes farther back: the walk stops at the 130 (>= 128, and
    at fast >= 32) and never sees the longer one"""
    y = di._fresh(rng, 300)
    return di._filler(rng, 2000) + y + di._filler(rng, 700) + y[:130] + b"\x01" + di._filler(rng, 900) + y + di._filler(rng, 500)


def ties(rng):
    """one 10-byte string at several distances, each copy followed by a different byte: equal lengths, the nearest wins"""
    z = di._fresh(rng, 10)
    return di._filler(rng, 1000) + b"".join(z + bytes([0x01 + i]) + di._filler(rng, 97 + 13 * i) for i in range(9)) + z + b"\x7f"


def tail_clip(rng):
    """a 300-byte string repeated at the very end: matches of the last 258 positions clip at n - p"""
    y = di._fresh(rng, 300)
    return di._filler(rng, 3000) + y + di._filler(rng, 2500) + y


def walk_inputs():
    """{name: (data, prime)}: inputs aimed at each rule of the walk"""
    rng = random.Random(2032)
    c = {"same_hash_runs": (same_hash_runs(rng), 0), "tile_crossings": (tile_crossings(rng), 0)}
    c["stale_heads"] = (di.stale_heads(rng), 0)
    c["window_32768"] = (di.window_edge(rng, 32768)[0], 0)
    c["window_32769"] = (di.window_edge(rng, 32769)[0], 0)
    c["collisions"] = (di.collisions(rng), 0)
    c["nice_stop"] = (nice_stop(rng), 0)
    c["ties"] = (ties(rng), 0)
    c["tail_clip"] = (tail_clip(rng), 0)
    primed = di.window_edge_primed(rng, 32768, seg=40960)[0][:40960 + 6000]
    c["primed"] = (primed, 32768)                  # a segment of 40960 + 6000 bytes primed with the 32 KiB before it
    for n in (1, 5, 2047, 2048, 2049, 2051, 4099):  # one tile, and last tiles with no position that can start a match
        c[f"short_{n}"] = ((same_hash_runs(rng) * 3)[:n], 0)
    return c
