"""Inputs built to reach every class of chunk of the device fold of the reference-flavour Adler-32 (adler_fold_kernel in
zipc_b200/csrc/adler32.cu) at the places where that fold hands its state from one tile to the next, and a plain
restatement of the reference's chunk recurrence (zipc_deflate.ml:166-206) that says which class every chunk of an input is
in.

The reference walks a buffer in chunks of 5552 bytes, the first one len mod 5552 bytes long (5552 when that is 0), and at
the end of every chunk computes s1' = rem(s1 + A), s2' = rem(wrap32(s2 + W)) with W = n s1 + B, A = sum b_i,
B = sum (n - i) b_i, and Int32.rem, which keeps the sign of a wrapped s2.  The fold classifies chunks by W alone
(adler32.cu:56-60), M = 65521:
    "L"       M <= W < 2^31 - M         no wrap, s2 ends non-negative whatever it was
    "H"       W >= 2^31 + M             wraps, s2 ends negative
    "low+"    W < M, s2 >= 0 before     no wrap, s2 stays non-negative
    "low-"    W < M, s2 < 0 before      no wrap, the sign depends on s2 (the fold walks it with the U chunks)
    "U"       otherwise, no wrap        the outcome depends on the exact s2: walked serially, in order
    "U-wrap"  otherwise, wraps
One CTA folds a tile of 16,384 chunks.  A tile that starts with low-W chunks waits for the state after its predecessor.

layout(name) builds one of LAYOUTS, an Input whose plan lists the (chunk index, class) pairs the generator aimed for;
Input.missed(classes) returns those of them the model does not find.  test_checksum_inputs_cpu.py holds every layout to
its plan and the model to zo.adler32 and zlib.adler32.  Seeded, plain Python and numpy, no GPU."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

CHUNK = 5552
M = 65521
TILE = 16384                 # chunks per CTA of adler_fold_kernel (kFoldTile)
TILE_BYTES = TILE * CHUNK    # 90,963,968
RED = 8192                   # chunks per CTA of adler_reduce_rfc_kernel (kRedThreads * kRedItems)
TWO31, TWO32 = 1 << 31, 1 << 32
LOW = ("low+", "low-")


# ---- the model ---------------------------------------------------------------------------------------------------------
def chunk_grid(n: int) -> tuple[int, int]:
    """(first chunk length, number of chunks) of an n-byte buffer on the reference's grid"""
    if n == 0:
        return 0, 0
    first = n % CHUNK or CHUNK
    return first, 1 + (n - first) // CHUNK


_WEIGHTS = np.arange(CHUNK, 0, -1, dtype=np.float64)


def chunk_sums(data) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(n, A, B) of every chunk, int64 arrays.  B < 2^32, so a float64 dot of the byte rows with the weights is exact."""
    v = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    first, nchunks = chunk_grid(v.size)
    n = np.full(nchunks, CHUNK, dtype=np.int64)
    A = np.empty(nchunks, dtype=np.int64)
    B = np.empty(nchunks, dtype=np.int64)
    if not nchunks:
        return n, A, B
    n[0] = first
    A[0] = int(v[:first].sum(dtype=np.int64))
    B[0] = int(np.dot(v[:first].astype(np.float64), _WEIGHTS[CHUNK - first:]))
    rows = v[first:].reshape(-1, CHUNK)
    for lo in range(0, rows.shape[0], 2048):
        r = rows[lo:lo + 2048]
        A[1 + lo:1 + lo + r.shape[0]] = r.sum(axis=1, dtype=np.int64)
        B[1 + lo:1 + lo + r.shape[0]] = (r.astype(np.float64) @ _WEIGHTS).astype(np.int64)
    return n, A, B


def srem(x: int) -> int:
    """Int32.rem x M: the remainder with the sign of x"""
    r = abs(x) % M
    return -r if x < 0 else r


def wrap32(x: int) -> int:
    x &= 0xFFFFFFFF
    return x - TWO32 if x >= TWO31 else x


def classify(W: int, s2: int) -> str:
    """the class adler_fold_kernel gives a chunk of weight W, refined by the sign of the exact s2 before it"""
    if M <= W < TWO31 - M:
        return "L"
    if W >= TWO31 + M:
        return "H"
    if W < M:
        return "low+" if s2 >= 0 else "low-"
    return "U-wrap" if s2 + W >= TWO31 else "U"


def step(s1: int, s2: int, n: int, a: int, b: int) -> tuple[int, int, int]:
    """one chunk of the reference's recurrence -> (s1', s2', W); s2 signed"""
    W = n * s1 + b                      # < 2^32: 5552 * 65520 + 255 * 5552 * 5553 / 2
    return srem(s1 + a), srem(wrap32(s2 + W)), W


def pack(s1: int, s2: int) -> int:
    return ((s2 << 16) + s1) & 0xFFFFFFFF


def model(data) -> tuple[int, list[str]]:
    """-> (the reference's Adler-32 of data, the class of every chunk)"""
    n, A, B = chunk_sums(data)
    s1, s2, classes = 1, 0, []
    for k, a, b in zip(n.tolist(), A.tolist(), B.tolist()):
        classes.append(classify(k * s1 + b, s2))
        s1, s2, _ = step(s1, s2, k, a, b)
    return pack(s1, s2), classes


def model_rfc1950(data) -> int:
    """the same chunk recurrence in exact arithmetic (RFC 1950): zlib.adler32 of data"""
    n, A, B = chunk_sums(data)
    s1, s2 = 1, 0
    for k, a, b in zip(n.tolist(), A.tolist(), B.tolist()):
        s1, s2 = (s1 + a) % M, (s2 + k * s1 + b) % M
    return (s2 << 16) | s1


# ---- the generator -----------------------------------------------------------------------------------------------------
@dataclass
class Input:
    name: str
    data: np.ndarray
    plan: list = field(default_factory=list)     # [(chunk index, class)]; "low" stands for either low class
    target: str = ""                              # what the layout is for, in words

    @property
    def nchunks(self) -> int:
        return chunk_grid(self.data.size)[1]

    def missed(self, classes) -> list:
        """the planned (index, class) pairs the chunks of data do not have, with the class they do have"""
        out = []
        for i, want in self.plan:
            got = classes[i] if i < len(classes) else None
            if got != want and not (want == "low" and got in LOW):
                out.append((i, want, got))
        return out


def _set_weight(chunk: np.ndarray, n: int, s1: int, W: int) -> None:
    """bytes of a chunk of n bytes with n s1 + B = W exactly: a fill, then single bytes raised by weight, heaviest first"""
    T = n * (n + 1) // 2
    R = W - n * s1
    if R < 0 or R > 255 * T:
        raise ValueError(f"weight {W} out of reach of a {n}-byte chunk at s1 = {s1}")
    f = min(R // T, 254)
    chunk[:] = f
    R -= f * T
    for i in range(n):
        if R == 0:
            break
        w = n - i
        k = min(255 - f, R // w)
        chunk[i] += k
        R -= k * w
    if R:
        raise ValueError(f"weight {W} out of reach of a {n}-byte chunk at s1 = {s1}")


def _lower_tail(chunk: np.ndarray, d: int) -> None:
    """lower the chunk's byte sum by d from its end (the lightest bytes), leaving its weight nearly unchanged"""
    i = chunk.size - 1
    while d and i >= 0:
        t = min(int(chunk[i]), d)
        chunk[i] -= t
        d -= t
        i -= 1
    if d:
        raise ValueError("chunk too light to bring s1 down")


def build(name: str, nchunks: int, first: int, plan: list, seed: int, target: str = "", s1_low: dict | None = None,
          wrap_slack: int = 1000) -> Input:
    """An input of nchunks chunks, the first one `first` bytes, random bytes except where plan says otherwise.

    Recipes, chunk by chunk in order while the exact state is tracked:
      "H": 0xFF;  "L": 0x40;  "low+" / "low-" / "low": zeros, which are low-W only when s1 <= 11 before them
      (5552 * 12 > M): so the chunk before a low-W run, whatever its class, has the byte sum of its tail lowered to bring
      s1 to s1_low.get(index of the run, 0) -- it keeps its class (checked);
      "U" / "U-wrap": a fill plus single bytes chosen by weight so that W lands just short of 2^31 - s2 (no wrap) or at
      or just past it (wrap), inside [2^31 - M, 2^31 + M); how far comes from the seed, at most wrap_slack.
    Whether the sign before a low-W chunk is what the plan says depends on the chunk before the run ("H": negative,
    "L": non-negative); Input.missed is the check."""
    rng = np.random.default_rng(seed)
    size = first + (nchunks - 1) * CHUNK
    assert chunk_grid(size) == (first, nchunks), (size, first, nchunks)
    data = np.frombuffer(rng.bytes(size), dtype=np.uint8).copy()
    want = dict(plan)
    for i, cls in plan:
        lo, hi = _bounds(i, first)
        if cls in ("H", "L") + LOW + ("low",):
            data[lo:hi] = {"H": 0xFF, "L": 0x40}.get(cls, 0)
    n, A, B = chunk_sums(data)
    s1, s2 = 1, 0
    s1_low = s1_low or {}
    for c in range(nchunks):
        k = int(n[c])
        lo, hi = _bounds(c, first)
        cls = want.get(c)
        if cls in ("U", "U-wrap"):
            slack = int(rng.integers(0, wrap_slack + 1))
            if cls == "U-wrap":
                W = TWO31 - s2 + min(slack, M - 1 + s2)          # < 2^31 + M
            else:
                W = TWO31 - s2 - 1 - min(slack, M - 1 - s2)      # >= 2^31 - M
            _set_weight(data[lo:hi], k, s1, W)
        nxt = want.get(c + 1)
        if nxt in LOW + ("low",) and want.get(c) not in LOW + ("low",):
            before = classify(k * s1 + _weight(data[lo:hi]), s2)
            t = s1_low.get(c + 1, 0)
            _lower_tail(data[lo:hi], (s1 + int(data[lo:hi].sum(dtype=np.int64)) - t) % M)
            after = classify(k * s1 + _weight(data[lo:hi]), s2)
            if after != before:
                raise ValueError(f"{name}: chunk {c} went from {before} to {after} when s1 was brought down")
        if cls is not None or nxt is not None:
            A[c], B[c] = int(data[lo:hi].sum(dtype=np.int64)), _weight(data[lo:hi])
        s1, s2, _ = step(s1, s2, k, int(A[c]), int(B[c]))
    return Input(name, data, list(plan), target)


def _bounds(c: int, first: int) -> tuple[int, int]:
    lo = 0 if c == 0 else first + (c - 1) * CHUNK
    return lo, lo + (first if c == 0 else CHUNK)


def _weight(chunk: np.ndarray) -> int:
    return int(np.dot(chunk.astype(np.float64), _WEIGHTS[CHUNK - chunk.size:]))


def _run(start: int, count: int, head: str) -> list:
    """a run of zero chunks: the first one with the given low class, the others either"""
    return [(start, head)] + [(start + j, "low") for j in range(1, count)]


# ---- the layouts -------------------------------------------------------------------------------------------------------
def _u_at_tile_edges():
    T = TILE
    plan = [(T - 1, "U-wrap"), (T, "U"), (2 * T - 1, "U"), (2 * T, "U-wrap"), (2 * T + 1, "U"), (3 * T - 1, "U-wrap"),
            (3 * T, "U-wrap"), (3 * T + 500, "U")]
    return build("u_at_tile_edges", 3 * T + 1001, 4321, plan, 11,
                 "U chunks as the last chunk of a tile (its sign out comes from the walk) and as the first chunk of the "
                 "next (its sign in is the tile's carry-in), wrapping and not")


def _h_then_low_head():
    T = TILE
    plan = [(T - 1, "H")] + _run(T, 40, "low-") + [(T + 39, "low+"), (T + 40, "U-wrap"), (2 * T - 1, "H")] + \
        _run(2 * T, 3, "low-") + [(2 * T + 2, "low-"), (2 * T + 3, "U")]
    return build("h_then_low_head", 3 * T - 17, 777, plan, 12,
                 "an H chunk ending a tile, then low-W chunks heading the next behind the negative state: the tile waits "
                 "for its predecessor's s2.  The first run turns the sign non-negative partway (s1 = 7); the second keeps "
                 "it negative (s1 = 0) up to a U chunk that does not wrap only because s2 is negative", s1_low={T: 7, 2 * T: 0})


def _low_tiles_behind_negative():
    T = TILE
    plan = [(T - 1, "H")] + [(T + j, "low-") for j in range(2 * T)] + [(3 * T, "U"), (3 * T + 1, "H")]
    return build("low_tiles_behind_negative", 3 * T + 2000, 5000, plan, 13,
                 "a whole tile of low-W chunks behind a negative state (s1 = 0: every chunk keeps it), then a second "
                 "such tile: two tiles in a row wait on the chain, each for the whole of its predecessor; the next tile "
                 "starts with a U chunk that does not wrap only because s2 is negative")


def _low_heads_behind_positive():
    T = TILE
    plan = [(T - 1, "L")] + _run(T, 30, "low+") + [(T + 29, "low+"), (2 * T - 1, "L")] + _run(2 * T, 5, "low+") + \
        [(2 * T + 5, "U")]
    return build("low_heads_behind_positive", 2 * T + 900, 5552, plan, 14,
                 "low-W chunks heading tiles behind a non-negative state (s1 = 11 and 3): the tiles wait, and resolve the "
                 "run as no-wrap chunks", s1_low={T: 11, 2 * T: 3})


def _nchunks(delta):
    def f():
        N = 2 * TILE + delta
        if delta > 0:   # a last tile of one low-W chunk behind a negative state: it waits, and gives the result its sign
            plan, last = [(TILE - 1, "U"), (N - 2, "H"), (N - 1, "low-")], "a low-W chunk behind a negative state"
        else:
            plan, last = [(TILE - 1, "U"), (N - 1, "U-wrap")], "a U chunk"
        return build(f"nchunks_2x16384{delta:+d}", N, 100 + delta, plan, 20 + delta,
                     f"2 * 16384 {delta:+d} chunks, a U chunk last in the first tile, {last} last in the input",
                     s1_low={N - 1: 0})
    return f


def _first(first, plan):
    def f():
        return build(f"first_chunk_{first}", TILE + 7, first, plan, 30 + first,
                     f"a first chunk of {first} bytes (len mod 5552), classes at the start")
    return f


LAYOUTS = {
    "u_at_tile_edges": _u_at_tile_edges,
    "h_then_low_head": _h_then_low_head,
    "low_tiles_behind_negative": _low_tiles_behind_negative,
    "low_heads_behind_positive": _low_heads_behind_positive,
    "nchunks_2x16384-1": _nchunks(-1),
    "nchunks_2x16384+0": _nchunks(0),
    "nchunks_2x16384+1": _nchunks(1),
    "first_chunk_1": _first(1, [(0, "low+"), (1, "U-wrap"), (TILE, "U")]),
    "first_chunk_5551": _first(5551, [(0, "U"), (1, "H")] + _run(2, 3, "low-") + [(TILE - 1, "U-wrap")]),
    "first_chunk_5552": _first(5552, [(0, "U-wrap"), (1, "U"), (TILE - 1, "L")] + _run(TILE, 7, "low+")),
}


def layout(name: str) -> Input:
    """the named layout (2 to 4 tiles), built anew"""
    inp = LAYOUTS[name]()
    assert inp.name == name
    return inp


def chained(ntiles: int, seed: int) -> Input:
    """ntiles tiles (the last one partial) in which every tile but the first starts with low-W chunks behind a negative
    state, followed by a U chunk, and ends with a U chunk and an H chunk: every tile waits on its predecessor, and walks.
    On odd tiles the run keeps s2 negative (s1 = 0) and the U chunk after it does not wrap only because of that; on even
    tiles the run turns the sign partway.  A prefix that ends on a chunk boundary keeps the chunk grid (the first chunk is
    the same) and so every class: prefix(k) is the first k tiles."""
    T = TILE
    plan = []
    for t in range(1, ntiles):
        plan += [(t * T - 2, "U" if t % 2 else "U-wrap"), (t * T - 1, "H")] + _run(t * T, 3 + t, "low-")
        if t % 2:
            plan += [(t * T + 3 + t, "U")]
    return build(f"chained_{ntiles}_{seed}", (ntiles - 1) * T + 333, 2024 + seed, plan, seed,
                 "low-W heads behind a negative state on every tile",
                 s1_low={t * T: 0 if t % 2 else 1 + t for t in range(1, ntiles)})


def prefix(inp: Input, ntiles: int) -> np.ndarray:
    """the input cut after its first ntiles tiles (at most): a prefix on the chunk grid, so with the same classes"""
    first, nchunks = chunk_grid(inp.data.size)
    k = min(nchunks, ntiles * TILE - 7)    # (a partial last tile)
    return inp.data[:first + (k - 1) * CHUNK]
