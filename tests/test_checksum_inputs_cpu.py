"""The generator's guarantee for test_gpu_checksum_edges.py: every layout of checksum_inputs reaches the chunk classes of its
plan at their planned indices, and the chunk model it is built on is the reference's Adler-32 (zo.adler32) bit for bit, and
zlib.adler32 in RFC 1950 arithmetic.  Without this the GPU tests of those layouts prove nothing.  No GPU."""
import zlib
from collections import Counter

import numpy as np
import pytest

import checksum_inputs as ci
from oracle import zipc_oracle as zo


@pytest.mark.parametrize("name", list(ci.LAYOUTS))
def test_layout_reaches_its_plan(name):
    inp = ci.layout(name)
    b = inp.data.tobytes()
    got, classes = ci.model(inp.data)
    assert inp.missed(classes) == [], f"{name}: planned (index, class, found) not reached"
    assert 2 <= -(-inp.nchunks // ci.TILE) <= 5
    assert got == zo.adler32(b)
    assert ci.model_rfc1950(inp.data) == zlib.adler32(b)
    # the layouts differ from the reference's RFC 1950 word where they should: every one has wrapping chunks
    assert Counter(classes)["H"] + Counter(classes)["U-wrap"] > 0 and got != zlib.adler32(b)
    print(name, inp.nchunks, "chunks:", dict(Counter(classes)), "| plan of", len(inp.plan), "reached")


def test_chained_input_and_its_prefixes():
    inp = ci.chained(4, 1)
    _, classes = ci.model(inp.data)
    assert inp.missed(classes) == []
    for k in (1, 2, 3, 4):
        p = ci.prefix(inp, k)
        got, pc = ci.model(p)
        assert got == zo.adler32(p.tobytes())
        assert pc == classes[:len(pc)], k                       # same grid, same classes
        assert -(-len(pc) // ci.TILE) == k


def test_model_on_random_and_crafted_data():
    rng = np.random.default_rng(3)
    cases = [b"", b"\x00", b"\xff", bytes(5551), b"\xff" * 5552, b"\xff" * 5553, bytes(range(256)) * 1000,
             b"\x80" * 300_000, b"\x81" * 300_001, b"\x7f" * 299_999]
    cases += [rng.bytes(int(n)) for n in rng.integers(1, 200_000, 40)]
    cases += [rng.integers(120, 140, int(n), dtype=np.uint8).tobytes() for n in rng.integers(5552, 400_000, 20)]
    seen = Counter()
    for d in cases:
        got, classes = ci.model(d)
        seen.update(classes)
        assert got == zo.adler32(d), len(d)
        assert ci.model_rfc1950(d) == zlib.adler32(d), len(d)
    assert set(seen) >= {"L", "H", "low+", "U"}, seen      # (the layouts reach the others on purpose)


def test_recipes_hit_the_wrap_boundary_exactly():
    """a U chunk aimed at W = 2^31 - s2 (slack 0) wraps, one aimed at 2^31 - s2 - 1 does not: the two sides of the boundary"""
    inp = ci.build("edge", 40, 5552, [(3, "U-wrap"), (4, "U"), (5, "H"), (6, "U-wrap"), (7, "U")], 5, wrap_slack=0)
    n, A, B = ci.chunk_sums(inp.data)
    s1, s2 = 1, 0
    for c in range(8):
        W = int(n[c]) * s1 + int(B[c])
        if c in (3, 6):
            assert s2 + W == 1 << 31
        if c in (4, 7):
            assert s2 + W == (1 << 31) - 1
        s1, s2, _ = ci.step(s1, s2, int(n[c]), int(A[c]), int(B[c]))
    got, classes = ci.model(inp.data)
    assert inp.missed(classes) == [] and got == zo.adler32(inp.data.tobytes())
