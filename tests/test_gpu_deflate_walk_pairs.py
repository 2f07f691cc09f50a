"""The kernel's chain walks against the host model, byte for byte, on inputs aimed at each rule of the walk
(tests/walk_pairs.py): more than 12 same-hash positions in a tile, chains crossing a tile boundary after 0 to 12 candidates
inside it, stale 16-bit heads, candidates at 32768 and 32769, hash collisions, the nice stop, ties, max_len clipping at the
end of a member, a primed segment and one-tile / empty-tail members.  All three levels; one CTA per member and many."""
import zlib

import pytest

import encoder_model as model
import walk_pairs as wp
from zipc_b200 import _lib
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu
LEVELS = ("fast", "default", "best")


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


@pytest.mark.parametrize("level", LEVELS)
def test_walk_inputs_equal_the_model(ctx, level, monkeypatch):
    inputs = wp.walk_inputs()
    names = [k for k, (_, prime) in inputs.items() if prime == 0]
    items = [inputs[k][0] for k in names]
    want = [model.deflate(d, level) for d in items]
    monkeypatch.setenv("ZIPC_B200_SPLIT_MIN", "0")      # one CTA per member, as the host model
    for batch in (items, items * 6):                     # alone, and after other members in the same CTA
        res = ctx.deflate_batch(batch, level, _lib.CK_CRC32)
        for i, (d, (st, cs, crc)) in enumerate(zip(batch, res)):
            cs = cs.tobytes()
            assert st == 0 and crc == zlib.crc32(d), names[i % len(names)]
            assert cs == want[i % len(names)], names[i % len(names)]
            assert zlib.decompress(cs, -15) == d


@pytest.mark.parametrize("level", LEVELS)
def test_primed_walk_input_equals_the_model(ctx, level):
    d, prime = wp.walk_inputs()["primed"]
    out, index, _ = ctx.deflate_segmented(d, level, prime, primed=True)
    starts = [int(x) for x in index[:, 1]]
    assert starts == [0, prime, len(d)]
    assert out.tobytes() == model.primed_segments(d, level, starts)
    assert zlib.decompress(out.tobytes(), -15) == d
