"""Deflate at the block boundaries: the encoder closes a block every 30 tiles of 2048 bytes and at the member's end.  Sizes
k * 61440 + {-1, 0, 1, 2048} make a block end exactly at the member's end, one byte or one tile before it, or leave the
member's last block one byte long; the kernel's bytes must equal the host encoder model's."""
import zlib

import pytest

from oracle import zipc_oracle as zo
import encoder_model as model
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu
BLOCK = 61440


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


def _boundary_corpus():
    t = synth.text_v1(3, 4 * BLOCK + 4096).tobytes()
    return {f"{k}x61440{d:+d}": t[:k * BLOCK + d] for k in range(1, 5) for d in (-1, 0, 1, 2048)}


@pytest.mark.parametrize("level", ["fast", "default", "best"])
def test_block_boundary_sizes_equal_the_model(ctx, level, monkeypatch):
    corpus = _boundary_corpus()
    names = list(corpus)
    monkeypatch.setenv("ZIPC_B200_SPLIT_MIN", str(1 << 40))   # (one CTA per member, as the host model)
    res = ctx.deflate_batch([corpus[k] for k in names], level, _lib.CK_CRC32)
    for k, (st, cs, crc) in zip(names, res):
        data = corpus[k]
        cs = cs.tobytes()
        assert st == 0 and crc == zo.crc32(data), k
        assert zlib.decompress(cs, -15) == data, k
        assert cs == model.deflate(data, level), k


@pytest.mark.parametrize("level", ["fast", "default"])
def test_block_boundary_sizes_in_a_full_batch(ctx, level, monkeypatch):
    """Many members per CTA: a member starts from the state its predecessor left behind on the same CTA."""
    corpus = _boundary_corpus()
    items = [corpus[k] for k in corpus] * 24
    monkeypatch.setenv("ZIPC_B200_SPLIT_MIN", str(1 << 40))
    res = ctx.deflate_batch(items, level, _lib.CK_CRC32)
    want = {k: model.deflate(d, level) for k, d in corpus.items()}
    for d, k, (st, cs, crc) in zip(items, list(corpus) * 24, res):
        assert st == 0 and crc == zlib.crc32(d) and cs.tobytes() == want[k], k


@pytest.mark.parametrize("level", ["fast", "default", "best"])
def test_primed_segments_at_block_boundaries(ctx, level):
    """Primed segments whose first block starts right after the prime and whose sizes put a block end at the segment's
    last tile, one tile before it, or at its very end; the non-final piece keeps BFINAL off."""
    s = synth.text_v1(78, 12 * BLOCK + 5000).tobytes()
    for seg in (BLOCK, BLOCK + 1, BLOCK + 2048, 2 * BLOCK, 2 * BLOCK + 2048):
        primed, index, crc = ctx.deflate_segmented(s, level, seg, primed=True)
        assert crc == zlib.crc32(s)
        assert zlib.decompress(bytes(primed), -15) == s, seg
        assert zo.inflate(bytes(primed)) == s, seg
    piece, _, _ = ctx.deflate_segmented(s[:4 * BLOCK], level, BLOCK + 2048, last_piece=False, primed=True)
    d = zlib.decompressobj(-15)
    assert d.decompress(bytes(piece)) == s[:4 * BLOCK] and not d.eof
