"""The kernel's deflate streams through the independent checker (tests/deflate_checker.py), on inputs built to reach each rule
of the encoder (tests/deflate_inputs.py): byte equality with the host model, one CTA per member and many members per CTA;
primed and plain segments against the model's segment entry; members split over CTAs by the public calls, segment by
segment, with the zlib trailer folded over the checker's blocks; and the device-resident entry point."""
import ctypes as C
import random
import zlib

import numpy as np
import pytest

import deflate_checker as dc
import deflate_inputs as di
import encoder_model as model
from oracle import zipc_oracle as zo
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu
LEVELS = ("fast", "default", "best")
BLOCK = 61440


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


@pytest.fixture(scope="module")
def corpus():
    return di.corpus()


_want = {}


def _model(data, level):
    key = (level, len(data), zlib.crc32(data))
    if key not in _want:
        _want[key] = model.deflate(data, level)
    return _want[key]


def _primes(starts):
    return [min(a, 32768) // 2048 * 2048 for a in starts]


@pytest.mark.parametrize("level", LEVELS)
def test_kernel_equals_model_and_passes_the_checker(ctx, corpus, level, monkeypatch):
    names = list(corpus)
    items = [corpus[k].data for k in names]
    monkeypatch.setenv("ZIPC_B200_SPLIT_MIN", "0")      # one CTA per member, as the host model
    res = ctx.deflate_batch(items, level, _lib.CK_CRC32)
    for k, d, (st, cs, crc) in zip(names, items, res):
        cs = cs.tobytes()
        assert st == 0 and crc == zlib.crc32(d), k
        assert cs == _model(d, level), k
        r = dc.check(cs, d)
        assert corpus[k].reached(d, r), (k, corpus[k].target)
    # many members per CTA: each starts from the shared-memory state the previous one left
    full = items * 8
    res = ctx.deflate_batch(full, level, _lib.CK_CRC32)
    for i, (d, (st, cs, crc)) in enumerate(zip(full, res)):
        assert st == 0 and crc == zlib.crc32(d) and cs.tobytes() == _model(d, level), (names[i % len(names)], i)


@pytest.mark.parametrize("level", LEVELS)
def test_primed_and_plain_segments_equal_the_model(ctx, level):
    s = (di._filler(random.Random(3), 200_000) + synth.text_v1(79, 200_000).tobytes() + synth.rand_v1(80, 30_000).tobytes()
         + di.fibonacci_lengths())
    pc = di.primed_corpus()
    for seg in (64 << 10, (96 << 10) + 1000, BLOCK + 1, 2 * BLOCK + 2048):
        primed, index, crc = ctx.deflate_segmented(s, level, seg, primed=True)
        starts = [int(x) for x in index[:, 1]]
        assert starts == list(range(0, len(s), seg)) + [len(s)]
        primed = primed.tobytes()
        assert primed == model.primed_segments(s, level, starts), seg
        dc.check(primed, s, _primes(starts[:-1]))
        plain, index, _ = ctx.deflate_segmented(s, level, seg, primed=False)
        want = b"".join(model.deflate_segment(s[a:b], level, 0, b < len(s)) for a, b in zip(starts, starts[1:]))
        assert plain.tobytes() == want, seg
    for name, inp in pc.items():
        primed, index, _ = ctx.deflate_segmented(inp.data, level, 64 << 10, primed=True)
        starts = [int(x) for x in index[:, 1]]
        primed = primed.tobytes()
        assert primed == model.primed_segments(inp.data, level, starts), name
        assert inp.reached(inp.data, dc.check(primed, inp.data, _primes(starts[:-1]))), name


def _split_members(corpus):
    """members over 320 KiB (split in a thin batch) holding the window-edge and collision inputs"""
    t = synth.text_v1(81, 600_000).tobytes()
    return [corpus["window_32768"].data + t[:300_000] + corpus["collisions"].data + corpus["window_32769"].data,
            t[:200_000] + corpus["stale_heads"].data + corpus["fib_distances"].data + t[200_000:400_000],
            (np.frombuffer(t, dtype=np.uint8) | 0x80).tobytes()]


def _check_split(cs, d, level):
    """the checker cuts the stream at its empty stored blocks; each segment equals the model's primed segment"""
    r = dc.check(cs, d, [0] + [32768] * 64)
    starts = [x[0] for x in r.segments] + [len(d)]
    assert len(starts) > 2
    assert r.segments[0][0] == 0
    want = model.primed_segments(d, level, starts)
    assert cs == want
    return r


@pytest.mark.parametrize("level", ["fast", "default"])
def test_split_members_through_the_public_calls(ctx, corpus, level):
    items = _split_members(corpus)
    res = ctx.deflate_batch(items, level, _lib.CK_CRC32)
    for d, (st, cs, crc) in zip(items, res):
        assert st == 0 and crc == zlib.crc32(d)
        _check_split(cs.tobytes(), d, level)
    res = ctx.zlib_compress_batch(items, level, _lib.ADLER_REF_COMPAT)
    for d, (st, zs, ad) in zip(items, res):
        zs = zs.tobytes()
        assert st == 0 and int.from_bytes(zs[-4:], "big") == ad
        r = _check_split(zs[2:-4], d, level)
        a = 1
        for b in r.blocks:    # the reference's Adler-32, folded block by block as its decoder sees them
            a = zo.adler32_update(a, d[b.src_start:b.src_start + b.src_len])
        assert a == ad


def test_device_entry_point_through_the_checker(ctx, corpus):
    """zipc_b200_deflate_batch_dev writes the same checked streams as the host call"""
    names = ["literal_only", "fib_lengths", "window_32768", "overhang", "deferred", "lazy_chain", "tiny3", "bfloat16"]
    items = [corpus[k].data for k in names]
    offs, pos = [], 64
    for d in items:
        offs.append(pos)
        pos += len(d) + 5
    src = np.zeros(pos + 64, dtype=np.uint8)
    for o, d in zip(offs, items):
        src[o:o + len(d)] = np.frombuffer(d, dtype=np.uint8)
    caps = [ctx.L.zipc_b200_deflate_bound(len(d)) for d in items]
    doffs, pos = [], 64
    for cap in caps:            # output slots must start 4-byte aligned
        doffs.append(pos)
        pos += (cap + 3) // 4 * 4
    dsize = pos + 64
    ps, pd = C.c_void_p(), C.c_void_p()
    ctx._check(ctx.L.zipc_b200_dev_alloc(ctx.h, src.size, C.byref(ps)), "dev_alloc")
    ctx._check(ctx.L.zipc_b200_dev_alloc(ctx.h, dsize, C.byref(pd)), "dev_alloc")
    try:
        ctx._check(ctx.L.zipc_b200_memcpy_h2d(ctx.h, ps.value, src.ctypes.data, src.size), "memcpy_h2d")
        n = len(items)
        sz = lambda v: (C.c_size_t * n)(*[int(x) for x in v])
        dl, cs, st = (C.c_size_t * n)(), (C.c_uint32 * n)(), (C.c_int * n)()
        for level in LEVELS:
            rc = ctx.L.zipc_b200_deflate_batch_dev(ctx.h, zd.LEVELS[level], _lib.CK_CRC32, _lib.ADLER_REF_COMPAT, n, ps.value,
                                                   sz(offs), sz([len(d) for d in items]), pd.value, sz(doffs), sz(caps),
                                                   dl, cs, st)
            assert rc == _lib.OK
            out = np.empty(dsize, dtype=np.uint8)
            ctx._check(ctx.L.zipc_b200_memcpy_d2h(ctx.h, out.ctypes.data, pd.value, dsize), "memcpy_d2h")
            for i, (k, d) in enumerate(zip(names, items)):
                got = out[doffs[i]:doffs[i] + dl[i]].tobytes()
                assert st[i] == 0 and cs[i] == zlib.crc32(d), k
                assert got == _model(d, level), (k, level)
                assert corpus[k].reached(d, dc.check(got, d)), (k, level)
    finally:
        ctx.L.zipc_b200_dev_free(ctx.h, ps.value)
        ctx.L.zipc_b200_dev_free(ctx.h, pd.value)
