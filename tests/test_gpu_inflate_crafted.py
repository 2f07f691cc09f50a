"""GPU parity of inflate on hand-built deflate streams (tests/deflate_writer.py) that sit on each acceptance rule of the
reference decoder, just inside and just outside it: code-length codes, run-length coded lengths, HLIT / HDIST / HCLEN
ranges, empty / single / 15-bit codes, 48-bit tokens across the input refills, distances equal to the output so far, stored
blocks at every bit phase, stream ends, and the per-block Adler-32 fold.  Encoders never write most of these shapes.

The expected status, bytes and checksum always come from the oracle.  The small streams go through the one-warp decoder
(host entry point at four output caps, device entry point at odd offsets, zlib framing); large streams built from the same
shapes go through the many-warp decoder (block-start search, speculative chunks, chain check, re-cuts, resolve)."""
import os
import random
import subprocess
import sys
import zlib

import pytest

import deflate_writer as dw
from oracle import zipc_oracle as zo
from test_gpu_device_entry_points import _check_inflate_dev, dev, oracle_inflate  # noqa: F401  (dev: the fixture)
from test_gpu_inflate_spec_plan import decode_pinned
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = dw.all_cases()
CKS = [(_lib.CK_NONE, 0), (_lib.CK_CRC32, 0), (_lib.CK_ADLER32, _lib.ADLER_REF_COMPAT), (_lib.CK_ADLER32, _lib.ADLER_RFC1950)]
CK_IDS = ["none", "crc32", "adler_ref", "adler_rfc"]


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


def _caps(kind, cases):
    exact = [len(c.out) for c in cases]
    return {"exact": exact, "minus1": [max(0, n - 1) for n in exact], "zero": [0] * len(cases), "none": [None] * len(cases)}[kind]


def _assert_like_oracle(cases, caps, res, ck, mode, what):
    for c, cap, (st, out, got) in zip(cases, caps, res):
        est, eout, eck = oracle_inflate(c.stream, cap, ck, mode)
        assert st == est, (what, c.name, cap, st, est)
        if est == _lib.OK:
            assert out.tobytes() == eout, (what, c.name, cap)
            assert got == eck, (what, c.name, cap, hex(got), hex(eck))
            if cap is None or cap >= len(c.out):
                assert eout == c.out, c.name


# ==== one-warp decoder ====================================================================================================
@pytest.mark.parametrize("ck,mode", CKS, ids=CK_IDS)
def test_crafted_streams_host_entry(ctx, monkeypatch, ck, mode):
    """every catalogue stream in one batch, at caps exact, exact - 1, 0 and None (the count-only pass first): SIZE_EXCEEDED
    and CORRUPTED come in the reference's order"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "0")
    streams = [c.stream for c in CASES]
    for kind in ("exact", "minus1", "zero", "none"):
        caps = _caps(kind, CASES)
        _assert_like_oracle(CASES, caps, ctx.inflate_batch(streams, caps, ck, mode), ck, mode, kind)
    # (both sides of every rule are in the batch)
    assert any(c.valid for c in CASES) and any(not c.valid for c in CASES)


@pytest.mark.parametrize("ck,mode", CKS, ids=CK_IDS)
def test_crafted_streams_device_entry(ctx, dev, monkeypatch, ck, mode):  # noqa: F811
    """zipc_b200_inflate_batch_dev: sources at every residue mod 16, slots back to back at odd offsets, caps exact and
    exact + 1; also the host path's (status, length, checksum)"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "0")
    streams = [c.stream for c in CASES]
    for extra in (0, 1):
        caps = [len(c.out) + extra for c in CASES]
        st = _check_inflate_dev(ctx, dev, streams, caps, ck, mode, [(3 * i + extra) % 16 for i in range(len(streams))])
        assert st.count(_lib.OK) == sum(c.valid for c in CASES)


def _zlib_frame(raw, adler):
    return b"\x78\x01" + raw + adler.to_bytes(4, "big")


@pytest.mark.parametrize("mode", [_lib.ADLER_REF_COMPAT, _lib.ADLER_RFC1950], ids=["ref", "rfc"])
def test_crafted_adler_blocks_under_zlib_framing(ctx, monkeypatch, mode):
    """blocks of 0xFF bytes of 0, 1, 5551, 5552, 5553 and 11104 bytes (stored, fixed, dynamic): the reference folds the
    Adler-32 block by block, the first round of each block over len mod 5552 bytes (possibly none).  Each stream carries the
    reference's checksum and RFC 1950's; the status and found checksum are the oracle's (REF_COMPAT) or zlib's (RFC1950)."""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "0")
    cases = [c for c in CASES if c.name.startswith("adler_")]
    items, want = [], []
    for c in cases:
        ref = zo.inflate_and_adler_32(c.stream)[1]
        for trailer in sorted({ref, zlib.adler32(c.out)}):
            z = _zlib_frame(c.stream, trailer)
            items.append(z)
            if mode == _lib.ADLER_REF_COMPAT:
                try:
                    out, found = zo.zlib_decompress(z)
                    want.append((_lib.OK, out, found))
                except zo.OracleError as e:
                    want.append((e.status, None, e.extra.get("found")))
            else:
                found = zlib.adler32(c.out)
                want.append((_lib.OK, c.out, found) if found == trailer else (_lib.ERR_CHECKSUM, None, found))
    assert any(w[0] == _lib.ERR_CHECKSUM for w in want) and any(w[0] == _lib.OK for w in want)
    res = ctx.zlib_decompress_batch(items, None, mode)
    for i, ((st, out, ex, fo), (wst, wout, wfo)) in enumerate(zip(res, want)):
        assert st == wst, (i, st, wst)
        assert fo == wfo, (i, hex(fo), hex(wfo))
        if wst == _lib.OK:
            assert out.tobytes() == wout, i


# ==== many-warp decoder ===================================================================================================
LIT_FULL = dw.complete_lengths(range(286), 286)
DIST_FULL = dw.complete_lengths(range(30), 30)
LIT_CHAIN = dw.chain_lengths(dw.LONG_LIT_SYMS, 286)
DIST_CHAIN = dw.chain_lengths(dw.LONG_DIST_SYMS, 30)
LIT_SHORT = dw.complete_lengths(range(270), 286)          # literal/length 270 .. 285 unused ...
DIST_SHORT = dw.complete_lengths(range(5, 30), 30)        # ... and distance 0 .. 4: one zero run across the boundary
DIST_ONE = [0] * 29 + [1]                                 # a single distance code: symbol 29 (24577 .. 32768)


def _tokens(w, rng, text, units, max_len, dists, lits=None, first=None):
    """a block's tokens: `first` (length, 32768) when the output reaches that far, then units of a few literals and matches
    whose distances reach back into earlier blocks (and, at this block size, across the 4 KiB chunks)"""
    if first and len(w.out) >= 32768:
        w.match(first, 32768)
    for _ in range(units):
        if lits is None:
            at = rng.randrange(len(text) - 64)
            w.literals(text[at:at + rng.randrange(8, 48)])
        else:
            w.literals(bytes(rng.choice(lits) for _ in range(rng.randrange(8, 40))))
        for _ in range(rng.randrange(0, 3) if dists else 0):
            lo, hi = dists
            hi = min(hi, len(w.out))
            if hi >= lo:
                w.match(rng.randrange(3, max_len + 1), rng.randrange(lo, hi + 1))


def _block(w, rng, text, shape, final=False):
    if shape == "full":              # HLIT 286 / HDIST 30
        w.dynamic(final, LIT_FULL, DIST_FULL)
        _tokens(w, rng, text, 300, 258, (1, 32768), first=258)
    elif shape == "chain15":         # literal/length and distance codes of every length up to 15
        w.dynamic(final, LIT_CHAIN, DIST_CHAIN)
        if len(w.out) >= 32768:
            w.match(258, 32768, lsym=284, lextra=31, dsym=29, dextra=8191)
        for _ in range(200):
            w.literals(bytes(rng.choice(b"abcdefghijklmn") for _ in range(rng.randrange(4, 30))))
            d = rng.choice(dw.LONG_DIST_SYMS)
            dist = dw.DIST_BASE[d] + rng.randrange(1 << dw.DIST_EXTRA[d])
            if dist <= len(w.out):
                w.match(227 + rng.randrange(32), dist, lsym=284)
    elif shape == "single_dist":     # one distance code of length 1
        w.dynamic(final, LIT_FULL, DIST_ONE)
        _tokens(w, rng, text, 300, 258, (24577, 32768), first=258)
    elif shape == "literal_only":    # no distance code at all
        w.dynamic(final, LIT_FULL, [0])
        _tokens(w, rng, text, 150, 0, None)
    elif shape == "boundary":        # an 18 across the HLIT / HDIST boundary
        w.dynamic(final, LIT_SHORT, DIST_SHORT)
        _tokens(w, rng, text, 300, 22, (7, 32768), first=22)
    else:
        raise ValueError(shape)
    w.eob()


SHAPES = ("full", "chain15", "single_dist", "literal_only", "boundary")


def _large(seed, out_bytes, insert=None, at=None):
    """a stream of many dynamic blocks of every shape; insert(w) writes an extra block before block `at`.  -> (stream, the
    output so far where the insert begins, writer output)"""
    rng = random.Random(seed)
    text = synth.text_v1(seed, 1 << 20).tobytes()
    w = dw.Writer()
    k, mark = 0, None
    while len(w.out) < out_bytes:
        if k == at:
            mark = len(w.out)
            insert(w)
        _block(w, rng, text, SHAPES[k % len(SHAPES)])
        k += 1
    w.fixed(True)
    w.literals(b"end")
    w.eob()
    return w.finish(), mark, bytes(w.out)


def _decode_like_oracle(ctx, s, caps, ck=_lib.CK_CRC32, mode=0):
    p0 = ctx.parallel_streams
    got = []
    for cap in caps:
        (st, out, c), = ctx.inflate_batch([s], [cap], ck, mode)
        est, eout, eck = oracle_inflate(s, cap, ck, mode)
        assert st == est, (cap, st, est)
        if est == _lib.OK:
            assert out.tobytes() == eout and c == eck, cap
        got.append(st)
    return got, p0, ctx.parallel_streams


def test_large_crafted_stream_many_warps(ctx, monkeypatch):
    """5 MiB of output from dynamic blocks of every shape above: the oracle's bytes and CRC, decoded in parallel"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "20000")
    monkeypatch.setenv("ZIPC_B200_PAR_CHUNK", "4096")
    s, _, want = _large(1, 5 << 20)
    assert zo.inflate(s) == want and len(s) > 40 * 4096
    st, p0, p1 = _decode_like_oracle(ctx, s, [len(want)])
    assert st == [_lib.OK]
    print("large crafted stream: %d bytes -> %d, (parallel, fallback) %s -> %s" % (len(s), len(want), p0, p1))
    assert p1[0] == p0[0] + 1, "the stream was not decoded in parallel"
    st, _, _ = _decode_like_oracle(ctx, s, [None, len(want) - 1], _lib.CK_ADLER32, _lib.ADLER_REF_COMPAT)
    assert st == [_lib.OK, _lib.ERR_SIZE_EXCEEDED]


def _bad_blocks():
    def hlit287(w):
        w.dynamic(False, LIT_FULL + [5], DIST_FULL)
    def oversubscribed(w):
        lit = list(LIT_FULL)
        lit[3] = 1
        w.dynamic(False, lit, DIST_FULL)
    def overrun(w):
        syms = dw.plain_symbols(LIT_FULL + DIST_SHORT[:18]) + [(18, 2)]
        h, cl = dw.clen_code_for(syms)
        w.dynamic_header(False, 286, 30, h, cl, syms)
    def dist_bit1(w):
        w.dynamic(False, LIT_FULL, [0, 0, 0, 1])
        w.sym(270)
        w.bits(0, 2)
        w.bits(1, 1)
    def eob_only_bit1(w):
        w.dynamic(False, [0] * 256 + [1], [0])
        w.bits(1, 1)
    def type3(w):
        w.header(False, 3)
    def no_eob(w):
        lit = dw.complete_lengths([s for s in range(286) if s != 256], 286)
        w.dynamic(False, lit, DIST_FULL)
    return {"hlit_287": hlit287, "lit_oversubscribed": oversubscribed, "rle_overrun": overrun, "dist_single_code_bit_1": dist_bit1,
            "lit_only_end_of_block_bit_1": eob_only_bit1, "block_type_3": type3, "no_end_of_block": no_eob}


@pytest.mark.parametrize("name", sorted(_bad_blocks()))
def test_large_crafted_stream_invalid_block_mid_stream(ctx, monkeypatch, name):
    """an invalid block in the middle of a 2 MiB stream: the oracle's status at caps exact, exact - 1 and None (exact: the
    output up to the invalid block)"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "20000")
    monkeypatch.setenv("ZIPC_B200_PAR_CHUNK", "4096")
    s, mark, _ = _large(2, 2 << 20, _bad_blocks()[name], at=23)
    with pytest.raises(zo.OracleError):
        zo.inflate(s)
    st, _, _ = _decode_like_oracle(ctx, s, [mark, mark - 1, None])
    assert st[0] == _lib.ERR_CORRUPTED and st[2] == _lib.ERR_CORRUPTED


def test_large_stream_match_before_the_start_in_a_later_chunk(ctx, monkeypatch):
    """a 10,000-byte stored block, then a dynamic block whose match reaches 20,000 back: the count pass accepts the stream
    without a cap (each chunk only knows its own output), so resolve has to catch it"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "20000")
    monkeypatch.setenv("ZIPC_B200_PAR_CHUNK", "4096")
    rng = random.Random(3)
    text = synth.text_v1(3, 1 << 20).tobytes()
    w = dw.Writer()
    w.stored(text[:10000])
    w.dynamic(False, LIT_FULL, DIST_FULL)
    w.literals(text[10000:10100])
    w.match(100, 20000)
    w.eob()
    for k in range(30):
        _block(w, rng, text, SHAPES[k % len(SHAPES)])
    w.fixed(True)
    w.eob()
    s = w.finish()
    assert len(s) > 8 * 4096
    with pytest.raises(zo.OracleError):
        zo.inflate(s)
    st, _, _ = _decode_like_oracle(ctx, s, [len(w.out), None])
    assert st == [_lib.ERR_CORRUPTED, _lib.ERR_CORRUPTED]


def test_large_stream_with_stored_deflate_streams_inside(ctx, monkeypatch):
    """stored blocks whose payload is itself a deflate stream (what storing a .gz or .png member gives), between text blocks:
    the block-start search finds valid headers inside the payloads and the re-cut has to recover -- one re-cut per payload,
    so twelve payloads take 13 of the 16 passes (24 of them used the passes up and fell back)"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "20000")
    monkeypatch.setenv("ZIPC_B200_PAR_CHUNK", "4096")
    rng = random.Random(4)
    text = synth.text_v1(4, 1 << 20).tobytes()
    w = dw.Writer()
    for k in range(12):
        _block(w, rng, text, SHAPES[k % len(SHAPES)])
        inner = zlib.compressobj(6, zlib.DEFLATED, -15, 1)
        at = rng.randrange(len(text) - 70000)
        payload = inner.compress(text[at:at + 60000 + k * 500]) + inner.flush()
        w.stored(payload[:65535])
    w.fixed(True)
    w.eob()
    s = w.finish()
    want = zo.inflate(s)
    assert want == bytes(w.out)
    plan = decode_pinned(ctx, s, [len(want), None], ((_lib.CK_CRC32, 0), (_lib.CK_ADLER32, _lib.ADLER_REF_COMPAT)))
    assert plan.outcome == "parallel" and plan.recuts == 12, plan.describe()


def test_sync_flushed_stream_over_the_block_list_falls_back(ctx, monkeypatch):
    """a text stream Z_SYNC_FLUSHed every ~30 bytes in its second half: far more than 256 non-empty blocks in one chunk, with
    Adler-32 (the chunks report the lengths of their blocks for the fold).  The chunk's list overflows, on the re-cut too,
    and the one-warp decoder gives the oracle's output and fold; block_list_256 of tests/par_inflate_inputs.py is a chunk of
    256 blocks that the many-warp decoder takes."""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "20000")
    monkeypatch.setenv("ZIPC_B200_PAR_CHUNK", "16384")
    data = synth.text_v1(5, 3 << 20).tobytes()
    half = len(data) // 2
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    parts = [c.compress(data[:half])]
    for i in range(half, half + 600_000, 30):
        parts.append(c.compress(data[i:i + 30]) + c.flush(zlib.Z_SYNC_FLUSH))
    parts.append(c.compress(data[half + 600_000:]) + c.flush())
    s = b"".join(parts)
    plan = decode_pinned(ctx, s, [len(data), None], ((_lib.CK_ADLER32, _lib.ADLER_REF_COMPAT), (_lib.CK_ADLER32, _lib.ADLER_RFC1950)),
                         chunk=16384)
    assert plan.outcome == "block_list", plan.describe()


# ==== the plan cache of the many-warp decoder ==============================================================================
_PLAN_CACHE_CHILD = r"""
import sys, zlib
sys.path[:0] = [%(root)r]
from oracle import zipc_oracle as zo
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

lanes = %(lanes)d
ctx = zd.Context(0)
text = lambda seed, n: synth.text_v1(seed, n).tobytes()
raw = lambda d: (lambda c: c.compress(d) + c.flush())(zlib.compressobj(6, zlib.DEFLATED, -15))
X = text(11, 6 << 20)
A = text(12, 8 << 20)
ys = {"zeros": text(13, 1 << 20) + bytes(7 << 20), "flip": text(14, 3 << 20)}
bad = 0
for yname, Y in ys.items():
    datas = [X, Y] if lanes == 1 else [A, X, Y]
    names = ["X", "Y"] if lanes == 1 else ["A", "X", "Y"]
    streams = [raw(d) for d in datas]
    if yname == "flip":
        s = bytearray(streams[-1])
        s[2 * len(s) // 3] ^= 0x10
        streams[-1] = bytes(s)
    zs = [zlib.compress(d, 6) for d in datas]
    if yname == "flip":
        zs[-1] = b"\x78\x9c" + streams[-1] + zs[-1][-4:]
    assert len(streams[0]) > len(streams[1]) and (lanes == 1 or len(streams[1]) > len(streams[2]))
    p0 = ctx.parallel_streams
    for name, s, (st, out, crc) in zip(names, streams, ctx.inflate_batch(streams, None, _lib.CK_CRC32)):
        try:
            want = (0,) + zo.inflate_and_crc_32(s)
        except zo.OracleError as e:
            want = (e.status, b"", 0)
        if (st, out.tobytes(), crc) != want:
            bad += 1
            print("inflate_batch lanes=%%d Y=%%s: %%s: status %%d (oracle %%d), %%d bytes (oracle %%d)"
                  %% (lanes, yname, name, st, want[0], len(out), len(want[1])))
    for name, z, (st, out, ex, fo) in zip(names, zs, ctx.zlib_decompress_batch(zs)):
        try:
            wout, wad = zo.zlib_decompress(z)
            want = (0, wout, wad)
        except zo.OracleError as e:
            want = (e.status, b"", e.extra.get("found", 0))
        if (st, out.tobytes() if st == 0 else b"", fo if st in (0, 6) else 0) != (want[0], want[1], want[2] if want[0] in (0, 6) else 0):
            bad += 1
            print("zlib_decompress_batch lanes=%%d Y=%%s: %%s: status %%d (oracle %%d), %%d bytes (oracle %%d)"
                  %% (lanes, yname, name, st, want[0], len(out), len(want[1])))
    print("lanes=%%d Y=%%s: (parallel, fallback) %%s -> %%s" %% (lanes, yname, p0, ctx.parallel_streams))
ctx.close()
sys.exit(1 if bad else 0)
"""


@pytest.mark.parametrize("lanes", [1, 2])
def test_plan_cache_never_serves_another_streams_chunks(lanes):
    """One call with unknown sizes decodes every large stream twice (sizing pass, then real pass), and the speculation plan
    of a stream is kept between the two.  A stream Y whose chain breaks after some accepted chunks (a 4 MB block of zeros
    behind 1 MiB of text, or a bit flip at 2/3) must not leave its chunks under the key of the stream X decoded before it on
    the same context: X would come back OK with Y's bytes.  ZIPC_B200_PAR_LANES is read once per process, hence the child."""
    env = dict(os.environ, ZIPC_B200_PAR_MIN="262144", ZIPC_B200_PAR_LANES=str(lanes))
    env.pop("ZIPC_B200_PAR_CHUNK", None)
    r = subprocess.run([sys.executable, "-c", _PLAN_CACHE_CHILD % {"root": ROOT, "lanes": lanes}], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
