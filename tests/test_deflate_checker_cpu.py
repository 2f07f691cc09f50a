"""The deflate checker (tests/deflate_checker.py) on the CPU: it flags streams that break one of the encoder's rules, each with
its own error; it passes the host model's streams for every input built to reach an encoder rule (tests/deflate_inputs.py),
whole and as primed segments; every such input reaches its rule; and the encoder's code length builder, driven directly, is
complete, within its limit, optimal where a Huffman code fits and never below the optimum length-limited code."""
import random
import zlib

import pytest

import deflate_checker as dc
import deflate_inputs as di
import deflate_writer as dw
import encoder_model as model

LEVELS = ("fast", "default", "best")


@pytest.fixture(scope="module")
def corpus():
    return di.corpus()


# ---- defective streams ----------------------------------------------------------------------------------------------
def _skewed(n=3000, seed=4):
    return di.no_repeat(n, 20, random.Random(seed), [1.0 / (1 + i) for i in range(20)])


def _dynamic(data, final=True, hlit=None, ll=None, rle=None, w=None):
    """a literal-only dynamic block of data as the encoder builds it, with the given parts replaced"""
    fl = [0] * dc.NUM_LIT
    for b in data:
        fl[b] += 1
    fl[256] += 1
    ell, edl, ehlit, ehdist, _, _, _, _ = dc._expected_header(fl, [0] * dc.NUM_DIST)
    ll = ell if ll is None else ll
    hlit = ehlit if hlit is None else hlit
    rle = dc.greedy_rle(ll[:hlit] + edl[:ehdist]) if rle is None else rle
    cf = [0] * dc.NUM_CLEN
    for s, _ in rle:
        cf[s] += 1
    cl = dc.encoder_lengths(cf, 7)
    hclen = max(4, max(i + 1 for i in range(dc.NUM_CLEN) if cl[dc.CLEN_ORDER[i]]))
    w = w or dw.Writer()
    w.dynamic_header(final, hlit, ehdist, hclen, [cl[dc.CLEN_ORDER[i]] for i in range(hclen)], rle)
    w.use(ll[:hlit], edl[:ehdist])
    w.literals(data)
    w.eob()
    return w


def _flags(rule, stream, data, valid=True, **kw):
    if valid:   # the stream itself is valid deflate
        assert zlib.decompressobj(-15).decompress(stream) == data
    with pytest.raises(dc.CheckError) as e:
        dc.check(stream, data, **kw)
    assert e.value.rule == rule, e.value


def test_the_checker_passes_a_stream_built_by_the_rules():
    data = _skewed()
    r = dc.check(_dynamic(data).finish(), data)
    (b,) = r.blocks
    assert b.type == "dynamic" and b.hdist == 1 and b.costs["dynamic"] < min(b.costs["fixed"], b.costs["stored"])


def test_fixed_where_dynamic_is_cheaper_is_flagged():
    data = _skewed()
    w = dw.Writer()
    w.fixed(True)
    w.literals(data)
    w.eob()
    _flags("block_type", w.finish(), data)


def test_untrimmed_hlit_is_flagged():
    _flags("hlit", _dynamic(_skewed(), hlit=286).finish(), _skewed())


def test_non_greedy_rle_is_flagged():
    data = _skewed()
    fl = [0] * dc.NUM_LIT
    for b in data:
        fl[b] += 1
    fl[256] += 1
    ll = dc.encoder_lengths(fl, 15)
    # the same lengths spelled one by one, no 16 / 17 / 18
    _flags("rle", _dynamic(data, rle=dw.plain_symbols(ll[:257] + [0])).finish(), data)


def _lengths(data):
    fl = [0] * dc.NUM_LIT
    for b in data:
        fl[b] += 1
    fl[256] += 1
    return fl, dc.encoder_lengths(fl, 15)


def test_suboptimal_lengths_are_flagged():
    data = _skewed()
    fl, ll = _lengths(data)
    used = sorted((f, s) for s, f in enumerate(fl) if f)
    lo, hi = used[0][1], used[-1][1]
    ll = list(ll)
    ll[lo], ll[hi] = ll[hi], ll[lo]     # still complete, but the most frequent symbol gets the longest code
    _flags("suboptimal", _dynamic(data, ll=ll).finish(), data)


def test_incomplete_lengths_are_flagged():
    data = _skewed()
    fl, ll = _lengths(data)
    ll = list(ll)
    ll[max((f, s) for s, f in enumerate(fl) if f)[1]] += 1   # Kraft sum below 1
    _flags("incomplete", _dynamic(data, ll=ll).finish(), data, valid=False)   # (zlib refuses an incomplete code)


def test_a_three_byte_match_is_flagged():
    data = b"abcdxyzabc" + b"q"
    w = dw.Writer()
    w.fixed(True)
    w.literals(b"abcdxyz")
    w.match(3, 7)
    w.literal(ord("q"))
    w.eob()
    _flags("match_length", w.finish(), data)


def test_a_distance_past_the_prime_is_flagged():
    rnd = random.Random(3)
    data = bytes(rnd.randrange(256) for _ in range(4096))
    data += data[-3000:-2900] + b"end"
    w = dw.Writer()
    w.stored(data[:4096])
    w.stored(b"")                           # end of segment 0
    w.fixed(True)
    w.match(100, 3000)
    w.literals(b"end")
    w.eob()
    s = w.finish()
    _flags("reach", s, data, primes=[0, 2048])
    dc.check(s, data, primes=[0, 4096])        # with a prime that covers it, the same distance is fine


def test_bfinal_on_a_non_final_piece_is_flagged():
    data = _skewed()
    _flags("bfinal", _dynamic(data, final=True).finish(), data, final=False)
    # the same piece without BFINAL and with its closing empty stored block passes
    w = _dynamic(data, final=False)
    w.stored(b"")
    dc.check(w.finish(), data, final=False)


def test_nonzero_pad_bits_are_flagged():
    data = _skewed()
    w = _dynamic(data)
    assert w.nacc
    w.pad_byte(1)
    _flags("pad", w.finish(), data)


# ---- the model's streams pass, and every input reaches its rule -----------------------------------------------------
@pytest.mark.parametrize("level", LEVELS)
def test_the_model_passes_the_checker_and_every_input_reaches_its_rule(corpus, level):
    for name, inp in corpus.items():
        cs = model.deflate(inp.data, level)
        r = dc.check(cs, inp.data)
        assert inp.reached(inp.data, r), (name, inp.target)


@pytest.mark.parametrize("level", LEVELS)
def test_the_model_passes_the_checker_as_primed_and_plain_segments(level):
    s = di._filler(random.Random(8), 150_000) + bytes(random.Random(9).randbytes(100_000)) + di.fibonacci_lengths()
    for seg in (64 << 10, (96 << 10) + 1000, 61441, 2 * 61440 + 2048):
        starts = list(range(0, len(s), seg)) + [len(s)]
        primes = [min(a, 32768) // 2048 * 2048 for a in starts[:-1]]
        cs = model.primed_segments(s, level, starts)
        r = dc.check(cs, s, primes)
        assert [x[0] for x in r.segments] == starts[:-1]
        with pytest.raises(dc.CheckError) as e:     # the primes are used: without them a match reaches too far
            dc.check(cs, s)
        assert e.value.rule == "reach"
        # not primed: every segment on its own, the last one a non-final piece
        plain = b"".join(model.deflate_segment(s[a:b], level, 0, True) for a, b in zip(starts, starts[1:]))
        dc.check(plain, s, final=False)
    for name, inp in di.primed_corpus().items():
        starts = list(range(0, len(inp.data), 64 << 10)) + [len(inp.data)]
        r = dc.check(model.primed_segments(inp.data, level, starts), inp.data,
                     [min(a, 32768) // 2048 * 2048 for a in starts[:-1]])
        assert inp.reached(inp.data, r), (name, inp.target)


def test_the_model_entry_for_segments_keeps_whole_members_unchanged():
    for data in (b"", b"a", b"hellohello", di._filler(random.Random(1), 70000)):
        for level in LEVELS:
            assert model.deflate_segment(data, level) == model.deflate(data, level)
    with pytest.raises(ValueError):
        model.deflate_segment(bytes(5000), "fast", 1000)     # a prime is whole tiles


# ---- the shared builder, driven directly --------------------------------------------------------------------------------
def _vectors(nsym, cap, count, seed):
    rnd = random.Random(seed)
    fib = [1, 1]
    while fib[-1] < cap:
        fib.append(fib[-1] + fib[-2])
    for i in range(count):
        k = rnd.randrange(2, nsym + 1)
        syms = rnd.sample(range(nsym), k)
        f = [0] * nsym
        kind = i % 3
        for j, s in enumerate(syms):
            if kind == 0:
                f[s] = rnd.randrange(1, max(2, cap // k))
            elif kind == 1:
                f[s] = fib[min(j, len(fib) - 1)] * rnd.randrange(1, 3)
            else:
                f[s] = max(1, int(cap * rnd.uniform(0.3, 0.9) ** j))
        total = sum(f)
        if total > cap:
            f = [x * cap // total + (1 if x else 0) for x in f]
        yield f


def test_the_builder_against_package_merge():
    """huff_lengths_from_sorted (zipc_model_huff_lengths) on 4500 seeded random, Fibonacci and geometric frequency vectors at
    the caps a block can reach: always a complete code within the limit, exactly the restated builder's lengths, the Huffman
    optimum whenever a Huffman code fits, never below package-merge.  Worst excess over package-merge on these vectors:
    literal/length 0.98 % (1534 bits), distance none, code-length 7.27 % (67 bits)."""
    worst = {}
    for nsym, limit, cap, seed in ((286, 15, 61698, 1), (30, 15, 15360, 2), (19, 7, 316, 3)):
        for f in _vectors(nsym, cap, 1500, seed):
            lens = model.huff_lengths(f, limit)
            assert lens == dc.encoder_lengths(f, limit)
            assert max(lens) <= limit and all(bool(a) == bool(b) for a, b in zip(f, lens))
            assert dc.kraft_ok(lens)
            cost = sum(a * b for a, b in zip(f, lens))
            hc, hd = dc.huffman_cost_depth(f)
            if hd <= limit:
                assert cost == hc, f
            pm = dc.package_merge_cost(f, limit)
            assert cost >= pm
            if cost > pm:
                gap = (cost - pm) / pm
                if gap > worst.get(nsym, (0, 0))[0]:
                    worst[nsym] = (gap, cost - pm)
    print("worst gap over package-merge by alphabet size:", {k: (f"{100 * g:.2f} %", b) for k, (g, b) in worst.items()})
