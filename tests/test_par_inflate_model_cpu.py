"""The plan model of the many-warp inflate (tests/par_inflate_model.py) and the crafted large streams
(tests/par_inflate_inputs.py), without a GPU: the block walker against the writer and the oracle, the finder against the
true block starts of writer-made streams, and every crafted input against the plan it was built to reach."""
import random

import pytest

import deflate_writer as dw
import par_inflate_inputs as pi
import par_inflate_model as pm
from oracle import zipc_oracle as zo

INPUTS = {i.name: i for i in pi.all_inputs()}


def _writer_stream(seed):
    """dynamic blocks of 8 .. 300 coded literal/length symbols, stored, fixed and empty blocks, headers noted as written"""
    rng = random.Random(seed)
    w = dw.Writer()
    heads = []
    for k in range(60):
        kind = rng.choice("ddddsfe")
        heads.append((w.nbits, kind))
        if kind == "s":
            w.stored(bytes(rng.randrange(256) for _ in range(rng.randrange(0, 300))))
            continue
        if kind == "f":
            w.fixed()
        else:
            ncoded = rng.choice([8, 11, 12, 13, 40, 200, 258]) if kind == "d" else 12
            syms = sorted(rng.sample(range(256), ncoded - 2)) + [256, 284]
            w.dynamic(False, dw.complete_lengths(syms, 286), dw.complete_lengths(range(30), 30))
        if kind != "e":
            for _ in range(rng.randrange(20, 400)):
                if rng.random() < 0.1 and len(w.out) > 300:
                    w.match(230 + rng.randrange(20), rng.randrange(1, min(len(w.out), 32768) + 1), lsym=284)
                else:
                    w.literal(rng.choice(syms[:-2]) if kind == "d" else rng.randrange(256))
        w.eob()
    heads.append((w.nbits, "final"))
    w.fixed(True)
    w.eob()
    return w.finish(), bytes(w.out), heads


@pytest.mark.parametrize("seed", range(4))
def test_walker_and_finder_on_writer_streams(seed):
    s, out, heads = _writer_stream(seed)
    w = pm.walk(s)
    assert w.error is None and w.out == out == zo.inflate(s)
    assert [b.start for b in w.blocks] == [h for h, _ in heads]
    assert [b.end for b in w.blocks[:-1]] == [h for h, _ in heads[1:]]
    assert [b.btype for b in w.blocks] == [{"s": 0, "f": 1, "final": 1}.get(k, 2) for _, k in heads]
    # the finder finds every non-final dynamic header with 12 coded symbols or more, and nothing else
    truth = []
    for b in w.blocks:
        if b.btype == 2 and not b.final and 8 * len(s) - b.start >= pm.FIND_TAIL:
            _, lit, _ = pm.read_dynamic_header(pm.Bits(s), b.start + 3)
            if sum(1 for x in lit if x) >= 12:
                truth.append(b.start)
    assert list(pm.valid_starts(s)) == truth
    assert any(sum(1 for x in pm.read_dynamic_header(pm.Bits(s), b.start + 3)[1] if x) == 11
               for b in w.blocks if b.btype == 2)   # (the substance rule is met on both sides)


def test_walker_stops_at_the_first_error():
    s, out, heads = _writer_stream(9)
    bad = bytearray(s)
    at = heads[30][0] // 8 + 2
    bad[at] ^= 0xFF
    w = pm.walk(bytes(bad))
    with pytest.raises(zo.OracleError):
        zo.inflate(bytes(bad), len(out))
    assert w.error is not None and w.error_bit <= 8 * at + 8 and w.out == out[:len(w.out)]


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_crafted_input_reaches_its_plan(name):
    i = INPUTS[name]
    w = pm.walk(i.stream)
    p = pm.plan(i.stream, pi.CHUNK, pi.PAR_MIN, w)
    print("%s (%s): %s" % (name, i.what, p.describe()))
    assert len(i.stream) >= pi.PAR_MIN
    if p.outcome == "match_before_start":
        with pytest.raises(zo.OracleError):
            zo.inflate(i.stream)
    else:
        assert w.out == i.out == zo.inflate(i.stream)
    assert i.intent(p, w) is None, "%s drifted: %s; the plan is %s" % (name, i.intent(p, w), p.describe())


def test_the_adler_quirk_input_differs_from_rfc1950():
    import zlib
    i = INPUTS["recuts_2_adler_quirk"]
    assert zo.inflate_and_adler_32(i.stream)[1] != zlib.adler32(i.out)


def test_counter_rules():
    """what one call moves the counters by, per outcome"""
    par = pm.Plan("parallel", [pm.Pass(0, [0, 9], [pm.Chunk(0, 9, 5, 1), pm.Chunk(9, 20, 5, 1)], "final")], 10)
    assert pm.calls(par, 10).tuple() == (1, 0, 1, 2)
    assert pm.calls(par, 9).tuple() == (0, 1, 1, 0)
    assert pm.calls(par, None).tuple() == (2, 0, 1, 2)        # the real pass takes the sizing pass's plan
    far = pm.Plan("match_before_start", par.passes, 10)
    assert pm.calls(far, 10).tuple() == (0, 1, 1, 2)
    assert pm.calls(far, None).tuple() == (1, 1, 1, 2)
    fb = pm.Plan("block_list", [pm.Pass(0, [0, 9], [], "failed block_list")])
    assert pm.calls(fb, None).tuple() == (0, 2, 2, 0)
    assert pm.calls(pm.Plan("not_tried", tried=False), None).tuple() == (0, 0, 0, 0)
