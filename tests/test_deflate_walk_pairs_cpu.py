"""The walk of levels fast and default as the kernel runs it (list the candidates, compare all of them, one max over keys)
gives every position the (len, dist, resume token) of the serial match_step walk: plain-Python restatements of both
(tests/walk_pairs.py) on inputs aimed at each rule of the walk and on C4-shaped text members.  Every input is also held to
the rule it is meant to reach."""
import numpy as np
import pytest

import deflate_inputs as di
import walk_pairs as wp
from zipc_b200 import synth

INPUTS = wp.walk_inputs()


@pytest.mark.parametrize("level", ["fast", "default"])
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_pair_walk_equals_serial_walk(name, level):
    d, prime = INPUTS[name]
    serial = wp.walks(d, level, wp.serial_walk, prime)
    assert wp.walks(d, level, wp.pair_walk, prime) == serial
    assert all(p >= prime for p in serial)


@pytest.mark.parametrize("level", ["fast", "default"])
def test_pair_walk_equals_serial_walk_on_text_members(level):
    sizes = synth.member_sizes(40, seed=3)            # the bench's C4 member sizes; the smallest few, whole
    for i, n in enumerate(sorted(int(x) for x in sizes)[:3]):
        d = synth.text_v1(1000 + i, n).tobytes()
        assert wp.walks(d, level, wp.pair_walk) == wp.walks(d, level, wp.serial_walk), (i, n)


def _details(name, level="default"):
    d, prime = INPUTS[name]
    return d, prime, wp.walk_details(d, level, prime), wp.walks(d, level, wp.serial_walk, prime)


def test_inputs_reach_their_rules():
    d = INPUTS["same_hash_runs"][0]
    h = [wp.hash4(d, p) for p in range(len(d) - 3)]
    assert any(max(np.unique(h[t:t + wp.TILE], return_counts=True)[1]) > 12 for t in range(0, len(h), wp.TILE))

    d, _, det, _ = _details("tile_crossings")
    inside = set()
    for p, cands in det.items():
        ts = p // wp.TILE * wp.TILE
        k = sum(p - x >= ts for x, _ in cands)
        if len(cands) > k or k == 12:                 # k candidates inside the tile, then the chain goes on below it
            inside.add(k)
    assert set(range(13)) <= inside

    assert di._stale_reached(INPUTS["stale_heads"][0], None)

    _, _, _, res = _details("window_32768")
    assert any(dist == 32768 and n >= 4 for n, dist, _ in res.values())
    d, _, det, res = _details("window_32769")
    assert all(x <= 32768 for c in det.values() for x, _ in c)
    assert 5000 + 32769 in res and res[5000 + 32769][0] == 0    # the second copy of the chunk: out of reach, no match

    _, _, det, _ = _details("collisions")
    assert any(n < 4 for c in det.values() for _, n in c)

    for level, nice in (("fast", 32), ("default", 128)):
        _, _, det, res = _details("nice_stop", level)
        assert any(res[p][0] >= nice and any(n > res[p][0] for _, n in c) for p, c in det.items()), level

    _, _, det, res = _details("ties")
    tied = [p for p, c in det.items() if len(c) > 1 and max(n for _, n in c) >= 4 and
            sum(n == max(m for _, m in c) for _, n in c) > 1]
    assert tied and all(res[p][1] == next(x for x, n in det[p] if n == res[p][0]) for p in tied)

    d, _, _, res = _details("tail_clip")
    assert any(4 <= n == len(d) - p < 258 for p, (n, _, _) in res.items())

    d, prime, _, res = _details("primed")
    assert min(res) == prime and any(dist == 32768 and p - dist < prime for p, (_, dist, _) in res.items())

    for level, steps in (("fast", 4), ("default", 12)):   # walks that ran out of budget leave their last candidate
        _, _, det, res = _details("same_hash_runs", level)
        assert any(len(c) == steps and res[p][2] != p & 0xFFFF for p, c in det.items())
