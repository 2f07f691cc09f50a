"""GPU: the many-warp inflate of large streams (DESIGN.md §4.6) held to the plan of tests/par_inflate_model.py as well as to
the oracle's bytes.  Every crafted input of tests/par_inflate_inputs.py goes through inflate_batch (no checksum, CRC-32,
Adler-32 in both flavours; caps exact, exact - 1 and unknown), zlib_decompress_batch and inflate_batch_dev at an odd offset.
Status, bytes and checksum are the oracle's; counters 1 to 4 of the context (parallel, fallback, speculation passes, chunks
resolved) move by exactly what the model predicts, so a stream cannot pass by falling back to the one-warp decoder."""
import os
import subprocess
import sys
import zlib

import pytest

import par_inflate_inputs as pi
import par_inflate_model as pm
from oracle import zipc_oracle as zo
from test_gpu_device_entry_points import _check_inflate_dev, dev, oracle_inflate  # noqa: F401  (dev: the fixture)
from zipc_b200 import _lib
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INPUTS = {i.name: i for i in pi.all_inputs()}
CKS = [(_lib.CK_NONE, 0), (_lib.CK_CRC32, 0), (_lib.CK_ADLER32, _lib.ADLER_REF_COMPAT), (_lib.CK_ADLER32, _lib.ADLER_RFC1950)]


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


@pytest.fixture
def small_chunks(monkeypatch):
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", str(pi.PAR_MIN))
    monkeypatch.setenv("ZIPC_B200_PAR_CHUNK", str(pi.CHUNK))


def _delta(a, b):
    return tuple(y - x for x, y in zip(a, b))


def decode_pinned(ctx, s, caps, cks=((_lib.CK_CRC32, 0),), chunk=pi.CHUNK, par_min=pi.PAR_MIN, plan=None):
    """inflate_batch of the one stream s at every cap and check: the oracle's status, bytes and checksum, and the counters
    moved as the model's plan says (ZIPC_B200_PAR_CHUNK / ZIPC_B200_PAR_MIN must be chunk / par_min).  -> the plan"""
    plan = plan or pm.plan(s, chunk, par_min)
    for ck, mode in cks:
        for cap in caps:
            c0 = ctx.parallel_counters
            (st, out, got), = ctx.inflate_batch([s], [cap], ck, mode)
            moved = _delta(c0, ctx.parallel_counters)
            est, eout, eck = oracle_inflate(s, cap, ck, mode)
            assert st == est, (cap, ck, mode, st, est)
            if est == _lib.OK:
                assert out.tobytes() == eout and got == eck, (cap, ck, mode)
            want = pm.calls(plan, cap).tuple()
            assert moved == want, "cap %s ck %d/%d: counters moved %s, the model says %s (%s)" % (
                cap, ck, mode, moved, want, plan.describe())
    return plan


def _size(i):
    return len(pm.walk(i.stream).out)


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_crafted_input_host_entry(ctx, small_chunks, name):
    i = INPUTS[name]
    n = _size(i)
    plan = decode_pinned(ctx, i.stream, [n, n - 1, None], CKS)
    print("%s: %s" % (name, plan.describe()))


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_crafted_input_zlib_framing(ctx, small_chunks, name):
    """the stream with its zlib framing, the reference's Adler-32 in the trailer: the body the decoder gets runs two bytes into
    the trailer (zipc_deflate.ml:732), and the plan is the model's over that body"""
    i = INPUTS[name]
    try:
        trailer = zo.inflate_and_adler_32(i.stream)[1]
    except zo.OracleError:
        trailer = zlib.adler32(b"")
    z = b"\x78\x01" + i.stream + trailer.to_bytes(4, "big")
    plan = pm.plan(z[2:-2], pi.CHUNK, pi.PAR_MIN)
    try:
        wout, wad = zo.zlib_decompress(z)
        want = (_lib.OK, wout, wad)
    except zo.OracleError as e:
        want = (e.status, None, e.extra.get("found"))
    c0 = ctx.parallel_counters
    (st, out, ex, fo), = ctx.zlib_decompress_batch([z])
    assert _delta(c0, ctx.parallel_counters) == pm.calls(plan, None).tuple(), plan.describe()
    assert st == want[0], (st, want[0])
    if st == _lib.OK:
        assert out.tobytes() == want[1] and fo == want[2]


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_crafted_input_device_entry(ctx, dev, small_chunks, name):  # noqa: F811
    """inflate_batch_dev: the source at an odd offset, the slot at an odd offset between canaries, caps exact and exact - 1"""
    i = INPUTS[name]
    plan = pm.plan(i.stream, pi.CHUNK, pi.PAR_MIN)
    n = _size(i)
    for ck, mode in CKS[1:3]:
        for cap in (n, n - 1):
            c0 = ctx.parallel_counters
            _check_inflate_dev(ctx, dev, [i.stream], [cap], ck, mode, [3], host=False)
            assert _delta(c0, ctx.parallel_counters) == pm.calls(plan, cap).tuple(), (cap, plan.describe())


_LANES_CHILD = r"""
import sys
sys.path[:0] = [%(root)r, %(tests)r]
import par_inflate_inputs as pi, par_inflate_model as pm
from test_gpu_device_entry_points import oracle_inflate
from zipc_b200 import _lib
from zipc_b200 import zipc_deflate as zd

ctx = zd.Context(0)
ins = [pi.recuts(2, high=True), pi.block_list(257), pi.chunk_count(33)]
plans = [pm.plan(i.stream, pi.CHUNK, pi.PAR_MIN) for i in ins]
bad = 0
for caps in ([len(i.out) for i in ins], [None] * len(ins)):
    for ck, mode in ((_lib.CK_CRC32, 0), (_lib.CK_ADLER32, _lib.ADLER_REF_COMPAT)):
        c0 = ctx.parallel_counters
        res = ctx.inflate_batch([i.stream for i in ins], caps, ck, mode)
        moved = tuple(b - a for a, b in zip(c0, ctx.parallel_counters))
        want = tuple(map(sum, zip(*(pm.calls(p, c).tuple() for p, c in zip(plans, caps)))))
        if moved != want:
            bad += 1
            print("caps %%s ck %%d: counters moved %%s, the model says %%s" %% (caps, ck, moved, want))
        for i, cap, (st, out, got) in zip(ins, caps, res):
            est, eout, eck = oracle_inflate(i.stream, cap, ck, mode)
            if (st, out.tobytes() if st == 0 else b"", got if st == 0 else 0) != (est, eout, eck if est == 0 else 0):
                bad += 1
                print("%%s: status %%d (oracle %%d)" %% (i.name, st, est))
ctx.close()
sys.exit(1 if bad else 0)
"""


def test_crafted_inputs_on_three_lanes():
    """three crafted streams in one batch on three lanes (host threads with a sub-context each): the counters are summed over
    the lanes, and each lane keeps its stream's plan from the sizing pass to the real pass.  ZIPC_B200_PAR_LANES is read once
    per process, hence the child."""
    env = dict(os.environ, ZIPC_B200_PAR_MIN=str(pi.PAR_MIN), ZIPC_B200_PAR_CHUNK=str(pi.CHUNK), ZIPC_B200_PAR_LANES="3")
    r = subprocess.run([sys.executable, "-c", _LANES_CHILD % {"root": ROOT, "tests": os.path.join(ROOT, "tests")}], env=env,
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
