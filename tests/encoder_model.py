"""Loader of the host-side encoder model (tools/deflate_model.cc): test scaffolding that drives the
same __host__ __device__ building blocks as the CUDA encoder, serially."""
import ctypes as C
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SO = os.path.join(ROOT, "tools", "libdeflate_model.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(ROOT, "tools", "deflate_model.cc")
        core = os.path.join(ROOT, "zipc_b200", "csrc", "deflate_core.h")
        if not os.path.exists(_SO) or max(os.path.getmtime(src), os.path.getmtime(core)) > os.path.getmtime(_SO):
            subprocess.run([os.path.join(ROOT, "tools", "build_model.sh")], check=True)
        L = C.CDLL(_SO)
        L.zipc_model_deflate.argtypes = [C.c_int, C.c_char_p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        L.zipc_model_deflate_ex.argtypes = [C.c_int, C.c_char_p, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(C.c_void_p),
                                            C.POINTER(C.c_uint64)]
        L.zipc_model_huff_lengths.argtypes = [C.POINTER(C.c_uint32), C.c_int, C.c_int, C.POINTER(C.c_uint8)]
        L.zipc_model_huff_lengths.restype = None
        _lib = L
    return _lib


LEVELS = {"fast": 1, "default": 2, "best": 3}


def deflate(data: bytes, level: str) -> bytes:
    o, n = C.c_void_p(), C.c_uint64()
    lib().zipc_model_deflate(LEVELS[level], data, len(data), C.byref(o), C.byref(n))
    out = C.string_at(o.value, n.value)
    lib().zipc_model_free(o)
    return out


def deflate_segment(data: bytes, level: str, prime: int = 0, not_final: bool = False) -> bytes:
    """One segment of a larger stream: data[:prime] is the input right before it (a multiple of 2048 bytes), only seen by
    the segment's matches; the segment is data[prime:].  not_final: BFINAL off, then an empty stored block."""
    o, n = C.c_void_p(), C.c_uint64()
    if lib().zipc_model_deflate_ex(LEVELS[level], data, len(data), prime, int(not_final), C.byref(o), C.byref(n)):
        raise ValueError(f"bad prime {prime} for a segment of {len(data) - prime} bytes")
    out = C.string_at(o.value, n.value)
    lib().zipc_model_free(o)
    return out


def primed_segments(data: bytes, level: str, starts, last_final: bool = True) -> bytes:
    """The concatenation of the segments [starts[k], starts[k + 1]) of data, each primed with the whole tiles of the (at most
    32 KiB of) input before it, as the split members and zipc_b200_deflate_primed cut them."""
    out = []
    for k in range(len(starts) - 1):
        a, b = starts[k], starts[k + 1]
        prime = min(a, 32768) // 2048 * 2048
        out.append(deflate_segment(data[a - prime:b], level, prime, k + 2 < len(starts) or not last_final))
    return b"".join(out)


def huff_lengths(freq, max_bits: int) -> list:
    """The encoder's code length builder (huff_lengths_from_sorted) over freq, limited to max_bits."""
    n = len(freq)
    f = (C.c_uint32 * n)(*freq)
    out = (C.c_uint8 * n)()
    lib().zipc_model_huff_lengths(f, n, max_bits, out)
    return list(out)
