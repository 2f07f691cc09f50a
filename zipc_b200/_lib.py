"""ctypes binding of libzipc_b200.so (the C ABI in include/zipc_b200.h).

The shared library is the product; this module only declares its signatures.  It is loaded from
inside the package directory (built in-tree by `make -C zipc_b200/csrc` or __graft_entry__.build()).
Importing never falls back to another implementation: a missing library raises ImportError.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ZIPC_B200_LIB: A/B testing of alternative builds of the same library (tuning only)
LIB_PATH = os.environ.get("ZIPC_B200_LIB") or os.path.join(_HERE, "libzipc_b200.so")

# status codes (include/zipc_b200.h)
OK, ERR_CORRUPTED, ERR_SIZE_EXCEEDED, ERR_ZLIB_METHOD, ERR_ZLIB_WINDOW, ERR_ZLIB_DICT = 0, 1, 2, 3, 4, 5
ERR_CHECKSUM, ERR_NOMEM, ERR_INVALID_ARG, ERR_CUDA, ERR_NO_DEVICE, ERR_DST_TOO_SMALL = 6, 7, 8, 9, 10, 11
ERR_ZIP_ENCRYPTED, ERR_ZIP_FORMAT = 31, 32
CK_NONE, CK_ADLER32, CK_CRC32 = 0, 1, 2
LEVEL_NONE, LEVEL_FAST, LEVEL_DEFAULT, LEVEL_BEST = 0, 1, 2, 3
ADLER_REF_COMPAT, ADLER_RFC1950 = 0, 1
SIZE_UNKNOWN = C.c_size_t(-1).value

EXPORTS = [
    "zipc_b200_version", "zipc_b200_strerror", "zipc_b200_device_count", "zipc_b200_ctx_create",
    "zipc_b200_ctx_destroy", "zipc_b200_last_error", "zipc_b200_ctx_stream", "zipc_b200_ctx_launches", "zipc_b200_ctx_counter",
    "zipc_b200_ctx_profile", "zipc_b200_ctx_kernel_ms",
    "zipc_b200_host_alloc", "zipc_b200_host_free", "zipc_b200_dev_alloc", "zipc_b200_dev_free",
    "zipc_b200_memcpy_h2d", "zipc_b200_memcpy_d2h", "zipc_b200_sync",
    "zipc_b200_crc32", "zipc_b200_crc32_dev", "zipc_b200_crc32_dev_async", "zipc_b200_adler32",
    "zipc_b200_adler32_dev", "zipc_b200_crc32_batch", "zipc_b200_crc32_combine", "zipc_b200_adler32_combine",
    "zipc_b200_inflate_batch", "zipc_b200_fetch", "zipc_b200_inflate_batch_dev", "zipc_b200_zlib_decompress_batch",
    "zipc_b200_deflate_batch", "zipc_b200_deflate_batch_dev", "zipc_b200_deflate_bound",
    "zipc_b200_zlib_compress_batch", "zipc_b200_zlib_decompress_batch_dev", "zipc_b200_zlib_compress_batch_dev",
    "zipc_b200_zlib_bound", "zipc_b200_deflate_segmented", "zipc_b200_deflate_primed", "zipc_b200_inflate_segmented", "zipc_b200_ptime_to_dos", "zipc_b200_ptime_of_dos", "zipc_b200_zip_parse",
    "zipc_b200_zip_encoding_size", "zipc_b200_zip_assemble", "zipc_b200_zip_extract_batch",
    "zipc_b200_zip_parse_ex", "zipc_b200_zip_encoding_size_ex", "zipc_b200_zip_assemble_ex", "zipc_b200_inflate_plan", "zipc_b200_zip_deflate_archive_ex",
    "zipc_b200_zip_deflate_archive", "zipc_b200_zip_parse_dev", "zipc_b200_zip_extract_batch_dev", "zipc_b200_free", "zipc_b200_synth_text", "zipc_b200_synth_rand",
    "zipc_b200_mctx_create", "zipc_b200_mctx_destroy", "zipc_b200_mctx_device_count", "zipc_b200_mctx_ctx",
    "zipc_b200_mctx_last_error", "zipc_b200_multi_crc32", "zipc_b200_multi_inflate_batch",
    "zipc_b200_multi_deflate_batch", "zipc_b200_multi_fetch",
]


class Member(C.Structure):
    """zipc_b200_member"""
    _fields_ = [("path", C.c_void_p), ("path_len", C.c_uint32), ("is_dir", C.c_int32), ("mode", C.c_int32),
                ("mtime", C.c_int64), ("version_made_by", C.c_int32), ("version_needed", C.c_int32),
                ("gp_flags", C.c_int32), ("compression", C.c_int32), ("compressed_bytes", C.c_void_p),
                ("start", C.c_uint64), ("compressed_size", C.c_uint64), ("decompressed_size", C.c_uint64),
                ("crc32", C.c_uint32), ("_pad", C.c_uint32)]


def _declare(L):
    vp, sz, u32, i32, u64 = C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, C.c_uint64
    P = C.POINTER
    szp, u32p, ip, vpp = P(sz), P(u32), P(i32), P(vp)
    sig = {
        "zipc_b200_version": (C.c_char_p, []),
        "zipc_b200_strerror": (C.c_char_p, [i32]),
        "zipc_b200_device_count": (i32, []),
        "zipc_b200_ctx_create": (i32, [i32, vpp]),
        "zipc_b200_ctx_destroy": (None, [vp]),
        "zipc_b200_last_error": (C.c_char_p, [vp]),
        "zipc_b200_ctx_stream": (vp, [vp]),
        "zipc_b200_ctx_launches": (u64, [vp]),
        "zipc_b200_ctx_counter": (u64, [vp, i32]),
        "zipc_b200_ctx_profile": (None, [vp, i32]),
        "zipc_b200_ctx_kernel_ms": (C.c_float, [vp]),
        "zipc_b200_host_alloc": (i32, [sz, vpp]),
        "zipc_b200_host_free": (None, [vp]),
        "zipc_b200_dev_alloc": (i32, [vp, sz, vpp]),
        "zipc_b200_dev_free": (None, [vp, vp]),
        "zipc_b200_memcpy_h2d": (i32, [vp, vp, vp, sz]),
        "zipc_b200_memcpy_d2h": (i32, [vp, vp, vp, sz]),
        "zipc_b200_sync": (i32, [vp]),
        "zipc_b200_crc32": (i32, [vp, vp, sz, u32p]),
        "zipc_b200_crc32_dev": (i32, [vp, vp, sz, u32p]),
        "zipc_b200_crc32_dev_async": (i32, [vp, vp, sz, vp]),
        "zipc_b200_adler32": (i32, [vp, vp, sz, i32, u32p]),
        "zipc_b200_adler32_dev": (i32, [vp, vp, sz, i32, u32p]),
        "zipc_b200_crc32_batch": (i32, [vp, sz, vpp, szp, u32p]),
        "zipc_b200_crc32_combine": (u32, [u32, u32, u64]),
        "zipc_b200_adler32_combine": (u32, [u32, u32, u64]),
        "zipc_b200_inflate_batch": (i32, [vp, i32, i32, sz, vpp, szp, szp, vp, sz, szp, szp, szp, u32p, ip]),
        "zipc_b200_fetch": (i32, [vp, vp, sz]),
        "zipc_b200_inflate_batch_dev": (i32, [vp, i32, i32, sz, vp, szp, szp, vp, szp, szp, szp, u32p, ip]),
        "zipc_b200_zlib_decompress_batch": (i32, [vp, i32, sz, vpp, szp, szp, vp, sz, szp, szp, szp, u32p, u32p, ip]),
        "zipc_b200_deflate_batch": (i32, [vp, i32, i32, i32, sz, vpp, szp, vp, sz, szp, szp, szp, u32p, ip]),
        "zipc_b200_deflate_batch_dev": (i32, [vp, i32, i32, i32, sz, vp, szp, szp, vp, szp, szp, szp, u32p, ip]),
        "zipc_b200_deflate_bound": (sz, [sz]),
        "zipc_b200_zlib_compress_batch": (i32, [vp, i32, i32, sz, vpp, szp, vp, sz, szp, szp, szp, u32p, ip]),
        "zipc_b200_zlib_decompress_batch_dev": (i32, [vp, i32, sz, vp, szp, szp, vp, szp, szp, szp, u32p, u32p, ip]),
        "zipc_b200_zlib_compress_batch_dev": (i32, [vp, i32, i32, sz, vp, szp, szp, vp, szp, szp, szp, u32p, ip]),
        "zipc_b200_zlib_bound": (sz, [sz]),
        "zipc_b200_deflate_segmented": (i32, [vp, i32, vp, sz, sz, i32, vp, sz, szp, P(u64), sz, szp, u32p]),
        "zipc_b200_deflate_primed": (i32, [vp, i32, vp, sz, sz, i32, vp, sz, szp, P(u64), sz, szp, u32p]),
        "zipc_b200_inflate_segmented": (i32, [vp, vp, sz, P(u64), sz, vp, sz, szp, u32p, ip]),
        "zipc_b200_ptime_to_dos": (None, [C.c_int64, ip, ip]),
        "zipc_b200_ptime_of_dos": (C.c_int64, [i32, i32]),
        "zipc_b200_zip_parse": (i32, [vp, sz, P(P(Member)), szp]),
        "zipc_b200_zip_encoding_size": (u64, [P(Member), sz]),
        "zipc_b200_zip_assemble": (i32, [P(Member), sz, C.c_char_p, vp, sz, szp]),
        "zipc_b200_inflate_plan": (None, [sz, szp, sz, C.c_char_p]),
        "zipc_b200_zip_parse_ex": (i32, [vp, sz, C.c_uint, P(P(Member)), szp]),
        "zipc_b200_zip_encoding_size_ex": (u64, [P(Member), sz, C.c_char_p, C.c_uint]),
        "zipc_b200_zip_assemble_ex": (i32, [P(Member), sz, C.c_char_p, C.c_uint, vp, sz, szp]),
        "zipc_b200_zip_extract_batch": (i32, [vp, P(Member), sz, vp, sz, szp, szp, szp, u32p, ip]),
        "zipc_b200_zip_deflate_archive": (i32, [vp, i32, sz, vpp, u32p, vpp, szp, P(C.c_int32), P(C.c_int64),
                                                C.c_char_p, vp, sz, szp]),
        "zipc_b200_zip_deflate_archive_ex": (i32, [vp, i32, sz, vpp, u32p, vpp, szp, P(C.c_int32), P(C.c_int64),
                                                   C.c_char_p, C.c_uint, vp, sz, szp]),
        "zipc_b200_zip_parse_dev": (i32, [vp, vp, sz, C.c_uint, P(P(Member)), szp]),
        "zipc_b200_zip_extract_batch_dev": (i32, [vp, P(Member), sz, vp, szp, szp, u32p, ip]),
        "zipc_b200_free": (None, [vp]),
        "zipc_b200_synth_text": (None, [u64, vp, sz]),
        "zipc_b200_synth_rand": (None, [u64, vp, sz]),
        "zipc_b200_mctx_create": (i32, [u64, vpp]),
        "zipc_b200_mctx_destroy": (None, [vp]),
        "zipc_b200_mctx_device_count": (i32, [vp]),
        "zipc_b200_mctx_ctx": (vp, [vp, i32]),
        "zipc_b200_mctx_last_error": (C.c_char_p, [vp]),
        "zipc_b200_multi_crc32": (i32, [vp, vp, sz, u32p]),
        "zipc_b200_multi_inflate_batch": (i32, [vp, i32, i32, sz, vpp, szp, szp, vp, sz, szp, szp, szp, u32p, ip]),
        "zipc_b200_multi_deflate_batch": (i32, [vp, i32, i32, i32, sz, vpp, szp, vp, sz, szp, szp, szp, u32p, ip]),
        "zipc_b200_multi_fetch": (i32, [vp, vp, sz]),
    }
    assert set(sig) == set(EXPORTS)
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError if the library does not export it
        fn.restype, fn.argtypes = res, args
    return L


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C zipc_b200/csrc` (or "
                "__graft_entry__.build()).  zipc_b200 has no CPU fallback.")
        _lib = _declare(C.CDLL(LIB_PATH))
    return _lib
