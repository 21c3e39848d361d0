"""ctypes binding of libzsgpu.so -- the C ABI declared in include/zsgpu.h.

This is the Python counterpart of the Node-API addon described in INTEGRATION.md: pure
marshalling, no compute.  There is NO CPU fallback: if the shared library is missing or no CUDA
device is usable, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libzsgpu.so")

# status codes (src/mod/common/constants.ts:21-29)
Z_OK, Z_STREAM_END, Z_NEED_DICT = 0, 1, 2
Z_ERRNO, Z_STREAM_ERROR, Z_DATA_ERROR, Z_MEM_ERROR, Z_BUF_ERROR, Z_VERSION_ERROR = -1, -2, -3, -4, -5, -6
ZS_E_CUDA = -100
# flush values (src/mod/common/constants.ts:13-19)
Z_NO_FLUSH, Z_PARTIAL_FLUSH, Z_SYNC_FLUSH, Z_FULL_FLUSH, Z_FINISH, Z_BLOCK = 0, 1, 2, 3, 4, 5
WRAP_RAW, WRAP_ZLIB, WRAP_GZIP = 0, 1, 2
MODE_INDEPENDENT, MODE_STITCHED = 0, 1
FLAG_PRIME, FLAG_NOT_FIRST, FLAG_NOT_LAST, FLAG_SYNC = 1, 2, 4, 8
KIND_ADLER32, KIND_CRC32 = 0, 1


class DeflateResult(C.Structure):
    _fields_ = [("total_out_bytes", C.c_uint64), ("total_out_bits", C.c_uint64), ("check", C.c_uint32),
                ("n_blocks", C.c_uint32)]


class ZStream(C.Structure):
    """zs_stream: the Stream carrier of src/mod/common/types.ts:1-15."""
    _fields_ = [("next_in", C.c_void_p), ("avail_in", C.c_uint64), ("total_in", C.c_uint64),
                ("next_out", C.c_void_p), ("avail_out", C.c_uint64), ("total_out", C.c_uint64),
                ("msg", C.c_char_p), ("adler", C.c_uint32), ("data_type", C.c_int32), ("state", C.c_void_p)]


class ZsError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ""):
        super().__init__(f"{where} failed with {code}" + (f": {detail}" if detail else ""))
        self.code = code


_PROTOTYPES = {
    "zs_version": (C.c_char_p, []),
    "zs_ctx_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "zs_ctx_destroy": (None, [C.c_void_p]),
    "zs_last_error": (C.c_char_p, [C.c_void_p]),
    "zs_ctx_synchronize": (C.c_int, [C.c_void_p]),
    "zs_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
    "zs_ctx_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "zs_ctx_profile_read": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint64]),
    "zs_deflate_bound": (C.c_uint64, [C.c_uint64, C.c_int]),
    "zs_deflate_batch_bound": (C.c_uint64, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int]),
    "zs_crc32_combine": (C.c_uint32, [C.c_uint32, C.c_uint32, C.c_uint64]),
    "zs_adler32_combine": (C.c_uint32, [C.c_uint32, C.c_uint32, C.c_uint64]),
    "zs_checksum_batch_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "zs_checksum_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32)]),
    "zs_checksum": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32)]),
    "zs_deflate_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32,
                                       C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p,
                                       C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_deflate_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int,
                                   C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.POINTER(DeflateResult)]),
    "zs_deflate_part": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_uint32,
                                  C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(DeflateResult)]),
    "zs_deflate_dict_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "zs_deflate_dict_id": (C.c_uint32, [C.c_void_p]),
    "zs_deflate_dict_destroy": (None, [C.c_void_p]),
    "zs_deflate_batch_dict_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32,
                                            C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_uint64,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_deflate_batch_dict": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32,
                                        C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.POINTER(DeflateResult)]),
    "zs_bit_concat_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]),
    "zs_huffman_blocks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_inflate_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "zs_inflate_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_uint64]),
    "zs_inflate_stream_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "zs_inflate_message": (C.c_char_p, [C.c_int]),
    "zs_inflate_last_details": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "zs_stream_deflate_init": (C.c_int, [C.c_void_p, C.POINTER(ZStream), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "zs_stream_deflate_set_dictionary": (C.c_int, [C.POINTER(ZStream), C.c_void_p, C.c_uint32]),
    "zs_stream_deflate": (C.c_int, [C.POINTER(ZStream), C.c_int]),
    "zs_stream_deflate_end": (C.c_int, [C.POINTER(ZStream)]),
    "zs_stream_deflate_reset": (C.c_int, [C.POINTER(ZStream)]),
    "zs_stream_deflate_params": (C.c_int, [C.POINTER(ZStream), C.c_int, C.c_int]),
    "zs_stream_deflate_pending": (C.c_int, [C.POINTER(ZStream), C.POINTER(C.c_uint32), C.POINTER(C.c_int)]),
    "zs_stream_deflate_set_header": (C.c_int, [C.POINTER(ZStream), C.c_void_p]),
    "zs_stream_inflate_get_header": (C.c_int, [C.POINTER(ZStream), C.c_void_p]),
    "zs_stream_inflate_init": (C.c_int, [C.c_void_p, C.POINTER(ZStream), C.c_int]),
    "zs_stream_inflate_set_dictionary": (C.c_int, [C.POINTER(ZStream), C.c_void_p, C.c_uint32]),
    "zs_stream_inflate": (C.c_int, [C.POINTER(ZStream), C.c_int]),
    "zs_stream_inflate_reset": (C.c_int, [C.POINTER(ZStream)]),
    "zs_stream_inflate_reset2": (C.c_int, [C.POINTER(ZStream), C.c_int]),
    "zs_stream_inflate_end": (C.c_int, [C.POINTER(ZStream)]),
}

class GzHeader(C.Structure):
    """zs_gz_header of include/zsgpu.h"""
    _fields_ = [("text", C.c_int32), ("time", C.c_uint32), ("xflags", C.c_int32), ("os", C.c_int32),
                ("extra", C.c_void_p), ("extra_max", C.c_uint32), ("extra_len", C.c_uint32),
                ("name", C.c_void_p), ("name_max", C.c_uint32), ("comment", C.c_void_p), ("comm_max", C.c_uint32),
                ("hcrc", C.c_int32), ("done", C.c_int32)]


EXPORTED_SYMBOLS = tuple(_PROTOTYPES)

_lib = None


def load() -> C.CDLL:
    """Load libzsgpu.so.  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
                "(nvcc, sm_100a).  zlib-streams-ts_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class Context:
    """zs_ctx: one engine context per CUDA device / stream."""

    def __init__(self, device: int = 0, cuda_stream: int | None = None):
        self._lib = load()
        h = C.c_void_p()
        rc = self._lib.zs_ctx_create(device, C.c_void_p(cuda_stream) if cuda_stream else None, C.byref(h))
        if rc != Z_OK:
            raise ZsError(rc, "zs_ctx_create", "no usable CUDA device (zsgpu has no CPU fallback)")
        self._h = h
        self.device = device

    @property
    def handle(self):
        return self._h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.zs_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def last_error(self) -> str:
        return (self._lib.zs_last_error(self._h) or b"").decode()

    def check(self, rc: int, where: str):
        if rc != Z_OK:
            raise ZsError(rc, where, self.last_error())

    def synchronize(self):
        self.check(self._lib.zs_ctx_synchronize(self._h), "zs_ctx_synchronize")

    @property
    def launch_count(self) -> int:
        return int(self._lib.zs_ctx_launch_count(self._h))

    def profile(self, enable: bool):
        self.check(self._lib.zs_ctx_profile(self._h, 1 if enable else 0), "zs_ctx_profile")

    def profile_read(self) -> dict:
        """{kernel name: (launches, total device ms)} since the last read (synchronises)."""
        buf = C.create_string_buffer(1 << 14)
        self.check(self._lib.zs_ctx_profile_read(self._h, buf, len(buf)), "zs_ctx_profile_read")
        out = {}
        for line in buf.value.decode().splitlines():
            name, n, ms = line.rsplit(" ", 2)
            out[name] = (int(n), float(ms))
        return out
