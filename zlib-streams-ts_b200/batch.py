"""Batch / chunked entry points: deflateBatch / inflateBatch / checksums.

These are the new entry points the north star adds next to the reference API (they have no
reference analogue; the results they must reproduce are those of deflate()/inflate() of
src/mod/deflate/deflate.ts:716 and src/mod/inflate/inflate.ts:332 applied per chunk / per stream).
PyTorch is used only for device memory and streams; all compute is in libzsgpu.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import capi
from .capi import (FLAG_NOT_FIRST, FLAG_NOT_LAST, FLAG_PRIME, FLAG_SYNC, MODE_INDEPENDENT, MODE_STITCHED,  # noqa: F401
                   WRAP_GZIP, WRAP_RAW, WRAP_ZLIB, Context, DeflateResult)

_contexts: dict = {}


def default_context(device: int | None = None) -> Context:
    """One context per device, bound to torch's current stream on that device."""
    if not torch.cuda.is_available():
        raise capi.ZsError(capi.ZS_E_CUDA, "default_context", "CUDA is not available and zsgpu has no CPU fallback")
    if device is None:
        device = torch.cuda.current_device()
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    ctx = _contexts.get(key)
    if ctx is None:
        # torch's default stream has handle 0; the C ABI reads NULL as "make your own stream", so
        # name the legacy default stream explicitly (cudaStreamLegacy == (cudaStream_t)1)
        ctx = Context(device, key[1] if key[1] else 1)
        _contexts[key] = ctx
    return ctx


def _ptr(t) -> C.c_void_p:
    if t is None:
        return None
    if t.numel() == 0:
        # torch reports a null data_ptr() for an empty view; the engine still needs the position of the
        # view inside its storage (the history of an empty part of a sharded stream lies before it)
        base = t.untyped_storage().data_ptr()
        return C.c_void_p(base + t.storage_offset() * t.element_size() if base else 0)
    return C.c_void_p(t.data_ptr())


def _as_u8(data) -> np.ndarray:
    if isinstance(data, np.ndarray):
        return np.ascontiguousarray(data.view(np.uint8).reshape(-1))
    return np.frombuffer(bytes(data) if not isinstance(data, (bytes, bytearray, memoryview)) else data, dtype=np.uint8)


def n_chunks_for(n: int, chunk_size: int) -> int:
    return max(1, -(-n // chunk_size))


@dataclass
class DeflateBatchDev:
    out: torch.Tensor        # uint8, capacity
    out_off: torch.Tensor    # uint64 as int64 [n+1]: byte offsets (INDEPENDENT) / bit offsets (STITCHED)
    out_bits: torch.Tensor   # int64 [n]
    checks: torch.Tensor | None
    result: torch.Tensor     # 24 raw bytes of zs_deflate_result (device)

    def read_result(self) -> DeflateResult:
        raw = self.result.cpu().numpy().tobytes()
        return DeflateResult.from_buffer_copy(raw)


class DeflateDictionary:
    """A preset dictionary prepared once for batch deflate (zs_deflate_dict_create): the device copy of its last
    32 KiB and the match finder's tables built from them.  `dict_id` is the DICTID a zlib stream made with it
    carries: adler32 of the whole dictionary.  Close it (or let it be collected) before its context goes."""

    def __init__(self, data, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        src = _as_u8(data)
        h = C.c_void_p()
        self._lib = capi.load()
        rc = self._lib.zs_deflate_dict_create(self.ctx.handle, src.ctypes.data if src.size else None, src.size, C.byref(h))
        self.ctx.check(rc, "zs_deflate_dict_create")
        self._h = h
        self.dict_id = int(self._lib.zs_deflate_dict_id(h))
        self.size = int(src.size)

    @property
    def handle(self):
        if not self._h:
            raise ValueError("DeflateDictionary is closed")
        return self._h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.zs_deflate_dict_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def deflate_batch_dev(d_in: torch.Tensor, chunk_size: int, level: int = 6, wrap: int = WRAP_RAW,
                      mode: int = MODE_INDEPENDENT, flags: int = 0, history: int = 0, in_off: torch.Tensor | None = None,
                      max_chunk: int | None = None, out: torch.Tensor | None = None, want_checks: bool = False,
                      ctx: Context | None = None, reuse: DeflateBatchDev | None = None,
                      dictionary: DeflateDictionary | None = None) -> DeflateBatchDev:
    """Enqueue one batch deflate on device-resident input (no synchronisation).

    `d_in` may be a view whose first `history` preceding bytes (same storage) are valid history.
    With `dictionary` every chunk is an independent stream that starts from it (zs_deflate_batch_dict_dev):
    mode must be INDEPENDENT, history 0, and flags the strategy alone; a zlib stream then carries FDICT + DICTID.
    """
    assert d_in.is_cuda and d_in.dtype == torch.uint8 and d_in.is_contiguous()
    ctx = ctx or default_context(d_in.device.index)
    n = d_in.numel()
    if in_off is None:
        n_chunks = n_chunks_for(n, chunk_size)
        mc = chunk_size
    else:
        n_chunks = in_off.numel() - 1
        mc = max_chunk if max_chunk is not None else int((in_off[1:] - in_off[:-1]).max().item())
    dev = d_in.device
    if reuse is not None:
        out, out_off, out_bits, checks, result = reuse.out, reuse.out_off, reuse.out_bits, reuse.checks, reuse.result
    else:
        if out is None:
            cap = int(capi.load().zs_deflate_batch_bound(n, n_chunks, mc, wrap, mode))
            if dictionary is not None:
                cap += 4 * n_chunks   # DICTID
            out = torch.empty(cap, dtype=torch.uint8, device=dev)
        out_off = torch.empty(n_chunks + 1, dtype=torch.int64, device=dev)
        out_bits = torch.empty(n_chunks, dtype=torch.int64, device=dev)
        checks = torch.empty(n_chunks, dtype=torch.int32, device=dev) if (want_checks or wrap != WRAP_RAW) else None
        result = torch.zeros(24, dtype=torch.uint8, device=dev)
    if dictionary is not None:
        if mode != MODE_INDEPENDENT or history:
            raise ValueError("a dictionary call is INDEPENDENT and takes no history")
        rc = capi.load().zs_deflate_batch_dict_dev(ctx.handle, dictionary.handle, _ptr(d_in), n, _ptr(in_off), n_chunks,
                                                   chunk_size, mc, level, wrap, flags, _ptr(out), out.numel(),
                                                   _ptr(out_off), _ptr(out_bits), _ptr(checks), _ptr(result))
        ctx.check(rc, "zs_deflate_batch_dict_dev")
        return DeflateBatchDev(out, out_off, out_bits, checks, result)
    rc = capi.load().zs_deflate_batch_dev(ctx.handle, _ptr(d_in), n, _ptr(in_off), n_chunks, chunk_size, mc, history,
                                          level, wrap, mode, flags, _ptr(out), out.numel(), _ptr(out_off),
                                          _ptr(out_bits), _ptr(checks), _ptr(result))
    ctx.check(rc, "zs_deflate_batch_dev")
    return DeflateBatchDev(out, out_off, out_bits, checks, result)


@dataclass
class DeflateBatchHost:
    data: bytes
    out_off: np.ndarray
    out_bits: np.ndarray
    checks: np.ndarray
    total_out_bytes: int
    total_out_bits: int
    check: int
    n_blocks: int

    def stream(self, i: int) -> bytes:
        """INDEPENDENT mode: the i-th complete stream."""
        return self.data[int(self.out_off[i]): int(self.out_off[i + 1])]


def deflate_batch(data, chunk_size: int = 65536, level: int = 6, wrap: int = WRAP_RAW, mode: int = MODE_INDEPENDENT,
                  flags: int = 0, in_off=None, ctx: Context | None = None,
                  dictionary: DeflateDictionary | None = None) -> DeflateBatchHost:
    """Host-buffer deflateBatch through zs_deflate_batch (H2D + kernels + D2H inside the call).

    With `dictionary`: zs_deflate_batch_dict, every chunk an independent stream that starts from it."""
    ctx = ctx or default_context()
    src = _as_u8(data)
    n = src.size
    if in_off is None:
        n_chunks = n_chunks_for(n, chunk_size)
        mc = chunk_size
        off_arr = None
    else:
        off_arr = np.ascontiguousarray(np.asarray(in_off, dtype=np.uint64))
        n_chunks = off_arr.size - 1
        mc = int((off_arr[1:] - off_arr[:-1]).max()) if n_chunks else 1
    lib = capi.load()
    cap = int(lib.zs_deflate_batch_bound(n, n_chunks, max(mc, 1), wrap, mode))
    if dictionary is not None:
        cap += 4 * n_chunks   # DICTID
    out = np.empty(cap, dtype=np.uint8)
    out_off = np.zeros(n_chunks + 1, dtype=np.uint64)
    out_bits = np.zeros(n_chunks, dtype=np.uint64)
    checks = np.zeros(n_chunks, dtype=np.uint32)
    res = DeflateResult()
    if dictionary is not None:
        if mode != MODE_INDEPENDENT:
            raise ValueError("a dictionary call is INDEPENDENT")
        rc = lib.zs_deflate_batch_dict(ctx.handle, dictionary.handle, src.ctypes.data if n else None, n,
                                       off_arr.ctypes.data if off_arr is not None else None, n_chunks, chunk_size, level,
                                       wrap, flags, out.ctypes.data, cap, out_off.ctypes.data, out_bits.ctypes.data,
                                       checks.ctypes.data, C.byref(res))
        ctx.check(rc, "zs_deflate_batch_dict")
    else:
        rc = lib.zs_deflate_batch(ctx.handle, src.ctypes.data if n else None, n,
                                  off_arr.ctypes.data if off_arr is not None else None, n_chunks, chunk_size, level, wrap,
                                  mode, flags, out.ctypes.data, cap, out_off.ctypes.data, out_bits.ctypes.data,
                                  checks.ctypes.data, C.byref(res))
        ctx.check(rc, "zs_deflate_batch")
    return DeflateBatchHost(out[: res.total_out_bytes].tobytes(), out_off, out_bits, checks, res.total_out_bytes,
                            res.total_out_bits, res.check, res.n_blocks)


@dataclass
class InflateBatchDev:
    out: torch.Tensor
    out_len: torch.Tensor   # int64 [n]
    in_used: torch.Tensor   # int64 [n]
    checks: torch.Tensor    # int32 [n] (bit pattern of the uint32 check)
    status: torch.Tensor    # int32 [n]


def inflate_batch_dev(d_in: torch.Tensor, in_off: torch.Tensor, out_off: torch.Tensor, window_bits: int = 15,
                      out: torch.Tensor | None = None, d_dict: torch.Tensor | None = None,
                      dict_rng: torch.Tensor | None = None, out_capacity: int | None = None,
                      ctx: Context | None = None, reuse: InflateBatchDev | None = None) -> InflateBatchDev:
    """Enqueue one batch inflate on device-resident streams (no synchronisation)."""
    assert d_in.is_cuda and d_in.dtype == torch.uint8
    ctx = ctx or default_context(d_in.device.index)
    n = in_off.numel() - 1
    dev = d_in.device
    if reuse is not None:
        out, out_len, in_used, checks, status = reuse.out, reuse.out_len, reuse.in_used, reuse.checks, reuse.status
    else:
        if out is None:
            if out_capacity is None:
                out_capacity = int(out_off[-1].item())
            out = torch.empty(out_capacity + 16, dtype=torch.uint8, device=dev)
        out_len = torch.zeros(n, dtype=torch.int64, device=dev)
        in_used = torch.zeros(n, dtype=torch.int64, device=dev)
        checks = torch.zeros(n, dtype=torch.int32, device=dev)
        status = torch.zeros(n, dtype=torch.int32, device=dev)
    rc = capi.load().zs_inflate_batch_dev(ctx.handle, _ptr(d_in), _ptr(in_off), n, window_bits, _ptr(out), _ptr(out_off),
                                          _ptr(out_len), _ptr(in_used), _ptr(checks), _ptr(status), _ptr(d_dict),
                                          _ptr(dict_rng))
    ctx.check(rc, "zs_inflate_batch_dev")
    return InflateBatchDev(out, out_len, in_used, checks, status)


@dataclass
class InflateBatchHost:
    data: bytes
    out_off: np.ndarray
    out_len: np.ndarray
    in_used: np.ndarray
    checks: np.ndarray
    status: np.ndarray
    details: np.ndarray

    def output(self, i: int) -> bytes:
        o = int(self.out_off[i])
        return self.data[o: o + int(self.out_len[i])]

    def message(self, i: int) -> str:
        return (capi.load().zs_inflate_message(int(self.details[i])) or b"").decode()


def inflate_batch(streams, window_bits: int = 15, out_caps=None, dictionaries=None,
                  ctx: Context | None = None) -> InflateBatchHost:
    """Host-buffer inflateBatch: `streams` is a list of bytes-like objects (independent streams).

    `out_caps[i]` is the output capacity given to stream i (avail_out of a one-shot
    inflate(strm, Z_FINISH)); `dictionaries[i]` an optional preset dictionary: a raw stream decodes against it,
    a zlib stream with FDICT when its DICTID is the dictionary's adler32 (Z_NEED_DICT otherwise).  None or an
    empty dictionary is no dictionary.
    """
    ctx = ctx or default_context()
    n = len(streams)
    lens = np.array([len(s) for s in streams], dtype=np.uint64)
    in_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lens, out=in_off[1:])
    blob = np.frombuffer(b"".join(bytes(s) for s in streams), dtype=np.uint8) if n else np.zeros(0, np.uint8)
    if out_caps is None:
        raise ValueError("out_caps is required (the output capacity per stream)")
    caps = np.asarray(out_caps, dtype=np.uint64)
    # slot i spans exactly caps[i] bytes (the avail_out of a one-shot call)
    out_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(caps, out=out_off[1:])
    lib = capi.load()
    out = np.zeros(int(out_off[-1]) + 16, dtype=np.uint8)
    out_len = np.zeros(n, dtype=np.uint64)
    in_used = np.zeros(n, dtype=np.uint64)
    checks = np.zeros(n, dtype=np.uint32)
    status = np.zeros(n, dtype=np.int32)
    details = np.zeros(n, dtype=np.int32)
    if n == 0:
        return InflateBatchHost(b"", out_off, out_len, in_used, checks, status, details)
    dict_blob = dict_rng = None
    dict_total = 0
    if dictionaries is not None:
        ds = [bytes(d) if d is not None else b"" for d in dictionaries]
        dict_rng = np.zeros(2 * n, dtype=np.uint64)
        pos = 0
        for i, d in enumerate(ds):
            dict_rng[2 * i] = pos
            pos += len(d)
            dict_rng[2 * i + 1] = pos
        dict_total = pos
        dict_blob = np.frombuffer(b"".join(ds) + b"\0", dtype=np.uint8)
    rc = lib.zs_inflate_batch(ctx.handle, blob.ctypes.data if blob.size else None, in_off.ctypes.data, n, window_bits,
                              out.ctypes.data, out_off.ctypes.data, out_len.ctypes.data, in_used.ctypes.data,
                              checks.ctypes.data, status.ctypes.data,
                              dict_blob.ctypes.data if dict_blob is not None else None,
                              dict_rng.ctypes.data if dict_rng is not None else None, dict_total)
    ctx.check(rc, "zs_inflate_batch")
    rc = lib.zs_inflate_last_details(ctx.handle, details.ctypes.data, n)
    ctx.check(rc, "zs_inflate_last_details")
    return InflateBatchHost(out[: int(out_off[-1])].tobytes(), out_off, out_len, in_used, checks, status, details)


def checksum(data, kind: int, init: int | None = None, ctx: Context | None = None) -> int:
    """adler32(adler, buf, len) / crc32(crc, buf, len) of a host buffer, computed on the GPU."""
    ctx = ctx or default_context()
    src = _as_u8(data)
    if init is None:
        init = 1 if kind == capi.KIND_ADLER32 else 0
    res = C.c_uint32(0)
    rc = capi.load().zs_checksum(ctx.handle, kind, src.ctypes.data if src.size else None, src.size, init, C.byref(res))
    ctx.check(rc, "zs_checksum")
    return res.value


def checksum_dev(t: torch.Tensor, kind: int, init: int | None = None, ctx: Context | None = None) -> int:
    ctx = ctx or default_context(t.device.index)
    if init is None:
        init = 1 if kind == capi.KIND_ADLER32 else 0
    res = C.c_uint32(0)
    rc = capi.load().zs_checksum_dev(ctx.handle, kind, _ptr(t), t.numel(), init, C.byref(res))
    ctx.check(rc, "zs_checksum_dev")
    return res.value


def checksum_batch_dev(t: torch.Tensor, off: torch.Tensor, kind: int, ctx: Context | None = None) -> torch.Tensor:
    ctx = ctx or default_context(t.device.index)
    n = off.numel() - 1
    out = torch.empty(n, dtype=torch.int32, device=t.device)
    rc = capi.load().zs_checksum_batch_dev(ctx.handle, kind, _ptr(t), _ptr(off), n, _ptr(out))
    ctx.check(rc, "zs_checksum_batch_dev")
    return out


def crc32_combine(c1: int, c2: int, len2: int) -> int:
    return int(capi.load().zs_crc32_combine(c1, c2, len2))


def adler32_combine(a1: int, a2: int, len2: int) -> int:
    return int(capi.load().zs_adler32_combine(a1, a2, len2))


def flag_strategy(strategy: int) -> int:
    """ZS_FLAG_STRATEGY: the strategy argument of deflateInit2_ carried in the batch flags."""
    return (strategy & 7) << 8


def huffman_blocks(freq, in_len, ctx: Context | None = None):
    """Huffman stage alone (zs_huffman_blocks): freq uint32 [n, 320], in_len uint32 [n] (numpy, host).

    Returns (code [n, 320] uint32 = code | length << 16, type [n] uint32, bits [n] uint64)."""
    import numpy as np
    freq = np.ascontiguousarray(freq, dtype=np.uint32)
    in_len = np.ascontiguousarray(in_len, dtype=np.uint32)
    n = freq.shape[0]
    assert freq.shape == (n, 320) and in_len.shape == (n,)
    ctx = ctx or default_context(0)
    code = np.zeros((n, 320), dtype=np.uint32)
    typ = np.zeros(n, dtype=np.uint32)
    bits = np.zeros(n, dtype=np.uint64)
    rc = capi.load().zs_huffman_blocks(ctx.handle, freq.ctypes.data, in_len.ctypes.data, n, code.ctypes.data,
                                       typ.ctypes.data, bits.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"zs_huffman_blocks failed: {rc} {ctx.last_error()}")
    return code, typ, bits
