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


def deflate_indexed_dev(d_in: torch.Tensor, chunk_size: int, level: int = 6, wrap: int = WRAP_ZLIB, flags: int = 0,
                        span: int = 1 << 20, in_off: torch.Tensor | None = None, max_chunk: int | None = None,
                        out: torch.Tensor | None = None, want_checks: bool = False,
                        ctx: Context | None = None) -> tuple[DeflateBatchDev, "InflateIndex"]:
    """One STITCHED stream from device-resident input and its index for `span` (zs_deflate_indexed_dev), without a
    decode: the DeflateBatchDev that deflate_batch_dev(mode=MODE_STITCHED) returns, and an InflateIndex whose source
    is the stream out[:total_out_bytes].  Synchronises."""
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
    if out is None:
        out = torch.empty(int(capi.load().zs_deflate_batch_bound(n, n_chunks, mc, wrap, MODE_STITCHED)), dtype=torch.uint8,
                          device=dev)
    out_off = torch.empty(n_chunks + 1, dtype=torch.int64, device=dev)
    out_bits = torch.empty(n_chunks, dtype=torch.int64, device=dev)
    checks = torch.empty(n_chunks, dtype=torch.int32, device=dev) if (want_checks or wrap != WRAP_RAW) else None
    result = torch.zeros(24, dtype=torch.uint8, device=dev)
    h = C.c_void_p()
    rc = capi.load().zs_deflate_indexed_dev(ctx.handle, _ptr(d_in), n, _ptr(in_off), n_chunks, chunk_size, mc, level, wrap,
                                            flags, span, _ptr(out), out.numel(), _ptr(out_off), _ptr(out_bits), _ptr(checks),
                                            _ptr(result), C.byref(h))
    ctx.check(rc, "zs_deflate_indexed_dev")
    batch = DeflateBatchDev(out, out_off, out_bits, checks, result)
    return batch, InflateIndex(h, ctx, out[: batch.read_result().total_out_bytes])


def deflate_indexed(data, chunk_size: int = 65536, level: int = 6, wrap: int = WRAP_ZLIB, flags: int = 0,
                    span: int = 1 << 20, in_off=None, ctx: Context | None = None) -> tuple[DeflateBatchHost, "InflateIndex"]:
    """One STITCHED stream from a host buffer and its index for `span` (zs_deflate_indexed), without a decode: the
    DeflateBatchHost that deflate_batch(mode=MODE_STITCHED) returns, and an InflateIndex whose source is its bytes."""
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
    cap = int(lib.zs_deflate_batch_bound(n, n_chunks, max(mc, 1), wrap, MODE_STITCHED))
    out = np.empty(cap, dtype=np.uint8)
    out_off = np.zeros(n_chunks + 1, dtype=np.uint64)
    out_bits = np.zeros(n_chunks, dtype=np.uint64)
    checks = np.zeros(n_chunks, dtype=np.uint32)
    res = DeflateResult()
    h = C.c_void_p()
    rc = lib.zs_deflate_indexed(ctx.handle, src.ctypes.data if n else None, n,
                                off_arr.ctypes.data if off_arr is not None else None, n_chunks, chunk_size, level, wrap, flags,
                                span, out.ctypes.data, cap, out_off.ctypes.data, out_bits.ctypes.data, checks.ctypes.data,
                                C.byref(res), C.byref(h))
    ctx.check(rc, "zs_deflate_indexed")
    stream = out[: res.total_out_bytes].tobytes()
    return (DeflateBatchHost(stream, out_off, out_bits, checks, res.total_out_bytes, res.total_out_bits, res.check,
                             res.n_blocks), InflateIndex(h, ctx, stream))


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


# zs_gz_member: one decoded member of a multi-member gzip file
GZ_MEMBER_DTYPE = np.dtype([("in_off", "<u8"), ("in_len", "<u8"), ("out_off", "<u8"), ("out_len", "<u8"),
                            ("crc32", "<u4"), ("_pad", "<u4")])
assert GZ_MEMBER_DTYPE.itemsize == C.sizeof(capi.GzMember)


@dataclass
class Gunzip:
    data: bytes | torch.Tensor   # the output (gunzip: bytes; gunzip_dev: the device buffer, valid to out_len)
    out_len: int
    in_used: int
    n_members: int
    status: int                  # Z_STREAM_END when every byte belonged to a member
    detail: int
    members: np.ndarray | None   # GZ_MEMBER_DTYPE [min(n_members, table size)] when asked for

    @property
    def message(self) -> str:
        return (capi.load().zs_inflate_message(int(self.detail)) or b"").decode()


def _gunzip_result(res: capi.GunzipResult, data, table: np.ndarray | None) -> Gunzip:
    members = table[: min(int(res.n_members), table.size)] if table is not None else None
    return Gunzip(data, int(res.out_len), int(res.in_used), int(res.n_members), int(res.status), int(res.detail), members)


def gunzip(data, out_cap: int | None = None, members: bool = False, ctx: Context | None = None) -> Gunzip:
    """Every member of a multi-member gzip file from a host buffer (zs_gunzip): what inflate(Z_FINISH) /
    inflateReset repeated until the input is used up produces, like gzip -d or Python's gzip.decompress -- but strict
    about trailing bytes, as that loop is.

    `out_cap` is the output room.  Without it the room starts at four times the input (at least 64 KiB) and is
    doubled for as long as the call ends with Z_BUF_ERROR on a full output, so the result is the one an unlimited
    room gives.  With `members` the result carries the member table (offsets, sizes and crc32 of each member)."""
    ctx = ctx or default_context()
    src = _as_u8(data)
    n = src.size
    lib = capi.load()
    grow = out_cap is None
    cap = max(4 * n, 1 << 16) if grow else int(out_cap)
    n_tab = n // 1024 + 1024 if members else 0
    while True:
        out = np.empty(cap + 16, dtype=np.uint8)
        table = np.zeros(n_tab, dtype=GZ_MEMBER_DTYPE) if members else None
        res = capi.GunzipResult()
        rc = lib.zs_gunzip(ctx.handle, src.ctypes.data if n else None, n, out.ctypes.data, cap, C.byref(res),
                           table.ctypes.data if members else None, n_tab)
        ctx.check(rc, "zs_gunzip")
        if grow and res.status == capi.Z_BUF_ERROR and res.out_len == cap:
            cap *= 2
            continue
        if members and res.n_members > n_tab:   # the table was too short: once more with the exact count
            n_tab = int(res.n_members)
            continue
        return _gunzip_result(res, out[: res.out_len].tobytes(), table)


def gunzip_dev(d_in: torch.Tensor, out_cap: int, members: int = 0, out: torch.Tensor | None = None,
               ctx: Context | None = None) -> Gunzip:
    """Every member of a multi-member gzip file in device memory (zs_gunzip_dev; synchronises).  `d_in` must start
    8-byte aligned (a fresh tensor does); the output goes to `out` (allocated with out_cap bytes when None).
    `members`: size of the member table to fill (0: none)."""
    assert d_in.is_cuda and d_in.dtype == torch.uint8 and d_in.is_contiguous()
    ctx = ctx or default_context(d_in.device.index)
    if out is None:
        out = torch.empty(out_cap + 16, dtype=torch.uint8, device=d_in.device)
    assert out.numel() >= out_cap
    table = np.zeros(members, dtype=GZ_MEMBER_DTYPE) if members else None
    res = capi.GunzipResult()
    rc = capi.load().zs_gunzip_dev(ctx.handle, _ptr(d_in), d_in.numel(), _ptr(out), out_cap, C.byref(res),
                                   table.ctypes.data if members else None, members)
    ctx.check(rc, "zs_gunzip_dev")
    return _gunzip_result(res, out, table)


@dataclass
class IndexBuild:
    """What zs_inflate_index_build_dev decoded: the zs_inflate_stream_dev result of the stream."""
    data: torch.Tensor   # device output, valid to out_len
    out_len: int
    in_used: int
    check: int
    status: int
    detail: int

    @property
    def message(self) -> str:
        return (capi.load().zs_inflate_message(int(self.detail)) or b"").decode()


@dataclass
class IndexExtract:
    """Ranges read from an index: range i is data[out_off[i]: out_off[i] + got[i]]."""
    data: bytes
    out_off: np.ndarray
    got: np.ndarray
    status: np.ndarray   # Z_OK, Z_BUF_ERROR (clipped at the end of the stream), Z_DATA_ERROR
    details: np.ndarray  # message codes (zs_inflate_message)

    def range(self, i: int) -> bytes:
        o = int(self.out_off[i])
        return self.data[o: o + int(self.got[i])]

    def message(self, i: int) -> str:
        return (capi.load().zs_inflate_message(int(self.details[i])) or b"").decode()


class InflateIndex:
    """Access points into one zlib, gzip or raw deflate stream (zs_inflate_index_*): block starts about every `span`
    bytes of output, each with the 32 KiB window before it, on the device.  Byte ranges of the stream are then read
    without decoding what comes before them, many at once.  Close it (or let it be collected) before its context goes.

    `source` is the stream the index was built from when build() had it (host bytes or a device tensor); extract()
    reads from it unless it is given another copy of the same stream."""

    def __init__(self, handle, ctx: Context, source=None):
        self._lib = capi.load()
        self._h = handle
        self.ctx = ctx
        self.source = source
        info = capi.InflateIndexInfo()
        ctx.check(self._lib.zs_inflate_index_info_get(handle, C.byref(info)), "zs_inflate_index_info_get")
        self.info = info

    @classmethod
    def build(cls, data, window_bits: int = 15, span: int = 1 << 20, dictionary=None, out_cap: int | None = None,
              ctx: Context | None = None):
        """Decode a whole stream (bytes or a CUDA uint8 tensor) as zs_inflate_stream_dev does and index it.  Returns
        (index, IndexBuild); the index is None unless the status is Z_STREAM_END.  Without `out_cap` the output room
        grows until a full-output Z_BUF_ERROR no longer occurs, as gunzip() does."""
        if isinstance(data, torch.Tensor):
            assert data.is_cuda and data.dtype == torch.uint8 and data.is_contiguous()
            ctx = ctx or default_context(data.device.index)
            d_in, source = data, data
        else:
            ctx = ctx or default_context()
            source = _as_u8(data)
            # (an empty stream still needs a real pointer: a slice of a small buffer)
            d_in = torch.from_numpy(source.copy()).to(f"cuda:{ctx.device}") if source.size else \
                torch.zeros(8, dtype=torch.uint8, device=f"cuda:{ctx.device}")[:0]
        d_dict = None
        if dictionary is not None and len(dictionary):
            d_dict = torch.from_numpy(_as_u8(dictionary).copy()).to(d_in.device)
        n = d_in.numel()
        grow = out_cap is None
        cap = max(4 * n, 1 << 16) if grow else int(out_cap)
        lib = capi.load()
        while True:
            out = torch.empty(cap + 16, dtype=torch.uint8, device=d_in.device)
            res = capi.InflateIndexResult()
            h = C.c_void_p()
            rc = lib.zs_inflate_index_build_dev(ctx.handle, _ptr(d_in), n, window_bits, span, _ptr(out),
                                                cap, _ptr(d_dict), d_dict.numel() if d_dict is not None else 0, C.byref(res),
                                                C.byref(h))
            ctx.check(rc, "zs_inflate_index_build_dev")
            if grow and res.status == capi.Z_BUF_ERROR and res.out_len == cap:
                cap *= 2
                continue
            built = IndexBuild(out, int(res.out_len), int(res.in_used), int(res.check), int(res.status), int(res.detail))
            return (cls(h, ctx, source) if h.value else None), built

    @classmethod
    def from_bytes(cls, blob, ctx: Context | None = None, source=None) -> "InflateIndex":
        """An index from to_bytes() output (zs_inflate_index_import): a malformed blob raises with Z_DATA_ERROR."""
        ctx = ctx or default_context()
        src = _as_u8(blob)
        h = C.c_void_p()
        rc = capi.load().zs_inflate_index_import(ctx.handle, src.ctypes.data if src.size else None, src.size, C.byref(h))
        ctx.check(rc, "zs_inflate_index_import")
        return cls(h, ctx, source)

    @property
    def handle(self):
        if not self._h:
            raise ValueError("InflateIndex is closed")
        return self._h

    @property
    def points(self) -> np.ndarray:
        """(n_points, 2) uint64: input bit and output offset of every access point."""
        n = int(self.info.n_points)
        bit = np.zeros(n, dtype=np.uint64)
        off = np.zeros(n, dtype=np.uint64)
        self.ctx.check(self._lib.zs_inflate_index_points(self.handle, bit.ctypes.data, off.ctypes.data, n),
                       "zs_inflate_index_points")
        return np.stack([bit, off], axis=1)

    def to_bytes(self) -> bytes:
        """The export format of include/zsgpu.h (version 1)."""
        n = C.c_uint64(0)
        self.ctx.check(self._lib.zs_inflate_index_export(self.handle, None, 0, C.byref(n)), "zs_inflate_index_export")
        buf = np.zeros(n.value, dtype=np.uint8)
        self.ctx.check(self._lib.zs_inflate_index_export(self.handle, buf.ctypes.data, n.value, C.byref(n)),
                       "zs_inflate_index_export")
        return buf.tobytes()

    def extract_dev(self, d_in: torch.Tensor, off: torch.Tensor, length: torch.Tensor, out: torch.Tensor,
                    out_off: torch.Tensor, got: torch.Tensor | None = None, status: torch.Tensor | None = None):
        """zs_inflate_index_extract_dev on device arrays (int64 off / length / out_off); no synchronisation.
        Returns (got, status) device tensors."""
        n = off.numel()
        got = got if got is not None else torch.zeros(n, dtype=torch.int64, device=off.device)
        status = status if status is not None else torch.zeros(n, dtype=torch.int32, device=off.device)
        rc = self._lib.zs_inflate_index_extract_dev(self.ctx.handle, self.handle, _ptr(d_in), d_in.numel(), _ptr(off),
                                                    _ptr(length), n, _ptr(out), _ptr(out_off), _ptr(got), _ptr(status))
        self.ctx.check(rc, "zs_inflate_index_extract_dev")
        return got, status

    def extract_ranges(self, off, length, data=None) -> IndexExtract:
        """Ranges [off[i], off[i] + length[i]) of the stream, packed one after the other, with their statuses and
        message codes.  A device source goes through extract_dev, a host one through zs_inflate_index_extract."""
        src = self.source if data is None else data
        if src is None:
            raise ValueError("the index has no source stream: pass the stream as `data`")
        off = np.ascontiguousarray(np.asarray(off, dtype=np.uint64).reshape(-1))
        length = np.ascontiguousarray(np.asarray(length, dtype=np.uint64).reshape(-1))
        n = off.size
        out_len = int(self.info.out_len)
        clipped = np.minimum(length, np.uint64(out_len) - np.minimum(off, np.uint64(out_len)))   # the bytes each range gets
        out_off = np.zeros(n, dtype=np.uint64)
        if n > 1:
            np.cumsum(clipped[:-1], out=out_off[1:])
        cap = int(clipped.sum()) if n else 0
        details = np.zeros(n, dtype=np.int32)
        if isinstance(src, torch.Tensor):
            dev = src.device
            t = lambda a: torch.from_numpy(a.view(np.int64)).to(dev)
            out = torch.zeros(cap + 16, dtype=torch.uint8, device=dev)
            got_t, status_t = self.extract_dev(src, t(off), t(length), out, t(out_off))
            got = got_t.cpu().numpy().view(np.uint64)
            status = status_t.cpu().numpy()
            data_out = out[:cap].cpu().numpy().tobytes()
        else:
            s = _as_u8(src)
            outb = np.zeros(cap + 16, dtype=np.uint8)
            got = np.zeros(n, dtype=np.uint64)
            status = np.zeros(n, dtype=np.int32)
            rc = self._lib.zs_inflate_index_extract(self.ctx.handle, self.handle, s.ctypes.data if s.size else None, s.size,
                                                    off.ctypes.data, length.ctypes.data, n, outb.ctypes.data, cap,
                                                    out_off.ctypes.data, got.ctypes.data, status.ctypes.data)
            self.ctx.check(rc, "zs_inflate_index_extract")
            data_out = outb[:cap].tobytes()
        if n:
            self.ctx.check(self._lib.zs_inflate_last_details(self.ctx.handle, details.ctypes.data, n), "zs_inflate_last_details")
        return IndexExtract(data_out, out_off, got, status, details)

    def extract(self, ranges, data=None) -> list:
        """[(off, length), ...] -> the bytes of each range (shorter where it runs past the end of the stream).  A range
        the stream does not decode for raises ZsError with Z_DATA_ERROR."""
        ranges = list(ranges)
        r = self.extract_ranges([o for o, _ in ranges], [n for _, n in ranges], data)
        bad = np.nonzero(r.status == capi.Z_DATA_ERROR)[0]
        if bad.size:
            raise capi.ZsError(capi.Z_DATA_ERROR, "zs_inflate_index_extract", f"range {int(bad[0])}: {r.message(int(bad[0]))}")
        return [r.range(i) for i in range(len(ranges))]

    def close(self):
        if getattr(self, "_h", None):
            self._lib.zs_inflate_index_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


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
