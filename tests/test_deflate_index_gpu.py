"""GPU tests of deflate with an index (zs_deflate_indexed / zs_deflate_indexed_dev).

The stream must be byte for byte what the STITCHED batch deflate writes with the same arguments, and the index made
from the encoder's block layout must be the one zs_inflate_index_build makes by decoding that stream: equal exports
(header, points, windows).  For some streams the points are also checked against the block starts C zlib's
inflate(Z_BLOCK) reports (zran_check.block_starts).  Reads through the index must give slices of the input, and the
call must run no decoder kernel."""
import ctypes as C
import random
import zlib

import numpy as np
import pytest

from conftest import make_mixed, make_text, pkg, rand_bytes
from zran_check import block_starts

pytestmark = pytest.mark.gpu

WB = {0: -15, 1: 15, 2: 31}   # the window_bits inflate reads each wrapper with
SYNC = 8
TEXT = make_text(1 << 20, 31)
MIXED = make_mixed(1 << 20, 32)
INPUTS = {"text": TEXT, "mixed": MIXED, "random": rand_bytes(600000, 33), "zeros": bytes(700000),
          "empty": b"", "one": b"x"}


def _rule(starts, span, out_len):
    """The access points: per m = 0, S, 2S, ... < out_len the first block start with offset >= m; the first start always."""
    pts = [starts[0]]
    m, k = span, 1
    while m < out_len:
        while k < len(starts) and starts[k][1] < m:
            k += 1
        if k == len(starts):
            break
        if starts[k] != pts[-1]:
            pts.append(starts[k])
        m = (starts[k][1] // span + 1) * span
    return pts


def _host(data, chunk=65536, level=6, wrap=1, flags=0, span=1 << 20, in_off=None):
    """The host call against zs_deflate_batch(STITCHED) and against the decode-based build; returns (batch, index)."""
    B = pkg("batch")
    got, ix = B.deflate_indexed(data, chunk, level, wrap, flags, span, in_off=in_off)
    ref = B.deflate_batch(data, chunk, level, wrap, B.MODE_STITCHED, flags, in_off=in_off)
    assert got.data == ref.data
    assert (got.out_off == ref.out_off).all() and (got.out_bits == ref.out_bits).all() and (got.checks == ref.checks).all()
    assert (got.total_out_bytes, got.total_out_bits, got.check, got.n_blocks) == \
        (ref.total_out_bytes, ref.total_out_bits, ref.check, ref.n_blocks)
    assert zlib.decompress(got.data, WB[wrap]) == bytes(data)
    built, res = B.InflateIndex.build(got.data, WB[wrap], span)
    assert res.status == pkg("capi").Z_STREAM_END
    assert ix.to_bytes() == built.to_bytes()
    return got, ix


def _dev(data, chunk=65536, level=6, wrap=1, flags=0, span=1 << 20, in_off=None):
    """The device call against zs_deflate_batch_dev(STITCHED) and the decode-based build; returns (batch, index)."""
    import torch
    B = pkg("batch")
    d_in = torch.frombuffer(bytearray(data) or bytearray(8), dtype=torch.uint8)[: len(data)].cuda()
    d_off = None if in_off is None else torch.tensor(np.asarray(in_off, dtype=np.int64), device="cuda")
    got, ix = B.deflate_indexed_dev(d_in, chunk, level, wrap, flags, span, in_off=d_off)
    ref = B.deflate_batch_dev(d_in, chunk, level, wrap, B.MODE_STITCHED, flags, in_off=d_off)
    torch.cuda.synchronize()
    r = got.read_result()
    n = r.total_out_bytes
    assert bytes(got.result.cpu().numpy()) == bytes(ref.result.cpu().numpy())
    assert torch.equal(got.out[:n], ref.out[:n])
    assert torch.equal(got.out_off, ref.out_off) and torch.equal(got.out_bits, ref.out_bits)
    assert (got.checks is None) == (ref.checks is None) and (got.checks is None or torch.equal(got.checks, ref.checks))
    stream = got.out[:n].cpu().numpy().tobytes()
    assert zlib.decompress(stream, WB[wrap]) == bytes(data)
    assert ix.source.data_ptr() == got.out.data_ptr() and ix.source.numel() == n
    built, _ = B.InflateIndex.build(ix.source, WB[wrap], span)
    assert ix.to_bytes() == built.to_bytes()
    return got, ix


@pytest.mark.parametrize("level", range(10))
def test_levels(gpu_ctx, level):
    _host(TEXT, level=level, span=65536)


@pytest.mark.parametrize("sync", [0, SYNC])
@pytest.mark.parametrize("wrap", [0, 1, 2])
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_wraps_levels_sync(gpu_ctx, level, wrap, sync):
    _host(MIXED, level=level, wrap=wrap, flags=sync, span=65536)
    _dev(MIXED[: 600000], level=level, wrap=wrap, flags=sync, span=65536)


@pytest.mark.parametrize("strategy", range(5))
def test_strategies(gpu_ctx, strategy):
    _host(MIXED, level=6, flags=strategy << 8, span=65536)
    _dev(TEXT, level=1, wrap=0, flags=(strategy << 8) | SYNC, span=4096)


@pytest.mark.parametrize("chunk", [4096, 65536, 262144])
def test_chunk_sizes(gpu_ctx, chunk):
    _host(TEXT, chunk=chunk, level=1, span=65536)
    _dev(MIXED, chunk=chunk, level=6, wrap=2, flags=SYNC, span=1 << 20)


@pytest.mark.parametrize("sync", [0, SYNC])
def test_ragged_chunks_with_empty_ones(gpu_ctx, sync):
    n = len(MIXED)
    in_off = [0, 0, 1000, 1000, 1000, 70000, 70001, 300000, 300000, 512 * 1024, n, n]
    _host(MIXED, level=6, flags=sync, span=65536, in_off=in_off)
    _dev(MIXED, level=1, wrap=0, flags=sync, span=4096, in_off=in_off)


@pytest.mark.parametrize("span", [1, 4096, 65536, 1 << 20])
@pytest.mark.parametrize("kind", ["text", "mixed", "random", "zeros"])
def test_spans_and_inputs(gpu_ctx, kind, span):
    _host(INPUTS[kind], chunk=65536, level=6, flags=SYNC if kind == "text" else 0, span=span)


@pytest.mark.parametrize("wrap", [0, 1, 2])
@pytest.mark.parametrize("kind", ["empty", "one"])
def test_tiny_inputs(gpu_ctx, kind, wrap):
    _, ix = _host(INPUTS[kind], wrap=wrap, span=1)
    assert ix.info.n_points == 1
    _dev(INPUTS[kind], wrap=wrap, span=4096)


@pytest.mark.parametrize("case", [("text_sync", TEXT, 6, 1, SYNC, 65536), ("mixed_l1", MIXED, 1, 0, 0, 4096),
                                  ("stored", INPUTS["random"], 0, 2, SYNC, 1), ("zeros_fixed", INPUTS["zeros"], 6, 1, 4 << 8, 65536)],
                         ids=lambda c: c[0])
def test_points_are_the_rule_over_zlib_block_starts(gpu_ctx, case):
    _, data, level, wrap, flags, span = case
    got, ix = _host(data, chunk=32768, level=level, wrap=wrap, flags=flags, span=span)
    want = _rule(block_starts(got.data, WB[wrap]), span, len(data))
    assert [tuple(map(int, p)) for p in ix.points] == want


def test_large_stream_through_the_pipelined_path(gpu_ctx):
    """64 MiB in 1024 chunks takes the sliced host path: every slice but the last ends with a sync marker, and with the
    span equal to the chunk size each marker starts the first block at a multiple of the span, so it is a point."""
    data = make_mixed(64 << 20, 34)
    span = 65536
    got, ix = _host(data, chunk=65536, level=1, span=span)
    pts = ix.points
    s = np.frombuffer(got.data, dtype=np.uint8)
    markers = []
    for bit, off in pts:
        bit, off = int(bit), int(off)
        if ((int(s[bit >> 3]) | int(s[(bit >> 3) + 1]) << 8) >> (bit & 7)) & 7 == 0:   # BFINAL 0, stored
            b = (bit + 3 + 7) >> 3
            if bytes(s[b: b + 4]) == b"\x00\x00\xff\xff":
                markers.append(off)
    assert markers, "no slice marker among the points"
    assert all(o % span == 0 for o in markers) and len(markers) < 64   # the slices' markers, not one per chunk


def test_reads_through_the_index(gpu_ctx):
    data = make_text(8 << 20, 35)
    B = pkg("batch")
    got, ix = _host(data, chunk=65536, level=6, span=262144)
    rng = random.Random(36)
    ranges = [(rng.randrange(len(data)), rng.randrange(1, 5000)) for _ in range(10000)]
    for src in (got.data, None):
        if src is None:
            import torch
            src = torch.frombuffer(bytearray(got.data), dtype=torch.uint8).cuda()
        r = ix.extract_ranges([o for o, _ in ranges], [n for _, n in ranges], src)
        for i, (o, n) in enumerate(ranges):
            assert r.range(i) == data[o: o + n]
        assert ix.extract([(0, len(data))], src)[0] == data
    again = B.InflateIndex.from_bytes(ix.to_bytes())
    assert again.to_bytes() == ix.to_bytes()
    assert again.extract([(123456, 7777)], got.data)[0] == data[123456: 123456 + 7777]
    _, dix = _dev(data, chunk=65536, level=1, span=65536)
    r = dix.extract_ranges([o for o, _ in ranges[:1000]], [n for _, n in ranges[:1000]])
    assert all(r.range(i) == data[o: o + n] for i, (o, n) in enumerate(ranges[:1000]))


def test_no_decoder_kernel_runs(gpu_ctx):
    import torch
    B = pkg("batch")
    d_in = torch.frombuffer(bytearray(MIXED), dtype=torch.uint8).cuda()
    for call in (lambda: B.deflate_indexed(MIXED, 65536, 6, 0, 0, 65536, ctx=gpu_ctx),
                 lambda: B.deflate_indexed_dev(d_in, 65536, 6, 1, SYNC, 65536, ctx=gpu_ctx)):
        gpu_ctx.profile(True)
        gpu_ctx.profile_read()
        call()
        prof = gpu_ctx.profile_read()
        gpu_ctx.profile(False)
        assert "deflate_record_kernel" in prof and "ix_gather_kernel" in prof and "encode_kernel" in prof
        assert not [k for k in prof if k.startswith(("inflate", "par_"))], sorted(prof)


def test_refusals(gpu_ctx):
    import torch
    lib, capi = pkg("capi").load(), pkg("capi")
    data = MIXED[:100000]
    src = np.frombuffer(data, dtype=np.uint8)
    nc = 2
    cap = int(lib.zs_deflate_batch_bound(len(data), nc, 65536, 1, 1))
    out = np.zeros(cap, dtype=np.uint8)
    res = capi.DeflateResult()
    d_in = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    d_res = torch.zeros(24, dtype=torch.uint8, device="cuda")

    def host(flags=0, span=65536, out_cap=cap, ptr=True, outp=True):
        h = C.c_void_p(12345)
        rc = lib.zs_deflate_indexed(gpu_ctx.handle, src.ctypes.data, len(data), None, nc, 65536, 6, 1, flags, span,
                                    out.ctypes.data if outp else None, out_cap, None, None, None, C.byref(res),
                                    C.byref(h) if ptr else None)
        return rc, h.value

    def dev(flags=0, span=65536, out_cap=cap, ptr=True, outp=True):
        h = C.c_void_p(12345)
        rc = lib.zs_deflate_indexed_dev(gpu_ctx.handle, C.c_void_p(d_in.data_ptr()), len(data), None, nc, 65536, 65536, 6, 1,
                                        flags, span, C.c_void_p(d_out.data_ptr()) if outp else None, out_cap, None, None,
                                        None, C.c_void_p(d_res.data_ptr()), C.byref(h) if ptr else None)
        return rc, h.value

    for call in (host, dev):
        for flags in (1, 2, 4, 1 | SYNC):
            assert call(flags=flags) == (capi.Z_STREAM_ERROR, None)
        assert call(span=0) == (capi.Z_STREAM_ERROR, None)
        assert call(outp=False) == (capi.Z_STREAM_ERROR, None)
        assert call(ptr=False)[0] == capi.Z_STREAM_ERROR
        assert call(out_cap=1000) == (capi.Z_BUF_ERROR, None)
        rc, h = call()
        assert rc == capi.Z_OK and h
        lib.zs_inflate_index_destroy(C.c_void_p(h))
    h = C.c_void_p(12345)
    assert lib.zs_deflate_indexed(None, src.ctypes.data, len(data), None, nc, 65536, 6, 1, 0, 65536, out.ctypes.data, cap,
                                  None, None, None, C.byref(res), C.byref(h)) == capi.Z_STREAM_ERROR
    assert h.value is None
