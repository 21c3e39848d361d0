"""GPU tests of zs_gunzip / zs_gunzip_dev: a whole multi-member gzip file in one call.  Every case is compared with the
reference's multi-member loop (gunzip_cases.oracle_gunzip): status, message, output, member count and, on
Z_STREAM_END, bytes used.  On an error, bytes used are the failing member's start plus what the engine's own batch
inflate reports for that member alone.  The host-buffer and device calls must agree, and member tables are checked
against the offsets the writer recorded."""
import zlib

import numpy as np
import pytest

from conftest import make_mixed, make_text, pkg, rand_bytes
from gunzip_cases import Writer, bgzf, gzip_member, oracle_gunzip

pytestmark = pytest.mark.gpu


def _dev_run(data, out_cap, table):
    import torch
    B = pkg("batch")
    d_in = torch.frombuffer(bytearray(data) or bytearray(8), dtype=torch.uint8)[: len(data)].cuda()
    r = B.gunzip_dev(d_in, out_cap, members=table)
    r.data = r.data[: r.out_len].cpu().numpy().tobytes()
    return r


def _check(oracle, data, out_cap=None, writer=None):
    """gunzip (host) and gunzip_dev == the oracle loop; returns the host result."""
    B = pkg("batch")
    total = writer.out_pos if writer is not None else None
    cap = out_cap if out_cap is not None else (total if total is not None else 4 * len(data) + (1 << 16))
    want = oracle_gunzip(oracle, data, cap)
    h = B.gunzip(data, cap, members=True)
    d = _dev_run(data, cap, max(want.members, 1))
    for r in (h, d):
        assert (r.status, r.message, r.n_members) == (want.ret, want.msg, want.members), (r.status, r.message, r.n_members)
        assert r.out_len == len(want.out) and r.data == want.out
    assert h.in_used == d.in_used
    assert np.array_equal(h.members, d.members)
    if want.ret == oracle.Z_STREAM_END:
        assert h.in_used == want.in_used == len(data)
    else:
        alone = B.inflate_batch([data[want.start:]], 31, [cap - want.out_start])
        assert h.in_used == want.start + int(alone.in_used[0])
        assert int(alone.status[0]) == want.ret and alone.message(0) == want.msg
    # the member table: contiguous, in file order, crc32 of each member's output
    m = h.members
    assert m.size == want.members
    if m.size:
        assert int(m["in_off"][0]) == 0 and int(m["out_off"][0]) == 0
        assert np.array_equal(m["in_off"][1:], m["in_off"][:-1] + m["in_len"][:-1])
        assert np.array_equal(m["out_off"][1:], m["out_off"][:-1] + m["out_len"][:-1])
        for k in np.linspace(0, m.size - 1, min(m.size, 50)).astype(int):
            o, n = int(m["out_off"][k]), int(m["out_len"][k])
            assert int(m["crc32"][k]) == zlib.crc32(want.out[o: o + n])
    if writer is not None and want.ret == oracle.Z_STREAM_END:
        t = np.array(writer.table, dtype=np.uint64).reshape(-1, 4)
        assert np.array_equal(np.stack([m["in_off"], m["in_len"], m["out_off"], m["out_len"]], 1), t)
    return h


@pytest.mark.parametrize("level", [1, 6, 9])
def test_bgzf(gpu_ctx, oracle, level):
    data = make_text(6 << 20, 40 + level) + make_mixed(2 << 20, 41)
    for n in (1000, len(data)):
        w = bgzf(data[:n], level)
        h = _check(oracle, w.data(), writer=w)
        assert h.status == 1 and h.data == data[:n]


def test_bgzf_64mib_and_no_out_cap(gpu_ctx, oracle):
    B = pkg("batch")
    data = make_mixed(64 << 20, 42)
    w = bgzf(data, 6)
    _check(oracle, w.data(), writer=w)
    r = B.gunzip(w.data())   # room grown from 4x the input
    assert r.status == 1 and r.data == data and r.n_members == len(w.table)
    z = zlib.compress(b"\0" * (40 << 20), 9, wbits=31)   # > 4000x: the room doubles many times
    r = B.gunzip(z + z)
    assert r.status == 1 and r.out_len == 80 << 20 and r.n_members == 2


@pytest.mark.parametrize("chunk", [4096, 65536])
def test_engine_independent_gzip_output(gpu_ctx, oracle, chunk):
    B = pkg("batch")
    data = make_text(5 << 20, 43)
    r = B.deflate_batch(data, chunk, 6, B.WRAP_GZIP, B.MODE_INDEPENDENT)
    h = _check(oracle, r.data, len(data))
    assert h.data == data
    n = -(-len(data) // chunk)
    assert np.array_equal(h.members["in_off"], r.out_off[:n]) and np.array_equal(h.members["out_off"], np.arange(n) * chunk)
    # chunks given by offsets, empty ones among them
    cuts = np.array([0, 0, 1000, 1000, 70000, 70000, 70001, len(data), len(data)], dtype=np.uint64)
    r = B.deflate_batch(data, chunk, 6, B.WRAP_GZIP, B.MODE_INDEPENDENT, in_off=cuts)
    h = _check(oracle, r.data, len(data))
    assert h.data == data and h.n_members == 8 and list(h.members["out_len"]) == list(np.diff(cuts))


def test_c_zlib_members_mixed_sizes_and_headers(gpu_ctx, oracle):
    text = make_text(40 << 20, 44)
    mixed = make_mixed(36 << 20, 45)
    w = Writer()

    def add(piece, **kw):
        w.add(gzip_member(piece, **kw), len(piece))

    add(b"")
    add(b"x", text=True)
    for i in range(3000):
        piece = text[i * 4096: (i + 1) * 4096]
        add(piece, level=(1, 6, 9)[i % 3], text=bool(i & 1), extra=b"ab" * (i % 5) if i % 7 == 0 else None,
            name=b"n%d" % i if i % 11 == 0 else None, comment=b"c%d" % i if i % 13 == 0 else None, hcrc=i % 17 == 0)
    add(text[: 33 << 20], level=6, name=b"big")                 # one go
    add(b"tiny", hcrc=True)
    add(mixed[: 32 << 20], level=1, sync_every=1 << 20)          # sync flush points every MiB
    add(text[5 << 20: (5 << 20) + 777], comment=b"last")
    h = _check(oracle, w.data(), writer=w)
    assert h.status == 1


def test_false_member_starts(gpu_ctx, oracle):
    B = pkg("batch")
    text = make_text(3 << 20, 46)
    inner = bgzf(text[: 1 << 20], 6).data()
    # level-0 members whose payload is a multi-member gzip file, between ordinary members
    w = Writer()
    for i in range(6):
        w.add(zlib.compress(inner, 0, wbits=31), len(inner))
        w.add(gzip_member(text[i * 5000: i * 5000 + 5000]), 5000)
    _check(oracle, w.data(), writer=w)
    # every member a stored wrapper of gzip files: nothing the batch plans holds
    w = Writer()
    for i in range(40):
        small = b"".join(zlib.compress(text[k * 300: k * 300 + 300 + i], 6, wbits=31) for k in range(20))
        w.add(zlib.compress(small, 0, wbits=31), len(small))
    _check(oracle, w.data(), writer=w)
    # a BGZF file whose BSIZE fields lie
    w = bgzf(text, 6, bsize_lie=1000)
    h = _check(oracle, w.data(), writer=w)
    assert h.data == text
    # a large member at an odd byte offset
    w = Writer()
    w.add(gzip_member(b"odd", name=b"abcd"), 3)
    assert w.in_pos & 7
    w.add(gzip_member(text, 6), len(text))
    w.add(gzip_member(text[:12345], 9), 12345)
    h = _check(oracle, w.data(), writer=w)
    assert h.data == b"odd" + text + text[:12345]
    # every tenth member a stored wrapper of a gzip file, among many small ones
    w = Writer()
    for i in range(400):
        piece = text[i * 3000: i * 3000 + 3000]
        if i % 10 == 3:
            inner = b"".join(zlib.compress(piece[k * 300: k * 300 + 300], 6, wbits=31) for k in range(10))
            w.add(zlib.compress(inner, 0, wbits=31), len(inner))
        else:
            w.add(gzip_member(piece, 6), len(piece))
    _check(oracle, w.data(), writer=w)
    # random bytes that look like headers inside stored data
    noise = bytearray(rand_bytes(1 << 20, 47))
    for k in range(0, len(noise) - 16, 4099):
        noise[k: k + 10] = b"\x1f\x8b\x08\x00\0\0\0\0\0\x03"
    w = Writer()
    for i in range(3):
        w.add(zlib.compress(bytes(noise), 0, wbits=31), len(noise))
        w.add(gzip_member(text[:100000], 6), 100000)
    _check(oracle, w.data(), writer=w)
    assert B.gunzip(w.data()).status == 1


def _members(n=12, seed=48, size=20000):
    text = make_text(n * size, seed)
    parts = [gzip_member(text[i * size: (i + 1) * size], 6) for i in range(n)]
    return text, parts


def test_corrupt_middle_member(gpu_ctx, oracle):
    text, parts = _members()
    big = gzip_member(make_text(3 << 20, 49), 6)
    for k, where in ((5, "body"), (5, "crc"), (5, "isize"), (6, "body")):
        ps = list(parts)
        if k == 6:
            ps.insert(6, big)
        m = bytearray(ps[k])
        off = {"body": len(m) // 2, "crc": len(m) - 6, "isize": len(m) - 2}[where]
        m[off] ^= 0x10
        ps[k] = bytes(m)
        h = _check(oracle, b"".join(ps))
        assert h.status in (-3, -5) and h.n_members == k


def test_truncated(gpu_ctx, oracle):
    _, parts = _members()
    whole = b"".join(parts)
    start = sum(len(p) for p in parts[:7])
    for cut in (start + 5, start + len(parts[7]) // 2, start + len(parts[7]) - 3):   # header, body, trailer
        h = _check(oracle, whole[:cut])
        assert h.status == -5 and h.n_members == 7


def test_trailing_bytes_and_not_gzip(gpu_ctx, oracle):
    _, parts = _members(4)
    whole = b"".join(parts)
    for tail in (b"garbage!", b"\0" * 512, b"\x1f", b"\x1f\x8b\x08\x00"):
        h = _check(oracle, whole + tail)
        assert h.status in (-3, -5) and h.n_members == 4
    h = _check(oracle, b"\0" * 1000 + whole)
    assert h.status == -3 and h.message == "incorrect header check" and h.n_members == 0
    h = _check(oracle, zlib.compress(b"zlib, not gzip" * 100))
    assert h.status == -3 and h.n_members == 0
    h = _check(oracle, b"", 100)
    assert h.status == -5 and h.n_members == 0 and h.out_len == 0


def test_room(gpu_ctx, oracle):
    text, parts = _members()
    large = make_text(2 << 20, 50)
    whole = b"".join(parts[:6]) + gzip_member(large, 6) + b"".join(parts[6:])
    size = 20000
    for cap in (0, 5 * size + 777, 6 * size, 6 * size + (1 << 20) + 3, 6 * size + len(large), 12 * size + len(large) - 1):
        h = _check(oracle, whole, cap)
        assert h.status == (1 if cap >= 12 * size + len(large) else -5)


def test_paths_taken(gpu_ctx, oracle):
    """BGZF: the locate kernel and the batch decoders, no segment-parallel decode; a 64 MiB member: the
    segment-parallel decoder."""
    B = pkg("batch")
    data = make_text(16 << 20, 51)
    w = bgzf(data, 6)
    gpu_ctx.profile(True)
    gpu_ctx.profile_read()
    r = B.gunzip(w.data(), len(data))
    prof = gpu_ctx.profile_read()
    assert r.status == 1 and r.data == data
    assert "gunzip_locate_kernel" in prof and "gunzip_verify_kernel" in prof, prof
    assert "inflate_kernel" in prof or "inflate_tps_kernel" in prof, prof
    assert "par_decode_kernel" not in prof, prof
    big = make_text(64 << 20, 52)
    z = gzip_member(b"head", 6) + gzip_member(big, 6) + gzip_member(b"tail", 6)
    r = B.gunzip(z, len(big) + 8)
    prof = gpu_ctx.profile_read()
    gpu_ctx.profile(False)
    assert r.status == 1 and r.data == b"head" + big + b"tail" and r.n_members == 3
    assert "par_decode_kernel" in prof and "gunzip_locate_kernel" in prof, prof


def test_header_lookalikes_without_end(gpu_ctx, oracle):
    """Input full of `1f 8b 08 08` (FNAME set) and no zero byte: every tenth byte looks like a member start whose file
    name never ends.  The candidates' header checks are bounded, so the call takes about as long as the loop does."""
    import time
    data = b"\x1f\x8b\x08\x08AAAAAA" * (400 << 10)
    t0 = time.perf_counter()
    h = _check(oracle, data, 1 << 20)
    assert time.perf_counter() - t0 < 60
    assert h.status == -5 and h.n_members == 0 and h.out_len == 0
    # the same after a real member, and a member whose header is longer than the bounded check
    m = gzip_member(b"payload" * 1000, name=b"n" * 5000, extra=b"e" * 3000)
    h = _check(oracle, m + m + data[: 1 << 20], 1 << 20)
    assert h.status == -5 and h.n_members == 2


def test_device_call_without_room_or_output_buffer(gpu_ctx):
    import ctypes as C
    import torch
    B, capi = pkg("batch"), pkg("capi")
    d_in = torch.frombuffer(bytearray(gzip_member(b"") * 3), dtype=torch.uint8).cuda()
    res = capi.GunzipResult()
    rc = capi.load().zs_gunzip_dev(gpu_ctx.handle, B._ptr(d_in), d_in.numel(), None, 0, C.byref(res), None, 0)
    assert rc == 0 and (res.status, res.n_members, res.out_len, res.in_used) == (1, 3, 0, d_in.numel())
    d_in = torch.frombuffer(bytearray(gzip_member(b"x")), dtype=torch.uint8).cuda()
    rc = capi.load().zs_gunzip_dev(gpu_ctx.handle, B._ptr(d_in), d_in.numel(), None, 0, C.byref(res), None, 0)
    assert rc == 0 and (res.status, res.n_members, res.out_len) == (-5, 0, 0)
