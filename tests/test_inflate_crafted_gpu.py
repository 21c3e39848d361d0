"""GPU: hand-built deflate streams (deflate_craft) through every decoder of the engine.

C zlib never writes these shapes: one-code and no-code distance sets, a literal/length set holding only EOB,
copies from 32768 back, length 258 as code 284 + 31, repeats across the tree boundary, 16 repeating a zero, 7-bit
code-length codes, table-filling sets with 15-bit codes, stored blocks at every bit phase, thousands of block starts
per MiB, junk bits behind the final block.  Nor does it write the errors: each block-layer message has a minimal
trigger, placed at the start of a stream, behind 32 KiB of output and several segments deep in a spliced stream.

Every decoder is held to the reference (the oracle's restatement of inflate()) and to its sibling path: the batch
kernels (warp and thread per stream), the segment-parallel decoder against the serial one, the index build and its
extracts, gunzip, and the streaming shim under call schedules."""
import os
import random
import zlib

import pytest

import deflate_craft as D
from conftest import pkg
from gunzip_cases import Writer
from test_gunzip_gpu import _check as gunzip_check
from test_inflate_index_gpu import _check_extract, _check_windows, _random_ranges, _rule, _stream_dev
from test_stream_inflate_schedules_gpu import check_schedule, random_schedule
from zran_check import block_starts

pytestmark = pytest.mark.gpu

PIECE = 256 << 10          # output of one bulk piece of a spliced stream
BEFORE = 3                 # bulk pieces ahead of the crafted blocks


def _deep(case, seed, sync_every=64 << 10):
    return D.deep_stream(case, False, seed, before=BEFORE, piece=PIECE, sync_every=sync_every, after=2)


def _behind(case, final=False):
    pieces = [D.bulk(D.text(40000, 11)), D.crafted(case, final)]
    return D.splice(pieces + ([] if final else [D.end_piece()]))


@pytest.fixture(scope="module")
def valid(oracle):
    return D.valid_cases(oracle)


def _errors(where, sync_every=64 << 10):
    """(name, raw stream, message) of every error case at one position (deep: spliced with flush points every
    `sync_every` bytes of output, or with none but the two around the crafted blocks)."""
    out = []
    for k, (name, case, msg, start_only) in enumerate(D.ERRORS):
        if where == "start":
            out.append((name, D.crafted(case, True), msg))
        elif start_only:
            continue
        elif where == "behind":
            out.append((name, D.splice([D.bulk(D.text(40000, 12)), D.crafted(case, False)]), msg))
        else:
            out.append((name, _deep(case, 100 + k, sync_every), msg))
    if where == "deep":   # the too-far trigger can only come first; the stream is long all the same
        out += [(name, D.deep_stream(case, False, 99, before=0, piece=PIECE, sync_every=sync_every, after=4), msg)
                for name, case, msg, start_only in D.ERRORS if start_only]
    return out


def _reference(oracle, s, wbits, cap, dictionary=None):
    st = oracle.InflateStream(wbits)
    if dictionary:
        assert st.set_dictionary(dictionary) == oracle.Z_OK
    ret, out, used = st.step(s, cap, oracle.Z_FINISH)
    msg = st.msg if ret == oracle.Z_DATA_ERROR else ""
    st.close()
    return ret, out, used, msg


def _batch_same_as_reference(oracle, streams, wbits, caps, names, dicts=None):
    r = pkg("batch").inflate_batch(streams, wbits, caps, dicts)
    for i, s in enumerate(streams):
        ret, out, used, msg = _reference(oracle, s, wbits, caps[i], dicts[i] if dicts else None)
        what = (names[i], wbits, int(r.status[i]), ret, r.message(i), msg)
        assert int(r.status[i]) == ret, what
        assert r.output(i) == out, (what, len(r.output(i)), len(out))
        if ret == oracle.Z_DATA_ERROR:
            assert r.message(i) == msg, what
        elif not (ret == oracle.Z_BUF_ERROR and len(out) == caps[i]):
            # (when the output room runs out, the reference's count holds the bytes it pulled for the symbol that did
            # not fit, and the kernels' count does not: a known difference, noted at store_result)
            assert int(r.in_used[i]) == used, (what, int(r.in_used[i]), used)
    return r


# ---- batch kernels -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("wbits", [-15, 15, 31, 47])
@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_batch_kernels(gpu_ctx, oracle, monkeypatch, valid, kernel, wbits):
    monkeypatch.setenv("ZS_INFLATE_TPS" if kernel == "thread" else "ZS_INFLATE_WARP", "1")
    names, streams, caps, msgs = [], [], [], []
    for name, case in valid:
        for where, raw in (("start", D.crafted(case, True)), ("behind", _behind(case))):
            out = zlib.decompressobj(-15).decompress(raw)
            names.append(f"{name}@{where}")
            streams.append(D.wrap(raw, wbits))
            caps.append(len(out) + 64)
            msgs.append(None)
    for where in ("start", "behind", "deep"):
        if where == "deep" and wbits not in (-15, 31):
            continue
        for name, raw, msg in _errors(where):
            names.append(f"{name}@{where}")
            streams.append(D.wrap(raw, wbits))
            caps.append(4 << 20)
            msgs.append(msg)
    assert len(streams) >= 32
    r = _batch_same_as_reference(oracle, streams, wbits, caps, names)
    for i, msg in enumerate(msgs):
        if msg is None:
            assert int(r.status[i]) == 1, (names[i], int(r.status[i]), r.message(i))
        else:
            assert int(r.status[i]) == -3 and r.message(i) == msg, (names[i], int(r.status[i]), r.message(i))
    if wbits == -15:   # copies that reach back to the first byte of a preset dictionary, with and without it
        s = D.crafted(D.dict_case, True)
        dicts = [D.DICT if i % 2 == 0 else None for i in range(32)]
        r = _batch_same_as_reference(oracle, [s] * 32, -15, [4096] * 32, [f"dict{i}" for i in range(32)], dicts)
        assert int(r.status[0]) == 1 and int(r.status[1]) == -3


@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_invalid_code_in_the_last_bits(gpu_ctx, oracle, monkeypatch, kernel):
    """An invalid code word that starts 1 ... 14 bits before the end of a raw stream: the reference's entry for it is
    one bit wide, so the verdict is a data error, not a want of input."""
    monkeypatch.setenv("ZS_INFLATE_TPS" if kernel == "thread" else "ZS_INFLATE_WARP", "1")
    names, streams, msgs = [], [], []
    for name, lit, dist, before, bit, msg in D.TAIL_TRIGGERS:
        for r in range(1, 15):
            names.append(f"{name}@last{r}")
            streams.append(D.tail_trigger(lit, dist, before, bit, r))
            msgs.append(msg)
    r = _batch_same_as_reference(oracle, streams, -15, [1024] * len(streams), names)
    for i, msg in enumerate(msgs):
        assert int(r.status[i]) == -3 and r.message(i) == msg, (names[i], int(r.status[i]), r.message(i))


@pytest.mark.parametrize("wbits", [-15, 15, 31, 47])
@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_truncation_and_output_room(gpu_ctx, oracle, monkeypatch, valid, kernel, wbits):
    """Every small valid case cut at every byte, and given every output room from 0 to its length."""
    monkeypatch.setenv("ZS_INFLATE_TPS" if kernel == "thread" else "ZS_INFLATE_WARP", "1")
    names, streams, caps = [], [], []
    for name, case in valid:
        raw = D.crafted(case, True)
        n = len(zlib.decompressobj(-15).decompress(raw))
        if n > 4096 or len(raw) > 4096:
            continue
        s = D.wrap(raw, wbits)
        for k in range(len(s)):
            names.append(f"{name}[:{k}]")
            streams.append(s[:k])
            caps.append(n + 64)
        for cap in range(n + 1):
            names.append(f"{name} cap {cap}")
            streams.append(s)
            caps.append(cap)
    _batch_same_as_reference(oracle, streams, wbits, caps, names)


# ---- the segment-parallel decoder ----------------------------------------------------------------------------

def _one(stream, wbits, cap, dictionary=None, serial=False):
    if serial:
        os.environ["ZS_INFLATE_SERIAL"] = "1"
    try:
        return pkg("batch").inflate_batch([stream], wbits, [cap], [dictionary] if dictionary else None)
    finally:
        os.environ.pop("ZS_INFLATE_SERIAL", None)


def _par_same_as_serial_and_reference(gpu_ctx, oracle, name, s, wbits, cap, dictionary=None):
    gpu_ctx.profile(True)
    gpu_ctx.profile_read()
    p = _one(s, wbits, cap, dictionary)
    prof = gpu_ctx.profile_read()
    gpu_ctx.profile(False)
    q = _one(s, wbits, cap, dictionary, serial=True)
    got = (int(p.status[0]), p.message(0), p.output(0), int(p.in_used[0]), int(p.checks[0]))
    assert got == (int(q.status[0]), q.message(0), q.output(0), int(q.in_used[0]), int(q.checks[0])), \
        (name, got[:2], int(q.status[0]), q.message(0))
    ret, out, used, msg = _reference(oracle, s, wbits, cap, dictionary)
    assert (got[0], got[1] if ret == oracle.Z_DATA_ERROR else "") == (ret, msg), (name, got[:2], ret, msg)
    assert got[2] == out, (name, len(got[2]), len(out))
    if ret != oracle.Z_DATA_ERROR:
        assert got[3] == used, (name, got[3], used)
    if ret == oracle.Z_STREAM_END and wbits > 0:
        st = zlib.adler32(out) if wbits == 15 else zlib.crc32(out)
        assert got[4] & 0xffffffff == st, name
    return p, prof


@pytest.mark.parametrize("variant", ["markers", "spec", "no_spec"])
def test_segment_parallel(gpu_ctx, oracle, monkeypatch, valid, variant):
    """Spliced streams with flush points every 64 KiB of output, or with none but the two around the crafted blocks
    (cuts at speculatively located block headers), the latter also with speculation off.  The parallel decoder must
    run on every stream, the error streams included."""
    if variant == "no_spec":
        monkeypatch.setenv("ZS_INFLATE_NO_SPEC", "1")
    every = (64 << 10) if variant == "markers" else 0
    for k, (name, case) in enumerate(valid):
        s = D.wrap(D.deep_stream(case, False, 200 + k, before=BEFORE, piece=PIECE, sync_every=every, after=2), 15)
        p, prof = _par_same_as_serial_and_reference(gpu_ctx, oracle, name, s, 15, 16 << 20)
        assert int(p.status[0]) == 1, (name, p.message(0))
        assert "par_decode_kernel" in prof, (name, sorted(prof))
    for name, raw, msg in _errors("deep", every):
        for wbits in (-15, 31):
            p, prof = _par_same_as_serial_and_reference(gpu_ctx, oracle, name, D.wrap(raw, wbits), wbits, 16 << 20)
            assert int(p.status[0]) == -3 and p.message(0) == msg, (name, wbits, p.message(0))
            assert "par_decode_kernel" in prof, (name, wbits, sorted(prof))
    s = D.deep_stream(D.dict_case, False, 14, before=0, piece=PIECE, sync_every=every, after=4)
    p, _ = _par_same_as_serial_and_reference(gpu_ctx, oracle, "dict", s, -15, 16 << 20, D.DICT)
    assert int(p.status[0]) == 1
    p, _ = _par_same_as_serial_and_reference(gpu_ctx, oracle, "dict missing", s, -15, 16 << 20)
    assert p.message(0) == "invalid distance too far back"


# ---- the index -------------------------------------------------------------------------------------------------

def test_index(gpu_ctx, oracle, valid):
    B = pkg("batch")
    rng = random.Random(4096)
    for k, (name, case) in enumerate(valid):
        data = D.wrap(_deep(case, 300 + k), 15)
        ret, out, _, _ = oracle.inflate(data, 15)
        assert ret == oracle.Z_STREAM_END, name
        cap = len(out) + 64
        want = _stream_dev(data, 15, None, cap)
        starts = block_starts(data, 15)
        ranges = _random_ranges(rng, len(out), 20)
        if name.startswith("far_"):             # ranges that start right before the 258-byte copies from 32768 back
            o = BEFORE * PIECE + len(D.HIST)
            ranges += [(o - 1, 300), (o, 258), (o - 5000, 10000), (o + 257, 2), (o - 40000, 41000)]
        for span in (4096, 65536):
            ix, built = B.InflateIndex.build(data, 15, span, out_cap=cap)
            got = (built.status, built.data[: built.out_len].cpu().numpy().tobytes(), built.out_len, built.in_used,
                   built.check & 0xffffffff, built.detail)
            assert got == want, name
            assert built.status == 1 and ix is not None, name
            assert [tuple(int(v) for v in p) for p in ix.points] == _rule(starts, span, len(out)), (name, span)
            if span == 65536:
                _check_windows(ix, data, out)
            _check_extract(ix, data, out, ranges)
            ix.close()
    for name, raw, msg in _errors("deep"):
        data = D.wrap(raw, 15)
        want = _stream_dev(data, 15, None, 16 << 20)
        ix, built = B.InflateIndex.build(data, 15, 65536, out_cap=16 << 20)
        got = (built.status, built.data[: built.out_len].cpu().numpy().tobytes(), built.out_len, built.in_used,
               built.check & 0xffffffff, built.detail)
        assert ix is None and got == want, name
        assert built.status == -3 and built.message == msg, (name, built.message)


# ---- gunzip ------------------------------------------------------------------------------------------------------

def _member(raw):
    return D.gzip_wrap(raw), len(zlib.decompressobj(-15).decompress(raw))


def test_gunzip(gpu_ctx, oracle, valid):
    """Files of crafted gzip members: small ones (decoded as a batch) and ones above 128 KiB of input (the one-stream
    path), then the same with each error case as the last member."""
    small = [_member(D.crafted(case, True)) for _, case in valid]
    big = [_member(D.deep_stream(case, True, 400 + k, before=2, piece=PIECE)) for k, (_, case) in enumerate(valid[:6])]
    assert all(len(m) > (128 << 10) for m, _ in big)
    for members in (small, big + small[:3], small[:2] + big[:2] + small[2:]):
        w = Writer()
        for m, n in members:
            w.add(m, n)
        h = gunzip_check(oracle, w.data(), out_cap=w.out_pos + 64, writer=w)
        assert h.status == 1 and h.n_members == len(members)
    for where in ("start", "deep"):
        for name, raw, msg in _errors(where):
            data = b"".join(m for m, _ in small[:2]) + D.gzip_wrap(raw)
            h = gunzip_check(oracle, data, out_cap=16 << 20)
            assert h.status == -3 and h.message == msg and h.n_members == 2, (name, where, h.message)


# ---- the streaming shim -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("wbits", [15, -15])
def test_stream_shim_schedules(gpu_ctx, oracle, valid, wbits):
    for k, (name, case) in enumerate(valid):
        raw = _deep(case, 500 + k)
        data = D.wrap(raw, wbits)
        expect = zlib.decompressobj(-15).decompress(raw)
        rng = random.Random(k)
        sched = random_schedule(rng, len(data), lo=4096, hi=1 << 20, forced=0.3, rooms=(1 << 20, 4 << 20))
        check_schedule(oracle, data, wbits, sched, seed=f"{name} {k}", expect=expect)
    for k, (name, raw, msg) in enumerate(_errors("deep")):
        rng = random.Random(1000 + k)
        data = D.wrap(raw, wbits)
        sched = random_schedule(rng, len(data), lo=4096, hi=1 << 20, forced=0.3, rooms=(1 << 20,))
        g = check_schedule(oracle, data, wbits, sched, seed=f"{name} {k}")
        assert g["msg"] == msg, (name, g["msg"])
