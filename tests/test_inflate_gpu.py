"""GPU parity: K6/K7 batch inflate against the oracle restatement of inflate.ts / inftrees.ts /
inffast.ts (incl. deflate64) and against the reference's known-answer vectors -- bit-exact output,
total_in / total_out, return code and message."""
import random
import zlib

import numpy as np
import pytest

from conftest import make_mixed, make_text, pkg, rand_bytes

pytestmark = pytest.mark.gpu


def _run(streams, wbits, caps, dicts=None):
    return pkg("batch").inflate_batch(streams, wbits, caps, dicts)


def _same_as_oracle(oracle, streams, wbits, caps, dicts=None, check_used=True):
    r = _run(streams, wbits, caps, dicts)
    for i, s in enumerate(streams):
        ret, out, used, check = oracle.inflate(s, wbits, int(caps[i]), dicts[i] if dicts else None)
        assert int(r.status[i]) == ret, (i, int(r.status[i]), ret, r.message(i))
        assert r.output(i) == out, (i, len(r.output(i)), len(out))
        if check_used and ret in (oracle.Z_STREAM_END, oracle.Z_DATA_ERROR):
            pass
        if ret == oracle.Z_STREAM_END:
            assert int(r.in_used[i]) == used, (i, int(r.in_used[i]), used)
    return r


def test_kats(gpu_ctx, oracle, kat):
    for v in kat["inflate"]:
        data = bytes.fromhex(v["in_hex"])
        r = _run([data], v["window_bits"], [1 << 17])
        ret = int(r.status[0])
        if "ret" in v:
            assert ret == v["ret"], v["ref"]
        if "ret_le" in v:
            assert ret <= v["ret_le"], v["ref"]
        if "ret_not" in v:
            assert ret not in v["ret_not"], v["ref"]
        if "out_hex" in v:
            assert r.output(0) == bytes.fromhex(v["out_hex"]), v["ref"]
        if "out_len" in v:
            assert r.output(0) == bytes([v["out_byte"]]) * v["out_len"], v["ref"]


def test_deflate64_fixtures(gpu_ctx, oracle, fixtures64):
    streams = [f["data"] for f in fixtures64]
    caps = [f["out_len"] + 100 for f in fixtures64]
    r = _same_as_oracle(oracle, streams, -16, caps)
    for i, f in enumerate(fixtures64):
        out = r.output(i)
        assert int(r.status[i]) == 1 and len(out) == f["out_len"], f["name"]
        assert zlib.crc32(out) == f["crc32"] and zlib.adler32(out) == f["adler32"], f["name"]
        assert int(r.checks[i]) == f["crc32"], f["name"]          # raw streams report crc32(out)
        assert int(r.in_used[i]) == f["length"]


@pytest.mark.parametrize("wbits", [15, -15, 31, 47])
def test_zlib_streams_all_levels(gpu_ctx, oracle, wbits):
    streams, datas = [], []
    enc_wbits = 31 if wbits == 47 else wbits
    for level in (0, 1, 6, 9):
        for data in (make_text(120000, level), make_mixed(90000, level), rand_bytes(70000, level), b"", b"a",
                     bytes(100000), bytes(j % 251 for j in range(60000))):
            co = zlib.compressobj(level, 8, enc_wbits)
            streams.append(co.compress(data) + co.flush())
            datas.append(data)
    caps = [len(d) + 16 for d in datas]
    r = _same_as_oracle(oracle, streams, wbits, caps)
    for i, d in enumerate(datas):
        assert int(r.status[i]) == 1 and r.output(i) == d
        if wbits == 15:
            assert int(r.checks[i]) == zlib.adler32(d)
        if wbits in (31, 47):
            assert int(r.checks[i]) == zlib.crc32(d)


def test_many_small_gzip_records(gpu_ctx, oracle):
    # config 4 shape: independent 4 KiB gzip records, ~5 % stored (random) records, crc32 verify
    rnd = random.Random(4)
    text = make_text(4096 * 400, 11)
    streams, datas = [], []
    for i in range(400):
        d = rnd.randbytes(4096) if rnd.random() < 0.05 else text[i * 4096: (i + 1) * 4096]
        co = zlib.compressobj(6, 8, 31)
        streams.append(co.compress(d) + co.flush())
        datas.append(d)
    r = _run(streams, 31, [4096] * 400)
    assert (r.status == 1).all()
    for i, d in enumerate(datas):
        assert r.output(i) == d and int(r.checks[i]) == zlib.crc32(d) and int(r.in_used[i]) == len(streams[i])


def test_errors_match_oracle(gpu_ctx, oracle):
    data = make_text(50000, 5)
    z = zlib.compress(data, 6)
    g = zlib.compressobj(6, 8, 31)
    gz = g.compress(data) + g.flush()
    streams, caps, wb = [], [], 15
    bad = bytearray(z); bad[-1] ^= 0xFF
    streams += [z[:-5], bytes(bad), z, z[:100], b"\x78", b"\x79\x9c\x03\x00", b"\x78\x9c\x07\x00"]
    caps += [60000, 60000, 1000, 60000, 100, 100, 100]
    r = _same_as_oracle(oracle, streams, wb, caps)
    assert int(r.status[1]) == -3 and r.message(1) == "incorrect data check"
    assert int(r.status[5]) == -3 and r.message(5) == "incorrect header check"
    assert int(r.status[6]) == -3 and r.message(6) == "invalid block type"
    badg = bytearray(gz); badg[-2] ^= 1
    r = _same_as_oracle(oracle, [gz, bytes(badg), gz[:-1]], 31, [60000, 60000, 60000])
    assert int(r.status[0]) == 1 and int(r.status[1]) == -3 and r.message(1) == "incorrect length check"
    assert int(r.status[2]) == -5
    # bit flips anywhere in the stream: same verdict, same output prefix as the oracle
    rnd = random.Random(9)
    streams = []
    for _ in range(300):
        junk = bytearray(z[:600])
        junk[rnd.randrange(2, 600)] ^= 1 << rnd.randrange(8)
        streams.append(bytes(junk))
    r = _same_as_oracle(oracle, streams, 15, [60000] * len(streams))
    msgs = {r.message(i) for i in range(len(streams)) if int(r.status[i]) == -3}
    assert msgs  # at least some data errors, all with reference messages
    # deflate64-specific header rule (coverage-too-many-len.spec.ts:28-46)
    def hdr(nlen, ndist):
        v = 0b101 | ((nlen - 257) << 3) | ((ndist - 1) << 8)
        return v.to_bytes(3, "little") + bytes(8)
    r = _same_as_oracle(oracle, [hdr(257, 31), hdr(287, 1)], -15, [64, 64])
    assert int(r.status[0]) == -3 and r.message(0) == "too many length or distance symbols"
    r = _same_as_oracle(oracle, [hdr(257, 31), hdr(287, 1)], -16, [64, 64])
    assert r.message(0) != "too many length" and r.message(1) == "too many length"


def test_preset_dictionary_raw(gpu_ctx, oracle):
    d = make_text(200000, 3)
    dic, body = d[:40000], d[40000:140000]
    co = zlib.compressobj(6, 8, -15, 8, 0, dic[-32768:])
    z = co.compress(body) + co.flush()
    r = _same_as_oracle(oracle, [z, z], -15, [len(body), len(body)], [dic[-32768:], None])
    assert int(r.status[0]) == 1 and r.output(0) == body
    assert int(r.status[1]) == -3 and r.message(1) == "invalid distance too far back"


def test_window_wrap_and_long_matches(gpu_ctx, oracle):
    # test-inffast-window-wrap.ts: 64 KiB+ of a 32-byte pattern; plus runs that use length 258
    pat = bytes(range(32)) * 4096
    runs = b"".join(bytes([i]) * 1000 for i in range(200))
    streams = [zlib.compress(pat, 9), zlib.compress(runs, 9), zlib.compress(pat + runs, 1)]
    r = _same_as_oracle(oracle, streams, 15, [len(pat), len(runs), len(pat) + len(runs)])
    assert (r.status == 1).all()


def test_thread_per_stream_kernel_matches_oracle(gpu_ctx, oracle, fixtures64, monkeypatch):
    # big batches (>= 16384 streams) take the thread-per-stream kernel; ZS_INFLATE_TPS forces it for
    # the sizes used here: same verdicts, bytes and counters as the oracle
    monkeypatch.setenv("ZS_INFLATE_TPS", "1")
    rnd = random.Random(21)
    text = make_text(1 << 20, 13)
    streams, caps, datas = [], [], []
    for i in range(1500):
        n = rnd.choice((0, 1, 5, 100, 700, 4096, 9000))
        d = rnd.randbytes(n) if i % 17 == 0 else text[i * 600: i * 600 + n]
        lvl = rnd.choice((0, 1, 6, 9))
        co = zlib.compressobj(lvl, 8, 31)
        s = co.compress(d) + co.flush()
        kind = i % 10
        cap = len(d)
        if kind == 7 and len(s) > 30:
            s = s[: rnd.randrange(11, len(s) - 1)]                        # truncated
        elif kind == 8 and len(s) > 30:
            b = bytearray(s); b[rnd.randrange(10, len(s))] ^= 1 << rnd.randrange(8); s = bytes(b)   # corrupted
        elif kind == 9 and n > 10:
            cap = n // 2                                                   # output too small
        streams.append(s); caps.append(cap); datas.append(d)
    r = _same_as_oracle(oracle, streams, 31, caps)
    good = [i for i in range(1500) if i % 10 < 7]
    for i in good:
        assert int(r.status[i]) == 1 and r.output(i) == datas[i] and int(r.checks[i]) == zlib.crc32(datas[i])
    # zlib wrapper, raw with dictionary, and deflate64 through the same kernel
    zs = [zlib.compress(text[i * 512: i * 512 + 3000], 6) for i in range(1100)]
    r = _same_as_oracle(oracle, zs, 15, [3000] * 1100)
    assert (r.status == 1).all()
    dic = text[:20000]
    raws, dicts = [], []
    for i in range(1100):
        co = zlib.compressobj(6, 8, -15, 8, 0, dic)
        raws.append(co.compress(text[30000 + i * 100: 33000 + i * 100]) + co.flush())
        dicts.append(dic if i % 2 == 0 else None)
    r = _same_as_oracle(oracle, raws, -15, [3000] * 1100, dicts)
    assert int(r.status[0]) == 1 and int(r.status[1]) == -3 and r.message(1) == "invalid distance too far back"
    f64 = [f for f in fixtures64 if f["out_len"] < 200000]
    streams = [f64[i % len(f64)]["data"] for i in range(1030)]
    caps = [f64[i % len(f64)]["out_len"] + 8 for i in range(1030)]
    r = _same_as_oracle(oracle, streams, -16, caps)
    for i in range(1030):
        f = f64[i % len(f64)]
        assert int(r.status[i]) == 1 and int(r.checks[i]) == f["crc32"], f["name"]
    kats = [bytes.fromhex("4b1cfdff07a3e5030000")] * 1024
    r = _run(kats, -16, [70000] * 1024)
    assert all(r.output(i) == b"a" * 66539 for i in (0, 511, 1023))


@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_generated_deflate64_streams(gpu_ctx, oracle, monkeypatch, kernel):
    """Config 5 of the scope table beyond the ten fixtures: raw deflate64 streams from the test-side
    encoder -- distances up to 65536 (codes 30/31), lengths up to 65538 (code 285 with 16 extra bits) --
    decoded with windowBits -16 by both kernels, bit-exact with the oracle; the same streams are a
    data error under windowBits -15."""
    monkeypatch.setenv("ZS_INFLATE_TPS" if kernel == "thread" else "ZS_INFLATE_WARP", "1")
    B = pkg("batch")
    rnd = np.random.default_rng(65)
    blk = rnd.integers(0, 256, 3000, dtype=np.uint8).tobytes()
    cases = []
    for i in range(48):
        gap = int(rnd.integers(33000, 62000))
        far = blk + rnd.integers(0, 256, gap, dtype=np.uint8).tobytes() + blk + bytes(int(rnd.integers(0, 50))) + blk
        runs = bytes(int(rnd.integers(300, 90000))) + b"xyz" * int(rnd.integers(100, 30000)) + bytes([i]) * int(rnd.integers(259, 70000))
        cases += [far, runs, make_text(int(rnd.integers(1, 200000)), 70 + i), b""]
    streams, raws = [], []
    for j, c in enumerate(cases):
        streams.append(oracle.deflate64_encode(c, 65538 if j % 3 else 258))
        raws.append(c)
    caps = [len(c) + 16 for c in raws]
    res = B.inflate_batch(streams, -16, caps, ctx=gpu_ctx)
    for j, c in enumerate(raws):
        assert res.status[j] == oracle.Z_STREAM_END, (j, res.status[j])
        assert res.output(j) == c, j
        assert int(res.in_used[j]) == len(streams[j])
    # plain deflate must reject what only deflate64 allows
    bad = B.inflate_batch(streams[:8], -15, caps[:8], ctx=gpu_ctx)
    for j in range(8):
        ret, _, _, _ = oracle.inflate(streams[j], -15, caps[j])
        assert bad.status[j] == ret, (j, bad.status[j], ret)


@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_fuzzed_streams_same_verdict_and_message(gpu_ctx, oracle, monkeypatch, kernel):
    """The reference's fuzz strategy (test/inflate/test-fuzz.ts) against the restated reference: bit flips,
    byte stomps and truncations of zlib / gzip / raw / deflate64 streams (stored, fixed and dynamic
    blocks).  Status, strm.msg and the bytes produced before the error must all be the reference's."""
    monkeypatch.setenv("ZS_INFLATE_TPS" if kernel == "thread" else "ZS_INFLATE_WARP", "1")
    rnd = random.Random(1234)
    text = make_text(6000, 81)
    bases = []
    for wb, zwb in ((15, 15), (31, 31), (-15, -15)):
        for level, strategy in ((0, 0), (1, 0), (6, 0), (6, zlib.Z_FIXED), (9, zlib.Z_HUFFMAN_ONLY)):
            co = zlib.compressobj(level, zlib.DEFLATED, zwb, 8, strategy)
            bases.append((wb, co.compress(text) + co.flush()))
    bases.append((-16, oracle.deflate64_encode(text + bytes(70000) + text, 65538)))
    per_wb = {}
    for wb, z in bases:
        lst = per_wb.setdefault(wb, [])
        for _ in range(60):
            s = bytearray(z)
            kind = rnd.randrange(4)
            if kind == 0:
                s[rnd.randrange(len(s))] ^= 1 << rnd.randrange(8)
            elif kind == 1:
                s[rnd.randrange(len(s))] = rnd.randrange(256)
            elif kind == 2:
                s = s[: rnd.randrange(1, len(s))]
            else:
                p = rnd.randrange(len(s))
                s[p: p + 3] = bytes(rnd.randrange(256) for _ in range(3))
            lst.append(bytes(s))
    n_err = 0
    for wb, streams in per_wb.items():
        cap = 100000 if wb == -16 else 8000
        r = _run(streams, wb, [cap] * len(streams))
        for i, s in enumerate(streams):
            st = oracle.InflateStream(wb)
            ret, out, used = st.step(s, cap, oracle.Z_FINISH)
            assert int(r.status[i]) == ret, (kernel, wb, i, int(r.status[i]), ret, r.message(i), st.msg)
            assert r.output(i) == out, (kernel, wb, i, len(r.output(i)), len(out))
            if ret == oracle.Z_DATA_ERROR:
                assert r.message(i) == st.msg, (kernel, wb, i, r.message(i), st.msg)
                n_err += 1
            st.close()
    assert n_err > 100


def _gzip_header(flg, method=8, hcrc_ok=True):
    h = bytes([0x1F, 0x8B, method, flg]) + (123456789).to_bytes(4, "little") + b"\x00\x03"
    if flg & 4:
        h += (5).to_bytes(2, "little") + b"ab\x00cd"
    if flg & 8:
        h += b"name.txt\x00"
    if flg & 16:
        h += b"a comment\x00"
    if flg & 2:
        h += ((zlib.crc32(h) & 0xFFFF) ^ (0 if hcrc_ok else 1)).to_bytes(2, "little")
    return h


def _zlib_header(cinfo=7, method=8, fdict=False, fcheck_ok=True):
    cmf, flg = cinfo << 4 | method, 0x80 | (0x20 if fdict else 0)
    flg += (31 - (cmf * 256 + flg) % 31) % 31
    return bytes([cmf, flg + (0 if fcheck_ok else 1)]) + (b"\x01\x02\x03\x04" if fdict else b"")


@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_wrapper_header_and_trailer_verdicts(gpu_ctx, oracle, monkeypatch, kernel):
    """zlib and gzip wrappers built by hand -- every combination of the gzip header fields, a right and a wrong
    header crc, truncation at every header byte and inside the trailer, reserved flags, other methods, a bad
    FCHECK, a window above 32 KiB, FDICT -- decoded as windowBits 15, 31 and 47 by both kernels: status,
    message, output and consumed input must be the reference's."""
    monkeypatch.setenv("ZS_INFLATE_TPS" if kernel == "thread" else "ZS_INFLATE_WARP", "1")
    data = make_text(3000, 17)
    co = zlib.compressobj(6, 8, -15)
    body = co.compress(data) + co.flush()
    gz_trailer = zlib.crc32(data).to_bytes(4, "little") + len(data).to_bytes(4, "little")
    z_trailer = zlib.adler32(data).to_bytes(4, "big")
    streams = []
    for flg in range(32):   # FTEXT 1, FHCRC 2, FEXTRA 4, FNAME 8, FCOMMENT 16
        streams.append(_gzip_header(flg) + body + gz_trailer)
        if flg & 2:
            streams.append(_gzip_header(flg, hcrc_ok=False) + body + gz_trailer)
    full = _gzip_header(31)
    streams += [full[:k] for k in range(len(full))]
    streams += [_gzip_header(8 | bit) + body + gz_trailer for bit in (0x20, 0x40, 0x80)]
    streams.append(_gzip_header(0, method=7) + body + gz_trailer)
    gz = _gzip_header(0) + body + gz_trailer
    streams += [gz[:-k] for k in range(1, 9)]
    for cinfo, method, ok in ((7, 8, True), (0, 8, True), (7, 7, True), (7, 8, False), (8, 8, True), (15, 8, True)):
        streams.append(_zlib_header(cinfo, method, fcheck_ok=ok) + body + z_trailer)
    zd = _zlib_header(fdict=True)
    streams += [zd[:k] for k in range(len(zd) + 1)] + [zd + body + z_trailer]
    zs = _zlib_header() + body + z_trailer
    streams += [zs[:-k] for k in range(1, 5)]
    streams += [streams[0]] * (32 - len(streams))   # ZS_INFLATE_TPS applies to batches of 32 streams or more
    cap = len(data) + 64
    seen = set()
    for wb in (15, 31, 47):
        r = _run(streams, wb, [cap] * len(streams))
        for i, s in enumerate(streams):
            st = oracle.InflateStream(wb)
            ret, out, used = st.step(s, cap, oracle.Z_FINISH)
            what = (kernel, wb, i, int(r.status[i]), ret, r.message(i), st.msg)
            assert int(r.status[i]) == ret, what
            assert r.output(i) == out, what
            if ret == oracle.Z_DATA_ERROR:
                # (after a data error the reference's count includes the bytes already in its bit buffer)
                assert r.message(i) == st.msg, what
            else:
                assert int(r.in_used[i]) == used, (what, int(r.in_used[i]), used)
            seen.add((ret, st.msg))
            st.close()
    assert {oracle.Z_STREAM_END, oracle.Z_NEED_DICT, oracle.Z_BUF_ERROR} <= {ret for ret, _ in seen}
    assert {"header crc mismatch", "unknown header flags set", "unknown compression method", "incorrect header check",
            "invalid window size"} <= {msg for _, msg in seen}


def test_randomised_soak_inflate_and_api(gpu_ctx):
    """tools/soak_inflate.py for a few seconds: random batches (valid, truncated, corrupted, too-small
    outputs; zlib / gzip / raw / auto / deflate64) on both kernels against the oracle, and random piece /
    flush patterns through the z_stream API against C zlib."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "tools", "soak_inflate.py"), "24", "3"], capture_output=True, text=True, timeout=400)
    assert p.returncode == 0 and p.stdout.count("soak ok") == 3, p.stdout[-2000:] + p.stderr[-2000:]


@pytest.mark.parametrize("n_streams", [12000, 40000])
def test_host_batch_pipelined_equals_unpipelined(gpu_ctx, monkeypatch, n_streams):
    """zs_inflate_batch slices a large batch (copies overlap the kernels); the results -- output bytes, lengths,
    consumed input, checksums, status and message of every stream, corrupt ones included -- must be those of the
    single-shot path (12000 streams: warp per stream; 40000: thread per stream in both)."""
    rnd = random.Random(n_streams)
    rec = 8192 if n_streams < 32768 else 2048
    text = make_text(rec * 512, 21)
    base = []
    for i in range(512):
        d = rnd.randbytes(rec) if i % 19 == 0 else text[i * rec: (i + 1) * rec]
        co = zlib.compressobj(6, 8, 31)
        base.append((co.compress(d) + co.flush(), d))
    streams, caps, want = [], [], []
    for i in range(n_streams):
        z, d = base[rnd.randrange(512)]
        if i % 997 == 5:                      # corrupt the deflate data of some records
            z = z[:20] + bytes([z[20] ^ 0x55]) + z[21:]
        if i % 1501 == 7:                     # and give some too little room
            caps.append(rec // 2)
        else:
            caps.append(rec)
        streams.append(z)
        want.append(d)
    assert sum(len(s) for s in streams) + sum(caps) >= 64 << 20
    r = _run(streams, 31, caps)
    monkeypatch.setenv("ZS_INFLATE_UNPIPELINED", "1")
    ref = _run(streams, 31, caps)
    monkeypatch.delenv("ZS_INFLATE_UNPIPELINED")
    assert np.array_equal(r.status, ref.status) and np.array_equal(r.out_len, ref.out_len)
    assert np.array_equal(r.in_used, ref.in_used) and np.array_equal(r.checks, ref.checks)
    assert np.array_equal(r.details, ref.details)
    assert all(r.output(i) == ref.output(i) for i in range(n_streams))
    ok = [i for i in range(n_streams) if i % 997 != 5 and i % 1501 != 7]
    assert all(int(r.status[i]) == 1 for i in ok)
    for i in ok[:: max(1, len(ok) // 300)]:
        assert r.output(i) == want[i] and int(r.checks[i]) == zlib.crc32(want[i])
    assert any(int(r.status[i]) != 1 for i in range(5, n_streams, 997))
