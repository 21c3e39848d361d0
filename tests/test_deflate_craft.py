"""The hand-built deflate streams of deflate_craft against C zlib and the oracle (no GPU): every valid case decodes to
the same bytes with both, every error case gives its named message from both, and the seeded search for
table-filling length sets finds what it found when it was written down."""
import zlib

import pytest

import deflate_craft as D

RAW = -15


def _zlib(stream, wbits=RAW, zdict=None):
    """C zlib: (output, None) or (output before the error, message)."""
    d = zlib.decompressobj(wbits, zdict=zdict) if zdict else zlib.decompressobj(wbits)
    try:
        out = d.decompress(stream)
    except zlib.error as e:
        return None, str(e).split(": ", 1)[1]
    assert d.eof, "C zlib wants more input"
    return out, None


def _oracle(oracle, stream, wbits=RAW, cap=1 << 22, dictionary=None):
    s = oracle.InflateStream(wbits)
    if dictionary:
        assert s.set_dictionary(dictionary) == oracle.Z_OK
    ret, out, used = s.step(stream, cap, oracle.Z_FINISH)
    msg = s.msg
    s.close()
    return ret, out, used, msg


def test_writer_bits_and_codes():
    w = D.BitWriter()
    w.bits(1, 1)
    w.bits(2, 2)
    w.code(0b110, 3)           # MSB first: bits 1, 1, 0
    assert w.n == 6 and w.data() == bytes([0b011101]) and w.data(fill=1) == bytes([0b11011101])
    assert D.canonical([2, 1, 3, 3]) == [0b10, 0b0, 0b110, 0b111]
    assert D.canonical([1, 0]) == [0, None]                                    # incomplete: one 1-bit code
    assert D.length_code(258) == (285, 0, 0) and D.length_code(257) == (284, 30, 5)
    assert D.dist_code(32768) == (29, 8191, 13) and D.dist_code(1) == (0, 0, 0)
    lens = [0] * 100 + [3, 3, 3] + [7] * 20 + [0] * 5
    assert D.rle_expand(D.rle(lens), len(lens)) == lens
    assert D.rle_expand(D.zero16(D.rle(lens)), len(lens)) == lens
    assert (18, 127) in D.rle([0] * 138) and (16, 0) in D.zero16(D.rle([0] * 20))
    assert (16, 0) in D.zero16(D.rle([1] + [0] * 20)) and (17, 0) in D.zero16(D.rle([1] + [0] * 6))


def test_repeats_cross_the_tree_boundary():
    """The default run-length code of the repeat cases runs one 16 over the literal/length -> distance boundary."""
    lit, dist = D._X8, [4] * 16
    pos, crossing = 0, False
    for s, x in D._X8_SEQ:
        n = 1 if s < 16 else (3 + x if s in (16, 17) else 11 + x)
        crossing |= s == 16 and pos < len(lit) < pos + n
        pos += n
    assert crossing and pos == len(lit) + len(dist)
    # 16 repeats a zero right after a 17 and right after an 18
    z = D.zero16(D._X8_SEQ)
    assert {z[i - 1][0] for i in range(1, len(z)) if z[i][0] == 16 and z[i - 1][0] in (17, 18)} == {17, 18}
    # the 7-bit code-length codes go to symbols the sequence writes
    cl = D.chain_cl(D._X8_SEQ)
    assert max(cl) == 7 and {s for s, _ in D._X8_SEQ if cl[s] == 7} == {17, 18}


@pytest.mark.parametrize("final", [True, False], ids=["alone", "spliced"])
def test_valid_cases_decode_alike(oracle, final):
    for name, case in D.valid_cases(oracle):
        s = D.crafted(case, final)
        if not final:
            s = D.splice([D.bulk(D.text(40000, 1)), s, D.end_piece()])
        want, msg = _zlib(s)
        assert msg is None, (name, msg)
        ret, out, used, _ = _oracle(oracle, s)
        assert ret == oracle.Z_STREAM_END and out == want and used == len(s), name
        for wbits in (15, 31):
            w = D.wrap(s, wbits)
            assert _zlib(w, wbits) == (want, None), (name, wbits)
            assert _oracle(oracle, w, wbits)[:2] == (oracle.Z_STREAM_END, want), (name, wbits)


def test_dictionary_case(oracle):
    s = D.crafted(D.dict_case, True)
    want, msg = _zlib(s, zdict=D.DICT)
    assert msg is None and want == D.DICT[:10] + b"a" + D.DICT[:20]
    assert _oracle(oracle, s, dictionary=D.DICT)[:2] == (oracle.Z_STREAM_END, want)
    assert _zlib(s)[1] == "invalid distance too far back"


@pytest.mark.parametrize("where", ["start", "behind_32k", "deep"])
def test_error_cases_name_their_message(oracle, where):
    for name, case, message, start_only in D.ERRORS:
        if start_only and where != "start":
            continue
        if where == "start":
            s = D.crafted(case, True)
        elif where == "behind_32k":
            s = D.splice([D.bulk(D.text(40000, 2)), D.crafted(case, False)])
        else:
            s = D.deep_stream(case, False, seed=3, before=2, piece=200 << 10, after=1)
        assert _zlib(s)[1] == message, (name, where, _zlib(s)[1])
        ret, _, _, msg = _oracle(oracle, s)
        assert ret == oracle.Z_DATA_ERROR and msg == message, (name, where, msg)


def test_invalid_code_in_the_last_bits(oracle):
    """An invalid code word 1 ... 14 bits before the end of a raw stream is a data error: the reference's
    invalid-code entry is one bit wide."""
    for name, lit, dist, before, bit, message in D.TAIL_TRIGGERS:
        for r in range(1, 15):
            s = D.tail_trigger(lit, dist, before, bit, r)
            assert _zlib(s)[1] == message, (name, r)
            ret, _, _, msg = _oracle(oracle, s)
            assert ret == oracle.Z_DATA_ERROR and msg == message, (name, r, ret, msg)


def test_one_code_distance_stream_from_the_issue(oracle):
    """14 bytes: a dynamic block whose distance set is one 1-bit code, then that set's unused bit value."""
    bad, good = bytes.fromhex("0dc0010900000080a0adfe3f517a"), bytes.fromhex("0dc0010900000080a0adfe3f515a")
    assert _zlib(good) == (b"aaaa", None) and _zlib(bad)[1] == "invalid distance code"
    ret, out, _, msg = _oracle(oracle, bad)
    assert (ret, out, msg) == (oracle.Z_DATA_ERROR, b"a", "invalid distance code")


def test_table_filling_search(oracle):
    """The seeded search over complete length sets: the most decode-table entries found for 286 literal/length codes
    (9 root bits, ceiling 852) and 30 distance codes (6 root bits, ceiling 592), with 15-bit codes in both."""
    lit, lit_used, dist, dist_used = D.table_filling_sets(oracle)
    assert (lit_used, dist_used) == (834, 584)
    assert len(lit) == 286 and len(dist) == 30 and max(lit) == 15 and max(dist) == 15
    for lens in (lit, dist):
        assert sum(2 ** (15 - l) for l in lens) == 2 ** 15              # complete
    assert D.table_used(oracle, 1, lit, 9) == (0, lit_used)
    assert D.table_used(oracle, 2, dist, 6) == (0, dist_used)
