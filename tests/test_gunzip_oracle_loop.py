"""CPU check of the multi-member reference loop the gunzip GPU tests compare with: on valid files it reads what
Python's own member loop (zlib.decompressobj(31) / unused_data) reads, member for member, including when the input and
the room are handed over in small pieces."""
import zlib

import pytest

from gunzip_cases import Writer, bgzf, gzip_member, oracle_gunzip, python_gunzip


def _files():
    text = bytes(range(256)) * 300 + b"the quick brown fox " * 5000
    w = Writer()
    for i, n in enumerate((0, 1, 4096, 70000, 3)):
        piece = text[i * 1000: i * 1000 + n]
        w.add(gzip_member(piece, 6, text=True, extra=b"xy" * i, name=b"f%d" % i if i & 1 else None,
                          comment=b"c" if i & 2 else None, hcrc=bool(i & 1)), n)
    yield "mixed headers", w.data(), w.out_pos
    b = bgzf(text * 3, 6)
    yield "bgzf", b.data(), b.out_pos
    yield "stored wrapping gzip", zlib.compress(b.data(), 0, wbits=31) + b.data(), 2 * b.out_pos
    yield "one member", zlib.compress(text, 9, wbits=31), len(text)


@pytest.mark.parametrize("step_in,step_out", [(1 << 20, 8 << 20), (777, 1000)])
def test_oracle_loop_matches_python_member_loop(oracle, step_in, step_out):
    for name, data, total in _files():
        want, members = python_gunzip(data)
        r = oracle_gunzip(oracle, data, total + 64, step_in, step_out)
        assert r.ret == oracle.Z_STREAM_END, name
        assert r.out == want and r.members == members and r.in_used == len(data), name


def test_oracle_loop_edges(oracle):
    m = zlib.compress(b"abc" * 1000, 6, wbits=31)
    r = oracle_gunzip(oracle, m + m + b"\0\0\0\0", 10000)
    assert (r.ret, r.msg, r.members, r.start) == (oracle.Z_DATA_ERROR, "incorrect header check", 2, 2 * len(m))
    r = oracle_gunzip(oracle, b"", 100)
    assert (r.ret, r.members, r.out) == (oracle.Z_BUF_ERROR, 0, b"")
    r = oracle_gunzip(oracle, m + m, 4500)
    assert (r.ret, r.members, len(r.out), r.start) == (oracle.Z_BUF_ERROR, 1, 4500, len(m))
