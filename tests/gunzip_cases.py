"""Multi-member gzip files and the reference loop that reads them, shared by the gunzip tests and tools/gunzipprof.py.

oracle_gunzip restates the reference's multi-member idiom (test/inflate/test-multistream.ts:16-79) with the oracle's
inflate: inflateInit2(31), inflate(Z_FINISH) on the rest of the input; on Z_STREAM_END inflateReset and go on behind
total_in.  The input and the output room are handed over in pieces (inflate is a resumable state machine, and with
Z_FINISH it returns Z_BUF_ERROR until it is done), so one oracle member step is one inflate(Z_FINISH) over the whole rest
of the file with all the room that is left, without copying the rest of a large file for every member.
"""
from __future__ import annotations

import struct
import zlib
from dataclasses import dataclass

BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
BGZF_BLOCK = 65280   # input bytes per BGZF block (bgzip's limit)


@dataclass
class LoopResult:
    ret: int
    msg: str
    out: bytes
    in_used: int        # total bytes consumed (file offset behind the last byte used)
    members: int        # members that ended with Z_STREAM_END
    start: int          # where the last member attempted starts
    out_start: int      # bytes produced before it


def oracle_gunzip(O, data: bytes, out_cap: int, step_in: int = 1 << 20, step_out: int = 8 << 20) -> LoopResult:
    mv = memoryview(data)
    s = O.InflateStream(31)
    pos = produced = members = 0
    out = []
    while True:
        fed = 0
        out_start = produced
        while True:
            chunk = mv[pos + fed: pos + fed + step_in]
            room = min(out_cap - produced, step_out)
            ret, o, used = s.step(chunk, room, O.Z_FINISH)
            out.append(o)
            produced += len(o)
            fed += used
            if ret == O.Z_BUF_ERROR:
                more_in = used == len(chunk) and pos + fed < len(data)
                more_out = len(o) == room and produced < out_cap
                if more_in or more_out:
                    continue
            break
        if ret == O.Z_STREAM_END:
            members += 1
            if pos + fed == len(data):
                s.close()
                return LoopResult(ret, "", b"".join(out), pos + fed, members, pos, out_start)
            pos += fed
            s.reset()
            continue
        msg = s.msg
        s.close()
        return LoopResult(ret, msg, b"".join(out), pos + fed, members, pos, out_start)


def python_gunzip(data: bytes) -> tuple[bytes, int]:
    """Python's own member loop (zlib.decompressobj(31) / unused_data) on a valid file: (output, members)."""
    out, members = [], 0
    rest = data
    while True:
        d = zlib.decompressobj(31)
        out.append(d.decompress(rest))
        assert d.eof, "not a complete member"
        members += 1
        rest = d.unused_data
        if not rest:
            return b"".join(out), members


class Writer:
    """Concatenates members and records (in_off, in_len, out_off, out_len) of each one."""

    def __init__(self):
        self.parts, self.table, self.in_pos, self.out_pos = [], [], 0, 0

    def add(self, member: bytes, out_len: int):
        self.parts.append(member)
        self.table.append((self.in_pos, len(member), self.out_pos, out_len))
        self.in_pos += len(member)
        self.out_pos += out_len

    def data(self) -> bytes:
        return b"".join(self.parts)


def raw_deflate(data: bytes, level: int, sync_every: int = 0) -> bytes:
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    if not sync_every:
        return co.compress(data) + co.flush()
    parts = []
    for i in range(0, len(data), sync_every):
        parts.append(co.compress(data[i: i + sync_every]))
        parts.append(co.flush(zlib.Z_SYNC_FLUSH))
    parts.append(co.flush())
    return b"".join(parts)


def gzip_member(data: bytes, level: int = 6, text: bool = False, extra: bytes | None = None, name: bytes | None = None,
                comment: bytes | None = None, hcrc: bool = False, sync_every: int = 0, body: bytes | None = None) -> bytes:
    """One gzip member with the header fields asked for (RFC 1952 2.3)."""
    flg = (1 if text else 0) | (2 if hcrc else 0) | (4 if extra is not None else 0) | (8 if name is not None else 0) | \
        (16 if comment is not None else 0)
    h = bytearray(b"\x1f\x8b\x08" + bytes([flg]) + struct.pack("<I", 0x5f000000) + b"\x00\x03")
    if extra is not None:
        h += struct.pack("<H", len(extra)) + extra
    if name is not None:
        h += name + b"\0"
    if comment is not None:
        h += comment + b"\0"
    if hcrc:
        h += struct.pack("<H", zlib.crc32(bytes(h)) & 0xffff)
    if body is None:
        body = raw_deflate(data, level, sync_every)
    return bytes(h) + body + struct.pack("<II", zlib.crc32(data), len(data) & 0xffffffff)


def bgzf(data: bytes, level: int, bsize_lie: int = 0) -> Writer:
    """A BGZF file (SAM/BAM specification 4.1): members of <= 65280 input bytes with the BC subfield, then the EOF
    block.  bsize_lie != 0 adds it to every BSIZE (a reader must not trust it)."""
    w = Writer()
    for i in range(0, len(data), BGZF_BLOCK):
        block = data[i: i + BGZF_BLOCK]
        cdata = raw_deflate(block, level)
        bsize = 18 + len(cdata) + 8 - 1 + bsize_lie
        h = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", bsize & 0xffff)
        w.add(h + cdata + struct.pack("<II", zlib.crc32(block), len(block)), len(block))
    w.add(BGZF_EOF, 0)
    return w
