"""CPU tests of the inflate index's test infrastructure and bindings: zran_check.block_starts (the zran.c method over
C zlib's inflate(Z_BLOCK)) and the Node addon's binding of the index calls."""
import os
import re
import shutil
import subprocess
import zlib

import pytest

from conftest import ROOT, make_text
from zran_check import block_starts, decode_from


def test_block_starts_behind_full_flush_points():
    data = make_text(600000, 4)
    c = zlib.compressobj(6)
    z, flush_at = b"", []
    for i in range(0, len(data), 150000):
        z += c.compress(data[i: i + 150000]) + c.flush(zlib.Z_FULL_FLUSH)
        flush_at.append((len(z) * 8, min(i + 150000, len(data))))
    z += c.flush()
    starts = block_starts(z, 15)
    assert starts[0] == (16, 0)
    assert [s[0] for s in starts] == sorted({s[0] for s in starts})
    for bit, off in flush_at:
        assert (bit, off) in starts          # the byte-aligned start right behind every flush marker
    # each start decodes with C zlib from its bit against the 32 KiB before it
    for bit, off in starts:
        assert decode_from(z, bit, data[max(0, off - 32768): off], 50000) == data[off: off + 50000]


def test_block_starts_raw_gzip_and_dictionary():
    data = make_text(200000, 5)
    for wbits in (-15, 31):
        c = zlib.compressobj(1, zlib.DEFLATED, wbits)
        z = c.compress(data) + c.flush()
        starts = block_starts(z, wbits)
        assert starts[0] == ((0 if wbits < 0 else 10 * 8), 0)
        for bit, off in starts:
            assert decode_from(z, bit, data[max(0, off - 32768): off], 20000) == data[off: off + 20000]
        assert all(b1 > b0 and o1 >= o0 for (b0, o0), (b1, o1) in zip(starts, starts[1:]))
    # a zlib stream that names a dictionary: the first block starts behind the 6-byte header with DICTID
    dic = data[-20000:]
    c = zlib.compressobj(6, zlib.DEFLATED, 15, 8, zlib.Z_DEFAULT_STRATEGY, dic)
    z = c.compress(data) + c.flush()
    starts = block_starts(z, 15, dic)
    assert starts[0] == (48, 0)
    for bit, off in starts:
        hist = (dic + data[:off])[-32768:]
        assert decode_from(z, bit, hist, 20000) == data[off: off + 20000]


@pytest.mark.skipif(shutil.which("g++") is None, reason="no g++")
def test_addon_binds_the_index_calls(tmp_path):
    obj = tmp_path / "addon.o"
    r = subprocess.run(["g++", "-std=c++17", "-Wall", "-Werror", "-c", "-fPIC", "-I" + os.path.join(ROOT, "tests", "stubs"),
                        "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "bindings", "node", "zsgpu_addon.cc"),
                        "-o", str(obj)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    need = set(re.findall(r"\bU (zs_\w+)", subprocess.run(["nm", "-u", str(obj)], capture_output=True, text=True).stdout))
    assert {"zs_inflate_index_build", "zs_inflate_index_extract", "zs_inflate_index_export", "zs_inflate_index_import",
            "zs_inflate_index_destroy"} <= need
    ts = open(os.path.join(ROOT, "bindings", "ts", "zlib-streams-gpu.ts")).read()
    assert "export class InflateIndex" in ts
