# Whole multi-member gzip files in one call (zs_gunzip_dev) against the ways to read them without it, on device-resident
# files larger than the 126 MB L2.  Shapes:
#  (a) BGZF (65280-byte blocks, level 6) of the 1 GiB text and mixed corpora -- the raw bodies come from the engine's
#      INDEPENDENT raw deflate, the BGZF framing from Python;
#  (b) 262144 x 4 KiB gzip records (the engine's INDEPENDENT gzip output, level 6, the records of configs[3]);
#  (c) the engine's INDEPENDENT gzip output with 64 KiB chunks (1 GiB text, level 6);
#  (d) 4 x 256 MiB members, each written in one go (STITCHED gzip without flush points, 1 GiB text, level 6);
#  (e) adversarial: 256 level-0 members, each wrapping a 1 MiB BGZF file (false member starts everywhere).
# Per shape, output GB/s of: zs_gunzip_dev; the ceiling, zs_inflate_batch_dev given the true member offsets and sizes
# ((d): zs_inflate_stream_dev per member); the existing one-stream path looped per member (zs_inflate_stream_dev on the
# rest of the file, aligned copy first, as its callers must; on the file cut behind >= 16 MiB of output, since that loop
# takes milliseconds per member; (e) whole); gzip.decompress on one core (the file cut behind >= 64 MiB of output); host-buffer
# zs_gunzip end to end; and the kernel split of one zs_gunzip_dev call (zs_ctx_profile).  CUDA events around
# synchronised calls after a warm-up call.  Then the large-member threshold (members of >= 128 KiB of input are decoded
# alone by the one-stream path, smaller ones in the batch), A/B through the ZS_GUNZIP_LARGE hook: the engine's
# INDEPENDENT gzip output of text at level 6 with 64 KiB (128 MiB in all), 1 MiB and 16 MiB chunks (1 GiB), each
# decoded with the default and with the other decoder forced.
#
# usage: python tools/gunzipprof.py [--out FILE] [--reps 3]
import argparse
import ctypes as C
import gzip
import importlib
import os
import struct
import subprocess
import sys
import time
import zlib

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

B = importlib.import_module("zlib-streams-ts_b200.batch")
capi = importlib.import_module("zlib-streams-ts_b200.capi")
corpus = importlib.import_module("zlib-streams-ts_b200.corpus")
GIB = 1 << 30


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        q = f"power limit unknown ({e})"
    return f"{name}, {q}"


def timed(fn, reps):
    """mean ms of one call, after a warm-up call"""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def bgzf_from_engine(data: bytes) -> bytes:
    blk = 65280
    r = B.deflate_batch(data, blk, 6, B.WRAP_RAW, B.MODE_INDEPENDENT)
    parts = []
    for i in range(len(r.out_off) - 1):
        body = r.stream(i)
        n = min(blk, len(data) - i * blk)
        h = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", 18 + len(body) + 8 - 1)
        parts.append(h + body + struct.pack("<II", int(r.checks[i]), n))
    parts.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    return b"".join(parts)


def shapes():
    text = corpus.text_numpy(GIB, 1).tobytes()
    mixed = corpus.mixed_numpy(GIB, 2).tobytes()
    yield "(a) BGZF text L6", bgzf_from_engine(text), GIB
    yield "(a) BGZF mixed L6", bgzf_from_engine(mixed), GIB
    yield "(b) 262144 x 4 KiB gzip records", B.deflate_batch(mixed, 4096, 6, B.WRAP_GZIP, B.MODE_INDEPENDENT).data, GIB
    yield "(c) INDEPENDENT gzip, 64 KiB chunks", B.deflate_batch(text, 65536, 6, B.WRAP_GZIP, B.MODE_INDEPENDENT).data, GIB
    q = 256 << 20
    yield "(d) 4 x 256 MiB members", b"".join(B.deflate_batch(text[i * q:(i + 1) * q], 262144, 6, B.WRAP_GZIP,
                                                               B.MODE_STITCHED).data for i in range(4)), GIB
    inner = bgzf_from_engine(text[: 1 << 20])
    adv = zlib.compress(inner, 0, wbits=31)
    yield "(e) 256 level-0 members wrapping BGZF", adv * 256, 256 * len(inner)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    lines = [f"# tools/gunzipprof.py on {card()}",
             "# output GB/s (decompressed bytes / time); device-resident input, synchronised calls, mean of --reps after a warm-up",
             f"{'shape':40s} {'members':>8s} {'in MiB':>8s} {'gunzip_dev':>10s} {'ceiling':>8s} {'ratio':>6s} "
             f"{'loop':>8s} {'gzip 1c':>8s} {'gunzip host':>11s}"]
    splits = []
    ctx = B.default_context(0)
    lib = capi.load()
    for name, data, total in shapes():
        d_in = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
        out = torch.empty(total + 64, dtype=torch.uint8, device="cuda")
        res = capi.GunzipResult()
        tab = np.zeros(len(data) // 18 + 2, dtype=B.GZ_MEMBER_DTYPE)
        rc = lib.zs_gunzip_dev(ctx.handle, B._ptr(d_in), len(data), B._ptr(out), total, C.byref(res), tab.ctypes.data,
                               tab.size)
        ctx.check(rc, "zs_gunzip_dev")
        assert res.status == 1 and res.out_len == total, (name, res.status, res.out_len)
        nm = int(res.n_members)
        mem = tab[:nm]

        def run():
            r = capi.GunzipResult()
            ctx.check(lib.zs_gunzip_dev(ctx.handle, B._ptr(d_in), len(data), B._ptr(out), total, C.byref(r), None, 0), "gunzip")

        t_dev = timed(run, args.reps)
        ctx.profile(True)
        ctx.profile_read()
        run()
        prof = ctx.profile_read()
        ctx.profile(False)
        splits.append((name, prof))
        # the ceiling: the true members handed to the decoders
        if name.startswith("(d)"):
            buf = torch.empty(max(int(x) for x in mem["in_len"]) + 64, dtype=torch.uint8, device="cuda")
            small = torch.zeros(8, dtype=torch.int64, device="cuda")

            def ceil():
                for e in mem:
                    o, n = int(e["in_off"]), int(e["in_len"])
                    buf[:n].copy_(d_in[o:o + n])
                    ctx.check(lib.zs_inflate_stream_dev(ctx.handle, B._ptr(buf), n, 31, B._ptr(out[int(e["out_off"]):]),
                                                        int(e["out_len"]), B._ptr(small), B._ptr(small[1:]),
                                                        B._ptr(small[2:]), B._ptr(small[3:]), None, 0), "stream")
        elif name.startswith("(e)"):
            ceil = None
        else:
            ioff = torch.from_numpy(np.append(mem["in_off"], len(data)).astype(np.int64)).cuda()
            ooff = torch.from_numpy(np.append(mem["out_off"], total).astype(np.int64)).cuda()
            prev = B.inflate_batch_dev(d_in, ioff, ooff, 31, out=out)

            def ceil():
                B.inflate_batch_dev(d_in, ioff, ooff, 31, out=out, reuse=prev)
        t_ceil = timed(ceil, args.reps) if ceil else float("nan")

        def prefix(nbytes):   # (input, output) bytes of the shortest run of whole members with >= nbytes of output
            k = min(int(np.searchsorted(mem["out_off"], nbytes)) + 1, nm)
            return int(mem["in_off"][k - 1] + mem["in_len"][k - 1]), int(mem["out_off"][k - 1] + mem["out_len"][k - 1])

        # the existing path looped per member over a file cut behind >= 16 MiB of output; (e) whole, since every step
        # of that loop there decodes the rest of the file
        pre_in, pre_out = (len(data), total) if name.startswith("(e)") else prefix(16 << 20)
        al = torch.empty(len(data) + 64, dtype=torch.uint8, device="cuda")
        small = torch.zeros(8, dtype=torch.int64, device="cuda")

        def loop():
            pos = produced = 0
            while pos < pre_in:
                n = pre_in - pos
                al[:n].copy_(d_in[pos:pre_in])
                ctx.check(lib.zs_inflate_stream_dev(ctx.handle, B._ptr(al), n, 31, B._ptr(out[produced:]), total - produced,
                                                    B._ptr(small), B._ptr(small[1:]), B._ptr(small[2:]), B._ptr(small[3:]),
                                                    None, 0), "stream")
                h = small.cpu()
                produced += int(h[0])
                pos += int(h[1])

        t0 = time.perf_counter()
        loop()
        torch.cuda.synchronize()
        t_loop = time.perf_counter() - t0
        t_loop_out = pre_out
        gz_in, gz_out = prefix(64 << 20)
        t0 = time.perf_counter()
        g = gzip.decompress(data[:gz_in])
        t_gz = time.perf_counter() - t0
        assert len(g) == gz_out
        B.gunzip(data, total)
        t0 = time.perf_counter()
        h = B.gunzip(data, total)
        t_host = time.perf_counter() - t0
        assert h.status == 1 and h.out_len == total
        gbs = lambda nbytes, s: nbytes / s / 1e9   # noqa: E731
        r_dev, r_ceil = gbs(total, t_dev / 1e3), gbs(total, t_ceil / 1e3)
        lines.append(f"{name:40s} {nm:8d} {len(data) / 2**20:8.1f} {r_dev:10.2f} {r_ceil:8.2f} {r_dev / r_ceil:6.2f} "
                     f"{gbs(t_loop_out, t_loop):8.3f} {gbs(gz_out, t_gz):8.3f} {gbs(total, t_host):11.2f}")
        print(lines[-1], flush=True)
        del d_in, out, al
        torch.cuda.empty_cache()
    lines.append("")
    lines.append("# large-member threshold: output GB/s of zs_gunzip_dev with the default (128 KiB) and with every member in the")
    lines.append("# batch (ZS_GUNZIP_LARGE=2^62) / every member alone (ZS_GUNZIP_LARGE=0)")
    lines.append(f"{'chunks':>8s} {'members':>8s} {'in KiB/member':>14s} {'default':>8s} {'batch':>8s} {'alone':>8s}")
    text = corpus.text_numpy(GIB, 1).tobytes()
    for chunk, total in ((64 << 10, 128 << 20), (1 << 20, GIB), (16 << 20, GIB)):
        data = B.deflate_batch(text[:total], chunk, 6, B.WRAP_GZIP, B.MODE_INDEPENDENT).data
        d_in = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
        out = torch.empty(total + 64, dtype=torch.uint8, device="cuda")
        rates = []
        for hook in (None, str(1 << 62), "0"):
            if hook is None:
                os.environ.pop("ZS_GUNZIP_LARGE", None)
            else:
                os.environ["ZS_GUNZIP_LARGE"] = hook

            def run():
                r = capi.GunzipResult()
                ctx.check(lib.zs_gunzip_dev(ctx.handle, B._ptr(d_in), len(data), B._ptr(out), total, C.byref(r), None, 0),
                          "gunzip")
                assert r.status == 1 and r.out_len == total

            rates.append(total / (timed(run, args.reps) / 1e3) / 1e9)
        os.environ.pop("ZS_GUNZIP_LARGE", None)
        n = total // chunk
        lines.append(f"{chunk >> 10:7d}K {n:8d} {len(data) / n / 1024:14.1f} {rates[0]:8.2f} {rates[1]:8.2f} {rates[2]:8.2f}")
        print(lines[-1], flush=True)
        del d_in, out
        torch.cuda.empty_cache()
    lines.append("")
    lines.append("# kernel split of one zs_gunzip_dev call: kernel launches total_ms")
    for name, prof in splits:
        lines.append(name)
        for k, (n, ms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
            lines.append(f"    {k:28s} {n:7d} {ms:9.3f}")
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
