# Random access into one deflate stream (zs_inflate_index_*), on device-resident streams larger than the 126 MB L2.
# Shapes:
#  (a) the 1 GiB mixed corpus as one zlib stream without flush points (the engine's STITCHED zlib output, level 6);
#  (b) a 256 MiB C zlib gzip stream at level 6 (the mixed corpus, written in one go);
#  (c) the engine's own 1 GiB SYNC stream (STITCHED + ZS_FLAG_SYNC, 64 KiB chunks, level 6, the text corpus).
# Per shape and span S in {256 KiB, 1 MiB, 4 MiB}:
#  1. build: zs_inflate_index_build_dev against zs_inflate_stream_dev on the same stream; the index's own kernels
#     (par_record_kernel: the record pass over the planned segments together with the serial walk; ix_gather_kernel) from
#     zs_ctx_profile; points and index size;
#  2. whole-stream extract: one range [0, out_len) through zs_inflate_index_extract_dev, GB/s of output;
#  3. 100 000 seeded 4 KiB reads in one call: device-resident (zs_inflate_index_extract_dev) and through the host-buffer
#     call from pinned memory (zs_inflate_index_extract), reads/s and GB/s;
#  4. CPU baseline: zran's method on one core (C zlib through ctypes: inflatePrime + inflateSetDictionary with the exported
#     window), on the first 300 of those reads.
# Device times: CUDA events around synchronised calls after a warm-up call (build: wall clock, it synchronises).
#
# usage: python tools/indexprof.py [--out FILE] [--reps 3]
import argparse
import importlib
import os
import random
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402
from zran_check import decode_from  # noqa: E402

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


def shapes():
    mixed = corpus.mixed_numpy(GIB, 2).tobytes()
    yield "(a) 1 GiB mixed, zlib, no flush points", B.deflate_batch(mixed, 262144, 6, B.WRAP_ZLIB, B.MODE_STITCHED).data, 15
    c = zlib.compressobj(6, zlib.DEFLATED, 31)
    q = mixed[: 256 << 20]
    yield "(b) 256 MiB C zlib gzip L6", c.compress(q) + c.flush(), 31
    del mixed, q
    text = corpus.text_numpy(GIB, 1).tobytes()
    yield "(c) 1 GiB engine SYNC stream", B.deflate_batch(text, 65536, 6, B.WRAP_ZLIB, B.MODE_STITCHED, B.FLAG_SYNC).data, 15


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "index_b200.txt"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    ctx = B.default_context(0)
    lib = capi.load()
    lines = [f"# tools/indexprof.py on {card()}", "# inputs larger than the 126 MB L2; times after a warm-up call", ""]

    def say(s):
        print(s, flush=True)
        lines.append(s)

    for name, data, wbits in shapes():
        say(f"## {name}: {len(data) / 2**20:.1f} MiB compressed")
        d_in = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        ix, built = B.InflateIndex.build(d_in, wbits, 1 << 20)
        out_len = built.out_len
        assert built.status == 1
        cap = out_len + 64
        out = built.data
        r = torch.zeros(4, dtype=torch.int64, device="cuda")

        def stream_dev():
            rc = lib.zs_inflate_stream_dev(ctx.handle, B._ptr(d_in), d_in.numel(), wbits, B._ptr(out), cap, B._ptr(r[0:1]),
                                           B._ptr(r[1:2]), B._ptr(r[2:3]), B._ptr(r[3:4]), None, 0)
            ctx.check(rc, "zs_inflate_stream_dev")

        t_stream = timed(stream_dev, args.reps)
        say(f"zs_inflate_stream_dev: {t_stream:.2f} ms, {out_len / t_stream / 1e6:.2f} GB/s of output ({out_len / 2**20:.0f} MiB)")
        ref = out[:out_len].clone()
        pinned = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).pin_memory()
        host_in = pinned.numpy()
        rng = random.Random(1234)
        reads = [rng.randrange(0, out_len - 4096) for _ in range(100000)]
        for span in (256 << 10, 1 << 20, 4 << 20):
            ix.close()
            ix, _ = B.InflateIndex.build(d_in, wbits, span, out_cap=cap)
            t0 = time.perf_counter()
            for _ in range(args.reps):
                ix.close()
                ix, _ = B.InflateIndex.build(d_in, wbits, span, out_cap=cap)
            t_build = (time.perf_counter() - t0) * 1e3 / args.reps
            ctx.profile(True)
            ix.close()
            ix, _ = B.InflateIndex.build(d_in, wbits, span, out_cap=cap)
            prof = ctx.profile_read()
            ctx.profile(False)
            rec = prof.get("par_record_kernel", (0, 0.0))[1]
            gat = prof.get("ix_gather_kernel", (0, 0.0))[1]
            size = len(ix.to_bytes())
            n = int(ix.info.n_points)
            say(f"S = {span >> 10} KiB: {n} points, index {size / 2**20:.1f} MiB exported")
            say(f"  build {t_build:.2f} ms = {t_build / t_stream:.2f} x zs_inflate_stream_dev; record pass + serial walk "
                f"{rec:.2f} ms, gather {gat:.2f} ms, the rest (decode, host merge, copies) {t_build - rec - gat:.2f} ms")
            # whole stream
            o1 = torch.zeros(out_len + 16, dtype=torch.uint8, device="cuda")
            z = torch.zeros(1, dtype=torch.int64, device="cuda")
            ln = torch.full((1,), out_len, dtype=torch.int64, device="cuda")
            got, st = torch.zeros(1, dtype=torch.int64, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
            t_whole = timed(lambda: ix.extract_dev(d_in, z, ln, o1, z, got, st), args.reps)
            assert int(st[0]) == 0 and torch.equal(o1[:out_len], ref)
            say(f"  whole-stream extract: {t_whole:.2f} ms, {out_len / t_whole / 1e6:.2f} GB/s "
                f"({t_stream / t_whole:.2f} x zs_inflate_stream_dev)")
            # random 4 KiB reads
            off = torch.tensor(reads, dtype=torch.int64, device="cuda")
            l4 = torch.full((len(reads),), 4096, dtype=torch.int64, device="cuda")
            ooff = torch.arange(len(reads), dtype=torch.int64, device="cuda") * 4096
            o2 = torch.zeros(len(reads) * 4096 + 16, dtype=torch.uint8, device="cuda")
            got2 = torch.zeros(len(reads), dtype=torch.int64, device="cuda")
            st2 = torch.zeros(len(reads), dtype=torch.int32, device="cuda")
            t_rand = timed(lambda: ix.extract_dev(d_in, off, l4, o2, ooff, got2, st2), args.reps)
            assert int((st2 != 0).sum()) == 0
            for k in range(0, len(reads), 9973):
                assert torch.equal(o2[k * 4096:(k + 1) * 4096], ref[reads[k]: reads[k] + 4096])
            say(f"  100000 x 4 KiB reads, device: {t_rand:.2f} ms, {len(reads) / t_rand * 1e3:.0f} reads/s, "
                f"{len(reads) * 4096 / t_rand / 1e6:.2f} GB/s")
            h_off = np.array(reads, dtype=np.uint64)
            h_len = np.full(len(reads), 4096, dtype=np.uint64)
            h_ooff = np.arange(len(reads), dtype=np.uint64) * 4096
            h_out = torch.zeros(len(reads) * 4096 + 16, dtype=torch.uint8).pin_memory().numpy()
            h_got = np.zeros(len(reads), dtype=np.uint64)
            h_st = np.zeros(len(reads), dtype=np.int32)

            def host():
                rc = lib.zs_inflate_index_extract(ctx.handle, ix.handle, host_in.ctypes.data, host_in.size, h_off.ctypes.data,
                                                  h_len.ctypes.data, len(reads), h_out.ctypes.data, len(reads) * 4096,
                                                  h_ooff.ctypes.data, h_got.ctypes.data, h_st.ctypes.data)
                ctx.check(rc, "zs_inflate_index_extract")

            t_host = timed(host, args.reps)
            assert int((h_st != 0).sum()) == 0 and bytes(h_out[:4096]) == ref[reads[0]: reads[0] + 4096].cpu().numpy().tobytes()
            say(f"  100000 x 4 KiB reads, host buffers (pinned): {t_host:.2f} ms, {len(reads) / t_host * 1e3:.0f} reads/s, "
                f"{len(reads) * 4096 / t_host / 1e6:.2f} GB/s")
            # zran on one core
            blob = ix.to_bytes()
            pts = ix.points
            wl = np.frombuffer(blob[56: 56 + 24 * n], dtype=np.uint64).reshape(n, 3)[:, 2] & 0xffffffff
            ws = np.concatenate([[0], np.cumsum(wl)]).astype(np.int64) + 56 + 24 * n
            poff = pts[:, 1].astype(np.int64)
            sub = reads[:300]
            t0 = time.perf_counter()
            for o in sub:
                p = int(np.searchsorted(poff, o, side="right")) - 1
                need = o - int(poff[p]) + 4096
                b = decode_from(data, int(pts[p][0]), blob[ws[p]: ws[p + 1]], need, max_in=2 * need + 65536)
                assert len(b) == need
            t_cpu = (time.perf_counter() - t0) * 1e3
            say(f"  CPU baseline (zran's method, C zlib, one core, {len(sub)} reads): {len(sub) / t_cpu * 1e3:.0f} reads/s; "
                f"device reads / CPU = {(len(reads) / t_rand) / (len(sub) / t_cpu):.0f} x")
        ix.close()
        say("")
        del d_in, out, ref, pinned
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    open(args.out, "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
