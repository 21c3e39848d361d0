# Deflate one stream and index it in the same call (zs_deflate_indexed*), against deflate followed by the decode-based
# build (zs_inflate_index_build_dev), on the 1 GiB mixed corpus (larger than the 126 MB L2), device-resident, zlib wrapper.
# Shapes: level 1 with 64 KiB chunks, and level 6 with 256 KiB chunks (bench.py's configs[2] shape).
# Per shape: plain STITCHED deflate (zs_deflate_batch_dev, then a synchronise); per span S in {256 KiB, 1 MiB, 4 MiB}:
#  1. zs_deflate_indexed_dev, and its overhead over the plain deflate (the two alternated, the median difference);
#  2. zs_deflate_batch_dev followed by zs_inflate_index_build_dev on its output (what a caller does without the call);
#  3. the indexed call's own kernels from zs_ctx_profile (deflate_record_kernel, ix_gather_kernel), points, export size;
#  4. the host-buffer calls from pinned memory: zs_deflate_indexed against zs_deflate_batch (STITCHED), alternated;
#  5. eight alternated plain / indexed calls at S = 1 MiB, each as kernel time (zs_ctx_profile) plus the rest.
# Every index is checked once against the build's (equal exports).  Times: host clock around calls that end in a
# synchronise, median of --reps calls after a warm-up call.
#
# usage: python tools/deflateindexprof.py [--out FILE] [--reps 7]
import argparse
import ctypes as C
import importlib
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
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


def wall(fn, reps):
    """median ms of one call that ends in a synchronise, after a warm-up call"""
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def paired(a, b, reps):
    """medians of a, of b and of b - a over `reps` rounds of a then b, after a warm-up round (work that shares the GPU
    slows both calls of a round alike, so the difference holds where the times themselves wander)"""
    a(), b()
    ta, tb = [], []
    for _ in range(reps):
        for fn, ts in ((a, ta), (b, tb)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ta)), float(np.median(tb)), float(np.median(np.subtract(tb, ta)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deflate_index_b200.txt"))
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    ctx = B.default_context(0)
    lib = capi.load()
    lines = [f"# tools/deflateindexprof.py on {card()}",
             "# 1 GiB mixed corpus, zlib wrapper; host clock around synchronised calls, median of "
             f"{args.reps} after a warm-up call", ""]

    def say(s):
        print(s, flush=True)
        lines.append(s)

    data = corpus.mixed_numpy(GIB, 2)
    n = data.size
    d_in = torch.from_numpy(data).cuda()
    pinned = torch.from_numpy(data).pin_memory()
    h_in = pinned.numpy()
    for level, chunk in ((1, 65536), (6, 262144)):
        nc = B.n_chunks_for(n, chunk)
        cap = int(lib.zs_deflate_batch_bound(n, nc, chunk, B.WRAP_ZLIB, B.MODE_STITCHED))
        out = torch.empty(cap, dtype=torch.uint8, device="cuda")
        out_off = torch.empty(nc + 1, dtype=torch.int64, device="cuda")
        out_bits = torch.empty(nc, dtype=torch.int64, device="cuda")
        checks = torch.empty(nc, dtype=torch.int32, device="cuda")
        res = torch.zeros(24, dtype=torch.uint8, device="cuda")
        args_dev = (B._ptr(d_in), n, None, nc, chunk, chunk)
        outs_dev = (B._ptr(out), cap, B._ptr(out_off), B._ptr(out_bits), B._ptr(checks), B._ptr(res))

        def plain():
            ctx.check(lib.zs_deflate_batch_dev(ctx.handle, *args_dev, 0, level, B.WRAP_ZLIB, B.MODE_STITCHED, 0, *outs_dev),
                      "zs_deflate_batch_dev")
            torch.cuda.synchronize()

        t_plain = wall(plain, args.reps)
        total = int(B.DeflateBatchDev(out, out_off, out_bits, checks, res).read_result().total_out_bytes)
        say(f"## level {level}, {chunk >> 10} KiB chunks: {total / 2**20:.1f} MiB compressed")
        say(f"plain STITCHED deflate (zs_deflate_batch_dev + synchronise): {t_plain:.2f} ms, {n / t_plain / 1e6:.2f} GB/s")
        stream = out[:total]
        h_out = torch.empty(cap, dtype=torch.uint8).pin_memory().numpy()
        h_res = capi.DeflateResult()

        def host_plain():
            ctx.check(lib.zs_deflate_batch(ctx.handle, h_in.ctypes.data, n, None, nc, chunk, level, B.WRAP_ZLIB,
                                           B.MODE_STITCHED, 0, h_out.ctypes.data, cap, None, None, None, C.byref(h_res)),
                      "zs_deflate_batch")

        for span in (256 << 10, 1 << 20, 4 << 20):
            handles = []

            def indexed():
                h = C.c_void_p()
                ctx.check(lib.zs_deflate_indexed_dev(ctx.handle, *args_dev, level, B.WRAP_ZLIB, 0, span, *outs_dev, C.byref(h)),
                          "zs_deflate_indexed_dev")
                handles.append(h)

            def deflate_then_build():
                plain()
                h = C.c_void_p()
                r = capi.InflateIndexResult()
                o = build_out
                ctx.check(lib.zs_inflate_index_build_dev(ctx.handle, B._ptr(stream), total, 15, span, B._ptr(o), n + 64, None, 0,
                                                         C.byref(r), C.byref(h)), "zs_inflate_index_build_dev")
                handles.append(h)

            def host_indexed():
                h = C.c_void_p()
                ctx.check(lib.zs_deflate_indexed(ctx.handle, h_in.ctypes.data, n, None, nc, chunk, level, B.WRAP_ZLIB, 0, span,
                                                 h_out.ctypes.data, cap, None, None, None, C.byref(h_res), C.byref(h)),
                          "zs_deflate_indexed")
                handles.append(h)

            def release():
                for h in handles:
                    lib.zs_inflate_index_destroy(h)
                handles.clear()

            t_plain, t_ix, d_ix = paired(plain, indexed, args.reps)
            release()
            ctx.profile(True)
            ctx.profile_read()
            indexed()
            prof = ctx.profile_read()
            ctx.profile(False)
            ix = B.InflateIndex(handles.pop(), ctx, stream)
            rec = prof.get("deflate_record_kernel", (0, 0.0))[1]
            gat = prof.get("ix_gather_kernel", (0, 0.0))[1]
            build_out = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
            t_build = wall(deflate_then_build, args.reps)
            built = B.InflateIndex(handles.pop(), ctx, stream)
            release()
            blob = ix.to_bytes()
            assert blob == built.to_bytes(), "the indexed call's index differs from the build's"
            built.close()
            del build_out
            torch.cuda.empty_cache()
            t_host_plain, t_host_ix, d_host = paired(host_plain, host_indexed, args.reps)
            release()
            say(f"S = {span >> 10} KiB: {int(ix.info.n_points)} points, export {len(blob) / 2**20:.2f} MiB (equal to the build's)")
            say(f"  zs_deflate_indexed_dev {t_ix:.2f} ms against plain {t_plain:.2f} ms: + {d_ix:.2f} ms "
                f"({d_ix / t_plain * 100:+.1f} %); deflate_record_kernel {rec:.3f} ms, ix_gather_kernel {gat:.3f} ms")
            say(f"  deflate + zs_inflate_index_build_dev {t_build:.2f} ms ({t_build / t_ix:.2f} x the indexed call)")
            say(f"  host buffers (pinned): zs_deflate_indexed {t_host_ix:.2f} ms against zs_deflate_batch {t_host_plain:.2f} ms: "
                f"+ {d_host:.2f} ms ({d_host / t_host_plain * 100:+.1f} %)")
            if span == 1 << 20:
                # where an indexed call's time goes, call by call: device time of its kernels (zs_ctx_profile) and the rest
                say("per call, plain / indexed alternated (S = 1 MiB): wall ms = kernels + host")
                ctx.profile(True)
                ctx.profile_read()
                for i in range(16):
                    fn = indexed if i % 2 else plain
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    t = (time.perf_counter() - t0) * 1e3
                    k = sum(v[1] for v in ctx.profile_read().values())
                    say(f"  {'indexed' if i % 2 else 'plain  '} {t:7.2f} = {k:7.2f} + {t - k:6.2f}")
                ctx.profile(False)
                release()
            ix.close()
        say("")
        del out, stream
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    open(args.out, "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
