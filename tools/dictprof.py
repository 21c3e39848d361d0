# Batch deflate of small JSON-like records against a prepared preset dictionary (zs_deflate_batch_dict_dev),
# next to the same records without one (zs_deflate_batch_dev, INDEPENDENT).  Records of 1, 4, 16 and 64 KiB,
# about 1 GiB per shape, cut at seeded offsets from a 64 MiB pool of rows (corpus.json_pool); dictionaries of
# 8 KiB and 30 000 bytes from the same generator (another seed); levels 1 and 6.  Per shape: input GB/s with
# and without the dictionary (device-resident input, CUDA events around each of 5 calls after a warm-up call:
# mean, and the slowest / fastest call), lz77 kernel time per call (zs_ctx_profile), the time to create one
# dictionary (zs_deflate_dict_create alone; it synchronises), and compressed sizes with and without it
# against C zlib (compressobj(level, zdict=D)) on the first 16 MiB of the same records.
#
# usage: python tools/dictprof.py [--gib 1] [--out FILE]
import argparse
import importlib
import os
import subprocess
import sys
import time
import zlib

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

B = importlib.import_module("zlib-streams-ts_b200.batch")
corpus = importlib.import_module("zlib-streams-ts_b200.corpus")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the numbers stand with the card name alone then
        q = f"power limit unknown ({e})"
    return f"{name}, {q}"


def timed(fn, reps=5):
    """(mean, min, max) ms of one call"""
    fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for i in range(reps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(reps)]
    return sum(ms) / reps, min(ms), max(ms)


def kernel_ms(ctx, fn, name):
    ctx.profile(True)
    ctx.profile_read()
    fn()
    prof = ctx.profile_read()
    ctx.profile(False)
    return prof.get(name, (0, 0.0))[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "dictprof measures on the GPU; there is nothing to measure without one"
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda:0")
    ctx = B.default_context(0)
    say(f"# dictprof on {card()}")
    t0 = time.time()
    pool = torch.frombuffer(bytearray(corpus.json_pool(64 << 20, 0xD1C7)), dtype=torch.uint8).to(dev)
    say(f"# pool: 64 MiB of JSON-like rows ({time.time() - t0:.1f} s to generate)")
    dicts = {8192: corpus.json_pool(8192, 0xD1C8), 30000: corpus.json_pool(30000, 0xD1C9)}
    for dl, D in dicts.items():
        B.DeflateDictionary(D, ctx).close()   # warm-up (module load, allocations)
        ms = []
        for _ in range(10):
            torch.cuda.synchronize()
            t = time.perf_counter()
            h = B.DeflateDictionary(D, ctx)   # zs_deflate_dict_create returns after a synchronise
            ms.append(1e3 * (time.perf_counter() - t))
            h.close()
        say(f"dictionary {dl} B: create {sum(ms) / len(ms):.2f} ms (min {min(ms):.2f}, max {max(ms):.2f}; host clock, 10 creates)")
    g = torch.Generator(device="cpu")
    say("record  dict  level | GB/s dict (min-max)      GB/s plain (min-max)    | lz77 ms/call dict  plain | sample bytes: dict  plain  zlib+zdict  (dict/zlib)")
    for rec_kib in (1, 4, 16, 64):
        rec = rec_kib << 10
        n_rec = int(args.gib * (1 << 30)) // rec
        g.manual_seed(rec_kib)
        starts = torch.randint(0, pool.numel() - rec, (n_rec,), generator=g).to(dev)
        data = pool.unfold(0, rec, 1)[starts].reshape(-1).contiguous()
        n = data.numel()
        sample_n = min(n_rec, (16 << 20) // rec)
        sample = data[: sample_n * rec].cpu().numpy().tobytes()
        for dl, D in dicts.items():
            h = B.DeflateDictionary(D, ctx)
            for level in (1, 6):
                rd = B.deflate_batch_dev(data, rec, level, B.WRAP_ZLIB, ctx=ctx, dictionary=h)
                rp = B.deflate_batch_dev(data, rec, level, B.WRAP_ZLIB, ctx=ctx)
                ms_d = timed(lambda: B.deflate_batch_dev(data, rec, level, B.WRAP_ZLIB, ctx=ctx, dictionary=h, reuse=rd))
                ms_p = timed(lambda: B.deflate_batch_dev(data, rec, level, B.WRAP_ZLIB, ctx=ctx, reuse=rp))
                k_d = kernel_ms(ctx, lambda: B.deflate_batch_dev(data, rec, level, B.WRAP_ZLIB, ctx=ctx, dictionary=h, reuse=rd),
                                "lz77_dict_kernel")
                k_p = kernel_ms(ctx, lambda: B.deflate_batch_dev(data, rec, level, B.WRAP_ZLIB, ctx=ctx, reuse=rp), "lz77_kernel")
                oo_d, oo_p = rd.out_off.cpu(), rp.out_off.cpu()
                s_d, s_p = int(oo_d[sample_n]), int(oo_p[sample_n])
                s_z = 0
                for i in range(sample_n):
                    c = zlib.compressobj(level, zlib.DEFLATED, 15, zdict=D)
                    s_z += len(c.compress(sample[i * rec: (i + 1) * rec]) + c.flush())
                gb = lambda t: f"{n / t[0] / 1e6:7.2f} ({n / t[2] / 1e6:.2f}-{n / t[1] / 1e6:.2f})"
                say(f"{rec_kib:3d} KiB {dl:6d} L{level}  | {gb(ms_d)}  {gb(ms_p)} | "
                    f"{k_d:10.2f}  {k_p:6.2f} | {s_d:11d} {s_p:10d} {s_z:10d}  ({s_d / s_z:.4f})")
                del rd, rp
            h.close()
        say(f"#   {rec_kib} KiB records: {n_rec} records, {n / (1 << 30):.2f} GiB; size sample = first {sample_n} records")
        del data, starts
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
