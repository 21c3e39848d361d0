#!/usr/bin/env python
"""bench.py -- headline benchmark of the deflate/inflate hot path (BASELINE.json).

N = 1  (config.workload = configs[1]): a 1 GiB synthetic text-like corpus, deflate-raw level 1, 64 KiB
       chunks each primed with the preceding 32 KiB, on one B200.
N > 1  (config.workload = configs[2], the north-star multi-GPU split, STRONG scaling): ONE 4 GiB mixed
       corpus (seed 0xB200) becomes ONE zlib stream at level 6 (lazy matching), 256 KiB chunks with 32 KiB
       dictionary priming; rank r deflates the contiguous chunk range [r*C/N, (r+1)*C/N) as one part of the
       stream (sharded.deflate_sharded), then the ranks all_gather (compressed bit length, adler32, length)
       -> exclusive scan (global bit offsets) -> adler32_combine (sharded.exchange_meta).  After the timed
       region the parts are gathered once on rank 0 (sharded.gather_stream, timed separately), decoded by C
       zlib and compared with the corpus (`verified`).  `inflate` holds the decode side of the same run: the
       stream inflated where it lies (every rank its own part, sharded.inflate_sharded) and configs[3], the
       corpus as independent 4 KiB gzip records block-partitioned over the ranks.

A step is one pass of the hot path over the whole corpus.
  value  input GB/s with the corpus resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e    the same metric through the C ABI's host-buffer calls (zs_deflate_batch / zs_deflate_part): pinned
         host input, H2D, kernels, D2H of the compressed bytes, all inside the timed region
  roofline / cpu_baseline / clocks / gpu_launches as the bench contract asks; `extra` (N = 1, rank 0) holds
  the other BASELINE configs: configs[2] shape on one GPU, configs[3] (gzip records inflate + crc verify),
  configs[4] (deflate64), the stream API with the reference's 32 KiB / 64 KiB slicing, checksums.
`--impl reference` times the CPU reference arm: the oracle port of the reference's deflate (the reference
itself is TypeScript and there is no JavaScript engine in this image; baseline/node_bench.mjs is run instead
when `node` is on PATH), one independent stream per host thread, on the same workload.
`--dump-outputs DIR` writes what the last timed step computed to DIR/<name>.npy (see dump_outputs), so that two
builds can be compared output for output on the same seeded corpus.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: the benchmark writes nothing into it

METRIC = "deflate_input_GBps"
UNIT = "GB/s"
CHUNK = 65536        # configs[1]
LEVEL = 1
CHUNK2 = 262144      # configs[2]
LEVEL2 = 6
SEED1 = 0xC0FFEE
SEED2 = 0xB200


def pkg(sub):
    return importlib.import_module("zlib-streams-ts_b200." + sub)


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def config1(n, n_chunks, world=1):
    return {"workload": "configs[1]: 1 GiB text-like corpus per GPU, deflate-raw level 1, 64 KiB chunks + 32 KiB dictionary priming",
            "bytes_per_gpu": n, "level": LEVEL, "chunk": CHUNK, "n_chunks": n_chunks, "wrapper": "deflate-raw",
            "cache": "input (1 GiB) larger than L2 (126 MB)", "parallelism": f"contiguous chunk ranges x{world}"}


def config2(total, n_chunks, world):
    return {"workload": "configs[2]: one 4 GiB mixed corpus -> one zlib stream, level 6 lazy matching, 256 KiB chunks + "
                        "32 KiB dictionary priming, sharded by contiguous chunk ranges",
            "total_bytes": total, "level": LEVEL2, "chunk": CHUNK2, "n_chunks": n_chunks, "wrapper": "zlib",
            "cache": "input per rank larger than L2 (126 MB)", "parallelism": f"contiguous chunk ranges x{world}"}


class ClockSampler:
    def __init__(self, device_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(device_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for k, nme in enumerate(names):
                    if r[3 + k].strip().lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["sm_max_mhz"] = max(mx)
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


def bind_numa(torch, local_rank):
    """Pin this rank's host threads (and so its pinned allocations, first touch) to the NUMA node of its
    GPU, when the box exposes one.  Returns the node or None."""
    try:
        props = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def copy_ceiling(torch, dist, world, dev, h_in, h_out, n_in, n_out):
    """What the host<->device copies of one e2e step cost with no kernels in between: n_in bytes H2D and n_out
    bytes D2H on two streams at once, all ranks together.  Returns ms (max over ranks)."""
    d_a = torch.empty(n_in, dtype=torch.uint8, device=dev)
    d_b = torch.empty(max(n_out, 1), dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def once():
        with torch.cuda.stream(s1):
            d_a.copy_(h_in[:n_in], non_blocking=True)
        with torch.cuda.stream(s2):
            h_out[:n_out].copy_(d_b[:n_out], non_blocking=True)
    once()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        once()
    torch.cuda.synchronize()
    ms = 1e3 * (time.perf_counter() - t0) / 3
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    del d_a, d_b
    return ms


def lz_issue(prof_key, n_bytes, lz_avg_ms, clocks, torch, dev, level):
    """Second yardstick: warp instructions per second against the SMs' issue rate (the kernel is issue bound,
    not DRAM bound).  Instructions per input byte come from the committed ncu capture."""
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        t = json.load(open(tpath))
        key = "lz77_kernel_warp_inst_per_input_byte" if level < 4 else "lz77_kernel_l6_warp_inst_per_input_byte"
        ipb = t[key]
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz")
        if lz_avg_ms > 0 and mhz:
            ach = ipb * n_bytes / (lz_avg_ms / 1e3) / 1e9
            pk = sms * 4 * mhz * 1e6 / 1e9
            return {"warp_inst_per_input_byte": ipb, "achieved_ginst_per_s": ach, "peak_ginst_per_s": pk,
                    "frac": ach / pk, "sm_mhz": mhz, "source": t.get("source", "profiles/") + " x this run's kernel time"}
    except Exception:
        pass
    return None


def sample_windows(n, budget=8 << 20, win=16384):
    """Start offsets and width of the windows dumped of an n-byte output: all of it up to `budget` bytes, else
    budget // win windows of `win` bytes at fixed, seeded positions, in order."""
    import numpy as np
    if n <= budget:
        return [0], n
    return (np.sort(np.random.default_rng(0).choice(n // win, budget // win, replace=False)) * win).tolist(), win


def dump_outputs(path, arrays):
    """--dump-outputs: each array as path/<name>.npy (float32 byte values, float64 offsets, lengths and checksums:
    both exact), at most 64 MB in all."""
    import numpy as np
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def lz_traffic(n_bytes, level):
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        t = json.load(open(tpath))
        key = "lz77_kernel_dram_bytes_per_input_byte" if level < 4 else "lz77_kernel_l6_dram_bytes_per_input_byte"
        return t[key] * n_bytes
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------------
# CPU reference arm
# ---------------------------------------------------------------------------------------------------
def cpu_deflate(sample, chunk, level, threads=0, repeats=1):
    """Oracle port (oracle/deflate.c), one stream per host thread, same chunk + dictionary plan."""
    from oracle import oracle as O
    import numpy as np
    L = O.lib()
    cores = L.zo_max_threads() if threads <= 0 else threads
    arr = np.ascontiguousarray(sample)
    best, total = None, 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        total = L.zo_deflate_chunks_mt(arr.ctypes.data, arr.size, chunk, level, 0, 1, cores)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return arr.size / best / 1e9, cores, total, best


def node_reference(args, workload):
    """The reference itself (TypeScript under Node, one stream per worker_thread) when a JavaScript engine
    exists on the box: baseline/node_bench.mjs prints one JSON object.  Returns it or None."""
    node = shutil.which("node")
    script = os.path.join(ROOT, "baseline", "node_bench.mjs")
    ref = os.environ.get("ZS_REFERENCE_DIR", "/root/reference")
    if not node or not os.path.exists(script) or not os.path.isdir(ref):
        return None
    try:
        out = subprocess.run([node, script, "--reference", ref, "--workload", workload,
                              "--steps", str(args.steps), "--warmup", str(args.warmup)], capture_output=True, text=True,
                             timeout=900)
        if out.returncode == 0:
            return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception:
        pass
    return None


def run_reference(args):
    """CPU reference arm on the host cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import oracle as O
    O.build()
    corpus = pkg("corpus")
    cores = O.lib().zo_max_threads()
    sharded = args.gpus > 1
    if sharded:
        total = args.total_mib << 20
        chunk, level = CHUNK2, LEVEL2
        # a bounded sample of the 4 GiB per step: the distinct 256 MiB of the corpus (it repeats after that)
        sample_bytes = min(total, 256 << 20)
        sample = corpus.mixed_numpy(sample_bytes, SEED2)
        cfg = config2(total, total // CHUNK2, args.gpus)
        what = f"the first {sample_bytes >> 20} MiB of the 4 GiB corpus per step (its 64 distinct tiles; the rest repeats them)"
    else:
        n = args.size_mib << 20
        chunk, level = CHUNK, LEVEL
        sample_bytes = n
        sample = corpus.text_numpy(n, SEED1)
        cfg = config1(n, n // CHUNK)
        what = f"the whole {n >> 20} MiB corpus per step"
    cfg["sample_bytes"] = sample_bytes
    nb = node_reference(args, "configs2" if sharded else "configs1")
    times = []
    for i in range(args.warmup + args.steps):
        gbs, cores, total_out, dt = cpu_deflate(sample, chunk, level)
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = sample_bytes / (ms / 1e3) / 1e9
    kind, how = "port", ("oracle/deflate.c, byte-exact with C zlib 1.3 -- an upper bound on the TypeScript original, "
                         "which cannot run here: no node")
    if nb and nb.get("value"):
        # the reference itself ran: report it as the arm's value, keep the port beside it
        kind, how = "reference", f"zlib-streams-ts under node {nb.get('node')}, {nb.get('cores')} worker_threads"
        port_value, value, ms, cores = value, float(nb["value"]), float(nb["ms_per_step"]), int(nb["cores"])
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if sharded else "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
        "compressed_ratio": total_out / sample_bytes,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{what}, same chunk + dictionary plan, one stream per host thread ({how})"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if kind == "reference":
        line["cpu_port_value"] = port_value
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# N = 1: configs[1]
# ---------------------------------------------------------------------------------------------------
def run_single(args, torch, dev, local_rank):
    import ctypes as C
    import numpy as np
    B, capi, corpus = pkg("batch"), pkg("capi"), pkg("corpus")
    ctx = B.default_context(local_rank)
    n = args.size_mib << 20
    data = corpus.text_torch(n, dev, seed=SEED1)
    n_chunks = B.n_chunks_for(n, CHUNK)
    flags = B.FLAG_PRIME
    torch.cuda.synchronize()

    def step(bufs):
        return B.deflate_batch_dev(data, CHUNK, LEVEL, B.WRAP_RAW, B.MODE_INDEPENDENT, flags, ctx=ctx, reuse=bufs,
                                   want_checks=False)

    bufs = step(None)
    for _ in range(max(args.warmup - 1, 0)):
        step(bufs)
    torch.cuda.synchronize()
    rr = bufs.read_result()
    out_bytes = int(rr.total_out_bytes)

    # ---- timed region: device-resident input ----
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    launches0 = ctx.launch_count
    ctx.profile(True)
    ctx.profile_read()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step(bufs)
    e1.record()
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    prof = ctx.profile_read()
    ctx.profile(False)
    launches = ctx.launch_count - launches0
    clocks = sampler.stop()
    ms_step = ms_total / args.steps
    value = n / (ms_step / 1e3) / 1e9
    if args.dump_outputs:
        # what deflate_batch_dev hands its caller after the last timed step: every chunk's byte offset and bit
        # length, the totals, and the concatenated raw streams (a seeded sample of them beyond 8 MiB)
        last = bufs.read_result()
        starts, win = sample_windows(int(last.total_out_bytes))
        dump_outputs(args.dump_outputs, {
            "chunk_byte_offsets": bufs.out_off.cpu().numpy().astype(np.float64),
            "chunk_bits": bufs.out_bits.cpu().numpy().astype(np.float64),
            "totals": np.array([last.total_out_bytes, last.total_out_bits, last.check, last.n_blocks], dtype=np.float64),
            "compressed_bytes": torch.cat([bufs.out[p: p + win] for p in starts]).cpu().numpy().astype(np.float32)})

    # ---- e2e: host buffers through zs_deflate_batch ----
    lib = capi.load()
    numa = bind_numa(torch, local_rank)
    h_in = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h_in.copy_(data)
    cap = int(lib.zs_deflate_batch_bound(n, n_chunks, CHUNK, B.WRAP_RAW, B.MODE_INDEPENDENT))
    h_out = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
    h_off = torch.empty(n_chunks + 1, dtype=torch.int64, pin_memory=True)
    h_bits = torch.empty(n_chunks, dtype=torch.int64, pin_memory=True)
    res = capi.DeflateResult()

    def e2e_step():
        rc = lib.zs_deflate_batch(ctx.handle, C.c_void_p(h_in.data_ptr()), n, None, n_chunks, CHUNK, LEVEL, B.WRAP_RAW,
                                  B.MODE_INDEPENDENT, flags, C.c_void_p(h_out.data_ptr()), cap,
                                  C.c_void_p(h_off.data_ptr()), C.c_void_p(h_bits.data_ptr()), None, C.byref(res))
        ctx.check(rc, "zs_deflate_batch")

    e2e_step()
    e2e_step()
    torch.cuda.synchronize()
    e2e_steps = max(1, min(args.steps, 5))
    t0 = time.perf_counter()
    e0.record()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1) / e2e_steps
    wall_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
    e2e_ms = max(e2e_ms, wall_ms)  # the call synchronises internally; never report less than wall time
    e2e_value = n / (e2e_ms / 1e3) / 1e9
    e2e_out = int(res.total_out_bytes)
    # the e2e stream must be the same stream the device path produced
    same = bool(torch.equal(h_out[:e2e_out].to(dev), bufs.out[:out_bytes])) if e2e_out == out_bytes else False
    d2h = e2e_out + 8 * (2 * n_chunks + 1) + 24
    ceil_ms = copy_ceiling(torch, None, 1, dev, h_in, h_out, n, e2e_out)

    # ---- roofline of the dominant kernel (lz77_kernel) ----
    peak, peak_src = hbm_peak()
    lz_n, lz_ms = prof.get("lz77_kernel", (0, 0.0))
    lz_avg_ms = lz_ms / max(lz_n, 1)
    algo_bytes = n + out_bytes + 32768 * (n_chunks - 1)   # SURVEY 8(d): in + compressed out + 32 KiB dictionary per chunk
    achieved = algo_bytes / (lz_avg_ms / 1e3) / 1e9 if lz_avg_ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": "lz77_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": lz_traffic(n, LEVEL), "peak_source": peak_src,
                "kernel_ms_per_launch": lz_avg_ms, "algorithmic_bytes_per_launch": algo_bytes,
                "kernel_share_of_step": lz_avg_ms / ms_step if ms_step else None,
                "per_kernel_ms_per_step": {k: v[1] / args.steps for k, v in sorted(prof.items())},
                # what actually limits the kernel (ncu --set full, profiles/): not DRAM
                "limiter": "integer ALU pipe / instruction issue (ncu: DRAM throughput < 1 %)",
                "issue": lz_issue("lz77_kernel", n, lz_avg_ms, clocks, torch, dev, LEVEL)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": config1(n, n_chunks),
        "compressed_ratio": out_bytes / n,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
                "identical_to_device_path": same, "copy_ceiling_GBps": n / (ceil_ms / 1e3) / 1e9,
                "copy_ceiling_note": "the step's H2D and D2H bytes copied concurrently with no kernels", "numa_node": numa},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "clocks": clocks,
    }

    if not args.no_cpu:
        from oracle import oracle as O
        O.build()
        cores = O.lib().zo_max_threads()
        sample_bytes = min(n, max(64 << 20, cores * (8 << 20)))
        sample = data[:sample_bytes].cpu().numpy()
        gbs, cores, total, dt = cpu_deflate(sample, CHUNK, LEVEL, repeats=2)
        line["cpu_baseline"] = {"value": gbs, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"first {sample_bytes >> 20} MiB of the corpus, same chunk+dictionary plan, "
                                          f"one stream per host thread, best of 2 ({dt:.2f} s)",
                                "compressed_ratio": total / sample_bytes}
        # ratio gate on the same sample (GPU bytes for those chunks / reference bytes)
        k = sample_bytes // CHUNK
        gpu_sample = int(bufs.out_off[k].item())
        line["size_vs_reference_level1"] = gpu_sample / total if total > 0 else None

    if not args.no_extra:
        try:
            line["extra"] = extras(args, torch, dev, ctx, data, bufs, n, n_chunks, h_in, h_out)
        except Exception as e:   # the headline must not die with a side table
            line["extra"] = {"error": repr(e)}
    print(json.dumps(line))


def timed(torch, fn, reps):
    """Average device ms of fn() over reps calls (one untimed call first)."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def extras(args, torch, dev, ctx, data, bufs, n, n_chunks, h_in, h_out):
    """The other BASELINE configs on one GPU (rank 0, outside the headline's timed region)."""
    import ctypes as C
    import numpy as np
    B, capi, corpus = pkg("batch"), pkg("capi"), pkg("corpus")
    lib = capi.load()
    peak = hbm_peak()[0]
    extra = {}
    use_cpu = not args.no_cpu
    if use_cpu:
        from oracle import oracle as O
        O.build()

    # ---- configs[2] shape on one GPU: mixed corpus, zlib level 6, 256 KiB chunks stitched into one stream ----
    m = min(args.total_mib << 20, 1 << 30)
    mixed = corpus.mixed_torch(m, dev, seed=SEED2)
    r6 = B.deflate_batch_dev(mixed, CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx)
    ctx.profile(True); ctx.profile_read()
    ms = timed(torch, lambda: B.deflate_batch_dev(mixed, CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx, reuse=r6), 3)
    prof6 = ctx.profile_read(); ctx.profile(False)
    rr6 = r6.read_result()
    lz6 = prof6.get("lz77_kernel", (1, 0.0))
    lz6_ms = lz6[1] / max(lz6[0], 1)
    c2 = {"workload": "configs[2] on one GPU: 1 GiB mixed corpus, zlib level 6, 256 KiB chunks + 32 KiB priming, one stream",
          "deflate_input_GBps": m / (ms / 1e3) / 1e9, "compressed_ratio": rr6.total_out_bytes / m,
          "lz77_kernel_ms": lz6_ms,
          "roofline_frac": ((m + rr6.total_out_bytes + 32768 * (m // CHUNK2 - 1)) / (lz6_ms / 1e3) / 1e9 / peak) if lz6_ms else None}
    if use_cpu:
        s = mixed[: 32 << 20].cpu().numpy().tobytes()
        ref6 = len(O.deflate(s, LEVEL2, 1))
        g6 = B.deflate_batch_dev(mixed[: 32 << 20], CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx).read_result()
        c2["size_vs_reference_level6"] = g6.total_out_bytes / ref6
        d = zlib.decompressobj(15)
        g = B.deflate_batch_dev(mixed[: 32 << 20], CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx)
        gs = bytes(g.out[: g.read_result().total_out_bytes].cpu().numpy())
        c2["decodes_with_c_zlib"] = bool(d.decompress(gs) + d.flush() == s and d.eof)
    # the same stream decoded again on this GPU: ONE stream without flush points, cut at located block headers
    try:
        S = pkg("sharded")
        zb = int(rr6.total_out_bytes)
        ip = S.inflate_part(r6.out, zb, m, B.WRAP_ZLIB, True, ctx=ctx)
        ms = timed(torch, lambda: S.inflate_part(r6.out, zb, m, B.WRAP_ZLIB, True, ctx=ctx, reuse=ip), 2)
        ip = S.inflate_part(r6.out, zb, m, B.WRAP_ZLIB, True, ctx=ctx, reuse=ip)
        c2["inflate_one_stream_output_GBps"] = m / (ms / 1e3) / 1e9
        c2["inflate_one_stream_bit_exact"] = bool(ip.status == 1 and ip.out_len == m and ip.in_used == zb
                                                  and torch.equal(ip.out[:m], mixed) and ip.check == int(rr6.check))
        del ip
    except Exception as e:
        c2["inflate_one_stream_error"] = repr(e)
    extra["configs2_single_gpu"] = c2
    # the same level-6 plan on the headline's text corpus (what round 1 reported as deflate_level6_input_GBps)
    view = data[: min(n, 512 << 20)]
    r6t = B.deflate_batch_dev(view, CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx)
    ms = timed(torch, lambda: B.deflate_batch_dev(view, CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx, reuse=r6t), 2)
    extra["deflate_level6_input_GBps"] = view.numel() / (ms / 1e3) / 1e9
    extra["level6_ratio"] = r6t.read_result().total_out_bytes / view.numel()
    if use_cpu:
        s = view[: 32 << 20].cpu().numpy().tobytes()
        g6 = B.deflate_batch_dev(view[: 32 << 20], CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx).read_result()
        extra["size_vs_reference_level6"] = g6.total_out_bytes / len(O.deflate(s, LEVEL2, 1))
    del r6, r6t, mixed

    # ---- inflate of the level-1 primed chunks (each chunk = independent raw stream + its dictionary) ----
    off = torch.arange(0, n_chunks + 1, dtype=torch.int64, device=dev) * CHUNK
    off[-1] = n
    starts = off[:-1]
    rng = torch.stack([torch.clamp(starts - 32768, min=0), starts], 1).reshape(-1).contiguous()
    inf = B.inflate_batch_dev(bufs.out, bufs.out_off, off, -15, d_dict=data, dict_rng=rng, out_capacity=n, ctx=ctx)
    ms = timed(torch, lambda: B.inflate_batch_dev(bufs.out, bufs.out_off, off, -15, d_dict=data, dict_rng=rng, ctx=ctx, reuse=inf), 2)
    extra["inflate_output_GBps"] = n / (ms / 1e3) / 1e9
    extra["inflate_roundtrip_bit_exact"] = bool((inf.status == 1).all().item()) and bool(torch.equal(inf.out[:n], data))
    del inf

    # ---- configs[3]: 131072 independent 4 KiB gzip records (reference-produced, ~5 % stored), inflate + crc verify ----
    if use_cpu:
        nrec, rec = 131072, 4096
        src = data[: nrec * rec].clone()
        g = torch.Generator(device=dev); g.manual_seed(3)
        stored = torch.arange(7, nrec, 20, device=dev)              # every 20th record is incompressible
        src.view(nrec, rec)[stored] = torch.randint(0, 256, (stored.numel(), rec), device=dev, generator=g, dtype=torch.uint8)
        host = src.cpu().numpy()
        slot = int(O.lib().zo_deflate_bound(rec, 2)) + 16
        zbuf = np.empty(nrec * slot, dtype=np.uint8)
        zoff = np.zeros(nrec + 1, dtype=np.uint64)
        t0 = time.perf_counter()
        ztotal = int(O.lib().zo_deflate_records_mt(host.ctypes.data, host.size, rec, 6, 2, zbuf.ctypes.data, slot, zoff.ctypes.data, 0))
        t_ref_deflate = time.perf_counter() - t0
        d_z = torch.from_numpy(zbuf[: ztotal + 8].copy()).to(dev)
        d_zoff = torch.from_numpy(zoff.astype(np.int64)).to(dev)
        ooff = torch.arange(0, nrec + 1, dtype=torch.int64, device=dev) * rec
        inf = B.inflate_batch_dev(d_z, d_zoff, ooff, 31, out_capacity=nrec * rec, ctx=ctx)
        ctx.profile(True); ctx.profile_read()
        ms = timed(torch, lambda: B.inflate_batch_dev(d_z, d_zoff, ooff, 31, ctx=ctx, reuse=inf), 3)
        prof3 = ctx.profile_read(); ctx.profile(False)
        ok = bool((inf.status == 1).all().item()) and bool(torch.equal(inf.out[: nrec * rec], src))
        # crc32 of every record against the CPU restatement's value for a sample of records
        ck = inf.checks.cpu().numpy().astype(np.uint32)
        sample_idx = list(range(0, nrec, 997))
        ok_crc = all(int(ck[i]) == O.crc32(host[i * rec:(i + 1) * rec].tobytes()) for i in sample_idx)
        # CPU restatement of inflate on the same records, all host threads
        out_cpu = np.empty(nrec * rec, dtype=np.uint8)
        ooff_h = (np.arange(nrec + 1, dtype=np.uint64) * rec)
        t0 = time.perf_counter()
        bad = int(O.lib().zo_inflate_batch_mt(zbuf.ctypes.data, zoff.ctypes.data, nrec, 31, out_cpu.ctypes.data, ooff_h.ctypes.data,
                                              None, None, None, 0))
        t_cpu = time.perf_counter() - t0
        extra["configs3_gzip_records"] = {
            "workload": "configs[3] per GPU: 131072 x 4 KiB gzip records deflated by the CPU restatement at level 6 "
                        "(5 % incompressible -> stored blocks), inflate + crc32 verify",
            "inflate_output_GBps": nrec * rec / (ms / 1e3) / 1e9, "records_per_s": nrec / (ms / 1e3),
            "compressed_bytes": ztotal, "roofline_frac": (ztotal + nrec * rec) / (ms / 1e3) / 1e9 / peak,
            "per_kernel_ms": {k: v[1] / 3 for k, v in sorted(prof3.items())},
            "bit_exact_and_status_ok": ok, "crc32_matches_oracle_on_sample": ok_crc,
            "cpu_port_inflate_GBps": nrec * rec / t_cpu / 1e9, "cpu_port_bad_streams": bad, "cpu_cores": O.lib().zo_max_threads()}
        # e2e through zs_inflate_batch: pinned host streams in, pinned host output out
        try:
            hz = torch.from_numpy(zbuf[: ztotal + 8]).pin_memory()
            hzoff = torch.from_numpy(zoff.astype(np.int64)).pin_memory()
            hooff = torch.from_numpy(ooff_h.astype(np.int64)).pin_memory()
            hlen = torch.empty(nrec, dtype=torch.int64, pin_memory=True)
            hst = torch.empty(nrec, dtype=torch.int32, pin_memory=True)
            hck = torch.empty(nrec, dtype=torch.int32, pin_memory=True)
            hout = h_in   # reuse the pinned 1 GiB buffer

            def inf_e2e():
                rc = lib.zs_inflate_batch(ctx.handle, C.c_void_p(hz.data_ptr()), C.c_void_p(hzoff.data_ptr()), nrec, 31,
                                          C.c_void_p(hout.data_ptr()), C.c_void_p(hooff.data_ptr()), C.c_void_p(hlen.data_ptr()),
                                          None, C.c_void_p(hck.data_ptr()), C.c_void_p(hst.data_ptr()), None, None, 0)
                ctx.check(rc, "zs_inflate_batch")
            inf_e2e()
            t0 = time.perf_counter()
            for _ in range(3):
                inf_e2e()
            e_ms = 1e3 * (time.perf_counter() - t0) / 3
            extra["configs3_gzip_records"]["e2e_output_GBps"] = nrec * rec / (e_ms / 1e3) / 1e9
            extra["configs3_gzip_records"]["e2e_ok"] = bool((hst == 1).all().item()) and bool(np.array_equal(hout[: nrec * rec].numpy(), host))
        except Exception as e:
            extra["configs3_gzip_records"]["e2e_error"] = repr(e)
        del inf, d_z, src

    # ---- configs[4]: raw deflate64 (64 KiB window) -- the reference's fixtures replicated to ~1 GiB of output ----
    try:
        meta = json.load(open(os.path.join(ROOT, "tests", "golden", "deflate64_fixtures.json")))
        blob = open(os.path.join(ROOT, "tests", "golden", "deflate64_fixtures.bin"), "rb").read()
        d64 = {}
        for name, reps in (("100k_lines.deflate64", 512), ("payload_64k.deflate64", 16384)):
            f = next(x for x in meta["fixtures"] if x["name"] == name)
            z = blob[f["offset"]: f["offset"] + f["length"]]
            zpad = z + bytes((-len(z)) % 8)
            din = torch.from_numpy(np.frombuffer(zpad * reps, dtype=np.uint8).copy()).to(dev)
            ioff = torch.arange(0, reps + 1, dtype=torch.int64, device=dev) * len(zpad)
            cap = (f["out_len"] + 15) & ~15
            ooff = torch.arange(0, reps + 1, dtype=torch.int64, device=dev) * cap
            inf = B.inflate_batch_dev(din, ioff, ooff, -16, out_capacity=cap * reps, ctx=ctx)
            ms = timed(torch, lambda: B.inflate_batch_dev(din, ioff, ooff, -16, ctx=ctx, reuse=inf), 3)
            ok = bool((inf.status == 1).all().item()) and bool((inf.out_len == f["out_len"]).all().item())
            first = bytes(inf.out[: f["out_len"]].cpu().numpy())
            ck = inf.checks.cpu().numpy().astype(np.uint32)
            d64[name] = {"streams": reps, "output_GBps": f["out_len"] * reps / (ms / 1e3) / 1e9, "status_ok": ok,
                         "crc32": "%08x" % zlib.crc32(first), "crc32_expected": f.get("crc32"),
                         "all_streams_same_crc": bool((ck == ck[0]).all()) and int(ck[0]) == zlib.crc32(first)}
            del inf, din
        extra["configs4_deflate64"] = d64
    except Exception as e:
        extra["configs4_deflate64"] = {"error": repr(e)}

    # ---- the drop-in stream API with the reference's slicing (streams.ts:7,78-93): 32 KiB in / 64 KiB out ----
    try:
        extra["stream_api"] = stream_api_bench(ctx, data[: 64 << 20].cpu().numpy(), capi)
    except Exception as e:
        extra["stream_api"] = {"error": repr(e)}

    # ---- the HBM-bound kernels of the path: per-chunk adler32 / crc32 of the same 1 GiB (64 KiB segments) ----
    for kind, name in ((0, "adler32"), (1, "crc32")):
        ms = timed(torch, lambda: B.checksum_batch_dev(data, off, kind, ctx=ctx), 3)
        gbps = n / (ms / 1e3) / 1e9
        extra[f"{name}_GBps"] = gbps
        extra[f"{name}_frac_of_hbm_peak"] = gbps / peak
    return extra


def stream_api_bench(ctx, host, capi, warm=True):
    """zs_stream_deflate / zs_stream_inflate driven like src/mod/streams.ts drives deflate()/inflate(): input in
    32 KiB slices (Z_NO_FLUSH, then Z_FINISH), output through 64 KiB buffers.  The loop itself is C
    (bindings/c/stream_pump.c: a Node-API call costs ~1 us, a ctypes call from Python 30-50 us, which at 32 KiB per
    call would cap the measurement near 1 GB/s whatever the library does)."""
    import ctypes as C
    import numpy as np
    from tools import streampump
    lib = capi.load()
    n = host.size
    big = np.zeros(n + (n >> 3) + (1 << 20), dtype=np.uint8)   # touched: the caller's output buffer exists before the stream starts
    big[::4096] = 1

    def run(init, fn, end, src):
        zs = capi.ZStream()
        assert init(zs) == 0
        t0 = time.perf_counter()
        rc, made, calls = streampump.pump(fn, zs, src, big)
        dt = time.perf_counter() - t0
        end(C.byref(zs))
        if rc != 1:
            raise RuntimeError(f"stream call failed: {rc}")
        return big[:made].copy(), dt, calls

    out = {"loop": "C (bindings/c/stream_pump.c), 32 KiB in / 64 KiB out"}
    if warm:   # one untimed pass: the first use of the stream paths grows their device scratch to this stream's size
        stream_api_bench(ctx, host, capi, warm=False)
    for level in (1, 6):
        comp, dt, calls = run(lambda zs: lib.zs_stream_deflate_init(ctx.handle, C.byref(zs), level, 8, 31, 8, 0),
                              lib.zs_stream_deflate, lib.zs_stream_deflate_end, host)
        out[f"CompressionStream_gzip_level{level}_input_GBps"] = n / dt / 1e9
        out[f"level{level}_ratio"] = comp.size / n
        out[f"level{level}_deflate_calls"] = calls
        out[f"level{level}_decodes_with_c_zlib"] = zlib.decompress(comp.tobytes(), 31) == host.tobytes()
        back, dt, calls = run(lambda zs: lib.zs_stream_inflate_init(ctx.handle, C.byref(zs), 31),
                              lib.zs_stream_inflate, lib.zs_stream_inflate_end, comp)
        out[f"DecompressionStream_own_level{level}_output_GBps"] = n / dt / 1e9
        out[f"level{level}_roundtrip_ok"] = bool(np.array_equal(back, host))
    # a C-zlib stream without flush points: cut at speculatively located block headers
    cz = np.frombuffer(zlib.compress(host.tobytes(), 6), dtype=np.uint8)
    back, dt, calls = run(lambda zs: lib.zs_stream_inflate_init(ctx.handle, C.byref(zs), 15),
                          lib.zs_stream_inflate, lib.zs_stream_inflate_end, cz)
    out["DecompressionStream_czlib_noflush_output_GBps"] = n / dt / 1e9
    out["czlib_noflush_ok"] = bool(np.array_equal(back, host))
    t0 = time.perf_counter()
    zlib.decompress(cz.tobytes())
    out["c_zlib_one_core_inflate_GBps"] = n / (time.perf_counter() - t0) / 1e9
    out["bytes"] = n
    return out


def sharded_inflate_legs(args, torch, dist, dev, rank, world, ctx, buf, hist, local, res, part_bytes, plan, total):
    """The inflate side of the multi-GPU run (outside the deflate line's timed region, same timing rules: barrier +
    synchronize on both sides, device events, max over ranks).
    (1) the stream deflate_sharded just produced, decoded where it lies: every rank inflates its own part with the
        32 KiB before its range as preset dictionary (each part goes through the segment-parallel decoder of one
        stream), the ranks fold adler32 and length with the exchange step, every rank compares its output with its
        shard of the corpus;
    (2) configs[3]: total / 4 KiB independent gzip records (1 M for the 4 GiB corpus), block-partitioned over the
        ranks with no communication, inflate + crc32 of every record checked on the device.
    A rank's own GPU work runs under try/except and the collectives run unconditionally, so that a failure on one
    rank shows up as `ok: false` instead of leaving the other ranks waiting in a collective."""
    B, S, capi = pkg("batch"), pkg("sharded"), pkg("capi")
    n = local.numel()
    out = {}
    d_hist = buf[:hist] if hist else None
    steps = max(1, min(args.steps, 5))
    errors = []

    def max_ms(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ok(ok):
        t = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    # (1) one stream, one part per rank: sharded.inflate_sharded spelled out (inflate_part + the exchange)
    state = {"ip": None}

    def step1():
        ip = None
        try:
            ip = S.inflate_part(res.out, part_bytes, n, B.WRAP_ZLIB, rank == 0, d_hist, ctx=ctx, reuse=state["ip"])
            state["ip"] = ip
        except Exception as e:
            errors.append(repr(e))
        meta = (ip.in_used * 8, ip.check, ip.out_len) if ip is not None else (0, 0, 0)
        return ip, S.exchange_meta(meta[0], meta[1], meta[2], capi.KIND_ADLER32, 0, device=dev)

    step1()
    step1()
    dist.barrier()
    torch.cuda.synchronize()
    ctx.profile(True); ctx.profile_read()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        ip, iplan = step1()
    e1.record()
    torch.cuda.synchronize()
    wall = 1e3 * (time.perf_counter() - t0)
    prof = ctx.profile_read(); ctx.profile(False)
    ms = max_ms(max(e0.elapsed_time(e1), wall) / steps)   # every step ends with a host read: wall == device
    want = 1 if (rank == world - 1) else -5                # Z_STREAM_END on the last part, Z_BUF_ERROR (input ran dry) before
    ok = False
    try:
        ok = (ip is not None and ip.status == want and ip.out_len == n and ip.in_used == part_bytes
              and bool(torch.equal(ip.out[:n], local)) and iplan.check == plan.check and iplan.total_len == total)
    except Exception as e:
        errors.append(repr(e))
    out["one_stream_sharded"] = {
        "workload": "the zlib stream of the deflate line, every rank inflating the part it holds (raw deflate + the 32 KiB "
                    "before its range as dictionary; rank 0 with the zlib header), adler32 folded across ranks",
        "output_GBps": total / (ms / 1e3) / 1e9, "ms_per_step": ms, "steps": steps,
        "bit_exact_and_adler32_ok": all_ok(ok), "adler32": "%08x" % iplan.check,
        "per_kernel_ms_per_step_rank0": {k: v[1] / steps for k, v in sorted(prof.items())}}
    state["ip"] = ip = None

    # (2) configs[3]: independent 4 KiB gzip records
    if not args.no_extra:
        rec = 4096
        nrec = n // rec
        ms, ok, zbytes = 0.0, False, 0
        try:
            src = local[: nrec * rec]
            z = B.deflate_batch_dev(src, rec, 6, B.WRAP_GZIP, B.MODE_INDEPENDENT, 0, ctx=ctx)
            ooff = torch.arange(0, nrec + 1, dtype=torch.int64, device=dev) * rec
            inf = B.inflate_batch_dev(z.out, z.out_off, ooff, 31, out_capacity=nrec * rec, ctx=ctx)
            B.inflate_batch_dev(z.out, z.out_off, ooff, 31, ctx=ctx, reuse=inf)
            torch.cuda.synchronize()
        except Exception as e:
            errors.append(repr(e))
            z = inf = None
        dist.barrier()
        torch.cuda.synchronize()
        try:
            if inf is not None:
                e0.record()
                for _ in range(steps):
                    B.inflate_batch_dev(z.out, z.out_off, ooff, 31, ctx=ctx, reuse=inf)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / steps
                crc = B.checksum_batch_dev(src, ooff, 1, ctx=ctx)
                ok = (bool((inf.status == 1).all().item()) and bool((inf.out_len == rec).all().item())
                      and bool(torch.equal(inf.out[: nrec * rec], src)) and bool(torch.equal(inf.checks, crc)))
                zbytes = int(z.read_result().total_out_bytes)
        except Exception as e:
            errors.append(repr(e))
        ms = max_ms(ms)
        cnt = torch.tensor([nrec, zbytes], dtype=torch.int64, device=dev)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        nrec_all, zbytes_all = int(cnt[0].item()), int(cnt[1].item())
        out["configs3_gzip_records"] = {
            "workload": "configs[3]: %d independent 4 KiB gzip records (the mixed corpus cut in records, deflated at level 6 "
                        "by this engine), block-partitioned over the ranks, inflate + crc32 of every record" % nrec_all,
            "records": nrec_all, "compressed_bytes": zbytes_all,
            "output_GBps": nrec_all * rec / (ms / 1e3) / 1e9 if ms else None,
            "records_per_s": nrec_all / (ms / 1e3) if ms else None, "ms_per_step": ms, "steps": steps,
            "roofline_frac_per_gpu": (zbytes_all + nrec_all * rec) / world / (ms / 1e3) / 1e9 / hbm_peak()[0] if ms else None,
            "bit_exact_status_and_crc32_ok": all_ok(ok)}
        z = inf = None
    if errors:
        out["errors_rank%d" % rank] = errors
    return out


# ---------------------------------------------------------------------------------------------------
# N > 1: configs[2], one stream sharded by contiguous chunk ranges (strong scaling)
# ---------------------------------------------------------------------------------------------------
def run_sharded(args, torch, dist, dev, rank, local_rank, world):
    import ctypes as C
    import numpy as np
    B, S, capi, corpus = pkg("batch"), pkg("sharded"), pkg("capi"), pkg("corpus")
    ctx = B.default_context(local_rank)
    lib = capi.load()
    total = args.total_mib << 20
    n_chunks_all = B.n_chunks_for(total, CHUNK2)
    lo, hi = S.shard_range(n_chunks_all, rank, world)
    b0, b1 = lo * CHUNK2, min(hi * CHUNK2, total)
    hist = min(b0, 32768)
    tiles = corpus.mixed_tiles_numpy(SEED2)
    buf = corpus.mixed_torch_range(b0 - hist, b1, dev, tiles=tiles)
    local = buf[hist:]
    n = local.numel()
    n_chunks = B.n_chunks_for(n, CHUNK2)
    torch.cuda.synchronize()

    state = {"bufs": None}

    def step():
        res, rr, plan = S.deflate_sharded(local, CHUNK2, LEVEL2, B.WRAP_ZLIB, local_is_shard=True, history=hist, ctx=ctx,
                                          reuse=state["bufs"])
        state["bufs"] = res
        return res, rr, plan

    for _ in range(max(args.warmup, 1)):
        res, rr, plan = step()
    torch.cuda.synchronize()
    out_bytes = int(rr.total_out_bytes)

    # ---- timed region: device-resident shards, the exchange step included ----
    dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    launches0 = ctx.launch_count
    ctx.profile(True)
    ctx.profile_read()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        res, rr, plan = step()
    e1.record()
    torch.cuda.synchronize()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    dist.barrier()
    ms_total = max(e0.elapsed_time(e1), wall_ms)     # every step ends with a host read of the result: wall == device
    prof = ctx.profile_read()
    ctx.profile(False)
    launches = ctx.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = total / (ms_step / 1e3) / 1e9
    lz_n, lz_ms = prof.get("lz77_kernel", (0, 0.0))
    lz_avg_ms = lz_ms / max(lz_n, 1)

    # ---- the stitched stream once, outside the timed region: gather on rank 0, decode with C zlib ----
    dist.barrier()
    t0 = time.perf_counter()
    stream = S.gather_stream(res, rr, plan, B.WRAP_ZLIB, dst=0)
    torch.cuda.synchronize()
    gather_ms = 1e3 * (time.perf_counter() - t0)
    verified, ratio = None, None
    if rank == 0:
        d = zlib.decompressobj(15)
        period = tiles.size
        pos, adler = 0, 1
        ok = stream[:2] == S.wrapper_header(B.WRAP_ZLIB, LEVEL2)

        def same(piece, at):
            arr = np.frombuffer(piece, dtype=np.uint8)
            p = 0
            while p < arr.size:
                o = (at + p) % period
                take = min(period - o, arr.size - p)
                if not np.array_equal(arr[p: p + take], tiles[o: o + take]):
                    return False
                p += take
            return True
        step_in = 16 << 20
        for o in range(0, len(stream), step_in):
            piece = d.decompress(stream[o: o + step_in])
            ok = ok and same(piece, pos)
            adler = zlib.adler32(piece, adler)
            pos += len(piece)
            if not ok:
                break
        if ok:
            piece = d.flush()
            ok = same(piece, pos)
            adler = zlib.adler32(piece, adler)
            pos += len(piece)
        verified = bool(ok and d.eof and pos == total and adler == plan.check and d.unused_data == b"")
        ratio = len(stream) / total
        if args.dump_outputs:
            # the last timed step's parts stitched into the one zlib stream, with the exchange step's plan
            s = np.frombuffer(stream, dtype=np.uint8)
            starts, win = sample_windows(s.size)
            dump_outputs(args.dump_outputs, {
                "part_bit_offsets": np.array(plan.bit_offset, dtype=np.float64),
                "totals": np.array([len(stream), plan.total_bits, plan.check, plan.total_len], dtype=np.float64),
                "compressed_bytes": np.concatenate([s[p: p + win] for p in starts]).astype(np.float32)})
    flag = torch.tensor([1 if (verified or rank != 0) else 0], device=dev)
    dist.broadcast(flag, 0)

    # ---- inflate, sharded the same way: every rank decodes the part it holds (sharded.inflate_sharded) ----
    inflate = None
    try:
        inflate = sharded_inflate_legs(args, torch, dist, dev, rank, world, ctx, buf, hist, local, res, out_bytes, plan, total)
    except Exception as e:   # the deflate line must not die with the inflate legs
        inflate = {"error": repr(e)}
    dist.barrier()

    # ---- e2e: every rank's shard from pinned host memory through zs_deflate_part + the exchange ----
    numa = bind_numa(torch, local_rank)
    h_buf = torch.empty(hist + n, dtype=torch.uint8, pin_memory=True)
    h_buf.copy_(buf)
    cap = int(lib.zs_deflate_batch_bound(n, n_chunks, CHUNK2, B.WRAP_ZLIB, B.MODE_STITCHED)) + 64
    h_out = torch.empty(cap, dtype=torch.uint8, pin_memory=True)

    def e2e_step():
        return S.deflate_sharded_host(h_buf, hist, CHUNK2, LEVEL2, B.WRAP_ZLIB, h_out, device=dev, ctx=ctx)

    e2e_step()
    e_res, e_plan = e2e_step()
    dist.barrier()
    torch.cuda.synchronize()
    e2e_steps = max(1, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e_res, e_plan = e2e_step()
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_out = int(e_res.total_out_bytes)
    # every rank decodes its own e2e part with C zlib (raw, primed with the 32 KiB before its range)
    part = h_out[:e2e_out].numpy().tobytes()
    if rank == 0:
        part = part[2:]
    dd = zlib.decompressobj(-15, zdict=bytes(h_buf[:hist].numpy())) if hist else zlib.decompressobj(-15)
    back = dd.decompress(part)
    e_ok = back == h_buf[hist:].numpy().tobytes() and (dd.eof if rank == world - 1 else True) and e_plan.check == plan.check
    okt = torch.tensor([1 if e_ok else 0], device=dev)
    dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    ceil_ms = copy_ceiling(torch, dist, world, dev, h_buf, h_out, hist + n, e2e_out)
    sizes = torch.tensor([hist + n, e2e_out], dtype=torch.int64, device=dev)
    dist.all_reduce(sizes, op=dist.ReduceOp.SUM)

    # ---- the same workload on ONE GPU (rank 0 alone, after the timed regions): the strong-scaling base ----
    single = None
    if rank == 0 and not args.no_extra:
        try:
            whole = corpus.mixed_torch_range(0, total, dev, tiles=tiles)
            r1 = B.deflate_batch_dev(whole, CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx)
            ms1 = timed(torch, lambda: (B.deflate_batch_dev(whole, CHUNK2, LEVEL2, B.WRAP_ZLIB, B.MODE_STITCHED, 0, ctx=ctx, reuse=r1).read_result()), 2)
            single = {"value": total / (ms1 / 1e3) / 1e9, "ms_per_step": ms1, "compressed_ratio": r1.read_result().total_out_bytes / total}
            del whole, r1
        except Exception as e:
            single = {"error": repr(e)}
    dist.barrier()

    if rank == 0:
        peak, peak_src = hbm_peak()
        algo_bytes = n + out_bytes + 32768 * (n_chunks - 1)
        achieved = algo_bytes / (lz_avg_ms / 1e3) / 1e9 if lz_avg_ms > 0 else 0.0
        roofline = {"bound": "hbm", "kernel": "lz77_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": lz_traffic(n, LEVEL2), "peak_source": peak_src,
                    "kernel_ms_per_launch": lz_avg_ms, "algorithmic_bytes_per_launch": algo_bytes,
                    "kernel_share_of_step": lz_avg_ms / ms_step if ms_step else None, "per_gpu": "rank 0's shard",
                    "per_kernel_ms_per_step": {k: v[1] / args.steps for k, v in sorted(prof.items())},
                    "limiter": "integer ALU pipe / instruction issue (ncu: DRAM throughput < 1 %)",
                    "issue": lz_issue("lz77_kernel", n, lz_avg_ms, clocks, torch, dev, LEVEL2)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config2(total, n_chunks_all, world),
            "compressed_ratio": ratio,
            "exchange": {"collective": "all_gather of (bit length, adler32, length) per rank -> exclusive scan -> adler32_combine",
                         "bit_offsets": plan.bit_offset, "total_bits": plan.total_bits, "adler32": "%08x" % plan.check,
                         "inside_timed_region": True},
            "verified": verified, "verification": "stream gathered on rank 0, decoded by C zlib, compared with the corpus, adler32 trailer checked",
            "gather_stream_ms": gather_ms,
            "e2e": {"value": total / (e2e_ms / 1e3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(sizes[0].item()),
                    "d2h_bytes_per_step": int(sizes[1].item()) + 24 * world, "ms_per_step": e2e_ms,
                    "verified": bool(okt.item()), "copy_ceiling_GBps": total / (ceil_ms / 1e3) / 1e9,
                    "copy_ceiling_note": "every rank's H2D and D2H bytes of one step copied concurrently with no kernels, max over ranks",
                    "numa_node_rank0": numa},
            "single_gpu_same_workload": single,
            "inflate": inflate,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "clocks": clocks,
        }
        if not args.no_cpu:
            from oracle import oracle as O
            O.build()
            sample = tiles[: 128 << 20]
            gbs, cores, tot, dt = cpu_deflate(sample, CHUNK2, LEVEL2)
            line["cpu_baseline"] = {"value": gbs, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"first {sample.size >> 20} MiB of the corpus, same chunk+dictionary plan, one stream per host thread ({dt:.2f} s)",
                                    "compressed_ratio": tot / sample.size}
            # size gate on rank 0's first chunks: GPU bits for the sample / reference bytes for the same plan
            k = sample.size // CHUNK2
            if k <= n_chunks:
                gpu_bits = int(res.out_off[k].item()) if k < n_chunks else int(rr.total_out_bits)
                line["size_vs_reference_level6"] = (gpu_bits / 8) / tot
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size-mib", type=int, default=1024, help="configs[1]: corpus size per GPU (MiB)")
    ap.add_argument("--total-mib", type=int, default=4096, help="configs[2]: size of the one sharded corpus (MiB)")
    ap.add_argument("--no-extra", action="store_true", help="skip the side measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--force-sharded", action="store_true", help="run the N > 1 code path with however many ranks there are "
                    "(one rank: a check of that path on a single GPU, not a bench line)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy: the "
                    "compressed bytes (a fixed, seeded 8 MiB sample of them when longer), offsets and totals")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has no such outputs")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 or args.force_sharded:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        os.environ.setdefault("RANK", "0")
        os.environ.setdefault("WORLD_SIZE", "1")
        dist.init_process_group("nccl", device_id=dev)
        run_sharded(args, torch, dist, dev, rank, local_rank, world)
        dist.barrier()
        dist.destroy_process_group()
    else:
        run_single(args, torch, dev, local_rank)


if __name__ == "__main__":
    main()
