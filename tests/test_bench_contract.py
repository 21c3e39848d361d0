"""CPU: what can be checked of bench.py without a GPU -- the reference arm (`--impl reference`: the oracle port of the
reference's deflate on the host cores, a bounded sample per step) prints ONE JSON line with the contract's keys for
the N = 1 and the N > 1 workload, a non-zero rank of a torchrun launch prints nothing, and the product arm refuses to
run without a CUDA device (there is no CPU fallback).  On a GPU: what --dump-outputs writes is the timed path's output."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT, pkg

BENCH = os.path.join(ROOT, "bench.py")


def _run(args, env=None):
    e = dict(os.environ)
    e.pop("RANK", None)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, timeout=300, env=e)


def test_reference_arm_lines():
    for args, workload, scaling in ((["--size-mib", "16"], "configs[1]", "weak"), (["--gpus", "2", "--total-mib", "32"], "configs[2]", "strong")):
        p = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", *args])
        assert p.returncode == 0, p.stderr[-2000:]
        lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
        assert len(lines) == 1
        d = json.loads(lines[0])
        assert d["impl"] == "reference" and d["metric"] == "deflate_input_GBps" and d["unit"] == "GB/s"
        assert d["higher_is_better"] is True and d["scaling"] == scaling and d["steps"] == 1 and d["warmup"] == 1
        assert d["config"]["workload"].startswith(workload) and d["value"] > 0 and d["ms_per_step"] > 0
        assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
        assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
        assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["dtype"] == "u8"
        assert 0.2 < d["compressed_ratio"] < 0.8
    # under torchrun only rank 0 runs the arm: the other ranks exit 0 without a line
    p = _run(["--impl", "reference", "--gpus", "2", "--total-mib", "32", "--steps", "1", "--warmup", "0"], env={"RANK": "1"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    p = _run(["--steps", "1", "--warmup", "1", "--size-mib", "16"])
    assert p.returncode != 0 and "no CUDA device" in (p.stderr + p.stdout)


def test_arguments_refused(tmp_path):
    """No timed step at all, and a dump of the reference arm (which computes nothing on the GPU), are usage errors."""
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        p = _run([*args, "--size-mib", "16"])
        assert p.returncode == 2 and "error" in p.stderr
    assert not any(tmp_path.iterdir())


def test_sample_windows():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", BENCH)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert bench.sample_windows(1000) == ([0], 1000)
    starts, win = bench.sample_windows(300 << 20)
    assert win == 16384 and len(starts) * win == 8 << 20 and starts == sorted(set(starts))
    assert all(p % win == 0 and p + win <= 300 << 20 for p in starts) and bench.sample_windows(300 << 20) == (starts, win)


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_path_outputs(gpu_ctx, tmp_path):
    """--dump-outputs of the N = 1 path: every chunk's raw stream, primed with the 32 KiB before it, decodes to the
    seeded corpus, and the offsets, bit lengths and totals agree with each other and with the JSON line."""
    import zlib

    import numpy as np
    import torch
    p = _run(["--steps", "2", "--warmup", "1", "--size-mib", "8", "--no-extra", "--no-cpu", "--dump-outputs", str(tmp_path)])
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2
    d = {f.stem: np.load(f) for f in tmp_path.iterdir()}
    assert sorted(d) == ["chunk_bits", "chunk_byte_offsets", "compressed_bytes", "totals"]
    assert d["compressed_bytes"].dtype == np.float32 and all(d[k].dtype == np.float64 for k in ("chunk_bits", "chunk_byte_offsets", "totals"))
    off = d["chunk_byte_offsets"].astype(np.int64)
    total = int(d["totals"][0])
    assert off.size == 129 and off[0] == 0 and off[-1] == total == d["compressed_bytes"].size   # 8 MiB compress to less than the 8 MiB dumped whole
    assert total == round(line["compressed_ratio"] * (8 << 20))
    assert np.all((d["chunk_bits"] + 7) // 8 == np.diff(off))
    corpus = pkg("corpus").text_torch(8 << 20, torch.device("cuda", 0), seed=0xC0FFEE).cpu().numpy().tobytes()
    z = d["compressed_bytes"].astype(np.uint8).tobytes()
    for i in range(off.size - 1):
        lo = i * 65536
        dec = zlib.decompressobj(-15, zdict=corpus[max(0, lo - 32768): lo]) if lo else zlib.decompressobj(-15)
        assert dec.decompress(z[off[i]: off[i + 1]]) == corpus[lo: lo + 65536] and dec.eof, i
