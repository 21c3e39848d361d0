"""Deterministic synthetic corpora of SURVEY.md section 8(d) (bench + tests; not part of the engine).

text   : word salad from a 4096-word vocabulary (words of 2-9 lowercase letters, 85 % space /
         15 % newline separators)
mixed  : 4 MiB tiles of 40 % text, 20 % ramp (j % 251), 20 % uniform random bytes, 10 % zeros /
         long runs, 10 % far repeats of 4 KiB blocks
Generated with numpy on the host (tests, CPU baseline samples) or with torch on the GPU (bench).
"""
from __future__ import annotations

import numpy as np


def _vocab(seed: int):
    rng = np.random.default_rng(seed)
    lens = rng.integers(2, 10, size=4096)
    W = np.zeros((4096, 10), dtype=np.uint8)
    for i, l in enumerate(lens):
        W[i, :l] = rng.integers(97, 123, size=l)
    return W, lens.astype(np.int64)


def text_numpy(n: int, seed: int = 0xC0FFEE) -> np.ndarray:
    """n bytes of word-salad text (host)."""
    W, lens = _vocab(seed)
    rng = np.random.default_rng(seed + 1)
    out = np.empty(n + 16, dtype=np.uint8)
    pos = 0
    while pos < n:
        k = max(1024, (n - pos) // 5 + 16)
        idx = rng.integers(0, 4096, size=k)
        sep = np.where(rng.random(k) < 0.85, 32, 10).astype(np.uint8)
        wl = lens[idx] + 1
        ends = np.cumsum(wl)
        total = int(ends[-1])
        starts = ends - wl
        word_of_byte = np.repeat(np.arange(k), wl)
        within = np.arange(total) - np.repeat(starts, wl)
        Wsep = W[idx].copy()
        Wsep[np.arange(k), lens[idx]] = sep
        piece = Wsep[word_of_byte, within]
        take = min(total, n - pos)
        out[pos:pos + take] = piece[:take]
        pos += take
    return out[:n]


def mixed_numpy(n: int, seed: int = 0xB200, tile: int = 4 << 20) -> np.ndarray:
    """n bytes of the mixed corpus (host)."""
    rng = np.random.default_rng(seed)
    out = np.empty(n, dtype=np.uint8)
    pos = 0
    t = 0
    while pos < n:
        size = min(tile, n - pos)
        parts = []
        a = int(size * 0.4)
        parts.append(text_numpy(a, seed + 7 * t + 1))
        b = int(size * 0.2)
        parts.append((np.arange(b, dtype=np.int64) % 251).astype(np.uint8))
        c = int(size * 0.2)
        parts.append(rng.integers(0, 256, size=c, dtype=np.uint8))
        d = int(size * 0.1)
        runs = np.zeros(d, dtype=np.uint8)
        if d > 4096:
            runs[d // 2:] = np.repeat(rng.integers(0, 256, size=(d - d // 2 + 511) // 512, dtype=np.uint8), 512)[: d - d // 2]
        parts.append(runs)
        e = size - a - b - c - d
        blk = rng.integers(0, 256, size=4096, dtype=np.uint8)
        rep = np.tile(blk, e // 4096 + 1)[:e].copy()
        if e > 8192:
            holes = rng.integers(0, e, size=e // 2048)
            rep[holes] = rng.integers(0, 256, size=holes.size, dtype=np.uint8)
        parts.append(rep)
        piece = np.concatenate(parts)[:size]
        out[pos:pos + size] = piece
        pos += size
        t += 1
    return out


def text_torch(n: int, device, seed: int = 0xC0FFEE, piece: int = 64 << 20):
    """n bytes of word-salad text generated on `device` (torch uint8 tensor)."""
    import torch

    W, lens = _vocab(seed)
    Wt = torch.from_numpy(W).to(device)
    Lt = torch.from_numpy(lens).to(device)
    g = torch.Generator(device=device)
    g.manual_seed(seed + 1)
    out = torch.empty(n, dtype=torch.uint8, device=device)
    pos = 0
    while pos < n:
        want = min(piece, n - pos)
        k = want // 5 + 64
        idx = torch.randint(0, 4096, (k,), device=device, generator=g)
        sep = torch.where(torch.rand(k, device=device, generator=g) < 0.85, 32, 10).to(torch.uint8)
        wl = Lt[idx] + 1
        ends = torch.cumsum(wl, 0)
        total = int(ends[-1].item())
        starts = ends - wl
        Wsep = Wt[idx].clone()
        Wsep[torch.arange(k, device=device), Lt[idx]] = sep
        word_of_byte = torch.repeat_interleave(torch.arange(k, device=device), wl)
        within = torch.arange(total, device=device) - torch.repeat_interleave(starts, wl)
        data = Wsep[word_of_byte, within]
        take = min(total, want)
        out[pos:pos + take] = data[:take]
        pos += take
        del idx, sep, wl, ends, starts, Wsep, word_of_byte, within, data
    return out


def mixed_torch(n: int, device, seed: int = 0xB200, tile: int = 4 << 20):
    """n bytes of the mixed corpus generated on `device`: 64 distinct 4 MiB tiles, then repeated."""
    import torch

    n_unique = min(64, -(-n // tile))
    uniq = torch.from_numpy(mixed_numpy(n_unique * tile, seed, tile)).to(device)
    reps = -(-n // uniq.numel())
    return uniq.repeat(reps)[:n].contiguous()


def mixed_tiles_numpy(seed: int = 0xB200, tile: int = 4 << 20, n_unique: int = 64) -> np.ndarray:
    """The distinct tiles of the mixed corpus (host): byte g of the corpus is tiles[g % tiles.size]."""
    return mixed_numpy(n_unique * tile, seed, tile)


def mixed_torch_range(lo: int, hi: int, device, seed: int = 0xB200, tile: int = 4 << 20, n_unique: int = 64, tiles=None):
    """Bytes [lo, hi) of mixed_torch(N >= hi, ...) without materialising the rest: what one rank of a
    sharded run holds (its chunk range plus the 32 KiB before it)."""
    import torch

    if tiles is None:
        tiles = mixed_tiles_numpy(seed, tile, n_unique)
    period = tiles.size
    uniq = torch.from_numpy(tiles).to(device)
    out = torch.empty(hi - lo, dtype=torch.uint8, device=device)
    pos = lo
    while pos < hi:
        o = pos % period
        take = min(period - o, hi - pos)
        out[pos - lo: pos - lo + take] = uniq[o: o + take]
        pos += take
    return out


_JSON_KEYS = ["id", "user", "name", "email", "created_at", "updated_at", "status", "type", "score", "tags", "region",
              "device", "session", "latency_ms", "bytes", "path", "method", "code", "message", "level", "version",
              "count", "enabled", "ratio", "parent", "owner", "priority", "source"]
_JSON_WORDS = ["active", "pending", "closed", "error", "warning", "info", "debug", "GET", "POST", "PUT", "eu-west-1",
               "us-east-2", "ap-south-1", "mobile", "desktop", "tablet", "admin", "guest", "premium", "trial", "/api/v1/items",
               "/api/v1/users", "/login", "/search", "timeout", "ok", "not found", "alpha", "beta", "gamma"]


def json_pool(n: int, seed: int = 0x4A53) -> bytes:
    """About n bytes of JSON-like rows (one object per line: a fixed key vocabulary, words, numbers, dates), the
    kind of small records a preset dictionary is for.  Deterministic in `seed`."""
    rng = np.random.default_rng(seed)
    rows = []
    size = 0
    while size < n:
        nk = int(rng.integers(4, 12))
        keys = rng.choice(len(_JSON_KEYS), size=nk, replace=False)
        parts = []
        for k in sorted(keys):
            key = _JSON_KEYS[k]
            kind = int(rng.integers(0, 5))
            if kind == 0:
                v = str(int(rng.integers(0, 10 ** int(rng.integers(1, 9)))))
            elif kind == 1:
                v = '"%s"' % _JSON_WORDS[int(rng.integers(0, len(_JSON_WORDS)))]
            elif kind == 2:
                v = "%.3f" % float(rng.random() * 1000)
            elif kind == 3:
                v = '"2026-%02d-%02dT%02d:%02d:%02dZ"' % tuple(int(x) for x in rng.integers([1, 1, 0, 0, 0], [13, 29, 24, 60, 60]))
            else:
                v = "true" if rng.random() < 0.5 else "false"
            parts.append('"%s": %s' % (key, v))
        row = ("{" + ", ".join(parts) + "}\n").encode()
        rows.append(row)
        size += len(row)
    return b"".join(rows)[:n]
