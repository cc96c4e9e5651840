"""Deterministic test inputs, independent of numpy's RNG streams (pure splitmix64 arithmetic).

`make_page(kind, n, seed)` kinds:
  R random bytes | T 4-letter text w.p. 3/4 else random byte | Z zeros with a 2-byte stamp |
  M second half repeats the first | P short period with sparse noise | A tiny alphabet |
  X segments of all of the above | S bench-stream chunk (edge_fuse_b200 generator, cid = seed)
"""
from __future__ import annotations

import numpy as np

G = np.uint64(0x9E3779B97F4A7C15)


def _mix(z: np.ndarray) -> np.ndarray:
    z = z.astype(np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def words(seed: int, count: int) -> np.ndarray:
    with np.errstate(over="ignore"):
        idx = (np.arange(1, count + 1, dtype=np.uint64) * G) + np.uint64(seed & 0xFFFFFFFFFFFFFFFF)
    return _mix(idx)


def rand_bytes(seed: int, n: int) -> np.ndarray:
    return words(seed, (n + 7) // 8).view(np.uint8)[:n].copy()


def make_page(kind: str, n: int, seed: int) -> np.ndarray:
    if n == 0:
        return np.zeros(0, dtype=np.uint8)
    if kind == "R":
        return rand_bytes(seed, n)
    if kind == "T":
        r = rand_bytes(seed, n)
        sel = rand_bytes(seed ^ 0x5151, n)
        text = (97 + (sel >> 2) % 4).astype(np.uint8)
        return np.where((sel & 3) != 0, text, r).astype(np.uint8)
    if kind == "Z":
        z = np.zeros(n, dtype=np.uint8)
        z[: min(2, n)] = rand_bytes(seed, 2)[: min(2, n)]
        return z
    if kind == "M":
        h = make_page("T", (n + 1) // 2, seed)
        return np.concatenate([h, h])[:n].copy()
    if kind == "P":
        w = words(seed, 4)
        period = int(w[0] % np.uint64(39)) + 1
        pat = rand_bytes(seed ^ 0x77, period)
        a = np.tile(pat, n // period + 1)[:n].copy()
        nn = int(w[1] % np.uint64(200))
        if nn:
            pos = (words(seed ^ 0x99, nn) % np.uint64(n)).astype(np.int64)
            a[pos] = rand_bytes(seed ^ 0xAB, nn)
        return a
    if kind == "A":
        k = int(words(seed, 1)[0] % np.uint64(4)) + 2
        return (rand_bytes(seed ^ 0x33, n) % k).astype(np.uint8)
    if kind == "X":
        out, tot, i = [], 0, 0
        lens = words(seed ^ 0xC0FFEE, 4096)
        while tot < n:
            k = int(lens[i] % np.uint64(3000)) + 1
            sub = "RTZMPA"[int(lens[i] >> np.uint64(40)) % 6] if k > 8 else "R"
            out.append(make_page(sub, k, seed + 1000 + i))
            tot += k
            i += 1
        return np.concatenate(out)[:n].copy()
    if kind == "S":
        import edge_fuse_b200 as E
        return E.gen_chunk_host(42, seed, n)
    raise ValueError(kind)


def pad_rows(pages: list[np.ndarray], stride: int | None = None) -> np.ndarray:
    n = max((len(p) for p in pages), default=0)
    stride = stride or max(16, (n + 15) // 16 * 16)
    buf = np.zeros((len(pages), stride), dtype=np.uint8)
    for i, p in enumerate(pages):
        buf[i, : len(p)] = p
    return buf


# The case list shared by the golden generator (tools/gen_golden.py), the oracle pin test and the
# GPU parity test: (kind, nbytes, accel, seed).
def codec_cases():
    cases = []
    for kind in "RTZMPAXS":
        for n in (4096, 32768, 65536, 131072):
            cases.append((kind, n, 12, 7 + len(cases)))
    for n in (65546, 65547, 8192, 16384, 100, 13, 12, 1, 5000):
        for kind in "RTZP":
            cases.append((kind, n, 12, 300 + len(cases)))
    for accel in (1, 3, 64, 1000, -5):
        for kind in "RTMX":
            cases.append((kind, 65536, accel, 500 + len(cases)))
    for cid in range(8):
        cases.append(("S", 65536, 12, cid))
    return cases


# The cases that the oracle and the CUDA encoder are compared on with the compiled reference
# (tests/golden/reference_lz4.json holds the reference's answers): (kind, nbytes, accel, seed).
def reference_lz4_cases():
    return [(kind, n, accel, 10_000 * rep + n + accel + ord(kind))
            for rep in range(2)
            for n in (4096, 16384, 65536, 131072, 65546, 65547, 13, 12, 1, 777)
            for accel in (12, 1, 0, 5, 200)
            for kind in "RTZMPAX"]


def reference_cuda_cases():
    return [("RTZMPAX"[i % 7], bs, 12, 9000 + i) for bs, n in ((65536, 84), (4096, 140)) for i in range(n)]
