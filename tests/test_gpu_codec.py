"""GPU parity, kernel level: the CUDA LZ4 encoder / decoder / key kernels against the oracle and
the committed golden vectors, through the C ABI.  Bit-exact (integer / byte work)."""
import hashlib
import json
import os

import numpy as np
import pytest

import datagen

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def _encode_group(E, pages, n, accel, fingerprints=False):
    return E.lz4_encode_batch(datagen.pad_rows(pages), nbytes=n, accel=accel, fingerprints=fingerprints)


def test_compose_and_keys(E, gpu, oracle):
    k = json.load(open(os.path.join(GOLD, "keys.json")))
    rng_off = datagen.words(1, 500)
    offs = np.concatenate([rng_off >> np.uint64(3), [np.uint64((1 << 44) << 16), np.uint64(65537), np.uint64(0)]])
    nh = datagen.words(2, len(offs))
    gen = (datagen.words(3, len(offs)) & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    for pshift in (12, 16, 17):
        addr, valid, key = E.compose_keys(offs, nh, gen, pshift)
        for i in range(len(offs)):
            exp = oracle.addr_compose(int(offs[i]), int(nh[i]), int(gen[i]), pshift)
            assert bool(valid[i]) == (exp is not None)
            if exp:
                assert (int(addr[i, 0]), int(addr[i, 1])) == exp
                assert int(key[i]) == oracle.addr_key(*exp)
    # golden address -> key vectors from the reference's own header
    u = np.array([int(a[0], 16) for a in k["addrs"]], dtype=np.uint64)
    l = np.array([int(a[1], 16) for a in k["addrs"]], dtype=np.uint64)
    page = l & np.uint64((1 << 44) - 1)
    gen = (l >> np.uint64(44)).astype(np.uint32)
    addr, valid, key = E.compose_keys(page << np.uint64(4), u, gen, 4)
    assert valid.all() and (addr[:, 1] == l).all()
    assert [int(x) for x in key] == [int(a[2], 16) for a in k["addrs"]]


def test_encode_golden_vectors(E, gpu, oracle):
    g = json.load(open(os.path.join(GOLD, "lz4_blocks.json")))["cases"]
    groups = {}
    for rec in g:
        groups.setdefault((rec["n"], rec["accel"]), []).append(rec)
    for (n, accel), recs in groups.items():
        if n == 0:
            continue
        pages = [datagen.make_page(r["kind"], n, r["seed"]) for r in recs]
        blocks, _ = _encode_group(E, pages, n, accel)
        for r, p, b in zip(recs, pages, blocks):
            assert len(b) == r["len"] and sha(b) == r["sha256"], (r["kind"], n, accel, len(b), r["len"])
            assert b == oracle.lz4_encode(p, accel)


def test_encode_matches_oracle_many(E, gpu, oracle):
    for n, accel, reps in ((65536, 12, 40), (4096, 12, 64), (131072, 12, 12), (32768, 1, 16), (65536, 97, 8)):
        pages = [datagen.make_page("RTZMPAXS"[i % 8], n, 9000 + 31 * i + n) for i in range(reps)]
        blocks, _ = _encode_group(E, pages, n, accel)
        for i, (p, b) in enumerate(zip(pages, blocks)):
            exp = oracle.lz4_encode(p, accel)
            assert b == exp, (n, accel, i, len(b), len(exp))


def test_encode_edge_inputs(E, gpu, oracle):
    n = 65536
    pages = [
        np.zeros(n, np.uint8),                                   # one giant match
        np.full(n, 0xAB, np.uint8),
        np.tile(np.arange(256, dtype=np.uint8), n // 256),       # period 256
        np.tile(np.array([1, 2, 3], np.uint8), n // 3 + 1)[:n],  # period 3 (overlapping matches)
        np.concatenate([datagen.make_page("R", n - 20, 4), np.zeros(20, np.uint8)]),   # match at the very end
        np.concatenate([np.zeros(20, np.uint8), datagen.make_page("R", n - 20, 5)]),
        np.concatenate([datagen.make_page("R", 5000, 6)] * 14)[:n],                   # far repeats
        np.concatenate([datagen.make_page("T", 300, 7)] * 219)[:n],
    ]
    blocks, _ = _encode_group(E, pages, n, 12)
    for p, b in zip(pages, blocks):
        assert b == oracle.lz4_encode(p, 12)
    assert len(blocks[0]) == 267                                  # SURVEY.md §8c known answer


def test_decode_matches_and_consumes(E, gpu, oracle):
    for n in (65536, 4096, 131072, 5000):
        pages = [datagen.make_page("RTZMPAXS"[i % 8], n, 50 + i + n) for i in range(24)]
        blocks = [oracle.lz4_encode(p, 12) for p in pages]
        out, used = E.lz4_decode_batch(blocks, n)
        for i, (p, b) in enumerate(zip(pages, blocks)):
            assert used[i] == len(b), (n, i, used[i], len(b))
            assert (out[i] == p).all(), (n, i)


def test_decode_rejects_malformed(E, gpu, oracle):
    page = datagen.make_page("T", 4096, 5)
    blk = oracle.lz4_encode(page, 12)
    bad = [blk[:-3], b"\x10\x41\x00\x00" + b"\0" * 16, blk[: len(blk) // 2]]
    _, used = E.lz4_decode_batch(bad, 4096)
    assert (used != np.array([len(b) for b in bad])).all()
    _, used = E.lz4_decode_batch([blk], 4095)
    assert used[0] != len(blk)


def test_roundtrip_full_size_properties(E, gpu):
    """BASELINE-size property check without the oracle: encode -> decode is the identity and the
    decoder consumes exactly what the encoder produced, on 2048 x 64 KiB stream chunks."""
    n, count = 65536, 2048
    pages = np.stack([E.gen_chunk_host(42, c, n) for c in range(count)])
    blocks, fps = E.lz4_encode_batch(pages, accel=12, fingerprints=True)
    out, used = E.lz4_decode_batch(blocks, n)
    assert (used == np.array([len(b) for b in blocks])).all()
    assert (out == pages).all()
    lens = np.array([len(b) for b in blocks])
    cls = (np.arange(count) + (np.arange(count) >> 3)) & 3
    assert (lens[cls == 0] == 65794).mean() > 0.9   # R: incompressible (a stray 4-byte match is possible)
    assert (lens[cls == 2] <= 300).all()            # Z chunks
    assert len({(int(a), int(b)) for a, b in fps}) == count


def test_fingerprint_matches_spec(E, gpu, oracle):
    for n in (65536, 4096, 131072, 513, 512, 100, 16, 8200):
        pages = [datagen.make_page("RTZM"[i % 4], n, 70 + i) for i in range(9)]
        fps = E.fingerprint_batch(datagen.pad_rows(pages), nbytes=n)
        for p, f in zip(pages, fps):
            assert (int(f[0]), int(f[1])) == oracle.fingerprint128(p), n
    # the fused kernel computes the same value
    pages = [datagen.make_page("X", 65536, 900 + i) for i in range(6)]
    _, fps = E.lz4_encode_batch(np.stack(pages), accel=12, fingerprints=True)
    for p, f in zip(pages, fps):
        assert (int(f[0]), int(f[1])) == oracle.fingerprint128(p)


def test_encode_fuzz_high_clash(E, gpu, oracle):
    """Many small pages built to stress the speculative batch: tiny alphabets and short periods
    (many lanes hashing to one table slot), matches at every distance, runs ending at every
    offset near the block end.  4-16 KiB so the oracle does 3000 pages in seconds."""
    pages_by_n = {}
    idx = 0
    for n in (4096, 8192, 16384):
        ps = []
        for i in range(1000 if n == 4096 else 500):
            w = datagen.words(777 + idx, 8)
            mode = int(w[0] % np.uint64(6))
            if mode == 0:      # alphabet of 2-4 symbols
                p = (datagen.rand_bytes(idx, n) % np.uint8(2 + int(w[1] % np.uint64(3)))).astype(np.uint8)
            elif mode == 1:    # period 1..64 with a few flipped bytes
                per = 1 + int(w[1] % np.uint64(64))
                p = np.tile(datagen.rand_bytes(idx, per), n // per + 1)[:n].copy()
                k = int(w[2] % np.uint64(12))
                if k:
                    p[(datagen.words(idx ^ 5, k) % np.uint64(n)).astype(np.int64)] ^= 0x55
            elif mode == 2:    # text-like with runs of zeros
                p = datagen.make_page("T", n, idx)
                a = int(w[1] % np.uint64(n - 600)); p[a:a + int(w[2] % np.uint64(600))] = 0
            elif mode == 3:    # copy of an earlier window at a random distance
                p = datagen.make_page("R", n, idx)
                d = 1 + int(w[1] % np.uint64(n // 2)); L = int(w[2] % np.uint64(n // 4))
                p[d + 100:d + 100 + L] = p[100:100 + L][: max(0, min(L, n - d - 100))]
            elif mode == 4:    # random bytes with the tail being a repeat (match runs into the end margin)
                p = datagen.make_page("R", n, idx)
                t = 5 + int(w[1] % np.uint64(40)); p[n - t:] = p[n - 2 * t:n - t]
            else:
                p = datagen.make_page("X", n, idx)
            ps.append(p)
            idx += 1
        pages_by_n[n] = ps
    for n, ps in pages_by_n.items():
        for accel in (12, 1):
            blocks, _ = E.lz4_encode_batch(np.stack(ps), accel=accel)
            bad = [i for i, (p, b) in enumerate(zip(ps, blocks)) if b != oracle.lz4_encode(p, accel)]
            assert not bad, (n, accel, bad[:5])


def test_encode_wide_mode_fuzz(E, gpu, oracle):
    """pshift 17 (byU32 table, 12-bit hash5, MAX_DISTANCE test): far matches beyond 64 KiB must be
    rejected, near ones taken."""
    n = 131072
    ps = []
    for i in range(48):
        w = datagen.words(4242 + i, 4)
        p = datagen.make_page("RTXM"[i % 4], n, 9100 + i)
        d = 60000 + int(w[0] % np.uint64(12000))          # straddles the 65535 limit
        L = 200 + int(w[1] % np.uint64(3000))
        p[d + 500:d + 500 + L] = p[500:500 + L]
        ps.append(p)
    blocks, _ = E.lz4_encode_batch(np.stack(ps), accel=12)
    for i, (p, b) in enumerate(zip(ps, blocks)):
        assert b == oracle.lz4_encode(p, 12), i
    out, used = E.lz4_decode_batch(blocks, n)
    assert (used == np.array([len(b) for b in blocks])).all() and (out == np.stack(ps)).all()


def test_plain_data_path_parity(gpu):
    """The encoder's other data path (CMB200_ENC_MODE=0: the page read through the L1 instead of the
    TMA ring — what accelerations above 12 and unaligned buffers take) must emit the same bytes; the
    mode is read once per process, so it runs in a child process over the golden vectors and a
    slice of the fuzz set."""
    import subprocess
    import sys
    code = r'''
import sys, os, json, hashlib
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import numpy as np, datagen, edge_fuse_b200 as E
from oracle import ef_oracle as O
g = json.load(open("tests/golden/lz4_blocks.json"))["cases"]
groups = {}
for r in g:
    if r["n"]: groups.setdefault((r["n"], r["accel"]), []).append(r)
for (n, accel), recs in groups.items():
    pages = [datagen.make_page(r["kind"], n, r["seed"]) for r in recs]
    blocks, fps = E.lz4_encode_batch(datagen.pad_rows(pages), nbytes=n, accel=accel, fingerprints=True)
    for r, p, b, f in zip(recs, pages, blocks, fps):
        assert hashlib.sha256(b).hexdigest() == r["sha256"], (r["kind"], n, accel)
        assert (int(f[0]), int(f[1])) == O.fingerprint128(p)
ps = [datagen.make_page("XTPA"[i % 4], 8192, 31 * i) for i in range(600)]
blocks, _ = E.lz4_encode_batch(np.stack(ps), accel=12)
assert all(b == O.lz4_encode(p, 12) for p, b in zip(ps, blocks))
eng = E.Engine(pshift=16, accel=12, capacity=2048, arena_bytes=128 << 20, max_batch=256, flags=E.FINGERPRINT)
pages = np.stack([E.gen_chunk_host(42, c, 65536) for c in range(64)])
u = np.full(64, 3, dtype=np.uint64); l = np.arange(64, dtype=np.uint64)
eng.put(u, l, pages); out, st = eng.get(u, l)
assert (st == E.HIT).all() and (out == pages).all()
fps, ok = eng.read_fingerprints(u, l)
assert ok.all() and (int(fps[5, 0]), int(fps[5, 1])) == O.fingerprint128(pages[5])
print("plain-path parity ok")
'''
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=dict(os.environ, CMB200_ENC_MODE="0"),
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "plain-path parity ok" in out.stdout, out.stdout + out.stderr


@pytest.mark.gpu
def test_cuda_blocks_equal_the_compiled_reference_directly(E, gpu, oracle):
    """CUDA == reference without the port in between: blocks and lengths of the GPU encoder against
    LZ4_compress_fast of oracle/_ref (the reference's own lz4.c compiled by oracle/Makefile), every
    content class, 64 KiB and 4 KiB pages, and the reference's LZ4_decompress_fast decodes them back.
    Without oracle/_ref the reference's blocks stored in golden/reference_lz4.json (each of which
    its decoder took back when they were recorded) stand in for it."""
    gold = json.load(open(os.path.join(GOLD, "reference_lz4.json")))["cuda_cases"]
    cases = datagen.reference_cuda_cases()
    assert [tuple(c[:4]) for c in gold] == cases and len(cases) == 224
    for bs in (65536, 4096):
        idx = [j for j, c in enumerate(cases) if c[1] == bs]
        pages = np.stack([datagen.make_page(kind, bs, seed) for kind, _, _, seed in (cases[j] for j in idx)])
        blocks, _ = E.lz4_encode_batch(pages, accel=12)
        for i, j in enumerate(idx):
            assert len(blocks[i]) == gold[j][4] and sha(blocks[i]) == gold[j][5], (bs, i)
            if oracle.ref() is not None:
                want = oracle.ref_lz4_encode(pages[i], 12)
                assert blocks[i] == want, (bs, i)
                back, used = oracle.ref_lz4_decode(want, bs)
                assert used == len(want) and back == pages[i].tobytes()
