#!/usr/bin/env python
"""Generates tests/golden/*.json from the reference itself (oracle/_ref/libcachemap_ref.so, i.e.
/root/reference/cachemap compiled unmodified, plus oracle/ref_kat.c built against the reference's
own uint128.h).  Run in the authoring container only; the fixtures it writes are committed and
are what pins the oracle (and, on the GPU box, the CUDA path) where /root/reference is absent.

    python tools/gen_golden.py [lz4 keys reference exerciser store]     (default: all of them)

`reference` and `exerciser` write the fixtures that stand in for the compiled reference in the tests
that compare with it live (reference_lz4.json, reference_records.json; reference_exerciser.json).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import datagen  # noqa: E402
from oracle import ef_oracle as O  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
REF = "/root/reference/cachemap"


def sha(b) -> str:
    return hashlib.sha256(bytes(b)).hexdigest()


def gen_lz4():
    out = []
    for kind, n, accel, seed in datagen.codec_cases():
        page = datagen.make_page(kind, n, seed)
        blk = O.ref_lz4_encode(page, accel)
        rec = {"kind": kind, "n": n, "accel": accel, "seed": seed, "in_sha256": sha(page),
               "len": len(blk), "sha256": sha(blk)}
        if len(blk) <= 300:
            rec["hex"] = blk.hex()
        if n:
            back, used = O.ref_lz4_decode(blk, n)
            assert back == page.tobytes() and used == len(blk)
        out.append(rec)
    with open(os.path.join(GOLD, "lz4_blocks.json"), "w") as f:
        json.dump({"generator": "tools/gen_golden.py", "reference": "LZ4_compress_fast of cachemap/lz4.c (v1.8.1), "
                   "called as filemap.c:126 does", "cases": out}, f, indent=0)
    print("lz4 cases:", len(out))


def gen_keys():
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_kat")
    subprocess.run(["gcc", "-O2", "-I" + REF, os.path.join(ROOT, "oracle", "ref_kat.c"), "-o", exe], check=True)
    data = json.loads(subprocess.run([exe], check=True, capture_output=True, text=True).stdout)
    data["generator"] = "oracle/ref_kat.c compiled against the reference's cachemap/uint128.h"
    with open(os.path.join(GOLD, "keys.json"), "w") as f:
        json.dump(data, f, indent=0)
    print("key KATs:", len(data["addrs"]))


def store_script(pshift=16):
    """The operation list of the store trace: C0 shape (16 x 64 KiB) plus the edge cases of
    SURVEY.md §8c.  Each op: [kind, offset, nhid, genid, content]; content = [kind, seed]."""
    import edge_fuse_b200 as E
    ops = []
    cids = list(range(16))
    off, nh = E.gen_addr(42, cids, pshift)
    for c in cids:                                   # 16 puts, config 0
        ops.append(["put", int(off[c]), int(nh[c]), 0, ["S", c]])
    for c in cids:
        ops.append(["get", int(off[c]), int(nh[c]), 0, None])
    ops.append(["put", 16 << pshift, int(nh[0]), 0, ["S", 3]])        # same content, new address
    ops.append(["get", 16 << pshift, int(nh[0]), 0, None])
    ops.append(["put", int(off[5]), int(nh[5]), 0, ["T", 999]])       # same address, new content
    ops.append(["get", int(off[5]), int(nh[5]), 0, None])
    ops.append(["get", 40 << pshift, int(nh[0]), 0, None])            # never stored
    ops.append(["get", (1 << pshift) + 1, int(nh[1]), 0, None])       # offset truncated by >> pshift
    ops.append(["get", int(off[2]), int(nh[2]), 7, None])             # other genid: miss
    ops.append(["put", int(off[2]), int(nh[2]), 7, ["Z", 5]])
    ops.append(["get", int(off[2]), int(nh[2]), 7, None])
    ops.append(["get", int(off[2]), int(nh[2]), 0, None])
    ops.append(["put", (1 << 44) << pshift, 1, 0, ["R", 1]])          # page number overflows 44 bits
    ops.append(["get", (1 << 44) << pshift, 1, 0, None])
    ops.append(["get", int(off[2]), int(nh[2]), (1 << 20) + 7, None]) # genid keeps its low 20 bits only
    ops.append(["put", int(off[9]), int(nh[9]), 0, ["R", 77]])
    ops.append(["put", int(off[9]), int(nh[9]), 0, ["M", 78]])        # twice in a row: last wins
    ops.append(["get", int(off[9]), int(nh[9]), 0, None])
    return ops


def gen_store():
    R = O.ref()
    pshift, accel = 16, 12
    ops = store_script(pshift)
    trace = []
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
        assert not R.cachemap_create(d.encode(), 1023, accel, pshift)         # n < 1024 -> NULL
        assert not R.cachemap_create((d + "/nope").encode(), 1024, accel, pshift)
        cm = R.cachemap_create(d.encode(), 1024, accel, pshift)
        assert cm
        libc = C.CDLL(None)
        libc.free.argtypes = [C.c_void_p]
        for kind, off, nh, gen, content in ops:
            if kind == "put":
                page = datagen.make_page(content[0], 1 << pshift, content[1])
                R.cachemap_put(cm, off, nh, gen, page.ctypes.data)
                trace.append(None)
            else:
                p = R.cachemap_get(cm, off, nh, gen)
                if p:
                    trace.append(sha(C.string_at(p, 1 << pshift)))
                    libc.free(p)
                else:
                    trace.append("miss")
        pages_ptr = C.cast(cm, C.POINTER(C.c_void_p))[0]                      # cm->pages
        entries = int(R.filemap_entries(pages_ptr))
        # struct cachemap tail: capacity, requests, hits are its last three u64 (cachemap.h:20-31)
        sz = 8 + 8 + 8 + 4 * 8 + 48 + 40 + 8 + 3 * 8
        raw = C.string_at(cm, sz)
        cap, req, hits = np.frombuffer(raw[-24:], dtype=np.uint64)
        assert cap == 1024, cap
        # deliberately no cachemap_free(): it can hang in the reference (SURVEY.md §5)
    with open(os.path.join(GOLD, "store_trace.json"), "w") as f:
        json.dump({"generator": "tools/gen_golden.py against libcachemap_ref.so (LMDB on tmpfs)",
                   "pshift": pshift, "accel": accel, "capacity": 1024, "ops": ops, "gets": trace,
                   "entries": entries, "requests": int(req), "hits": int(hits),
                   "create_null": ["capacity 1023", "missing directory"]}, f, indent=0)
    print("store trace ops:", len(ops), "entries", entries, "requests", int(req), "hits", int(hits))
    os._exit(0)


def _write(name, data):
    with open(os.path.join(GOLD, name), "w") as f:
        json.dump(data, f, indent=0)


def gen_reference_lz4():
    """The reference's blocks for the cases that test_oracle_vs_reference_live and
    test_cuda_blocks_equal_the_compiled_reference_directly compare with."""
    def case(kind, n, accel, seed):
        page = datagen.make_page(kind, n, seed)
        blk = O.ref_lz4_encode(page, accel)
        back, used = O.ref_lz4_decode(blk, n)
        assert back == page.tobytes() and used == len(blk)
        return [kind, n, accel, seed, len(blk), sha(blk)]
    _write("reference_lz4.json", {
        "generator": "tools/gen_golden.py reference: LZ4_compress_fast of cachemap/lz4.c; every block decodes "
                     "back with its LZ4_decompress_fast",
        "version": O.ref().LZ4_versionString().decode(),
        "oracle_cases": [case(*c) for c in datagen.reference_lz4_cases()],
        "cuda_cases": [case(*c) for c in datagen.reference_cuda_cases()]})
    print("reference lz4 cases written")


def _ref_child(body: str):
    """Runs `body` in a child with R = the compiled reference, under a watchdog: its cachemap_create
    starts the put threads before it initialises their mutex and condition variable
    (cachemap.c:123-138), and a child that loses that race never gets going."""
    code = ("import sys, ctypes as C, numpy as np\n"
            f"sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})\n"
            "import datagen\nfrom oracle import ef_oracle as O\nR = O.ref()\n" + body +
            "\nprint('child ok', flush=True)\nimport os; os._exit(0)\n")
    for _ in range(6):
        try:
            r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
        except subprocess.TimeoutExpired:
            continue
        assert r.returncode == 0 and "child ok" in r.stdout, r.stdout + r.stderr
        return
    raise RuntimeError("the reference library hung at start-up in every attempt")


def _lmdb_records(exe, d, tmp):
    """{(u, l): sha256 of the LMDB value without its 4 unspecified pad bytes} of a reference directory."""
    from oracle import snapshot as S
    snap = os.path.join(tmp, "from.snap")
    subprocess.run([exe, "from-lmdb", d, snap, "16"], check=True, capture_output=True)
    pshift, flags, recs = S.read_snapshot(snap)
    assert pshift == 16 and flags == 0 and all(ts > 0 for ts, _, _, _ in recs)
    out = {}
    for _, _, _, rec in recs:
        u, l = np.frombuffer(rec[:16], dtype=np.uint64)
        out[(int(u), int(l))] = sha(rec[:20] + rec[24:])
    return out


def gen_reference_records():
    """The records the reference keeps in its LMDB files for the puts of
    test_snapshot_lmdb_interchange_on_the_reference_side and
    test_cache_directory_interchange_with_the_reference, read back through tools/snap2lmdb."""
    import pathlib
    from test_oracle_pin import _build_snap2lmdb
    with tempfile.TemporaryDirectory() as tmp:
        exe = _build_snap2lmdb(pathlib.Path(tmp))
        dirs = {k: os.path.join(tmp, k) for k in ("roundtrip", "gpu_to_ref", "ref_to_gpu")}
        for d in dirs.values():
            os.mkdir(d)
        _ref_child(f"pages = O.gen_chunks(42, np.arange(24, dtype=np.uint64), 65536, 2)\n"
                   f"cm = R.cachemap_create({dirs['roundtrip']!r}.encode(), 2048, 12, 16)\n"
                   "for i in range(24):\n"
                   "    R.cachemap_put(cm, i << 16, 777, 3, pages[i].ctypes.data)\n")
        pages = "pages = np.stack([datagen.make_page('RTZMPAX'[i % 7], 65536, 300 + i) for i in range(48)])\n"
        _ref_child(pages + f"cm = R.cachemap_create({dirs['gpu_to_ref']!r}.encode(), 2048, 12, 16)\n"
                   "for i in range(48):\n"
                   "    R.cachemap_put(cm, i << 16, 4242, 5, pages[i].ctypes.data)\n")
        _ref_child(pages + f"cm = R.cachemap_create({dirs['ref_to_gpu']!r}.encode(), 2048, 12, 16)\n"
                   "for i in range(48):\n"
                   "    R.cachemap_put(cm, i << 16, 99, 7, pages[47 - i].ctypes.data)\n")
        rt = _lmdb_records(exe, dirs["roundtrip"], tmp)
        g2r = _lmdb_records(exe, dirs["gpu_to_ref"], tmp)
        r2g = _lmdb_records(exe, dirs["ref_to_gpu"], tmp)
    assert len(rt) == 24 and len(g2r) == 48 and len(r2g) == 48
    _write("reference_records.json", {
        "generator": "tools/gen_golden.py reference: cachemap_put of the compiled reference, its LMDB files read back "
                     "with tools/snap2lmdb from-lmdb; sha256 of each value without its 4 unspecified pad bytes",
        "roundtrip": sorted(rt.values()),
        "gpu_to_ref": [g2r[(4242, (5 << 44) | i)] for i in range(48)],
        "ref_to_gpu": [r2g[(99, (7 << 44) | i)] for i in range(48)]})
    print("reference records written")


def gen_reference_exerciser():
    """Per-phase hits of tests/c/exerciser.c linked against the compiled reference.  One seed: most
    starts of the reference lose its start-up race on a small host (see _ref_child)."""
    import re
    ref = os.path.join(ROOT, "oracle", "_ref", "libcachemap_ref.so")
    runs = []
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "exer_ref")
        subprocess.run(["gcc", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "exerciser.c"),
                        "-o", exe, ref, f"-Wl,-rpath,{os.path.dirname(ref)}", "-lpthread"], check=True)
        for seed in (1,):
            out = None
            for _ in range(12):
                with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
                    try:
                        out = subprocess.run([exe, d, "32768", "15", str(seed)], capture_output=True, text=True,
                                             timeout=150, check=True).stdout
                        break
                    except subprocess.TimeoutExpired:
                        continue
            assert out is not None, "the reference library hung at start-up in every attempt"
            runs.append({"seed": seed,
                         "hits": {m.group(1): [int(m.group(2)), int(m.group(3))]
                                  for m in re.finditer(r"phase (\w+) hits (\d+) of (\d+)", out)},
                         "entries": [int(x) for x in re.findall(r"entries_after_\w+ (\d+)", out)]})
    _write("reference_exerciser.json", {
        "generator": "tools/gen_golden.py reference: tests/c/exerciser.c linked against the compiled reference, "
                     "32 768 objects of 32 KiB, LMDB on tmpfs",
        "runs": runs})
    print("reference exerciser runs:", runs)


if __name__ == "__main__":
    assert O.ref() is not None, "oracle/_ref/libcachemap_ref.so missing: run make -C oracle"
    os.makedirs(GOLD, exist_ok=True)
    which = sys.argv[1:] or ["lz4", "keys", "reference", "exerciser", "store"]
    if "lz4" in which:
        gen_lz4()
    if "keys" in which:
        gen_keys()
    if "reference" in which:
        gen_reference_lz4()
        gen_reference_records()
    if "exerciser" in which:
        gen_reference_exerciser()
    if "store" in which:
        gen_store()                                   # last: it ends the process (see gen_store)
