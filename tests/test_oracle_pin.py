"""Pins the CPU oracle (oracle/) to the reference: against the committed golden vectors that
tools/gen_golden.py produced with the compiled reference, and — when oracle/_ref is present —
against the compiled reference live.  CPU only."""
import hashlib
import json
import os

import numpy as np
import pytest

import datagen

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def load(name):
    with open(os.path.join(GOLD, name)) as f:
        return json.load(f)


def test_fnv_and_key_kats(oracle):
    k = load("keys.json")
    assert k["sizeof_uint128"] == 16
    for s, h in k["strings"]:
        assert oracle.fnv1a64(s.encode()) == int(h, 16)
    for u, l, h in k["addrs"]:
        assert oracle.addr_key(int(u, 16), int(l, 16)) == int(h, 16)
    # SURVEY.md §8c known answers
    assert oracle.fnv1a64(b"") == 0xcbf29ce484222325
    assert oracle.addr_key(0x1122334455667788, (7 << 44) | 3) == 0x1e041ed74a444846
    assert oracle.addr_key(0x1122334455667788, (7 << 44) | 3) & 31 == 6


def test_addr_compose(oracle):
    assert oracle.addr_compose(65537, 9, 0, 16) == (9, 1)            # offset truncated, no alignment check
    assert oracle.addr_compose(3 << 16, 9, 7, 16) == (9, (7 << 44) | 3)
    assert oracle.addr_compose((1 << 44) << 16, 9, 0, 16) is None    # cachemap.c:160-161
    assert oracle.addr_compose(((1 << 44) - 1) << 12, 9, 0, 12) == (9, (1 << 44) - 1)
    assert oracle.addr_compose(0, 9, (1 << 20) + 7, 16) == (9, 7 << 44)   # genid keeps 20 bits
    assert oracle.record_prefix(1, 2, 267) == (1).to_bytes(8, "little") + (2).to_bytes(8, "little") + \
        (267).to_bytes(4, "little") + b"\0" * 4


def test_lz4_golden_vectors(oracle):
    g = load("lz4_blocks.json")
    assert len(g["cases"]) == len(datagen.codec_cases())
    for rec in g["cases"]:
        page = datagen.make_page(rec["kind"], rec["n"], rec["seed"])
        assert sha(page) == rec["in_sha256"], rec
        blk = oracle.lz4_encode(page, rec["accel"])
        assert len(blk) == rec["len"] and sha(blk) == rec["sha256"], rec
        if "hex" in rec:
            assert blk.hex() == rec["hex"]
        if rec["n"]:
            back, used = oracle.lz4_decode(blk, rec["n"])
            assert used == len(blk) and back == page.tobytes(), rec


def test_lz4_known_answers(oracle):
    # SURVEY.md §8c: incompressible 64 KiB -> 65 794 bytes; zero page -> 267 bytes; bound
    assert oracle.lib().ef_lz4_bound(65536) == 65809
    assert len(oracle.lz4_encode(datagen.make_page("R", 65536, 1), 12)) == 65794
    assert len(oracle.lz4_encode(np.zeros(65536, dtype=np.uint8), 12)) == 267


def test_decoder_rejects_malformed(oracle):
    page = datagen.make_page("T", 4096, 5)
    blk = oracle.lz4_encode(page, 12)
    assert oracle.lz4_decode(blk[:-3], 4096)[1] < 0               # truncated
    assert oracle.lz4_decode(blk, 4095)[1] != len(blk)            # wrong size never "consumes" all
    assert oracle.lz4_decode(b"\x10\x41\x00\x00", 4096)[1] < 0    # offset 0


def test_oracle_vs_reference_live(oracle):
    """The oracle's blocks against the reference's: against its stored answers
    (golden/reference_lz4.json) always, and against the compiled reference itself when oracle/_ref
    was built."""
    g = load("reference_lz4.json")
    cases = datagen.reference_lz4_cases()
    assert g["version"] == "1.8.1" and len(cases) == 700
    assert [tuple(c[:4]) for c in g["oracle_cases"]] == cases
    R = oracle.ref()
    if R is not None:
        assert R.LZ4_versionString() == b"1.8.1"
    for kind, n, accel, seed, ref_len, ref_sha in g["oracle_cases"]:
        page = datagen.make_page(kind, n, seed)
        a = oracle.lz4_encode(page, accel)
        assert len(a) == ref_len and sha(a) == ref_sha, (kind, n, accel)
        back, used = oracle.lz4_decode(a, n)
        assert back == page.tobytes() and used == len(a)
        if R is not None:
            assert a == oracle.ref_lz4_encode(page, accel), (kind, n, accel)
            back, used = oracle.ref_lz4_decode(a, n)
            assert back == page.tobytes() and used == len(a)


def test_store_model_matches_reference_trace(oracle):
    t = load("store_trace.json")
    m = oracle.StoreModel(t["pshift"], t["accel"])
    gets = []
    for kind, off, nh, gen, content in t["ops"]:
        if kind == "put":
            m.put(off, nh, gen, datagen.make_page(content[0], 1 << t["pshift"], content[1]))
            gets.append(None)
        else:
            p = m.get(off, nh, gen)
            gets.append("miss" if p is None else sha(p))
    assert gets == t["gets"]
    assert (m.entries(), m.requests, m.hits) == (t["entries"], t["requests"], t["hits"])


def test_fingerprint_self_consistency(oracle):
    """EF128 has no reference definition (parity unpinned): frozen KATs of this oracle plus
    basic sanity (length sensitivity, single-bit sensitivity, padding is not aliasing)."""
    f = oracle.fingerprint128
    assert f(b"") == (16344626119028627888, 17509804346615072515)
    assert f(b"abc") == (8640923672218744830, 2380023549751616974)
    a = datagen.make_page("R", 65536, 3)
    b = a.copy(); b[40000] ^= 1
    assert f(a) != f(b)
    assert f(a[:65535]) != f(a) and f(np.append(a, np.uint8(0))) != f(a)
    z1, z2 = np.zeros(512, np.uint8), np.zeros(513, np.uint8)
    assert f(z1) != f(z2)
    seen = {f(datagen.make_page("Z", 4096, s)) for s in range(200)}
    assert len(seen) == len({bytes(datagen.make_page("Z", 4096, s)) for s in range(200)})


def test_stream_generators_agree(oracle, E):
    """oracle/streamgen.c and the product's generator (csrc/streamgen.cuh, host form) are two
    independent statements of the benchmark stream: same pages, addresses and duplicate pattern."""
    import numpy as np
    cids = np.concatenate([np.arange(0, 24, dtype=np.uint64), np.array([16383, 16384, 70001, 2**33 + 5], dtype=np.uint64)])
    for bsize in (4096, 65536, 131072):
        pages = oracle.gen_chunks(42, cids, bsize, threads=3)
        for i, c in enumerate(cids):
            assert (pages[i] == E.gen_chunk_host(42, int(c), bsize)).all(), (bsize, int(c))
    off_o, nh_o = oracle.gen_addr(42, cids, 16)
    off_p, nh_p = E.gen_addr(42, cids, 16)
    assert (off_o == off_p).all() and (nh_o == nh_p).all()
    for dup in (0.0, 0.3, 0.5):
        a, da = oracle.gen_stream_ids(5000, dup)
        b, db = E.gen_stream_ids(5000, dup)
        assert da == db and (a == b).all()


def test_parity_gate_detects_a_wrong_record(oracle):
    """The bench's parity gate (oracle.parity_records) accepts the reference's records and flags a
    single flipped byte, a wrong length and a wrong prefix."""
    import numpy as np
    cids = np.arange(12, dtype=np.uint64)
    pages = oracle.gen_chunks(42, cids, 65536, threads=2)
    u = np.arange(12, dtype=np.uint64) + 7
    l = np.arange(12, dtype=np.uint64)
    recs = np.zeros((12, 24 + 65536 + 1024), dtype=np.uint8)
    lens = np.zeros(12, dtype=np.int32)
    for i in range(12):
        blk = oracle.ref_lz4_encode(pages[i]) if oracle.ref() is not None else oracle.lz4_encode(pages[i])
        rec = oracle.record_prefix(int(u[i]), int(l[i]), len(blk)) + blk
        recs[i, :len(rec)] = np.frombuffer(rec, dtype=np.uint8)
        lens[i] = len(rec)
    ok = oracle.parity_records(pages, u, l, recs, lens, lens - 24, threads=3)
    assert ok["mismatches"] == 0 and ok["chunks"] == 12
    bad = recs.copy(); bad[5, 100] ^= 1
    assert oracle.parity_records(pages, u, l, bad, lens, threads=3)["mismatches"] == 1
    assert oracle.parity_records(pages, u, l, bad, lens, threads=3)["first_mismatch"] == 5
    l2 = lens.copy(); l2[0] -= 1
    assert oracle.parity_records(pages, u, l, recs, l2, threads=1)["mismatches"] == 1
    assert oracle.parity_records(pages, u + np.uint64(1), l, recs, lens, threads=2)["mismatches"] == 12


def _build_snap2lmdb(tmp_path):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref_dir, ora_dir = os.path.join(root, "oracle", "_ref"), os.path.join(root, "oracle")
    exe = str(tmp_path / "snap2lmdb")
    subprocess.check_call(["gcc", "-O2", "-I", os.path.join(root, "include"), os.path.join(root, "tools", "snap2lmdb.c"), "-o", exe,
                           "-L", ref_dir, "-L", ora_dir, "-l:libcachemap_ref.so", "-l:liboracle.so",
                           f"-Wl,-rpath,{ref_dir}", f"-Wl,-rpath,{ora_dir}", "-lpthread"])
    return exe


def test_snapshot_lmdb_interchange_on_the_reference_side(oracle, tmp_path):
    """tools/snap2lmdb (test infrastructure linking the compiled reference): an LMDB cache directory
    written by the reference becomes a snapshot file in this library's format and back; the
    reference reads every page again, and the snapshot parses with the independent reader.
    Without oracle/_ref the records the reference stored (golden/reference_records.json) stand in
    for its LMDB directory."""
    import ctypes as C
    import subprocess
    import numpy as np
    from oracle import snapshot as S
    pages = oracle.gen_chunks(42, np.arange(24, dtype=np.uint64), 65536, 2)
    want = {oracle.record_prefix(777, (3 << 44) | i, len(oracle.lz4_encode(pages[i])))[:20] + oracle.lz4_encode(pages[i]) for i in range(24)}
    assert sorted(sha(r) for r in want) == load("reference_records.json")["roundtrip"]
    R = oracle.ref()
    if R is None:
        return
    exe = _build_snap2lmdb(tmp_path)
    a, b = tmp_path / "lmdb_a", tmp_path / "lmdb_b"
    a.mkdir(); b.mkdir()
    cm = R.cachemap_create(str(a).encode(), 2048, 12, 16)
    for i in range(24):
        R.cachemap_put(cm, i << 16, 777, 3, pages[i].ctypes.data)
    snap = str(tmp_path / "cachemap_b200.snap")
    assert "24 records" in subprocess.run([exe, "from-lmdb", str(a), snap, "16"], capture_output=True, text=True, check=True).stdout
    pshift, flags, recs = S.read_snapshot(snap)
    assert pshift == 16 and flags == 0 and len(recs) == 24 and all(ts > 0 for ts, _, _, _ in recs)
    got = {bytes(rec[:20]) + bytes(rec[24:]) for _, _, _, rec in recs}          # the 4 pad bytes are unspecified in the reference
    assert got == want
    out = subprocess.run([exe, "to-lmdb", snap, str(b), "2048", "16"], capture_output=True, text=True, check=True).stdout
    assert "24 of 24" in out
    cm2 = R.cachemap_create(str(b).encode(), 2048, 12, 16)
    for i in range(24):
        p = R.cachemap_get(cm2, i << 16, 777, 3)
        assert p and bytes((C.c_uint8 * 65536).from_address(p)) == pages[i].tobytes()
