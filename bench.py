#!/usr/bin/env python
"""bench.py — GiB/s through the cachemap put path (fingerprint -> LZ4 encode -> key-table insert)
on 64 KiB chunks, BASELINE.json's metric.

A step = one pass of the hot path over one batch = the whole 1 GiB synthetic stream of config 1
(16 384 x 64 KiB chunks, 0 % duplicates, classes R/T/Z/M round-robin, SURVEY.md §8d) put into the
cache under fresh addresses (genid = step).  Per GPU the work is fixed (weak scaling): with N
ranks the global stream is N GiB and chunk k belongs to rank k mod N; after each step the ranks
all-gather their new key records over NCCL (side stream, overlapping the next step's encode) and
import them into their index replica.

  value      device-timed (CUDA events on the engine's stream, max over ranks), pages resident in HBM
  e2e        same metric through the C-ABI with page-locked HOST pages: H2D of every page and D2H
             of the per-chunk stored lengths inside the timed region.  Headline = the write-behind
             call cmb200_put_step with two steps in flight; the strictly synchronous
             cmb200_put_batch figure is reported beside it (e2e.synchronous_call)
  roofline   the encode kernel alone: algorithmic bytes / its CUDA-event duration vs measured HBM peak
  parity     the measured run's own records against the reference's LZ4_compress_fast + data_prefix
             (oracle/_ref); any mismatch fails the run (SURVEY.md §8d "voids the throughput number")
  integrity  dropped_puts == 0 and entries == the number of distinct keys written, after every pass
  configs    C2 (50 % same-address duplicates), C3 (read-hit: lookup + LZ4 decode, with its own
             roofline and an end-to-end figure), and for N > 1 C4 (30 % duplicates across ranks,
             final index checked against a sequential model)
  cpu_baseline  the reference's own CPU path (oracle/_ref, else the oracle port) on a bounded sample

`--impl reference` times the reference CPU implementation instead (same metric/config); that arm
never imports the product library.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CHUNK = 65536
PSHIFT = 16
ACCEL = 12
SEED = 42
METRIC = "GiB/s hash+LZ4+dedup on 64 KiB chunks"
GIB = float(1 << 30)
WORST = CHUNK + 1056            # arena bytes one incompressible 64 KiB page can take (prefix + block, rounded)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def workload_config(gpus: int, chunks: int) -> dict:
    return {"workload": f"config 1: {chunks * CHUNK / GIB:g} GiB synthetic stream per GPU per step, 64 KiB fixed "
                        "chunks, 0% duplicates, classes R/T/Z/M round-robin, EF128 fingerprint + LZ4(accel 12) "
                        "encode + key-table insert",
            "chunk_bytes": CHUNK, "chunks_per_gpu_per_step": chunks, "pshift": PSHIFT, "accel": ACCEL,
            "sharding": f"chunk k -> rank k mod {gpus}" if gpus > 1 else "single GPU",
            "l2": "per-step input (1 GiB) is larger than the 126 MB L2; no explicit flush"}


# -------------------------------------------------------------------------------------------------
# reference / CPU arm  (imports oracle/ only — never the product library)
# -------------------------------------------------------------------------------------------------

def reference_store_child(n: int, threads: int) -> int:
    """(child process of reference_store_rates) cachemap_put / cachemap_get of the reference's own
    library over the first n chunks of the stream, `threads` pthreads, LMDB on tmpfs; one JSON line."""
    import ctypes as C
    import tempfile
    from oracle import ef_oracle as O
    L, R = O.lib(), O.ref()
    cids = np.arange(n, dtype=np.uint64)
    pages = O.gen_chunks(SEED, cids, CHUNK, threads)
    off, nh = O.gen_addr(SEED, cids, PSHIFT)
    offs = np.ascontiguousarray(off, dtype=np.uint64)
    nhs = np.ascontiguousarray(nh, dtype=np.uint64)
    out3 = (C.c_double * 3)()
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=base) as d:
        cm = R.cachemap_create(d.encode(), max(1024, 2 * n), ACCEL, PSHIFT)
        assert cm, "reference cachemap_create failed"
        L.ef_cpu_bench_store(C.cast(R.cachemap_put, C.c_void_p), C.cast(R.cachemap_get, C.c_void_p),
                             C.c_void_p(cm), pages.ctypes.data, n, CHUNK, offs.ctypes.data,
                             nhs.ctypes.data, threads, 1, out3)
        assert out3[2] == 0, "reference get returned different bytes"
        print(json.dumps({"put_gibs": n * CHUNK / GIB / out3[0], "get_gibs": n * CHUNK / GIB / out3[1]}), flush=True)
        # no cachemap_free(): it can hang in the reference (SURVEY.md §5); the process just ends and the
        # LMDB files go away with the temporary directory
        sys.stdout.flush()
        os._exit(0)


def reference_store_rates(n: int, threads: int) -> dict:
    """The reference's full put / get path over the first n chunks, measured in a child process under
    a watchdog: cachemap_create starts its put threads before it initialises the mutex and condition
    variable they use (cachemap.c:123-138), and a process that loses that race sleeps forever before
    the first put (seen in ~3 % of the starts on the 128-thread GPU host, in half of them on a small
    one).  Such a child is killed and the measurement repeated; the numbers come from a run that ran."""
    import subprocess
    limit = 40 + 30 * n // 16384                          # a healthy child needs a few seconds even for the whole 1 GiB step
    for attempt in range(5):
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--ref-store-child", str(n), str(threads)],
                                 capture_output=True, text=True, timeout=limit)
        except subprocess.TimeoutExpired:
            continue
        lines = [x for x in out.stdout.splitlines() if x.startswith("{")]
        assert out.returncode == 0 and lines, f"reference store run failed: {out.stdout[-300:]} {out.stderr[-600:]}"
        return json.loads(lines[-1])
    raise RuntimeError("the reference library hung at start-up in five attempts")


def cpu_reference_run(pages: np.ndarray, off: np.ndarray, nh: np.ndarray, threads: int, codec: bool = True):
    """Times the reference's CPU path on `pages` ([n, 65536] host array).  Returns a dict with the
    full-path put/get rate (cachemap_put / cachemap_get on a tmpfs store) and, with codec=True, the
    codec-only rate (LZ4_compress_fast / LZ4_decompress_fast, no LMDB), wall clock, `threads` pthreads."""
    import ctypes as C
    import tempfile
    from oracle import ef_oracle as O
    L = O.lib()
    R = O.ref()
    n = len(pages)
    res = {"kind": "reference" if R is not None else "port", "cores": threads}
    if codec or R is None:
        out4 = (C.c_double * 4)()
        if R is not None:
            enc, dec = C.cast(R.LZ4_compress_fast, C.c_void_p), C.cast(R.LZ4_decompress_fast, C.c_void_p)
        else:
            enc, dec = C.cast(L.ef_port_compress_fast, C.c_void_p), C.cast(L.ef_port_decompress_fast, C.c_void_p)
        L.ef_cpu_bench_codec(enc, dec, pages.ctypes.data, n, CHUNK, ACCEL, threads, out4)
        assert out4[2] == 0, "CPU codec round trip mismatch"
        res.update({"codec_encode_gibs": n * CHUNK / GIB / out4[0], "codec_decode_gibs": n * CHUNK / GIB / out4[1],
                    "ratio": out4[3] / (n * CHUNK)})
    if R is not None:
        res.update(reference_store_rates(n, threads))
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import ef_oracle as O
    assert "edge_fuse_b200" not in sys.modules
    threads = os.cpu_count() or 1
    n = args.chunks                                    # the same step as the CUDA arm: the whole 1 GiB stream
    cids = np.arange(n, dtype=np.uint64)
    pages = O.gen_chunks(SEED, cids, CHUNK, threads)
    off, nh = O.gen_addr(SEED, cids, PSHIFT)
    runs = []
    for it in range(args.warmup + args.steps):
        r = cpu_reference_run(pages, off, nh, threads, codec=(it == args.warmup))
        if it >= args.warmup:
            runs.append(r)
    # metric of a step = the put path of the reference: cachemap_put (fingerprint-less: the
    # reference has no content hash) when the reference compiled, else the codec-only port
    key = "put_gibs" if "put_gibs" in runs[0] else "codec_encode_gibs"
    value = float(np.median([r[key] for r in runs]))
    assert "edge_fuse_b200" not in sys.modules, "the reference arm must not load the product library"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": n * CHUNK / GIB / value * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.gpus, args.chunks),
        "cpu_baseline": {"value": value, "unit": "GiB/s", "cores": threads, "kind": runs[0]["kind"],
                         "sample": f"the whole step: {n} chunks ({n * CHUNK >> 20} MiB) per step, generated by "
                                   f"oracle/streamgen.c; "
                                   f"{'cachemap_put on a tmpfs LMDB store' if key == 'put_gibs' else 'LZ4 encode only'}, "
                                   f"{threads} threads",
                         "codec_encode_gibs": runs[0].get("codec_encode_gibs"),
                         "codec_decode_gibs": runs[0].get("codec_decode_gibs"),
                         "get_gibs": float(np.median([r["get_gibs"] for r in runs])) if "get_gibs" in runs[0] else None},
        "e2e": {"value": value, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# -------------------------------------------------------------------------------------------------
# CUDA arm
# -------------------------------------------------------------------------------------------------

def bind_to_gpu_numa_node(torch, local: int):
    """Runs this rank on the CPUs next to its GPU (NVML's ideal affinity) so that the page-locked
    staging buffers it allocates are first-touched on that NUMA node; with 8 ranks on a two-socket
    host the H2D rate otherwise depends on where the allocator happened to put them.  Returns the
    previous affinity (restored before the CPU baseline, which uses every host thread)."""
    try:
        before = os.sched_getaffinity(0)
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(local).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return before
    except Exception:
        return None


def next_pow2(v: int) -> int:
    p = 1
    while p < v:
        p <<= 1
    return p


class DevView:
    """torch view of a raw device allocation (on-device comparisons only)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def pinned(E, nbytes: int, dtype=np.uint8):
    ptr = E.lib().cmb200_host_alloc(nbytes)
    assert ptr, "page-locked host buffer"
    arr = np.ctypeslib.as_array((np.ctypeslib.ctypes.c_uint8 * nbytes).from_address(ptr)).view(dtype)
    return ptr, arr


def parity_gate(O, eng, pages: np.ndarray, u, l, put_lens, threads: int) -> dict:
    """Records of the measured run vs the reference's LZ4_compress_fast + data_prefix."""
    recs, rec_lens = eng.read_records_raw(u, l)
    return O.parity_records(pages, u, l, recs, rec_lens, put_lens, ACCEL, threads)


def dump_outputs(out_dir: str, eng, u, l, lens) -> None:
    """Writes what the put path returned and stored for the last timed device-resident step: the
    stored block length of every chunk, its 128-bit fingerprint (four 32-bit limbs), and the LZ4
    blocks of a fixed, seeded sample of 64 chunks (byte values, -1 past the block's end).  The
    pages are a function of the chunk ids and SEED alone, so two builds can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    fps, ok = eng.read_fingerprints(u, l)
    assert ok.all(), "a chunk of the last step has no fingerprint"
    limbs = np.stack([fps[:, 0] >> np.uint64(32), fps[:, 0] & np.uint64(0xFFFFFFFF),
                      fps[:, 1] >> np.uint64(32), fps[:, 1] & np.uint64(0xFFFFFFFF)], axis=1)
    pick = np.sort(np.random.default_rng(SEED).choice(len(u), size=min(64, len(u)), replace=False))
    recs, rec_lens = eng.read_records_raw(u[pick], l[pick])
    blocks = np.full((len(pick), recs.shape[1] - 24), -1.0, dtype=np.float32)
    for i, n in enumerate(rec_lens):
        blocks[i, :max(0, n - 24)] = recs[i, 24:n]
    np.save(os.path.join(out_dir, "stored_lengths.npy"), np.asarray(lens, dtype=np.float64))
    np.save(os.path.join(out_dir, "fingerprints.npy"), limbs.astype(np.float64))
    np.save(os.path.join(out_dir, "block_sample_chunks.npy"), pick.astype(np.float64))
    np.save(os.path.join(out_dir, "block_sample.npy"), blocks)


def run_config_2_3(args, E, O, torch, local, d_pages, h_ptr, h_pages, peak, threads):
    """BASELINE configs 2 and 3 on this GPU (SURVEY.md §8d): a stream with 50 % same-address
    duplicates through put (key table insert / overwrite in place), then the read-hit path over
    everything that is resident: lookup + LZ4 decode, device-timed, and end to end into host memory."""
    S = args.chunks
    n2 = int(args.c2_gib * GIB) // CHUNK
    cids, distinct = E.gen_stream_ids(n2, 0.5)
    off, nh = E.gen_addr(SEED, cids, PSHIFT)
    page = off >> np.uint64(PSHIFT)
    eng = E.Engine(pshift=PSHIFT, accel=ACCEL, capacity=2 * distinct, table_slots=next_pow2(4 * distinct),
                   arena_bytes=distinct * WORST + (5 << 30), max_batch=args.max_batch, flags=E.FINGERPRINT, device=local)
    main = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    s0 = eng.stats()
    put_ms = 0.0
    stored = 0.0
    for at in range(0, n2, S):
        m = min(S, n2 - at)
        eng.gen_chunks_dev(SEED, cids[at:at + m], d_pages)
        ev[0].record(main)
        lens = eng.put(nh[at:at + m], page[at:at + m], d_pages, on_dev=True)
        ev[1].record(main)
        torch.cuda.synchronize()
        put_ms += ev[0].elapsed_time(ev[1])
        stored += float(lens[lens > 0].sum())
    s1 = eng.stats()
    enc_s = (s1["encode_kernel_ns"] - s0["encode_kernel_ns"]) * 1e-9
    assert s1["dropped_puts"] == 0, f"config 2 dropped {s1['dropped_puts']} puts"
    assert s1["entries"] == distinct, f"config 2: {s1['entries']} entries, {distinct} distinct keys"
    # parity of a sample of the distinct keys (a repeat carries the same chunk id, i.e. the same content)
    ns = min(args.parity_chunks // 4, distinct)
    qs = np.linspace(0, distinct - 1, ns).astype(np.uint64)
    so, sn = E.gen_addr(SEED, qs, PSHIFT)
    par2 = parity_gate(O, eng, O.gen_chunks(SEED, qs, CHUNK, threads), sn, so >> np.uint64(PSHIFT), None, threads)
    assert par2["mismatches"] == 0, f"config 2 parity: {par2}"
    c2 = {"workload": f"{n2 * CHUNK / GIB:g} GiB stream, {n2} chunks, 50% same-address duplicates ({distinct} distinct keys), "
                      "put incl. key-table insert / in-place overwrite, pages resident",
          "put_gibs": n2 * CHUNK / GIB / (put_ms * 1e-3), "put_gibs_encode_kernel_only": n2 * CHUNK / GIB / enc_s,
          "entries": s1["entries"], "distinct": distinct, "dropped_puts": s1["dropped_puts"],
          "arena_used_gib": s1["arena_used"] / GIB, "arena_garbage_gib": s1["arena_garbage"] / GIB,
          "roofline_frac": (n2 * (CHUNK + 88) + stored) / enc_s / 1e9 / peak,
          "parity": par2, "gate": "entries == distinct keys, dropped_puts == 0, sampled records == oracle"}

    # ---- C3: read-hit path over everything resident ----
    qc = np.arange(distinct, dtype=np.uint64)
    qo, qn = E.gen_addr(SEED, qc, PSHIFT)
    qp = qo >> np.uint64(PSHIFT)
    d_out = eng.dev_alloc(S * CHUNK)
    t_in = torch.as_tensor(DevView(d_pages, S * CHUNK), device="cuda")
    t_out = torch.as_tensor(DevView(d_out, S * CHUNK), device="cuda")
    get_ms, bad, rec_bytes = 0.0, 0, 0.0
    s2 = eng.stats()
    for at in range(0, distinct, S):
        m = min(S, distinct - at)
        ev[0].record(main)
        _, status = eng.get(qn[at:at + m], qp[at:at + m], out=d_out, on_dev=True)
        ev[1].record(main)
        torch.cuda.synchronize()
        get_ms += ev[0].elapsed_time(ev[1])
        assert (status == E.HIT).all(), "config 3: a resident key missed"
        eng.gen_chunks_dev(SEED, qc[at:at + m], d_pages)
        torch.cuda.synchronize()
        bad += int((t_in[: m * CHUNK] != t_out[: m * CHUNK]).any().item())
    s3 = eng.stats()
    dec_s = (s3["decode_kernel_ns"] - s2["decode_kernel_ns"]) * 1e-9
    assert bad == 0, "config 3: decoded pages differ from the regenerated stream"
    rec_bytes = float(s1["arena_used"] - s1["arena_garbage"])      # live records = what the decoder reads
    # end to end: every page back into page-locked host memory through cmb200_get_batch
    e2e_n = min(distinct, (int(args.c3_e2e_gib * GIB) // CHUNK) // S * S) or min(distinct, S)
    t0 = time.perf_counter()
    host_bad = 0
    for at in range(0, e2e_n, S):
        m = min(S, e2e_n - at)
        _, status = eng.get(qn[at:at + m], qp[at:at + m], out=h_ptr, on_dev=False)
        host_bad += int((status != E.HIT).sum())
    e2e_s = time.perf_counter() - t0
    assert host_bad == 0
    # the last slice now sits in h_pages: check a sample of it against the CPU generator
    last0 = (e2e_n - 1) // S * S
    mlast = e2e_n - last0
    pick = np.linspace(0, mlast - 1, min(512, mlast)).astype(np.int64)
    want = O.gen_chunks(SEED, qc[last0 + pick], CHUNK, threads)
    assert (h_pages.reshape(-1, CHUNK)[pick] == want).all(), "config 3 e2e: host pages differ from the generator"
    alg3 = distinct * (CHUNK + 32 + 24) + (rec_bytes - 24 * distinct if rec_bytes > 24 * distinct else stored)
    c3 = {"workload": f"read-hit path: {distinct} resident keys ({distinct * CHUNK / GIB:g} GiB of pages), k_lookup + k_decode, pages written to HBM",
          "get_gibs": distinct * CHUNK / GIB / (get_ms * 1e-3), "get_gibs_decode_kernel_only": distinct * CHUNK / GIB / dec_s,
          "roofline": {"bound": "hbm", "kernel": "k_decode", "achieved": alg3 / dec_s / 1e9, "peak": peak, "unit": "GB/s",
                       "frac": alg3 / dec_s / 1e9 / peak, "algorithmic_bytes_per_chunk": alg3 / distinct},
          "e2e": {"value": e2e_n * CHUNK / GIB / e2e_s, "unit": "GiB/s", "chunks": e2e_n,
                  "call": "cmb200_get_batch into page-locked host memory (D2H of every page inside the region)",
                  "d2h_bytes": int(e2e_n * (CHUNK + 4)), "h2d_bytes": int(e2e_n * 16)},
          "hits": int(s3["get_hits"] - s2["get_hits"]),
          "gate": "every key hits, decoded pages == regenerated input (all, on device; e2e sample vs CPU generator)"}
    eng.dev_free(d_out)
    eng.close()
    return c2, c3


def run_config_4(args, E, O, torch, dist, rank, world, local, d_pages, threads, h_ptr=None, h_pages=None):
    """N > 1: a stream with 30 % same-address duplicates sharded round-robin, so that the same key is
    written by different ranks inside one step; afterwards every rank's index replica must equal the
    outcome of a sequential pass over the global stream (SURVEY.md App. B rule 4)."""
    from edge_fuse_b200 import sharding
    n = args.chunks
    steps = args.c4_steps
    n_tot = world * n * steps
    cids, distinct = E.gen_stream_ids(n_tot, 0.3)
    off, nh = E.gen_addr(SEED + 1, cids, PSHIFT)                 # its own objects
    page = off >> np.uint64(PSHIFT)
    eng = E.Engine(pshift=PSHIFT, accel=ACCEL, capacity=2 * distinct, table_slots=next_pow2(4 * distinct),
                   arena_bytes=(distinct // world + n) * WORST + (5 << 30), max_batch=args.max_batch,
                   flags=E.FINGERPRINT, device=local)
    xch = sharding.StepExchange(eng, n, rank, world, torch.device("cuda", local))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = 0.0
    for s in range(steps):
        base = s * world * n
        mine = base + rank + world * np.arange(n)
        eng.gen_chunks_dev(SEED + 1, cids[mine], d_pages)
        dist.barrier(); torch.cuda.synchronize()
        ev[0].record(xch.main)
        xch.step(nh[mine], page[mine], d_pages, True, next_seq=1 + base + rank)
        if s == steps - 1:
            xch.flush()
        ev[1].record(xch.main)
        torch.cuda.synchronize()
        ms += ev[0].elapsed_time(ev[1])
    eng.sync(); torch.cuda.synchronize(); dist.barrier()
    # sequential model: the last position of every key decides its owner
    last = np.zeros(distinct, dtype=np.int64)
    last[cids.astype(np.int64)] = np.arange(n_tot)               # later positions overwrite earlier ones
    exp_owner = last % world
    qc = np.arange(distinct, dtype=np.uint64)
    qo, qn = E.gen_addr(SEED + 1, qc, PSHIFT)
    status, owner = eng.locate(qn, qo >> np.uint64(PSHIFT))
    ok = bool(((status == E.HIT) == (exp_owner == rank)).all()
              and (owner[status == E.REMOTE] == exp_owner[status == E.REMOTE]).all()
              and ((status == E.HIT) | (status == E.REMOTE)).all())
    st = eng.stats()
    ok = ok and st["dropped_puts"] == 0 and st["entries"] + st["remote_entries"] == distinct
    # the records this rank owns are the reference's bytes
    own = np.nonzero(exp_owner == rank)[0][: args.parity_chunks // 8]
    par = parity_gate(O, eng, O.gen_chunks(SEED + 1, qc[own], CHUNK, max(1, threads // world)), qn[own],
                      (qo >> np.uint64(PSHIFT))[own], None, max(1, threads // world))
    # cross-GPU read path: keys whose newest record lives on another rank are read out of the owner's
    # arena over NVLink (CUDA IPC peer mapping) and decoded here
    remote = {"served": False}
    if h_ptr is not None:
        sharding.open_peers(eng, rank, world)
        dist.barrier()
        theirs = np.nonzero(exp_owner != rank)[0]
        pick = theirs[np.linspace(0, len(theirs) - 1, min(len(theirs), 2048)).astype(np.int64)]
        qp = (qo >> np.uint64(PSHIFT))[pick]
        eng.get_small(qn[pick[:64]], qp[:64], out=h_ptr)                        # warm-up
        t0 = time.perf_counter()
        _, gst = eng.get_small(qn[pick], qp, out=h_ptr)
        dt = time.perf_counter() - t0
        want = O.gen_chunks(SEED + 1, qc[pick], CHUNK, max(1, threads // world))
        good = bool((gst == E.HIT).all() and (h_pages.reshape(-1, CHUNK)[: len(pick)] == want).all())
        ok = ok and good
        remote = {"served": good, "gets": int(len(pick)), "gibs_per_rank": len(pick) * CHUNK / GIB / dt,
                  "path": "cmb200_get_small: record copied from the owner's arena over NVLink (peer memory), LZ4 decode on the "
                          "requesting GPU, page written to page-locked host memory"}
        eng.close_peers()
        dist.barrier()                                      # nobody frees its arena while a peer still maps it
    t = torch.tensor([int(ok), st["entries"], par["mismatches"], ms], dtype=torch.float64, device="cuda")
    tmin, tsum, tmax = t.clone(), t.clone(), t.clone()
    dist.all_reduce(tmin, op=dist.ReduceOp.MIN); dist.all_reduce(tsum); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    all_ok = bool(tmin[0].item() == 1 and int(tsum[1].item()) == distinct and int(tsum[2].item()) == 0)
    eng.close()
    res = {"workload": f"{n_tot * CHUNK / GIB:g} GiB stream, 30% same-address duplicates, sharded k mod {world}, "
                       f"{steps} steps x {n} chunks per rank, one all-gather + replica import per step",
           "put_gibs": n_tot * CHUNK / GIB / (float(tmax[3].item()) * 1e-3), "distinct": distinct,
           "entries_sum_over_ranks": int(tsum[1].item()), "index_matches_sequential": all_ok,
           "parity_mismatches": int(tsum[2].item()), "parity_chunks_per_rank": par["chunks"],
           "remote_gets_rank0": remote,
           "gate": "every key HIT on the rank of its last writer and REMOTE(owner) elsewhere; sum of entries == distinct; "
                   "owned records == oracle; pages fetched from other ranks' arenas == generator"}
    assert all_ok, f"config 4: index replica differs from the sequential model on rank {rank}: {res}"
    return res


def run_ours(args):
    import torch
    import edge_fuse_b200 as E
    from edge_fuse_b200 import sharding
    from oracle import ef_oracle as O          # the checker (parity gate, cpu_baseline); never on the timed path

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert E.device_count() > local, f"no CUDA device for rank {rank}: {E.last_error()}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity_before = bind_to_gpu_numa_node(torch, local)
    host_threads = os.cpu_count() or 1

    n = args.chunks
    K, W = args.steps, args.warmup
    T = W + K
    PASSES = 3                                    # device-resident, e2e synchronous, e2e write-behind
    # Arena: every put of every pass goes to a fresh address, sized for the WORST case (incompressible
    # pages) so that no put can be dropped; if K is so large that this does not fit in HBM the
    # addresses recycle every R steps (records of equal size are then rewritten in place).
    free_b, _ = torch.cuda.mem_get_info(local)
    budget = int(free_b * 0.60) - (6 << 30)
    R = max(1, min(T, budget // (PASSES * n * WORST)))
    arena = PASSES * R * n * WORST + (5 << 30)    # + room for the per-warp arena segments in flight
    keys_all_ranks = PASSES * R * n * world
    eng = E.Engine(pshift=PSHIFT, accel=ACCEL, capacity=keys_all_ranks, table_slots=next_pow2(2 * keys_all_ranks),
                   arena_bytes=arena, max_batch=args.max_batch, flags=E.FINGERPRINT, device=local)
    cids = np.arange(n, dtype=np.uint64) * np.uint64(world) + np.uint64(rank)     # round-robin shard
    off, nh = E.gen_addr(SEED, cids, PSHIFT)
    d_pages = eng.dev_alloc(n * CHUNK)
    eng.gen_chunks_dev(SEED, cids, d_pages)
    h_ptr, h_pages = pinned(E, n * CHUNK)
    eng.d2h(h_pages, d_pages)
    page_no = off >> np.uint64(PSHIFT)
    ts = np.full(n, 1, dtype=np.uint64)
    sampler = ClockSampler(local)
    sync_all = (lambda: (dist.barrier(), torch.cuda.synchronize())) if dist else torch.cuda.synchronize
    written = set()                               # (step % R, pass) pairs put so far

    def addr_for(step: int, lane: int):
        # fresh addresses every step: genid = 3 * (step mod R) + pass (low 20 bits kept, cachemap.c:163)
        written.add((step % R, lane))
        return nh, page_no | (np.uint64(PASSES * (step % R) + lane) << np.uint64(44))

    def seq_base(counter=[0]):
        base = 1 + counter[0] * world * n
        counter[0] += 1
        return base

    def check_integrity(what: str) -> dict:
        st = eng.stats()
        expect = len(written) * n
        assert st["dropped_puts"] == 0, f"{what}: {st['dropped_puts']} puts were dropped (arena {st['arena_used']}/{st['arena_bytes']})"
        assert st["entries"] == expect, f"{what}: {st['entries']} local entries, expected {expect}"
        assert st["remote_entries"] == expect * (world - 1), f"{what}: {st['remote_entries']} remote entries, expected {expect * (world - 1)}"
        return st

    xch = sharding.StepExchange(eng, n, rank, world, dev, timing=True)
    main = xch.main

    # ---- pass 0: device-resident -> value ----
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    ev_all = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    st0 = None
    for it in range(T):
        if it == W:
            xch.flush()
            sync_all()
            xch.times = {"allgather": [], "import": []}
            sampler.start()
            st0 = eng.stats()
            t_wall0 = time.perf_counter()
            ev_all[0].record(main)
        if it >= W:
            ev[it - W][0].record(main)
        u, l = addr_for(it, 0)
        xch.step(u, l, d_pages, True, ts=ts, next_seq=seq_base() + rank)
        if it >= W:
            ev[it - W][1].record(main)
    xch.flush()                                   # the last step's records are imported inside the region
    ev_all[1].record(main)
    sync_all()
    t_wall = time.perf_counter() - t_wall0
    st1 = eng.stats()
    lens = xch.last_lens()
    u_last, l_last = addr_for(T - 1, 0)
    dev_ms_steps = [a.elapsed_time(b) for a, b in ev]
    dev_ms_total = ev_all[0].elapsed_time(ev_all[1])
    breakdown = xch.breakdown_ms()
    if dist:
        tt = torch.tensor([dev_ms_total, t_wall * 1e3], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_ms_total, wall_ms_total = float(tt[0].item()), float(tt[1].item())
    else:
        wall_ms_total = t_wall * 1e3
    step_ms = dev_ms_total / K
    value = world * n * CHUNK / GIB / (step_ms * 1e-3)
    integrity = {"after_resident_pass": {k: check_integrity("device-resident pass")[k] for k in ("entries", "dropped_puts")}}

    # ---- e2e: host pages through the C ABI ----
    # (1) synchronous calls, one step at a time, each bracketed by a barrier + synchronize
    e2e_t = []
    lens_e = None
    for it in range(T):
        u, l = addr_for(it, 1)
        sync_all()
        t0 = time.perf_counter()
        base = seq_base()
        eng.set_stream_order(base + rank, world)
        lens_e = eng.put(u, l, h_ptr, ts=ts, on_dev=False)
        if dist:
            pos = sharding.shard_positions(rank, world, n, base)
            rec = torch.from_numpy(sharding.pack_records(u, l, pos, rank, lens_e)).cuda(non_blocking=True)
            sharding.import_gathered(eng, sharding.all_gather_records(rec), rank)
        sync_all()
        if it >= W:
            e2e_t.append(time.perf_counter() - t0)
    e2e_sync_s = float(np.mean(e2e_t))
    integrity["after_synchronous_e2e_pass"] = {k: check_integrity("synchronous e2e pass")[k] for k in ("entries", "dropped_puts")}

    # (2) the write-behind call (cmb200_put_step): step k+1 is submitted before step k's result is
    # read, so its host-to-device copy overlaps the tail of step k's encode.  Every step still copies
    # its own inputs from page-locked host memory and reads its own result (the stored lengths) back
    # inside the timed region; the region ends after the last result is in.
    lens_pin = [pinned(E, n * 4, np.int32) for _ in range(2)]
    h_ptr_b, h_pages_b = pinned(E, n * CHUNK)     # step k+1's pages must not be the buffer step k is still copied from
    h_pages_b[:] = h_pages
    h_ptr2 = (h_ptr, h_ptr_b)

    def pipelined(first_step: int, count: int):
        inflight = None
        for k in range(count):
            u, l = addr_for(first_step + k, 2)
            # host pages stay untouched until the step's ticket is done (mode 2): the call does not
            # wait for its own copies, so the copy engine never idles between steps
            tk = xch.step(u, l, h_ptr2[k & 1], 2, ts=ts, lens=lens_pin[k & 1][0], next_seq=seq_base() + rank)
            if inflight is not None:
                eng.wait(inflight[0])                   # step k-1's stored lengths are on the host
            inflight = (tk, lens_pin[k & 1][1])
        xch.flush()
        eng.wait(inflight[0])
        return inflight[1]

    pipelined(0, W)
    sync_all()
    t0 = time.perf_counter()
    lens_p = pipelined(W, K)
    sync_all()
    e2e_s = (time.perf_counter() - t0) / K
    assert (lens_p == lens_e).all() and (lens_p == lens).all(), "the three passes stored different lengths"
    clocks = sampler.stop()
    if dist:
        tt = torch.tensor([e2e_s, e2e_sync_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s, e2e_sync_s = float(tt[0].item()), float(tt[1].item())
    e2e = world * n * CHUNK / GIB / e2e_s
    e2e_sync = world * n * CHUNK / GIB / e2e_sync_s
    final = check_integrity("write-behind e2e pass")
    integrity["after_write_behind_e2e_pass"] = {k: final[k] for k in ("entries", "dropped_puts")}
    integrity.update({"dropped_puts": final["dropped_puts"], "local_entries": final["entries"],
                      "expected_local_entries": len(written) * n, "remote_entries": final["remote_entries"],
                      "distinct_steps_before_addresses_recycle": R, "arena_gib": final["arena_bytes"] / GIB,
                      "arena_used_gib": final["arena_used"] / GIB})

    # ---- parity gate on the measured run's own records (every rank checks its shard) ----
    if affinity_before:
        os.sched_setaffinity(0, affinity_before)
    S = min(n, args.parity_chunks if world == 1 else max(256, args.parity_chunks // world))
    par_threads = max(1, host_threads // world)
    parity = parity_gate(O, eng, h_pages.reshape(n, CHUNK)[:S], u_last[:S], l_last[:S], lens[:S].astype(np.int32), par_threads)
    if dist:
        tt = torch.tensor([parity["mismatches"], parity["chunks"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt)
        parity["mismatches"], parity["chunks"] = int(tt[0].item()), int(tt[1].item())
    parity["what"] = ("records of the last device-resident step read back from the arena (cmb200_read_records) and its reported "
                      "stored lengths vs LZ4_compress_fast(accel 12) + data_prefix of the same pages")
    assert parity["mismatches"] == 0, f"parity gate failed: {parity}"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, u_last, l_last, lens)

    # ---- roofline of the dominant kernel (k_encode) ----
    peak, peak_src = peaks()
    enc_ns = st1["encode_kernel_ns"] - st0["encode_kernel_ns"]
    enc_launches = st1["encode_kernel_launches"] - st0["encode_kernel_launches"]
    stored = float(lens[lens > 0].sum())
    alg_bytes_step = n * (CHUNK + 24 + 64) + stored          # SURVEY.md §8d: 65 624 + c per chunk
    achieved = alg_bytes_step * K / (enc_ns * 1e-9) / 1e9 if enc_ns else 0.0
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "encode_traffic.json")) as f:
            tj = json.load(f)
        traffic = tj["dram_bytes_per_launch"] * (n / max(1, enc_launches // K)) / tj["chunks_per_launch"]
        traffic_src = f"static: {tj['source']} (ncu --set full capture of this launch shape; not re-measured per run)"
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "k_encode (LZ4 encode + EF128 fingerprint along the parse + record in place + slot publish)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": alg_bytes_step / max(1, enc_launches // K),
                "avg_launch_ms": enc_ns / 1e6 / max(1, enc_launches),
                "read_form_frac": n * CHUNK * K / (enc_ns * 1e-9) / 1e9 / peak if enc_ns else 0.0,
                "stored_ratio": stored / (n * CHUNK)}
    launches = (st1["kernel_launches"] - st0["kernel_launches"]) // K

    # ---- the other BASELINE configs, each with its gate ----
    eng.close()                                   # frees the arena for the config engines
    configs = {}
    if not args.no_configs:
        if world == 1:
            configs["C2"], configs["C3"] = run_config_2_3(args, E, O, torch, local, d_pages, h_ptr, h_pages, peak, host_threads)
        else:
            configs["C4"] = run_config_4(args, E, O, torch, dist, rank, world, local, d_pages, host_threads, h_ptr, h_pages)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        eng_tmp_pages = O.gen_chunks(SEED, cids[: args.cpu_sample_chunks], CHUNK, host_threads)
        r = cpu_reference_run(eng_tmp_pages, off[: args.cpu_sample_chunks], nh[: args.cpu_sample_chunks], host_threads)
        key = "put_gibs" if "put_gibs" in r else "codec_encode_gibs"
        cpu = {"value": r[key], "unit": "GiB/s", "cores": r["cores"], "kind": r["kind"],
               "sample": f"first {args.cpu_sample_chunks} chunks ({args.cpu_sample_chunks * CHUNK >> 20} MiB) of the same stream; "
                         f"{'cachemap_put on a tmpfs LMDB store' if key == 'put_gibs' else 'LZ4 encode only'}",
               "codec_encode_gibs": r["codec_encode_gibs"], "codec_decode_gibs": r["codec_decode_gibs"],
               "get_gibs": r.get("get_gibs")}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(world, n),
            "timing": {"clock": "CUDA events on the engine's stream around the K timed steps (incl. the replica import of every step), max over ranks",
                       "device_ms_total": dev_ms_total, "wall_ms_between_barriers": wall_ms_total,
                       "per_step_ms_rank0": dev_ms_steps,
                       "step_breakdown_ms_rank0": {"encode_ms": enc_ns / 1e6 / max(1, K), **breakdown}},
            "e2e": {"value": e2e, "unit": "GiB/s", "h2d_bytes_per_step": int(n * (CHUNK + 16 + 8)),
                    "d2h_bytes_per_step": int(n * 4),
                    "call": "cmb200_put_step (write-behind) + cmb200_wait, 2 steps in flight from 2 page-locked input "
                            "buffers (step k+1 submitted before step k's stored lengths are read); all K steps, "
                            "copies and reads inside one timed region",
                    "synchronous_call": {"value": e2e_sync, "unit": "GiB/s",
                                         "call": "cmb200_put_batch, one step at a time, barrier + synchronize around each"}},
            "gpu_launches": int(launches * K), "gpu_launches_per_step": int(launches),
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "parity": parity, "integrity": integrity, "configs": configs,
            "index": {"local_entries": final["entries"], "remote_entries": final["remote_entries"],
                      "exchange": "1 all-gather of 32-byte key records per step (NCCL on a side stream, overlapping the next "
                                  "step's encode; records packed and imported on the device)" if dist else "none (single GPU)"},
        }
        print(json.dumps(line))
    E.lib().cmb200_dev_free(None, d_pages)
    E.lib().cmb200_host_free(h_ptr)
    E.lib().cmb200_host_free(h_ptr_b)
    for p, _ in lens_pin:
        E.lib().cmb200_host_free(p)
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    if len(sys.argv) == 4 and sys.argv[1] == "--ref-store-child":     # see reference_store_rates
        return reference_store_child(int(sys.argv[2]), int(sys.argv[3]))
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunks", type=int, default=16384, help="chunks per GPU per step (16384 = 1 GiB)")
    ap.add_argument("--max-batch", type=int, default=16384, help="chunks per kernel launch (resident pages)")
    ap.add_argument("--cpu-sample-chunks", type=int, default=8192)
    ap.add_argument("--parity-chunks", type=int, default=8192, help="chunks of the measured run checked against the oracle")
    ap.add_argument("--c2-gib", type=float, default=16.0, help="stream size of config 2 (and thereby the resident set of config 3)")
    ap.add_argument("--c3-e2e-gib", type=float, default=4.0, help="pages read back to the host in config 3's end-to-end leg")
    ap.add_argument("--c4-steps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                    "(rank 0's shard)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
