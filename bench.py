#!/usr/bin/env python
"""bench.py -- stage-1 structural indexing throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--check] [--dump-outputs DIR]

One "step" = one stage-1 pass (structural indexing + UTF-8 validation) over one batch of synthetic input per GPU.

Configurations (`--config`, BASELINE.json `configs`):
  stage1_64m   (default) configs[1]: synthetic 64 MiB random-structure JSON, stage 1 on 1xB200.  At N>1 every rank
               holds one 64 MiB shard of ONE N x 64 MiB document (a JSON array cut after line feeds, so no shard is a
               document of its own); every step is a sharded pass through sjb200_stage1_sharded: the scan kernel itself
               stores each shard's {count, state, transducer, flags} record into every rank's exchange window over
               NVLink (the path's one exchange, SURVEY.md 8e), the host folds state / index base -> weak scaling.
  jsonexamples configs[0]: twitter.json / citm_catalog.json / amazon_cellphones.ndjson (latency-bound: one launch each)
  ndjson_1g    configs[2]: 1 GiB NDJSON (amazon_cellphones-style rows), streaming_final; N>1: cut after line feeds
  utf8_minify_256m  configs[3]: validate_utf8 on 256 MiB mixed ASCII / UTF-8 text, minify on 256 MiB pretty JSON
  concat_8g    configs[4]: twitter + citm repeated to 8 GiB, 8 shards of ~1 GiB with 64-bit index bases, round-robin
               over the N ranks
  tokens_64m   SURVEY.md 8(f) row 4 (not a BASELINE config): stage-2-lite (sjb200_tokens_dev) on the 64 MiB document
`--check` runs the parity gate of the multi-rank path on adversarial cuts (mid-row, mid-string: carry-in != 0, second
round, re-scans) through the real IPC / NCCL plumbing and prints one JSON line; exit code 1 on a mismatch.

The JSON line carries:
  value     input GB/s with the input resident in HBM (device-timed, max over ranks)
  e2e       the same metric through the reference's own boundary: libsimdjson_b200.so (the C++ plug-in),
            get_active_implementation()->create_dom_parser_implementation()->stage1() on a PAGEABLE padded_string;
            H2D copy, scan and the indexes' way back to the parser's structural_indexes inside the timed region
  roofline  algorithmic bytes (1 B read per input byte + 4 B written per structural + 12 B of sentinels, SURVEY.md
            section 8(d)) / the scan kernel's mean duration, measured with CUDA events recorded around every scan kernel
            of the timed region on its launch stream, against MEASURED_PEAKS.json hbm_gbs
  parity    every distinct document of the timed region: (n + 3) index words of its last step against the CPU oracle
  cpu_baseline  the reference's own CPU stage 1 (oracle/_ref, the unmodified reference) on this box's host cores:
            pre-spawned threads, one private copy of the document per thread; all cores and one core
`--impl reference` times that CPU implementation as its own arm (rank 0 only).

`--dump-outputs DIR` (stage1_64m) writes what the last timed step returned, as float64 .npy files under DIR (see
dump_outputs), so that two builds can be compared output for output: the inputs are seeded, the same on every run.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # bench.py writes nothing into the tree it runs from, bytecode caches of its modules included

DOC_BYTES = 64 << 20
ROTATE = 4  # distinct 64 MiB inputs used round-robin: 256 MiB > 126 MB of L2, so no step finds its input in L2
METRIC = "stage1 GB/s (bytes in / s) vs HBM roofline at 1/2/4/8 B200; CPU ref GB/s"
UNIT = "GB/s"
PLUGIN = os.path.join(ROOT, "simdjson_b200", "plugin", "libsimdjson_b200.so")
DUMP_LIMIT = 64_000_000  # bytes of --dump-outputs in all, .npy headers included
KERNEL_SOURCES = ["sjb200_scan4.cuh", "sjb200_bits.cuh", "sjb200_simt.cuh", "sjb200_params.h", "sjb200_kernels.cu", "sjb200_utf8.cuh"]


def workload_name(world):
    if world == 1:
        return "synthetic 64 MiB random-structure JSON, stage1 index on 1xB200 (BASELINE.json configs[1])"
    return f"synthetic {world} x 64 MiB random-structure JSON, stage1 sharded by byte range over {world}xB200 (BASELINE.json configs[1] per GPU)"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def kernel_source_hash():
    h = hashlib.sha256()
    for f in KERNEL_SOURCES:
        with open(os.path.join(ROOT, "simdjson_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel="scan4_kernel"):
    """DRAM bytes of one launch of the kernel (substring of its name) on the bench document, from an `ncu --set full`
    capture summarised under profiles/ -- reported ONLY when that capture was taken from the kernel sources this run was
    built from (the summary records their hash); otherwise null: a stale constant is worse than no number."""
    want = kernel_source_hash()
    best = None
    pdir = os.path.join(ROOT, "profiles")
    for name in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if not name.endswith("_ncu_full.json"):
            continue
        try:
            d = json.load(open(os.path.join(pdir, name)))
            for e in (d if isinstance(d, list) else [d]):
                kn = e.get("Kernel Name", "")
                if (kernel + "(") not in kn and not kn.startswith(kernel) and ("::" + kernel + "(") not in kn:
                    continue
                if e.get("kernel_src_sha16") != want:
                    continue
                unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                tot = 0.0
                for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    v, u = e[k]
                    tot += float(v) * unit[u]
                best = (int(tot), os.path.join("profiles", name))
        except Exception:  # noqa: BLE001
            continue
    return best if best else (None, f"no ncu capture of kernel sources {want} under profiles/")


class ClockSampler:
    """samples SM clocks / throttle reasons through NVML while the timed region runs (every ~1 ms; the timed region
    of a 64 MiB stage-1 pass is milliseconds long, far shorter than one `nvidia-smi` invocation)"""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.rows, self.stop, self.th, self.h = index, [], threading.Event(), None, None
        try:
            if os.environ.get("SJB200_BENCH_NVML") == "0":  # diagnostic: no sampling thread at all
                raise RuntimeError("disabled")
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv, self.h, self.max_sm = None, None, None

    def _run(self):
        while not self.stop.is_set():
            try:
                sm = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                try:
                    rs = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    rs = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, rs))
            except Exception:  # noqa: BLE001
                pass
            self.stop.wait(0.001)

    def __enter__(self):
        if self.h is not None:
            self.th = threading.Thread(target=self._run, daemon=True)
            self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.th:
            self.th.join(timeout=2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["nvml unavailable"], "samples": 0}
        sm = sorted(r[0] for r in self.rows)
        reasons = set()
        for _, rs in self.rows:
            for bit, nm in self.REASONS.items():
                if rs & bit:
                    reasons.add(nm)
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_max_mhz": float(self.max_sm), "reasons": sorted(reasons), "samples": len(self.rows)}


# =============================================================================== workloads
def make_doc(seed_offset):
    from simdjson_b200 import corpus
    return corpus.random_json(DOC_BYTES, seed=corpus.SEED + 7919 * seed_offset)


def make_stream(world, k):
    """ONE document of world x 64 MiB: '[' + pieces separated by ',\\n' + ']' -- a single JSON array, so that a shard cut
    anywhere is not a document of its own.  Deterministic in (world, k); every rank builds the same buffer."""
    from simdjson_b200 import corpus
    total = world * DOC_BYTES
    parts, size = [b"["], 1
    i = 0
    while True:
        piece = bytes(corpus.random_json(8 << 20, seed=corpus.SEED + 104729 * k + 31 * i))
        extra = len(piece) + (2 if i else 0)
        if size + extra + 64 > total:
            break
        if i:
            parts.append(b",\n")
        parts.append(piece)
        size += extra
        i += 1
    pad = total - size - len(b',\n"') - len(b'"]')
    parts.append(b',\n"' + b"x" * pad + b'"]')
    doc = np.frombuffer(b"".join(parts), dtype=np.uint8)
    assert len(doc) == total
    return doc


STREAM_PIECE = 8 << 20


def _stream_layout(world):
    """(number of 8 MiB pieces, end of the last piece, total) of make_stream(world, k): piece i occupies
    [1 + i * (P + 2), ... + P), ',\n' in front of every piece but the first"""
    total = world * DOC_BYTES
    size, i = 1, 0
    while True:
        extra = STREAM_PIECE + (2 if i else 0)
        if size + extra + 64 > total:
            break
        size += extra
        i += 1
    return i, size, total


def stream_range(world, k, lo, hi, cache=None):
    """bytes [lo, hi) of make_stream(world, k) without building the rest: only the 8 MiB pieces that overlap are generated
    (a rank of an N-GPU run needs its own 64 MiB shard, not N x 64 MiB -- at N = 8 the full stream costs minutes of Python per rank)"""
    from simdjson_b200 import corpus
    npieces, end_pieces, total = _stream_layout(world)
    lo, hi = max(0, lo), min(total, hi)
    out = np.empty(hi - lo, dtype=np.uint8)
    cache = {} if cache is None else cache

    def put(start, data):  # data = stream bytes [start, start + len(data))
        a, b = max(lo, start), min(hi, start + len(data))
        if a < b:
            out[a - lo: b - lo] = np.frombuffer(data, dtype=np.uint8)[a - start: b - start] if isinstance(data, (bytes, bytearray)) else data[a - start: b - start]
    put(0, b"[")
    for i in range(npieces):
        start = 1 + i * (STREAM_PIECE + 2)
        if i:
            put(start - 2, b",\n")
        if start < hi and start + STREAM_PIECE > lo:
            if i not in cache:
                cache[i] = np.asarray(corpus.random_json(STREAM_PIECE, seed=corpus.SEED + 104729 * k + 31 * i), dtype=np.uint8)
                assert len(cache[i]) == STREAM_PIECE
            put(start, cache[i])
    tail_head = b',\n"'
    put(end_pieces, tail_head)
    xs, xe = end_pieces + len(tail_head), total - 2  # the padding string's body
    a, b = max(lo, xs), min(hi, xe)
    if a < b:
        out[a - lo: b - lo] = ord("x")
    put(total - 2, b'"]')
    return out


def make_shard(world, k, rank, window=1 << 20):
    """rank's shard of make_stream(world, k) cut the way sharding.shard_cuts_at_lines cuts it, built from the pieces around it only"""
    from simdjson_b200 import sharding
    L = sharding._lib()
    total = world * DOC_BYTES
    cache = {}

    def cut(j):
        if j == 0:
            return 0
        if j >= world:
            return total
        nominal = (total * j) // world
        base = max(0, nominal - window)
        loc = np.ascontiguousarray(stream_range(world, k, base, min(total, nominal + 8), cache))
        return base + int(L.sjb200_shard_cut_line(loc.ctypes.data, len(loc), nominal - base, window))
    c0 = cut(rank)
    c1 = max(c0, cut(rank + 1))  # (shard_cuts_at_lines keeps cuts monotonic the same way; nominal cuts are 64 MiB apart, the window is 1 MiB)
    return np.ascontiguousarray(stream_range(world, k, c0, c1, cache))


def oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    return O


def raw_scan(O, port, buf, state_in=0):
    """the oracle's raw structural list of a buffer entered in state_in (no finish() logic)"""
    L = port.L
    L.sjo_scan_shard.restype = C.c_uint64
    L.sjo_scan_shard.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32)]
    a = np.ascontiguousarray(buf, dtype=np.uint8)
    idx = np.zeros(len(a) + 1, dtype=np.uint32)
    so = C.c_uint32(0)
    n = L.sjo_scan_shard(a.ctypes.data, len(a), state_in, idx.ctypes.data, C.byref(so))
    return idx[:n], int(so.value)


def cpu_baseline(doc, steps=3):
    """the reference's CPU stage 1 on this host: all cores (pre-spawned threads, one private copy of the document per
    thread: DRAM-bound, not cache-luck-bound) and one core; a bounded sample (a few rounds)"""
    O = oracle()
    cores = os.cpu_count() or 1
    if O.have_ref():
        ref = O.Ref("")
        threads = max(1, min(cores, int(os.environ.get("SJB200_REF_THREADS", cores))))
        best1, mean1, _ = ref.time_rounds(0, doc, 0, 1, 1, 3)
        bestn, meann, err = ref.time_rounds(0, doc, 0, threads, 1, max(2, steps))
        return {"value": round(threads * len(doc) / meann / 1e9, 3), "unit": UNIT, "cores": threads, "kind": "reference",
                "value_best_round": round(threads * len(doc) / bestn / 1e9, 3), "one_core": round(len(doc) / mean1 / 1e9, 3),
                "sample": f"{ref.name} kernel; {threads} pre-spawned threads x one private {len(doc) >> 20} MiB document each, mean of {max(2, steps)} rounds after 1 warm-up round",
                "error_code": err}
    port = O.Port()
    t0 = time.perf_counter()
    port.stage1(doc[: 16 << 20], 0)
    dt = time.perf_counter() - t0
    return {"value": round((16 << 20) / dt / 1e9, 3), "unit": UNIT, "cores": 1, "kind": "port", "sample": "scalar C port, 16 MiB prefix, one pass"}


def dump_sample(n, k):
    """positions of the k of n index words that --dump-outputs keeps when all n do not fit: fixed by the seed, sorted"""
    return np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def dump_outputs(out_dir, rank, world, scalars, words):
    """--dump-outputs: the last timed step's results (scalars: name -> value) and index words, as float64 .npy files (exact
    for 32-bit values), named rank<r>_<name>.npy when world > 1.  The index words go out whole when they fit this rank's
    share of DUMP_LIMIT, else as words[dump_sample(len(words), cap)]; len(words) is n_structural_indexes + 3 at one rank
    and count at several."""
    os.makedirs(out_dir, exist_ok=True)
    cap = (DUMP_LIMIT // world - 4096) // 8  # float64 words; 4 KiB covers the .npy headers of this rank's files
    if len(words) > cap:
        words = words[dump_sample(len(words), cap)]
    arrays = dict(scalars, structural_indexes=words)
    prefix = f"rank{rank}_" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, dtype=np.float64).reshape(-1))


# =============================================================================== reference arm
def run_reference(args, rank, world):
    """the reference's own CPU stage 1 (oracle/_ref = unmodified reference, compiled in the build container) on this box's
    host cores; else the oracle port.  Rank 0 only."""
    if rank != 0:
        return
    doc = make_doc(0)
    cb = cpu_baseline(doc, steps=max(2, min(args.steps, 8)))
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(len(doc) * cb["cores"] / (cb["value"] * 1e9) * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": workload_name(max(1, args.gpus)), "bytes_per_call": DOC_BYTES, "threads": cb["cores"],
                   "how": "CPU reference: every host thread runs the whole 64 MiB stage-1 call on its own copy of the document (the reference has no intra-call parallelism)"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# =============================================================================== e2e through the plug-in
def plugin_e2e(doc, iters, want_words=None):
    """stage 1 through libsimdjson_b200.so on a pageable padded_string (dropin_stage1_timed, plugin/dropin_harness.cpp)"""
    L = C.CDLL(PLUGIN)
    L.dropin_stage1_timed.restype = C.c_int
    L.dropin_stage1_timed.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.c_void_p, C.c_size_t,
                                      C.POINTER(C.c_ulonglong)]
    secs = (C.c_double * 2)()
    n = C.c_uint32(0)
    calls = C.c_ulonglong(0)
    idx = np.zeros(len(doc) // 4 + 16, dtype=np.uint32)
    rc = L.dropin_stage1_timed(1, doc.ctypes.data, len(doc), iters, secs, C.byref(n), idx.ctypes.data, len(idx), C.byref(calls))
    ok = None
    if want_words is not None:
        ok = bool(rc == 0 and np.array_equal(idx[: len(want_words)], want_words))
    return {"rc": rc, "n": int(n.value), "seconds_total": secs[0], "seconds_best": secs[1], "gpu_calls": int(calls.value), "parity": ok}


# =============================================================================== our arm
def run_ours(args, rank, world):
    import torch
    import torch.distributed as dist

    import simdjson_b200 as sj
    from simdjson_b200 import capi, sharding

    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    impl = sj.get_active_implementation(local)
    L = sj.lib()
    O = oracle()
    port = O.Port()

    rc, parser = impl.create_dom_parser_implementation(DOC_BYTES)
    if rc != sj.SUCCESS:
        raise RuntimeError("create_dom_parser_implementation failed: " + capi.ERROR_NAMES.get(rc, str(rc)))
    parser.set_option("time_kernel", 1)
    stream = torch.cuda.Stream(device=dev)  # the stream every scan of the timed region is launched on
    torch.cuda.set_stream(stream)
    words = L.sjb200_index_words(DOC_BYTES)
    d_idxs = [torch.empty(words, dtype=torch.int32, device=dev) for _ in range(ROTATE)]  # one per distinct input: the last step's output of each stays for the parity gate

    # ---- workload, resident in HBM before the timed region
    if world == 1:
        docs = [make_doc(k) for k in range(ROTATE)]
        shards, cuts = docs, None
    else:
        shards = [make_shard(world, k, rank) for k in range(ROTATE)]  # = make_stream(world, k) cut by sharding.shard_cuts_at_lines, rank's part
        cuts = None
    d_docs = [torch.from_numpy(d.copy()).to(dev) for d in shards]
    comm = None
    if world > 1:
        comm = sharding.Comm(parser, rank, world)

        def all_gather_bytes(h):
            t = torch.from_numpy(h.copy()).to(dev)
            out = torch.empty(world * t.numel(), dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(out, t)  # NCCL: the 64-byte IPC handles of the exchange windows, once per job
            return out.cpu().numpy()
        comm.connect(all_gather_bytes)

    kernel_ms, n_struct, results = [], [], {}
    host_ms = {"enqueue": 0.0, "finish": 0.0, "finish_max": 0.0}

    def run_steps(k, record):
        t_ev0, t_ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        parser.get_stat("kernel_ms_mean")  # reset the per-launch event log
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t_ev0.record(stream)
        if world == 1:
            # K steps = K documents through the batch entry point: every scan is queued back to back on `stream`
            res = parser.stage1_device_batch([d_docs[i % ROTATE] for i in range(k)], [d_idxs[i % ROTATE] for i in range(k)], sj.REGULAR, stream=stream)
            for i, (err, n) in enumerate(res):
                if err != sj.SUCCESS:
                    raise RuntimeError("stage1 failed: " + capi.ERROR_NAMES.get(err, str(err)) + " " + parser.last_cuda_error())
                if record:
                    n_struct.append(n)
                    results[i % ROTATE] = (n, 0, 0)
        else:
            # sharded passes, up to 24 in flight: enqueue (scan + fused exchange, no host round trip), then finish
            # (fold state / base from the local exchange window; re-scan + second round only on a wrong speculation)
            i = 0
            while i < k:
                w = min(24, k - i)
                th0 = time.perf_counter()
                for j in range(i, i + w):
                    rcq = comm.enqueue(d_docs[j % ROTATE], d_idxs[j % ROTATE], rank == world - 1, stream)
                    if rcq != 0:
                        raise RuntimeError("sharded enqueue failed: " + parser.last_cuda_error())
                host_ms["enqueue"] += (time.perf_counter() - th0) * 1e3
                for j in range(i, i + w):
                    th1 = time.perf_counter()
                    rcf, res = comm.finish()
                    dt = (time.perf_counter() - th1) * 1e3
                    host_ms["finish"] += dt
                    host_ms["finish_max"] = max(host_ms["finish_max"], dt)
                    if rcf != 0:
                        raise RuntimeError("sharded finish failed: " + parser.last_cuda_error())
                    if record:
                        n_struct.append(int(res.count))
                        results[j % ROTATE] = (int(res.count), int(res.base), int(res.state_in), int(res.rescanned), int(res.total_count))
                i += w
        t_ev1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        if record:
            kernel_ms.append(parser.get_stat("kernel_ms_mean"))
        return t_ev0.elapsed_time(t_ev1)

    # warm-up: at least W steps; for sharded passes at least one full pipeline (24 passes in flight) so that every event,
    # window slot and peer mapping the timed region uses has been used once (a 2 ms timed region has no room for first uses)
    warmup_steps = max(3, args.warmup) if world == 1 else max(3, args.warmup, min(args.steps, 24))
    run_steps(warmup_steps, False)
    launches1 = parser.get_stat("launches")
    with ClockSampler(local) as clocks:
        total_ms = run_steps(args.steps, True)
    launches2 = parser.get_stat("launches")
    sharded_host = None
    if world > 1:  # where the host's time went in the timed region (and the warm-up): per rank on stderr, rank 0's in the line
        sharded_host = {"enqueue_ms": round(host_ms["enqueue"], 3), "finish_ms": round(host_ms["finish"], 3), "finish_max_ms": round(host_ms["finish_max"], 3),
                        "window_polls": int(parser.get_stat("xchg_polls")), "poll_wait_ms": round(parser.get_stat("xchg_wait_ms"), 3),
                        "own_scan_wait_ms": round(parser.get_stat("xchg_evsync_ms"), 3), "second_rounds": int(parser.get_stat("xchg_second_rounds")),
                        "note": "host wall time over warm-up + timed passes of this rank"}
        print(f"[rank {rank}] total_ms {total_ms:.3f} {sharded_host}", file=sys.stderr, flush=True)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * DOC_BYTES / (ms_per_step * 1e-3) / 1e9

    if args.dump_outputs:
        last = (args.steps - 1) % ROTATE  # the input (and index buffer) of the last timed step
        got = d_idxs[last].cpu().numpy().view(np.uint32)
        if world == 1:
            n = results[last][0]
            dump_outputs(args.dump_outputs, rank, world, {"n_structural_indexes": n}, got[: n + 3])
        else:
            count, base, _state_in, _rescanned, total = results[last]
            dump_outputs(args.dump_outputs, rank, world, {"count": count, "base": base, "total_count": total}, got[:count])

    # ---- parity gate: the output every distinct input left behind in the timed region, against the oracle
    parity_ok, checked, rescans = True, 0, 0
    first_words = None
    for k in range(min(ROTATE, args.steps)):
        got = d_idxs[k].cpu().numpy().view(np.uint32)
        if world == 1:
            want = port.stage1(shards[k], 0)
            n = results[k][0]
            okk = want.err == 0 and want.n == n and np.array_equal(got[: n + 3], want.words())
            if k == 0:
                first_words = want.words().copy()
        else:
            count, base, state_in, rescanned, total = results[k]
            widx, _ = raw_scan(O, port, shards[k], state_in)
            counts = torch.tensor([count], dtype=torch.int64, device=dev)
            allc = torch.empty(world, dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(allc, counts)
            allc = allc.cpu().numpy()
            okk = len(widx) == count and np.array_equal(got[:count], widx) and base == int(allc[:rank].sum()) and total == int(allc.sum())
            rescans += rescanned
        parity_ok = parity_ok and bool(okk)
        checked += 1
    if world > 1:
        flag = torch.tensor([1 if parity_ok else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity_ok = bool(flag.item())

    # ---- e2e: stage 1 through the plug-in (the reference's own boundary), pageable input, every rank its own shard
    e2e_steps = max(3, min(args.steps, 10))
    if world > 1:
        dist.barrier()
    e2e_info = None
    if os.path.exists(PLUGIN):
        r = plugin_e2e(shards[0], e2e_steps, first_words)
        e2e_s, e2e_n = r["seconds_total"], r["n"]
        e2e_info = {"through": "libsimdjson_b200.so: create_dom_parser_implementation()->stage1() on a pageable padded_string", "rc": r["rc"], "parity": r["parity"],
                    "gbs_best_call": round(len(shards[0]) / r["seconds_best"] / 1e9, 3), "gpu_stage1_calls": r["gpu_calls"]}
    else:  # the plug-in needs the reference headers to build; without it the same C-ABI call through the Python mirror, pageable numpy input
        host = shards[0].copy()
        for _ in range(2):
            parser.stage1(host, sj.REGULAR)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            rcx = parser.stage1(host, sj.REGULAR)
        e2e_s, e2e_n = time.perf_counter() - t0, parser.n_structural_indexes
        e2e_info = {"through": "sjb200_stage1 (C ABI, Python mirror), pageable input", "rc": rcx}
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * DOC_BYTES * e2e_steps / float(te.item()) / 1e9

    if rank == 0:
        peak, peak_src = peaks()
        kms = float(np.mean(kernel_ms))
        nmean = float(np.mean(n_struct))
        algo_bytes = DOC_BYTES + 4.0 * nmean + 12.0
        achieved = algo_bytes / (kms * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic("scan4_kernel")
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup_steps,
            "ms_per_step": round(ms_per_step, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_name(world), "bytes_per_gpu_per_step": DOC_BYTES, "mode": "regular" if world == 1 else "shard", "structurals_per_step": int(nmean),
                       "l2": f"{ROTATE} distinct inputs used round-robin ({ROTATE * DOC_BYTES >> 20} MiB > 126 MB L2)",
                       "content": "random sequence of 48 distinct 96 KiB random subtrees per document (corpus.random_json): DRAM behaviour of 64 MiB, 4.6 MB of distinct structure",
                       "api": "sjb200_stage1_dev_batch: the K documents of the timed region are queued back to back on one stream" if world == 1 else
                              "sjb200_stage1_sharded_enqueue / _finish: exchange record stored by the scan kernel into every rank's window over NVLink (CUDA IPC); NCCL only for the handle exchange at start-up"},
            "clocks": clocks.summary(),
            "parity": {"ok": parity_ok, "documents_checked": checked, "against": "CPU oracle (oracle/sj_oracle.c), (n+3) index words" if world == 1 else "CPU oracle raw scan of every rank's shard + index bases", "rescans": rescans},
            "e2e": dict({"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": DOC_BYTES, "d2h_bytes_per_step": int(4 * e2e_n + 24), "steps": e2e_steps}, **(e2e_info or {})),
            "gpu_launches": int(launches2 - launches1),
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
                         "traffic_source": traffic_src, "peak_source": peak_src, "kernel": "sjb200::scan4_kernel (sjb200_scan4.cuh)", "kernel_ms": round(kms, 5), "algorithmic_bytes": int(algo_bytes),
                         "input_gbs_kernel_only": round(DOC_BYTES / (kms * 1e-3) / 1e9, 1), "kernel_src_sha16": kernel_source_hash()},
        }
        if sharded_host is not None:
            line["sharded_host"] = sharded_host
        line["cpu_baseline"] = cpu_baseline(shards[0])
        print(json.dumps(line), flush=True)
    if comm is not None:
        comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not parity_ok:
        sys.exit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="stage1_64m", choices=["stage1_64m", "jsonexamples", "ndjson_1g", "utf8_minify_256m", "concat_8g", "tokens_64m"])
    ap.add_argument("--check", action="store_true", help="parity gate of the multi-rank path on adversarial cuts")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.check or args.config != "stage1_64m"):
        ap.error("--dump-outputs writes the outputs of --impl ours --config stage1_64m")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and args.gpus > 1:
        sys.stderr.write(f"bench.py: --gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})\n")
    if args.check or args.config != "stage1_64m":
        import bench_configs
        bench_configs.run(args, rank, world)
        return
    run_ours(args, rank, world)


if __name__ == "__main__":
    main()
