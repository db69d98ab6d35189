"""bench_configs.py -- the BASELINE.json configurations beyond the headline one, and the multi-rank parity gate.

Called by bench.py for `--config NAME` (other than the default stage1_64m) and for `--check`.  Same contract: one JSON
line on rank 0; every number device-timed with CUDA events around the scan kernels, every output compared with the CPU
oracle (tests/oracle_lib.py -> oracle/) before the line is printed; exit code 1 on a mismatch.
"""
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

import bench as B

ROOT = B.ROOT


def _setup(rank, world):
    import torch
    import torch.distributed as dist

    import simdjson_b200 as sj
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    return torch, dist, sj, dev, local


def _connect(torch, dist, sharding, parser, rank, world, dev):
    comm = sharding.Comm(parser, rank, world)

    def all_gather_bytes(h):
        t = torch.from_numpy(h.copy()).to(dev)
        out = torch.empty(world * t.numel(), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(out, t)
        return out.cpu().numpy()
    comm.connect(all_gather_bytes)
    return comm


def _max_over_ranks(torch, dist, dev, world, x):
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _all_ok(torch, dist, dev, world, ok):
    t = torch.tensor([1 if ok else 0], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


def _roofline(algo_bytes, kms, kernel):
    peak, src = B.peaks()
    ach = algo_bytes / (kms * 1e-3) / 1e9
    traffic, tsrc = B.ncu_traffic(kernel)
    return {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4), "traffic": traffic, "traffic_source": tsrc,
            "peak_source": src, "kernel_ms": round(kms, 5), "algorithmic_bytes": int(algo_bytes), "kernel_src_sha16": B.kernel_source_hash()}


def _warmup(args):
    """untimed passes before the timed ones, the same floor as bench.py's default config"""
    return max(3, args.warmup)


def _line(args, world, value, ms_per_step, config, extra):
    d = {"metric": B.METRIC, "value": round(value, 2), "unit": B.UNIT, "n_gpus": world, "steps": args.steps, "warmup": _warmup(args), "ms_per_step": round(ms_per_step, 5),
         "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config}
    d.update(extra)
    return d


# =============================================================================== configs[0]: jsonexamples
def run_jsonexamples(args, rank, world):
    torch, dist, sj, dev, local = _setup(rank, world)
    if rank != 0:
        return True
    O = B.oracle()
    port = O.Port()
    rc, parser = sj.get_active_implementation(local).create_dom_parser_implementation(4 << 20)
    parser.set_option("time_kernel", 1)
    files, ok = [], True
    steps = args.steps
    for name, mode in (("twitter.json", 0), ("citm_catalog.json", 0), ("amazon_cellphones.ndjson", 2)):
        data = np.frombuffer(O.jsonexample(name), dtype=np.uint8).copy()
        d = torch.from_numpy(data).to(dev)
        want = port.stage1(data, mode)
        for _ in range(_warmup(args)):
            parser.stage1_device(d, mode)
        parser.get_stat("kernel_ms_mean")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            rcs = parser.stage1_device(d, mode)
        e1.record()
        torch.cuda.synchronize()
        kms = parser.get_stat("kernel_ms_mean")
        got = parser.device_index_buffer().cpu().numpy().view(np.uint32)
        same = rcs == want.err and parser.n_structural_indexes == want.n and np.array_equal(got[: want.n + 3], want.words())
        ok = ok and bool(same)
        e2e = B.plugin_e2e(data, 10, want.words() if mode == 0 else None) if os.path.exists(B.PLUGIN) and mode == 0 else None
        ref1 = None
        if O.have_ref():
            b1, m1, _ = O.Ref("").time_rounds(0, data, mode, 1, 1, 5)
            ref1 = round(len(data) / m1 / 1e9, 3)
        files.append({"file": name, "bytes": int(len(data)), "mode": mode, "n_structural_indexes": int(want.n), "parity": bool(same), "kernel_ms": round(kms, 5),
                      "gbs_kernel": round(len(data) / kms / 1e6, 2), "gbs_call": round(len(data) * steps / e0.elapsed_time(e1) / 1e6, 2),
                      "e2e_gbs_plugin": round(len(data) * 10 / e2e["seconds_total"] / 1e9, 3) if e2e else None, "e2e_parity": e2e["parity"] if e2e else None,
                      "cpu_reference_1core_gbs": ref1})
    f0 = files[0]
    line = _line(args, 1, f0["gbs_call"], f0["bytes"] / (f0["gbs_call"] * 1e6) if f0["gbs_call"] else 0.0,
                 {"workload": "jsonexamples/twitter.json single-doc stage1 (BASELINE.json configs[0]); also citm_catalog.json, amazon_cellphones.ndjson",
                  "note": "latency-bound: a 0.6-1.7 MB document is one launch of ~10-27 elements; one CPU core is the natural reference here", "files": files},
                 {"parity": {"ok": ok, "documents_checked": len(files), "against": "CPU oracle, (n+3) index words"},
                  "e2e": {"value": f0["e2e_gbs_plugin"], "unit": B.UNIT, "h2d_bytes_per_step": f0["bytes"], "d2h_bytes_per_step": 4 * f0["n_structural_indexes"] + 24},
                  "gpu_launches": steps * len(files), "roofline": _roofline(f0["bytes"] + 4 * f0["n_structural_indexes"] + 12, f0["kernel_ms"], "scan4_kernel")})
    print(json.dumps(line), flush=True)
    parser.close()
    return ok


# =============================================================================== configs[2]: 1 GiB NDJSON
def run_ndjson(args, rank, world, total=1 << 30):
    torch, dist, sj, dev, local = _setup(rank, world)
    from simdjson_b200 import corpus, sharding
    O = B.oracle()
    port = O.Port()
    doc = corpus.ndjson_rows(total)
    cuts = sharding.shard_cuts_at_lines(doc, world) if world > 1 else [0, len(doc)]
    shard = np.ascontiguousarray(doc[cuts[rank]: cuts[rank + 1]])
    del doc
    rc, parser = sj.get_active_implementation(local).create_dom_parser_implementation(len(shard))
    parser.set_option("time_kernel", 1)
    d = torch.from_numpy(shard).to(dev)
    d_idx = torch.empty(int(sj.lib().sjb200_index_words(len(shard))), dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    comm = _connect(torch, dist, sharding, parser, rank, world, dev) if world > 1 else None
    steps = args.steps
    last = None

    def one_pass():
        nonlocal last
        if world == 1:
            rcs = parser.stage1_device(d, sj.STREAMING_FINAL, d_idx=d_idx, stream=stream)
            last = (rcs, parser.n_structural_indexes)
        else:
            rcs, res = comm.scan(d, d_idx, rank == world - 1, stream)
            if rcs != 0:
                raise RuntimeError("sharded scan failed: " + parser.last_cuda_error())
            last = (rcs, int(res.count), int(res.base), int(res.state_in), int(res.total_count), int(res.rescanned))
    for _ in range(_warmup(args)):
        one_pass()
    parser.get_stat("kernel_ms_mean")
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        one_pass()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = _max_over_ranks(torch, dist, dev, world, e0.elapsed_time(e1)) / steps
    kms = parser.get_stat("kernel_ms_mean")
    got = d_idx.cpu().numpy().view(np.uint32)
    if world == 1:
        want = port.stage1(shard, sj.STREAMING_FINAL)
        ok = last[0] == want.err and last[1] == want.n and np.array_equal(got[: want.n + 3], want.words())
        n = int(want.n)
    else:
        widx, _ = B.raw_scan(O, port, shard, last[3])
        counts = torch.tensor([last[1]], dtype=torch.int64, device=dev)
        allc = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allc, counts)
        allc = allc.cpu().numpy()
        ok = len(widx) == last[1] and np.array_equal(got[: last[1]], widx) and last[2] == int(allc[:rank].sum()) and last[4] == int(allc.sum())
        n = int(allc.sum())
    ok = _all_ok(torch, dist, dev, world, bool(ok))
    if rank == 0:
        line = _line(args, world, total / (ms * 1e-3) / 1e9, ms,
                     {"workload": f"1 GiB NDJSON (amazon_cellphones-style rows), stage1 " + ("streaming_final on 1xB200" if world == 1 else f"sharded after line feeds over {world}xB200") + " (BASELINE.json configs[2])",
                      "bytes_total": total, "structurals": n, "l2": "1 GiB input >> 126 MB L2",
                      "api": "sjb200_stage1_dev" if world == 1 else "sjb200_stage1_sharded (exchange fused into the scan kernel)"},
                     {"parity": {"ok": ok, "against": "CPU oracle on the whole shard of every rank" + (" + 64-bit index bases" if world > 1 else ", (n+3) index words")},
                      "gpu_launches": int(steps), "roofline": _roofline(len(shard) + 4 * (last[1]) + 12, kms, "scan4_kernel"),
                      "e2e": {"value": None, "unit": B.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "device-resident configuration; e2e is reported by the default config"}})
        print(json.dumps(line), flush=True)
    if comm:
        comm.close()
    parser.close()
    return ok


# =============================================================================== configs[3]: validate_utf8 + minify, 256 MiB
def run_utf8_minify(args, rank, world, size=256 << 20):
    torch, dist, sj, dev, local = _setup(rank, world)
    if rank != 0:
        return True
    from simdjson_b200 import corpus
    O = B.oracle()
    port = O.Port()
    steps, warm = args.steps, _warmup(args)
    rc, parser = sj.get_active_implementation(local).create_dom_parser_implementation(size)
    parser.set_option("time_kernel", 1)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # ---- validate_utf8
    u = corpus.random_utf8(size).copy()
    du = torch.from_numpy(u).to(dev)
    ok = parser.validate_utf8_device(du) == 1 and port.validate_utf8(u)
    for where in (5, size // 2, size - 2):  # three corrupted copies: start / middle / last bytes
        bad = du.clone()
        bad[where] = 0xFF
        ok = ok and parser.validate_utf8_device(bad) == 0
        del bad
    ts = []
    for it in range(warm + steps):
        flush.fill_(it)
        torch.cuda.synchronize()
        parser.validate_utf8_device(du)
        ts.append(parser.get_stat("kernel_ms"))
    ums = float(np.mean(ts[warm:]))
    del du
    # ---- minify
    j = corpus.random_json(size, pretty_bias=0.8, utf8_rate=0.15).copy()
    dj = torch.from_numpy(j).to(dev)
    dst = torch.zeros(len(j), dtype=torch.uint8, device=dev)
    werr, wout = port.minify(j)
    rcm, dl = parser.minify_device(dj, dst)
    okm = rcm == werr and dl == len(wout) and torch.equal(dst[:dl].cpu(), torch.from_numpy(np.frombuffer(wout, dtype=np.uint8).copy()))
    ts = []
    for it in range(warm + steps):
        flush.fill_(it)
        torch.cuda.synchronize()
        parser.minify_device(dj, dst)
        ts.append(parser.get_stat("kernel_ms"))
    mms = float(np.mean(ts[warm:]))
    ok = bool(ok and okm)
    line = _line(args, 1, size / (ums * 1e-3) / 1e9, ums,
                 {"workload": "validate_utf8 + minify on 256 MiB mixed-ASCII/UTF-8 synthetic, 1xB200 (BASELINE.json configs[3])", "bytes": size,
                  "l2": "a 256 MiB buffer is written between launches (cold L2)", "value_is": "validate_utf8 input GB/s (kernel); minify below"},
                 {"parity": {"ok": ok, "against": "CPU oracle: verdict (valid + 3 corrupted copies), whole minified buffer"}, "gpu_launches": 2 * (warm + steps) + 5,
                  "roofline": dict(_roofline(size, ums, "utf8v2_kernel"), kernel="sjb200::utf8v2_kernel (sjb200_utf8.cuh)"),
                  "minify": {"input_gbs": round(size / (mms * 1e-3) / 1e9, 1), "kept_fraction": round(dl / size, 4), "kernel_ms": round(mms, 5),
                             "roofline": dict(_roofline(size + dl, mms, "scan4_minify_kernel"), kernel="sjb200::scan4_minify_kernel (1 B read + kept bytes written per input byte)")},
                  "e2e": {"value": None, "unit": B.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "device-resident configuration"}})
    print(json.dumps(line), flush=True)
    parser.close()
    return ok


# =============================================================================== SURVEY 8(f) row 4: stage-2-lite on the 64 MiB document
def run_tokens(args, rank, world, size=64 << 20):
    """sjb200_tokens_dev behind stage 1 on BASELINE.json configs[1]'s document: token types / payloads / string buffer.
    Timed with CUDA events around the three launches of one call (cold L2), whole-output parity against the oracle."""
    torch, dist, sj, dev, local = _setup(rank, world)
    if rank != 0:
        return True
    from simdjson_b200 import corpus
    O = B.oracle()
    port = O.Port()
    steps, warm = args.steps, _warmup(args)
    doc = corpus.random_json(size).copy()
    d = torch.from_numpy(doc).to(dev)
    rc, parser = sj.get_active_implementation(local).create_dom_parser_implementation(size)
    assert parser.stage1_device(d, sj.REGULAR) == 0
    parser.set_option("tok_stage", int(os.environ.get("SJB200_TOK_STAGE", "1")))  # 0: A/B baseline without shared-memory staging
    n = parser.n_structural_indexes
    d_idx = parser.device_index_buffer()
    cap = int(sj.lib().sjb200_string_buf_capacity(size))
    d_type = torch.empty(n, dtype=torch.uint8, device=dev)
    d_payload = torch.empty(n, dtype=torch.int64, device=dev)
    d_strbuf = torch.empty(cap, dtype=torch.uint8, device=dev)
    res = sj.capi.TokensResult()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    ts = []
    for it in range(warm + steps):
        flush.fill_(it)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        sj.lib().sjb200_tokens_dev(parser._ctx, d.data_ptr(), size, d_idx.data_ptr(), n, d_type.data_ptr(), d_payload.data_ptr(), d_strbuf.data_ptr(), cap,
                                   C.byref(res), C.c_void_p(stream.cuda_stream))
        e1.record(stream)
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = float(np.mean(ts[warm:]))
    r = port.stage1(doc)
    t0 = time.time()
    want = port.tokens(doc, r.idx, r.n, strbuf_cap=cap)
    cpu_s = time.time() - t0
    ok = (res.error == want[0] == 0 and n == r.n and bytes(d_type.cpu().numpy()) == bytes(want[1]) and np.array_equal(d_payload.cpu().numpy().view(np.uint64), want[2])
          and res.string_bytes == want[4] and res.n_strings == want[5]
          and bytes(d_strbuf[: res.string_bytes].cpu().numpy()) == bytes(want[3]))
    # algorithmic bytes: the document once + the index array in, type + payload + string buffer out
    algo = size + 4 * n + 9 * n + int(res.string_bytes)
    line = _line(args, 1, size / (ms * 1e-3) / 1e9, ms,
                 {"workload": "stage-2-lite (token types, integer values, string buffer) on the synthetic 64 MiB document of BASELINE.json configs[1], 1xB200 (SURVEY.md 8(f) row 4)",
                  "bytes": size, "structurals": int(n), "strings": int(res.n_strings), "string_buf_bytes": int(res.string_bytes),
                  "l2": "a 256 MiB buffer is written between calls (cold L2)", "value_is": "document bytes per second through sjb200_tokens_dev (3 launches + the 24-byte result)",
                  "api": "sjb200_tokens_dev", "tok_stage": int(os.environ.get("SJB200_TOK_STAGE", "1"))},
                 {"parity": {"ok": bool(ok), "against": "CPU oracle (sjo_tokens): every type, payload and string-buffer byte"}, "gpu_launches": 3 * (warm + steps),
                  "roofline": dict(_roofline(algo, ms, "token_scan_kernel"), kernel="sjb200::token_scan_kernel + tile_scan_kernel + string_write_kernel (sjb200_tape.cu), one call",
                                   note="the call's three launches together; strings are walked twice (length, then copy)"),
                  "cpu_baseline": {"value": round(size / cpu_s / 1e9, 3), "unit": B.UNIT, "cores": 1, "kind": "port", "sample": "sjo_tokens (oracle/sj_oracle.c) on the whole 64 MiB document, one call"},
                  "e2e": {"value": None, "unit": B.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "device-resident configuration"}})
    print(json.dumps(line), flush=True)
    parser.close()
    return ok


# =============================================================================== configs[4]: 8 GiB of twitter + citm, 8 shards
def run_concat(args, rank, world, nshards=8, shard_target=1 << 30):
    torch, dist, sj, dev, local = _setup(rank, world)
    from simdjson_b200 import sharding
    O = B.oracle()
    port = O.Port()
    if nshards % world != 0:
        raise SystemExit("concat_8g needs 1, 2, 4 or 8 ranks")
    unit = b"".join(O.jsonexample(f) + b"\n" for f in ("twitter.json", "citm_catalog.json"))
    unit_a = np.frombuffer(unit, dtype=np.uint8)
    reps = shard_target // len(unit)
    shard = np.tile(unit_a, reps)  # every shard is the same bytes: reps whole (twitter, citm) pairs, cut at a document boundary
    uidx, ustate = B.raw_scan(O, port, unit_a, 0)
    assert ustate == 0
    rc, parser = sj.get_active_implementation(local).create_dom_parser_implementation(len(shard))
    parser.set_option("time_kernel", 1)
    d = torch.from_numpy(shard).to(dev)
    d_idx = torch.empty(int(sj.lib().sjb200_index_words(len(shard))), dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    comm = _connect(torch, dist, sharding, parser, rank, world, dev) if world > 1 else sharding.Comm(parser, 0, 1)
    rounds = nshards // world
    steps = args.steps

    def whole_job():
        """8 shards: `rounds` sharded passes of `world` shards each; 64-bit bases accumulate over the rounds on the host"""
        base, out = 0, []
        for q in range(rounds):
            rcs, res = comm.scan(d, d_idx, (q == rounds - 1) and rank == world - 1, stream)
            if rcs != 0 or res.final_state != 0:
                raise RuntimeError("sharded scan failed: " + parser.last_cuda_error())
            out.append((q * world + rank, base + int(res.base), int(res.count), int(res.rescanned)))
            base += int(res.total_count)
        return out, base
    for _ in range(_warmup(args)):
        whole_job()
    parser.get_stat("kernel_ms_mean")
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        out, total = whole_job()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = _max_over_ranks(torch, dist, dev, world, e0.elapsed_time(e1)) / steps
    kms = parser.get_stat("kernel_ms_mean")
    # parity: the shard is `reps` copies of the unit -> its index list must be the unit's list, shifted, `reps` times
    got = d_idx.cpu().numpy().view(np.uint32)[: out[-1][2]]
    ok = len(got) == reps * len(uidx)
    if ok:
        g = got.reshape(reps, len(uidx)).astype(np.int64) - (np.arange(reps, dtype=np.int64) * len(unit))[:, None]
        ok = bool((g == uidx.astype(np.int64)[None, :]).all())
    for shard_no, base, count, rescanned in out:
        ok = ok and base == shard_no * reps * len(uidx) and count == reps * len(uidx) and rescanned == 0
    ok = ok and total == nshards * reps * len(uidx)
    ok = _all_ok(torch, dist, dev, world, bool(ok))
    if rank == 0:
        nbytes = nshards * len(shard)
        line = _line(args, world, nbytes / (ms * 1e-3) / 1e9, ms,
                     {"workload": f"8 GB concatenated jsonexamples corpus (twitter/citm_catalog repeated), stage1 sharded across {world}xB200 with carry fixup (BASELINE.json configs[4])",
                      "bytes_total": int(nbytes), "shards": nshards, "shard_bytes": int(len(shard)), "passes_per_job": rounds, "structurals_total": int(total),
                      "bases": "64-bit: shard-relative uint32 indexes + uint64 base per shard (document_stream-inl.h L250)",
                      "api": "sjb200_stage1_sharded: exchange record stored by the scan kernel into every rank's window (CUDA IPC over NVLink)"},
                     {"parity": {"ok": ok, "against": "CPU oracle on one (twitter, citm) unit; every repetition of every shard compared with it, bases checked"},
                      "gpu_launches": int(steps * rounds), "roofline": _roofline(len(shard) + 4 * out[-1][2] + 12, kms, "scan4_kernel"),
                      "e2e": {"value": None, "unit": B.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "device-resident configuration"}})
        print(json.dumps(line), flush=True)
    comm.close()
    parser.close()
    return ok


# =============================================================================== --check: the multi-rank path on adversarial cuts
def run_check(args, rank, world, total=256 << 20):
    """ONE NDJSON buffer cut at arbitrary character boundaries (mid-row, mid-string): carry-in != 0, wrong speculations,
    second exchange round and re-scans, through the real plumbing (CUDA IPC windows; NCCL for the handles).  Every rank
    compares its base + indexes with the oracle's scan of the whole prefix.  With one process (no torchrun) the ranks run
    as threads of this process on one GPU."""
    torch, dist, sj, dev, local = _setup(rank, world)
    from simdjson_b200 import corpus, sharding
    O = B.oracle()
    port = O.Port()
    nranks = world if world > 1 else max(2, args.gpus if args.gpus > 1 else 4)
    doc = corpus.ndjson_rows(total)
    cuts = list(sharding.shard_cuts(doc, nranks))
    # every odd cut is moved INTO a string value (the first byte after an opening quote): the rank behind it speculates
    # "not in a string", is told otherwise in the first exchange round, re-scans and republishes in the second
    raw = doc.tobytes() if hasattr(doc, "tobytes") else bytes(doc)
    for k in range(1, nranks, 2):
        pos = cuts[k]
        for _ in range(64):
            hit = raw.find(b',"', pos)
            if hit < 0 or hit + 3 >= cuts[k + 1]:
                break
            cand = hit + 2
            row0 = raw.rfind(b"\n", 0, cand) + 1
            if B.raw_scan(O, port, doc[row0:cand], 0)[1] & 2:  # bit 1: in a string
                cuts[k] = cand
                break
            pos = hit + 1
    del raw
    report = {"ranks": nranks, "bytes": total, "cuts": "character boundaries (sjb200_shard_cut), every odd cut moved inside a string value", "processes": world}

    def verify(r, res, got):
        want_all, state_before = B.raw_scan(O, port, doc[: cuts[r]], 0) if r else (np.zeros(0, np.uint32), 0)
        widx, _ = B.raw_scan(O, port, doc[cuts[r]: cuts[r + 1]], state_before)
        return (res.state_in == state_before and res.base == len(want_all) and res.count == len(widx) and np.array_equal(got[: res.count], widx)
                and res.rescanned == (1 if state_before else 0)), int(res.rescanned), int(state_before)

    if world > 1:
        rc, parser = sj.get_active_implementation(local).create_dom_parser_implementation(cuts[rank + 1] - cuts[rank])
        comm = _connect(torch, dist, sharding, parser, rank, world, dev)
        d = torch.from_numpy(np.ascontiguousarray(doc[cuts[rank]: cuts[rank + 1]])).to(dev)
        d_idx = torch.empty(int(sj.lib().sjb200_index_words(d.numel())), dtype=torch.int32, device=dev)
        rcs, res = comm.scan(d, d_idx, rank == world - 1)
        torch.cuda.synchronize()
        ok, resc, st = verify(rank, res, d_idx.cpu().numpy().view(np.uint32)) if rcs == 0 else (False, 0, 0)
        info = torch.tensor([resc, st], dtype=torch.int64, device=dev)
        allinfo = torch.empty(2 * world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allinfo, info)
        ok = _all_ok(torch, dist, dev, world, ok)
        report.update({"rescans": int(allinfo.view(world, 2)[:, 0].sum().item()), "states_in": [int(x) for x in allinfo.view(world, 2)[:, 1].cpu()]})
        comm.close()
        parser.close()
    else:
        parsers, comms = [], []
        for r in range(nranks):
            rc, p = sj.get_active_implementation(local).create_dom_parser_implementation(cuts[r + 1] - cuts[r])
            parsers.append(p)
            comms.append(sharding.Comm(p, r, nranks))
        sharding.Comm.connect_local(comms)
        outs = [None] * nranks

        def work(r):
            torch.cuda.set_device(local)
            d = torch.from_numpy(np.ascontiguousarray(doc[cuts[r]: cuts[r + 1]])).to(dev)
            d_idx = torch.empty(int(sj.lib().sjb200_index_words(d.numel())), dtype=torch.int32, device=dev)
            rcs, res = comms[r].scan(d, d_idx, r == nranks - 1, torch.cuda.Stream(device=dev))
            torch.cuda.synchronize()
            outs[r] = verify(r, res, d_idx.cpu().numpy().view(np.uint32)) if rcs == 0 else (False, 0, 0)
        th = [threading.Thread(target=work, args=(r,)) for r in range(nranks)]
        [t.start() for t in th]
        [t.join() for t in th]
        ok = all(o is not None and o[0] for o in outs)
        report.update({"rescans": sum(o[1] for o in outs if o), "states_in": [o[2] for o in outs if o]})
        for c in comms:
            c.close()
        for p in parsers:
            p.close()
    if rank == 0:
        report["ok"] = bool(ok)
        print(json.dumps({"check": "sharded stage 1, carry-in != 0 (BASELINE.json configs[2] cut mid-row)", "result": report}), flush=True)
    return ok


def run(args, rank, world):
    import torch.distributed as dist
    t0 = time.time()
    if args.check:
        ok = run_check(args, rank, world)
    elif args.config == "jsonexamples":
        ok = run_jsonexamples(args, rank, world)
    elif args.config == "ndjson_1g":
        ok = run_ndjson(args, rank, world)
    elif args.config == "utf8_minify_256m":
        ok = run_utf8_minify(args, rank, world)
    elif args.config == "tokens_64m":
        ok = run_tokens(args, rank, world)
    else:
        ok = run_concat(args, rank, world)
    _ = t0
    if world > 1 and dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        sys.exit(1)
