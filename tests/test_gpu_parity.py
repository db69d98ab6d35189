"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle
(oracle/libsj_oracle.so, pinned to the reference by test_oracle_pinning.py) and against the
committed golden vectors the reference itself produced.  Bar: bit-exact error code,
n_structural_indexes and the (n+3) index words; minified bytes; UTF-8 verdict."""
import hashlib
import json
import os
import random
import threading

import numpy as np
import torch
import pytest

import oracle_lib as O
import simdjson_b200 as sj
from simdjson_b200 import corpus

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
TILE = 32768


@pytest.fixture(scope="module")
def port():
    return O.Port()


@pytest.fixture(scope="module")
def parser():
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(8 << 20)
    assert rc == sj.SUCCESS, sj.ERROR_NAMES.get(rc, rc)
    yield p
    p.close()


def _load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def run_stage1(p, buf, mode):
    """host-pointer call; returns an oracle_lib.Stage1Result-alike"""
    p.n_structural_indexes = O.N_SENTINEL
    err = p.stage1(buf, mode)
    return O.Stage1Result(err, p.n_structural_indexes, p.structural_indexes)


def assert_same(got, want, ctx=None):
    assert got.err == want.err, (ctx, got.err, want.err, got.n, want.n)
    assert got.n == want.n, (ctx, got.err, got.n, want.n)
    if want.wrote:
        a, b = got.words(), want.words()
        if not np.array_equal(a, b):
            k = int(np.argmax(a != b))
            raise AssertionError((ctx, "first differing word", k, a[max(0, k - 3):k + 4], b[max(0, k - 3):k + 4]))


# --------------------------------------------------------------------------- golden vectors
def test_golden_stage1(parser):
    for c in _load("stage1.json")["cases"]:
        r = run_stage1(parser, bytes.fromhex(c["hex"]), c["mode"])
        assert r.err == c["err"], c
        if c["n"] is None:
            assert r.n == O.N_SENTINEL, c
        else:
            assert r.n == c["n"], c
            assert [int(x) for x in r.words()] == c["words"], c


def test_golden_minify_and_utf8(parser):
    impl = sj.get_active_implementation()
    for c in _load("minify.json")["cases"]:
        err, out = impl.minify(bytes.fromhex(c["hex"]))
        assert (err, bytes(out).hex()) == (c["err"], c["out"]), c
    for c in _load("utf8.json")["cases"]:
        assert impl.validate_utf8(bytes.fromhex(c["hex"])) == c["valid"], c


def test_golden_corpora(parser):
    import torch
    impl = sj.get_active_implementation()
    for f in _load("corpora.json")["files"]:
        data = np.frombuffer(O.jsonexample(f["file"]), dtype=np.uint8).copy()
        r = run_stage1(parser, data, f["mode"])
        assert (r.err, r.n) == (f["err"], f["n"]), f["file"]
        assert hashlib.sha256(r.words().tobytes()).hexdigest() == f["idx_sha256"], f["file"]
        # device-resident call gives the same array
        d = torch.from_numpy(data).cuda()
        parser.n_structural_indexes = O.N_SENTINEL
        rc = parser.stage1_device(d, f["mode"])
        got = parser.device_index_buffer().cpu().numpy().view(np.uint32)
        assert (rc, parser.n_structural_indexes) == (f["err"], f["n"])
        assert hashlib.sha256(got[: f["n"] + 3].tobytes()).hexdigest() == f["idx_sha256"], f["file"]
        err, out = impl.minify(data)
        assert (err, len(out), hashlib.sha256(bytes(out)).hexdigest()) == (f["minify_err"], f["minify_len"], f["minify_sha256"])
        assert impl.validate_utf8(data) == f["utf8"]


# --------------------------------------------------------------------------- seeded fuzz vs the oracle
def _fuzz_inputs(rng, n):
    for i in range(n):
        kind = i % 4
        if kind == 0:
            yield corpus.adversarial(rng), rng.choice(O.ALL_MODES)
        elif kind == 1:
            yield corpus.multi_document(rng), rng.choice([1, 2])
        elif kind == 2:
            yield b"\x1e" + corpus.multi_document(rng, sep=b"\x1e"), rng.choice([3, 4])
        else:
            yield corpus.multi_document(rng, sep=b","), rng.choice([5, 6])


@pytest.mark.parametrize("use_tma", [1, 0])
def test_fuzz_small_all_modes(parser, port, use_tma):
    parser.set_option("use_tma", use_tma)
    try:
        rng = random.Random(corpus.SEED + use_tma)
        impl = sj.get_active_implementation()
        for k, (b, mode) in enumerate(_fuzz_inputs(rng, 1500)):
            assert_same(run_stage1(parser, b, mode), port.stage1(b, mode), (b, mode))
            if k % 4 == 0:
                err, out = impl.minify(b)
                assert (err, bytes(out)) == port.minify(b), b
                assert impl.validate_utf8(b) == port.validate_utf8(b), b
    finally:
        parser.set_option("use_tma", 1)


def _big_adversarial(rng, nbytes):
    """many adversarial snippets, with backslash runs and quotes planted on lane / warp / tile boundaries"""
    out = bytearray()
    while len(out) < nbytes:
        out += corpus.adversarial(rng, 900)
    out = out[:nbytes]
    for boundary in range(128, nbytes - 300, 128):
        r = rng.random()
        if boundary % TILE == 0 or boundary % 4096 == 0 or r < 0.05:
            run = rng.choice([1, 2, 3, 5, 127, 128, 129, 255, 256, 4095, 4096, 4097])
            if rng.random() < 0.7:
                run = rng.choice([1, 2, 3, 4, 5])
            start = max(0, boundary - rng.randint(0, run))
            out[start:start + run] = b"\\" * run
            if rng.random() < 0.7:
                out[start + run:start + run + 1] = b'"'
        elif r < 0.10:
            s = rng.choice([b"\xe2\x82\xac", b"\xf0\x9f\x98\x80", b"\xc3\xa9", b"\xf0\x9f\x98", b"\xe2\x82"])
            at = boundary - rng.randint(0, len(s))
            out[at:at + len(s)] = s
    return bytes(out[:nbytes])


@pytest.mark.parametrize("use_tma", [1, 0])
def test_fuzz_multi_tile(parser, port, use_tma):
    """documents of several 64 KiB elements: tickets, look-back chain, emit pipeline"""
    parser.set_option("use_tma", use_tma)
    try:
        rng = random.Random(corpus.SEED ^ 0x77 ^ use_tma)
        impl = sj.get_active_implementation()
        sizes = [TILE - 1, TILE, TILE + 1, 2 * TILE, 3 * TILE + 17, 5 * TILE - 128, 9 * TILE + 4095, 40 * TILE + 1, 64 * TILE]
        for n in sizes:
            for rep in range(3):
                b = _big_adversarial(rng, n)
                for mode in (0, 2):
                    assert_same(run_stage1(parser, b, mode), port.stage1(b, mode), (n, rep, mode))
                err, out = impl.minify(b)
                werr, wout = port.minify(b)
                assert err == werr and bytes(out) == wout, (n, rep)
                assert impl.validate_utf8(b) == port.validate_utf8(b), (n, rep)
    finally:
        parser.set_option("use_tma", 1)


def test_stage1_sizes_across_the_pipeline(port):
    """sizes from one partial block to more elements than one wave of CTAs holds, so that the ticket and summary rings
    wrap and the emit pipeline drains: host-pointer calls in two modes, one large device-resident call"""
    rc, parser = sj.get_active_implementation().create_dom_parser_implementation(32 << 20)
    assert rc == sj.SUCCESS
    try:
        rng = random.Random(corpus.SEED ^ 0x4D)
        sizes = [1, 4095, 4096, 4097, TILE, TILE + 1, 2 * TILE, 2 * TILE + 1, 7 * TILE + 4100, 300 * TILE + 77]
        for n in sizes:
            b = _big_adversarial(rng, n) if n < (8 << 20) else (_big_adversarial(rng, 1 << 20) * 32)[:n]
            for mode in (0, 2):
                assert_same(run_stage1(parser, b, mode), port.stage1(b, mode), (n, mode))
        doc = corpus.random_json(20 << 20)
        d = torch.from_numpy(doc.copy()).cuda()
        want = port.stage1(doc, 0)
        rc = parser.stage1_device(d, 0)
        got = parser.device_index_buffer().cpu().numpy().view(np.uint32)
        assert rc == want.err and parser.n_structural_indexes == want.n
        assert np.array_equal(got[: want.n + 3], want.words())
    finally:
        parser.close()


def test_emit_warp_kernel_for_large_launches(port):
    """launches of at least `ew_min_bytes` run the emit-warp build of the stage-1 kernel (sjb200_kernels_ew.cu: scan warps
    never emit, the masks wait in an L2-resident ring): same index arrays, all modes' scans, ring wrap (more elements per
    CTA than the ring holds), partial last block, streaming mode, and back to the default kernel on the same context"""
    rc, parser = sj.get_active_implementation().create_dom_parser_implementation(48 << 20)
    assert rc == sj.SUCCESS
    try:
        parser.set_option("ew_min_bytes", 64 << 10)
        rng = random.Random(corpus.SEED ^ 0xE3)
        before = parser.get_stat("ew_launches")
        for n, mode in [(2 * TILE, 0), (2 * TILE + 1, 0), (9 * TILE + 4100, 2), (40 << 20, 0), ((40 << 20) - 4097, 2)]:
            doc = np.frombuffer((_big_adversarial(rng, 1 << 20) * 41)[:n], dtype=np.uint8) if n > (8 << 20) else np.frombuffer(_big_adversarial(rng, n), dtype=np.uint8)
            d = torch.from_numpy(doc.copy()).cuda()
            want = port.stage1(doc.tobytes(), mode)
            parser.n_structural_indexes = O.N_SENTINEL
            rc = parser.stage1_device(d, mode)
            got = O.Stage1Result(rc, parser.n_structural_indexes, parser.device_index_buffer().cpu().numpy().view(np.uint32))
            assert_same(got, want, (n, mode))
        assert parser.get_stat("ew_launches") >= before + 5
        parser.set_option("ew_min_bytes", 0)
        doc = corpus.random_json(20 << 20)
        d = torch.from_numpy(doc.copy()).cuda()
        want = port.stage1(doc, 0)
        mid = parser.get_stat("ew_launches")
        rc = parser.stage1_device(d, 0)
        got = parser.device_index_buffer().cpu().numpy().view(np.uint32)
        assert rc == want.err and parser.n_structural_indexes == want.n and np.array_equal(got[: want.n + 3], want.words())
        assert parser.get_stat("ew_launches") == mid
    finally:
        parser.close()


def test_minify_sizes_and_alignments(port):
    """minify (scan4 structure: kept bytes compacted per block, output as aligned 16-byte vectors) over the same range of
    sizes, and with the device destination at every alignment class"""
    rc, parser = sj.get_active_implementation().create_dom_parser_implementation(32 << 20)
    assert rc == sj.SUCCESS
    try:
        rng = random.Random(corpus.SEED ^ 0x3141)
        for n in [1, 127, 4095, 4096, 4097, 2 * TILE, 2 * TILE + 1, 7 * TILE + 4100, 300 * TILE + 77]:
            b = _big_adversarial(rng, n)
            err, out = parser._minify_host(b)
            werr, wout = port.minify(b)
            assert err == werr and bytes(out) == wout, n
        doc = corpus.random_json(20 << 20, pretty_bias=0.8, utf8_rate=0.15)
        d = torch.from_numpy(doc.copy()).cuda()
        dst = torch.empty(len(doc) + 16, dtype=torch.uint8, device="cuda")
        for shift in (0, 1, 7):  # destination alignment
            rcm, dl = parser.minify_device(d, dst[shift:])
            werr, wout = port.minify(doc)
            assert rcm == werr and dl == len(wout) and bytes(dst[shift:shift + dl].cpu().numpy()) == wout, shift
    finally:
        parser.close()


def test_valid_documents_and_streams(parser, port):
    impl = sj.get_active_implementation()
    d = corpus.random_json(3 * (1 << 20) + 12345)
    assert_same(run_stage1(parser, d, 0), port.stage1(d, 0))
    err, out = impl.minify(d)
    werr, wout = port.minify(d)
    assert err == werr == 0 and bytes(out) == wout
    nd = corpus.ndjson_rows(2 << 20)
    for mode in (1, 2):
        assert_same(run_stage1(parser, nd, mode), port.stage1(nd, mode))
    cut = nd[: (1 << 20) + 123]  # mid-row: streaming_partial must stop at the last complete row
    r = run_stage1(parser, cut, 1)
    assert_same(r, port.stage1(cut, 1))
    assert r.err == 0 and r.idx[r.n] < len(cut)
    u = corpus.random_utf8(1 << 20)
    assert impl.validate_utf8(u)
    for pos in (0, 1, len(u) // 2, 32767, 32768, len(u) - 2, len(u) - 1):
        v = u.copy()
        v[pos] = 0xFF
        assert not impl.validate_utf8(v), pos
    t = u.copy()  # truncated sequence exactly at the end of the input
    t[-3:] = np.frombuffer(b"\xf0\x9f\x98", dtype=np.uint8)
    assert impl.validate_utf8(t) == port.validate_utf8(t) is False


def test_capacity_and_empty(parser, port):
    doc = b'{"a":[1,2,3]}'
    rc, small = sj.get_active_implementation().create_dom_parser_implementation(8)
    assert rc == 0
    small.n_structural_indexes = 77
    assert small.stage1(doc, 0) == sj.CAPACITY and small.n_structural_indexes == 77  # untouched, like the reference
    assert small.stage1(b"", 0) == sj.EMPTY and small.n_structural_indexes == 77
    assert small.set_capacity(1 << 33) == sj.CAPACITY
    assert small.set_capacity(64) == 0 and small.stage1(doc, 0) == 0
    small.close()
    for b in (b" ", b"   \n\t ", b'"', b'"abc', b'["a\x01b"]', b'["a\xffb"]', b"\xe2\x82", b"\\"):
        for mode in O.ALL_MODES:
            assert_same(run_stage1(parser, b, mode), port.stage1(b, mode), (b, mode))


# --------------------------------------------------------------------------- entry-point variants
def test_device_resident_matches_host_path(parser, port):
    import torch
    rng = random.Random(99)
    for n in (1, 63, 64, 65, 4097, TILE + 5, 7 * TILE + 1234):
        b = _big_adversarial(rng, max(n, 400))[:n]
        for mode in (0, 1, 2, 3, 6):
            want = port.stage1(b, mode)
            d = torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()).cuda()
            parser.n_structural_indexes = O.N_SENTINEL
            rc = parser.stage1_device(d, mode)
            got = O.Stage1Result(rc, parser.n_structural_indexes, parser.device_index_buffer().cpu().numpy().view(np.uint32))
            assert_same(got, want, (n, mode))
        # minify / utf8 device entry points
        d = torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()).cuda()
        dst = torch.empty(max(n, 1), dtype=torch.uint8, device="cuda")
        rc, dl = parser.minify_device(d, dst)
        werr, wout = port.minify(b)
        assert rc == werr and bytes(dst[:dl].cpu().numpy()) == wout
        assert parser.validate_utf8_device(d) == int(port.validate_utf8(b))


def test_batch_entry_point(parser, port):
    """sjb200_stage1_dev_batch == a loop of sjb200_stage1_dev"""
    import torch
    rng = random.Random(77)
    docs = [_big_adversarial(rng, n) for n in (100, TILE + 3, 5 * TILE, 17, 9 * TILE + 4000)] + [b'{"a":1} [1,2', b"", b'"open']
    for mode in (0, 1, 2):
        d_bufs = [torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()).cuda() if len(b) else torch.empty(0, dtype=torch.uint8, device="cuda") for b in docs]
        d_idxs = [torch.zeros(sj.lib().sjb200_index_words(max(len(b), 1)), dtype=torch.int32, device="cuda") for b in docs]
        res = parser.stage1_device_batch(d_bufs, d_idxs, mode)
        for b, (err, n), di in zip(docs, res, d_idxs):
            want = port.stage1(b, mode)
            assert err == want.err, (len(b), mode, err, want.err)
            if want.wrote:
                assert n == want.n
                assert np.array_equal(di.cpu().numpy().view(np.uint32)[: n + 3], want.words()), (len(b), mode)


def test_unaligned_device_pointer(parser, port):
    """a device buffer that is not 16-byte aligned cannot use TMA; the plain-load path must agree"""
    import torch
    b = np.frombuffer(_big_adversarial(random.Random(5), 3 * TILE + 100), dtype=np.uint8)
    base = torch.zeros(len(b) + 64, dtype=torch.uint8, device="cuda")
    for off in (1, 3, 8, 13):
        view = base[off: off + len(b)]
        view.copy_(torch.from_numpy(b.copy()))
        want = port.stage1(b, 0)
        parser.n_structural_indexes = O.N_SENTINEL
        rc = parser.stage1_device(view, 0)
        got = O.Stage1Result(rc, parser.n_structural_indexes, parser.device_index_buffer().cpu().numpy().view(np.uint32))
        assert_same(got, want, off)
        assert parser.validate_utf8_device(view) == int(port.validate_utf8(b))


def test_chunked_host_pipeline_carries(port):
    """host path with tiny chunks: every chunk boundary exercises the carry hand-off between launches"""
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(1 << 20)
    assert rc == 0
    rng = random.Random(1234)
    for chunk in (TILE, 2 * TILE, 8 * TILE):
        p.set_option("chunk_bytes", chunk)
        b = _big_adversarial(rng, 11 * TILE + 77)
        for mode in (0, 2):
            assert_same(run_stage1(p, b, mode), port.stage1(b, mode), (chunk, mode))
        err, out = p._minify_host(b)
        werr, wout = port.minify(b)
        assert err == werr and bytes(out) == wout, chunk
        assert p._validate_utf8_host(b) == port.validate_utf8(b), chunk
    p.close()


def test_sharded_scan_matches_single_scan(port):
    """section 8(e): byte-range shards + a fold of 6-bit transducers == one scan of the whole buffer"""
    import torch
    L = sj.lib()
    rng = random.Random(4242)
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(4 << 20)
    assert rc == 0
    docs = [np.frombuffer(_big_adversarial(rng, 6 * TILE + 999), dtype=np.uint8), corpus.random_json(1 << 20), corpus.ndjson_rows(1 << 20)]
    for doc in docs:
        want = port.stage1(doc, 2)  # streaming_final tolerates an unclosed tail; gives the raw structurals
        raw_n = int(np.count_nonzero(want.idx[: want.n] < 2**32)) if want.wrote else 0
        for nshards in (2, 3, 8):
            cuts = [0]
            for k in range(1, nshards):
                nominal = (len(doc) * k) // nshards
                cuts.append(int(L.sjb200_shard_cut(doc.ctypes.data, len(doc), nominal)))
            cuts.append(len(doc))
            shards = [doc[cuts[k]: cuts[k + 1]] for k in range(nshards)]
            tts, counts, idxs, flags = [], [], [], 0
            for k, sh in enumerate(shards):
                d = torch.from_numpy(sh.copy()).cuda()
                rc, res = p.stage1_shard_device(d, 0, k == nshards - 1)
                assert rc == 0
                tts.append(res.ttable)
                import ctypes as C
                state_in = L.sjb200_fold_state((C.c_uint32 * len(tts))(*tts), k)
                if state_in != 0:  # speculation was wrong for this shard: scan again with the true state
                    rc, res = p.stage1_shard_device(d, state_in, k == nshards - 1)
                    assert rc == 0 and res.ttable == tts[-1]
                counts.append(res.count)
                flags |= res.flags
                idxs.append(p.device_index_buffer().cpu().numpy().view(np.uint32)[: res.count].astype(np.int64) + cuts[k])
            allidx = np.concatenate(idxs) if idxs else np.zeros(0, np.int64)
            # compare with the single-scan raw structural list (before the streaming fix-ups trimmed the tail)
            single = port.stage1(doc, 0)
            if single.err in (0, sj.UTF8_ERROR, sj.EMPTY) and single.wrote:
                assert len(allidx) == single.n and np.array_equal(allidx, single.idx[: single.n].astype(np.int64)), nshards
                assert bool(flags & 1) == (not port.validate_utf8(doc))
            _ = raw_n
    p.close()


def test_two_parsers_in_two_threads(port):
    """document_stream's stage-1 worker runs a second parser concurrently (dom/document_stream-inl.h L16-85)"""
    impl = sj.get_active_implementation()
    docs = [bytes(corpus.random_json(700000 + 4096 * k, seed=k)) for k in range(2)]
    wants = [port.stage1(d, 0) for d in docs]
    errors = []

    def work(k):
        try:
            rc, p = impl.create_dom_parser_implementation(1 << 20)
            assert rc == 0
            for _ in range(20):
                assert_same(run_stage1(p, docs[k], 0), wants[k], k)
            p.close()
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    th = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errors, errors


# --------------------------------------------------------------------------- BASELINE.json sizes
def test_config2_64mib_random_json(port):
    """configs[1]: synthetic 64 MiB random-structure JSON, stage1 on 1xB200 -- full array compared"""
    import torch
    doc = corpus.random_json(64 << 20)
    want = port.stage1(doc, 0)
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(len(doc))
    assert rc == 0
    d = torch.from_numpy(doc).cuda()
    rc = p.stage1_device(d, 0)
    got = p.device_index_buffer().cpu().numpy().view(np.uint32)
    assert rc == want.err == 0 and p.n_structural_indexes == want.n
    assert np.array_equal(got[: want.n + 3], want.words())
    # size-independent properties: strictly increasing, every index addresses a non-whitespace byte
    idx = got[: want.n].astype(np.int64)
    assert np.all(np.diff(idx) > 0)
    assert not np.any(np.isin(doc[idx], [0x20, 0x0A, 0x0D, 0x09]))
    # the host-pointer path (chunked H2D pipeline) agrees
    assert_same(run_stage1(p, doc, 0), want)
    # minify: idempotent and equal to the oracle
    dst = torch.empty(len(doc), dtype=torch.uint8, device="cuda")
    rc, dl = p.minify_device(d, dst)
    werr, wout = port.minify(doc)
    assert rc == werr == 0 and dl == len(wout)
    assert bytes(dst[:dl].cpu().numpy()) == wout
    dst2 = torch.empty(dl, dtype=torch.uint8, device="cuda")
    rc, dl2 = p.minify_device(dst[:dl].clone(), dst2)
    assert rc == 0 and dl2 == dl and torch.equal(dst2[:dl2], dst[:dl])
    p.close()


def test_config4_utf8_256mib(port):
    """configs[3]: validate_utf8 on 256 MiB mixed ASCII/UTF-8; valid -> true, three corrupted copies -> false"""
    import torch
    u = corpus.random_utf8(256 << 20)
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(0)
    assert rc == 0
    d = torch.from_numpy(u).cuda()
    assert p.validate_utf8_device(d) == 1
    for pos in (0, len(u) // 2 + 1, len(u) - 2):
        saved = int(d[pos])
        d[pos] = 0xFF
        assert p.validate_utf8_device(d) == 0, pos
        d[pos] = saved
    assert p.validate_utf8_device(d) == 1
    p.close()
    assert port.validate_utf8(u[: 1 << 20])


# --------------------------------------------------------------------------- host-pointer pipeline (every input / output path)
def test_host_pointer_paths(port):
    """sjb200_stage1 / _minify / _validate_utf8 with host buffers: pageable input through the staging ring (copy
    threads), through the driver, page-locked input; indexes stored by the kernel into the page-locked caller array or
    copied back chunk by chunk -- all bit-identical to the oracle (include/simdjson/internal/dom_parser_implementation.h L80)."""
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(40 << 20)
    assert rc == sj.SUCCESS
    try:
        rng = random.Random(corpus.SEED ^ 0x7077)
        docs = [corpus.random_json(n) for n in (100, (1 << 20) - 3, (5 << 20) + 17, (33 << 20) + 4099)]
        docs.append(_big_adversarial(rng, 3 * (1 << 20) + 333))
        want = [(port.stage1(d, 0), port.stage1(d, 2)) for d in docs]
        for threads, zero_copy, chunk in ((8, 1, 2 << 20), (3, 1, 1 << 20), (0, 1, 4 << 20), (5, 0, 2 << 20), (0, 0, 64 << 10)):
            p.set_option("copy_threads", threads)
            p.set_option("zero_copy_out", zero_copy)
            p.set_option("chunk_bytes", chunk)
            p.set_option("stage_min_bytes", 1 << 20)
            for d, (w0, w2) in zip(docs, want):
                assert_same(run_stage1(p, d, 0), w0, ("pageable", threads, zero_copy, len(d)))
                assert p.get_stat("input_path") == (1 if threads and len(d) >= (1 << 20) else 0)
                assert p.get_stat("output_path") == zero_copy
                assert_same(run_stage1(p, d, 2), w2, ("pageable streaming_final", threads, zero_copy, len(d)))
            pinned = torch.from_numpy(docs[2].copy()).pin_memory()
            assert_same(run_stage1(p, pinned.numpy(), 0), want[2][0], ("page-locked input", threads))
            assert p.get_stat("input_path") == 2
            # the same pipeline feeds minify and validate_utf8
            werr, wout = port.minify(docs[3])
            err, out = p._minify_host(docs[3])
            assert err == werr and bytes(out) == wout
            assert p._validate_utf8_host(docs[3]) == port.validate_utf8(docs[3])
            bad = docs[2].copy()
            bad[len(bad) - 70000] = 0xFF
            assert p._validate_utf8_host(bad) is False
            assert_same(run_stage1(p, bad, 0), port.stage1(bad, 0), ("invalid utf-8", threads))
    finally:
        p.close()


# --------------------------------------------------------------------------- sharded scan, exchange fused into the scan kernel
def _raw_scan(port, doc):
    """the oracle's raw structural list of a whole buffer (no finish() logic): what the shards together must reproduce"""
    import ctypes as C
    L = port.L
    L.sjo_scan_shard.restype = C.c_uint64
    L.sjo_scan_shard.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32)]
    idx = np.zeros(len(doc) + 1, dtype=np.uint32)
    so = C.c_uint32(0)
    n = L.sjo_scan_shard(doc.ctypes.data, len(doc), 0, idx.ctypes.data, C.byref(so))
    return idx[:n].astype(np.int64), int(so.value)


def _run_ranks_in_threads(doc, cuts, device=0):
    """one sjb200_comm per rank, all ranks in this process (connect_local), one thread per rank like one process per GPU"""
    from simdjson_b200 import sharding
    world = len(cuts) - 1
    impl = sj.get_active_implementation(device)
    parsers, comms = [], []
    for r in range(world):
        rc, p = impl.create_dom_parser_implementation(max(cuts[r + 1] - cuts[r], 64))
        assert rc == sj.SUCCESS
        parsers.append(p)
        comms.append(sharding.Comm(p, r, world))
    sharding.Comm.connect_local(comms)
    out = [None] * world

    def work(r):
        try:
            torch.cuda.set_device(device)
            shard = torch.from_numpy(doc[cuts[r]: cuts[r + 1]].copy()).cuda()
            d_idx = torch.empty(int(sj.lib().sjb200_index_words(shard.numel())), dtype=torch.int32, device="cuda")
            stream = torch.cuda.Stream()
            results = []
            for rep in range(3):  # several passes in flight: enqueue all, then finish all
                assert comms[r].enqueue(shard, d_idx, r == world - 1, stream) == 0
            for rep in range(3):
                rc, res = comms[r].finish()
                results.append((rc, res.count, res.base, res.total_count, res.state_in, res.final_state, res.flags_all, res.rescanned))
            torch.cuda.synchronize()
            idx = d_idx.cpu().numpy().view(np.uint32)[: results[-1][1]].astype(np.int64) + cuts[r]
            out[r] = (results, idx)
        except Exception as e:  # noqa: BLE001
            out[r] = e

    th = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    [t.start() for t in th]
    [t.join(timeout=300) for t in th]
    for c in comms:
        c.close()
    for p in parsers:
        p.close()
    for o in out:
        if isinstance(o, Exception) or o is None:
            raise AssertionError(o)
    return out


def test_sharded_scan_fused_exchange(port):
    """SURVEY.md 8(e) through sjb200_stage1_sharded: ONE buffer cut into 2 / 4 / 8 shards -- at arbitrary character
    boundaries (mid-row, mid-string: carry-in != 0, wrong speculations, second round) and at line feeds (the sharder's
    choice: no rank scans twice) -- every rank's base + indexes against one scan of the whole buffer by the oracle."""
    from simdjson_b200 import sharding
    rng = random.Random(corpus.SEED ^ 0x5a5a)
    docs = [corpus.ndjson_rows(24 << 20), corpus.random_json((6 << 20) + 4321, pretty_bias=0.9),
            np.frombuffer(_big_adversarial(rng, 9 * TILE + 777), dtype=np.uint8).copy()]
    for di, doc in enumerate(docs):
        want, want_state = _raw_scan(port, doc)
        utf8_ok = port.validate_utf8(doc)
        for world in (2, 4, 8):
            for mode, cuts in (("bytes", sharding.shard_cuts(doc, world)), ("lines", sharding.shard_cuts_at_lines(doc, world))):
                if any(cuts[k + 1] <= cuts[k] for k in range(world)):
                    continue
                out = _run_ranks_in_threads(doc, cuts)
                got = np.concatenate([o[1] for o in out])
                assert len(got) == len(want) and np.array_equal(got, want), (di, world, mode)
                base = 0
                for r, (results, idx) in enumerate(out):
                    for rc, count, b, total, state_in, final_state, flags_all, rescanned in results:
                        assert rc == 0 and b == base and total == len(want) and count == len(idx), (di, world, mode, r)
                        assert final_state == want_state and bool(flags_all & 1) == (not utf8_ok)
                        assert rescanned == (1 if state_in != 0 else 0)
                    base += len(idx)
                if mode == "lines" and di < 2:
                    assert all(res[7] == 0 for o in out for res in o[0]), "valid JSON cut after a line feed never needs a second scan"
        if di == 0:  # arbitrary cuts of NDJSON land inside strings: the second round really ran
            out = _run_ranks_in_threads(doc, sharding.shard_cuts(doc, 8))
            assert any(res[7] for o in out for res in o[0])


# --------------------------------------------------------------------------- streams of documents, epilogue on the device
def _doc_starts(doc, idx):
    """python restatement of the boundary predicate (find_next_document_index.h L60-88) applied to every structural"""
    role = {ord(":"): 1, ord(","): 1, ord("{"): 2, ord("}"): 3, ord("["): 4, ord("]"): 5}
    r = np.array([role.get(int(b), 0) for b in doc[idx]], dtype=np.int64) if len(idx) < 200000 else None
    if r is None:
        lut = np.zeros(256, dtype=np.int64)
        for k, v in role.items():
            lut[k] = v
        r = lut[doc[idx]]
    cur, before = r[1:], r[:-1]
    start = ~np.isin(cur, (1, 3, 5)) & ~np.isin(before, (1, 2, 4))
    return np.concatenate([[0], np.nonzero(start)[0] + 1]) if len(idx) else np.zeros(0, np.int64)


def test_device_stream_epilogue_and_document_table(port):
    """streaming_partial / streaming_final with device-resident data: finish() incl. find_next_document_index runs on the
    device behind the scan (sjb200_docs.cu) -- same n, same sentinel words, same error code as the oracle; the document
    boundary table lists every document start in stream order (SURVEY.md 8(f) rows 1-2)."""
    import ctypes as C
    rng = random.Random(corpus.SEED ^ 0xd0c5)
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(8 << 20)
    assert rc == sj.SUCCESS
    try:
        inputs = [corpus.multi_document(rng) for _ in range(60)]
        inputs += [corpus.adversarial(rng) for _ in range(40)]
        inputs += [bytes(corpus.ndjson_rows(3 << 20)), bytes(corpus.ndjson_rows(3 << 20))[:-777], b"[1,2,3]  {\"a\":1} [1,2  ", b"{\"a\":[1,2", b"   ", b"1 2 3",
                   bytes(corpus.tile_documents([b'{"k":[1,2,{"z":null}]}', b"[]", b"7", b'"s"'], 2 << 20)), b"\"unclosed", b"[1,2] \xe2\x82", b"\xe2\x82"]
        for b in inputs:
            a = np.frombuffer(bytes(b), dtype=np.uint8)
            if len(a) == 0:
                continue
            d = torch.from_numpy(a.copy()).cuda()
            for mode in (1, 2):
                want = port.stage1(a, mode)
                p.n_structural_indexes = O.N_SENTINEL
                rcd = p.stage1_device(d, mode)
                got = O.Stage1Result(rcd, p.n_structural_indexes, p.device_index_buffer().cpu().numpy().view(np.uint32))
                assert_same(got, want, ("device stream epilogue", mode, len(a), bytes(b[:40])))
        # RS-delimited (RFC 7464) and comma-delimited streams: the filters are device compactions of the index array
        for b, mode in _fuzz_inputs(rng, 600):
            a = np.frombuffer(bytes(b), dtype=np.uint8)
            if len(a) == 0 or mode < 3:
                continue
            d = torch.from_numpy(a.copy()).cuda()
            for md in ((3, 4) if mode in (3, 4) else (5, 6)):
                want = port.stage1(a, md)
                p.n_structural_indexes = O.N_SENTINEL
                rcd = p.stage1_device(d, md)
                got = O.Stage1Result(rcd, p.n_structural_indexes, p.device_index_buffer().cpu().numpy().view(np.uint32))
                assert_same(got, want, ("device filter", md, len(a), bytes(b[:60])))
        big_rs = b"\x1e" + b"\x1e".join(bytes(corpus.random_json(20000 + 977 * k, seed=k)) + b"\n" for k in range(40))
        big_comma = b",".join(bytes(corpus.random_json(20000 + 977 * k, seed=100 + k)) for k in range(40))
        for a, modes in ((np.frombuffer(big_rs, dtype=np.uint8), (3, 4)), (np.frombuffer(big_comma, dtype=np.uint8), (5, 6)),
                         (np.frombuffer(big_rs[:-5000], dtype=np.uint8), (3, 4)), (np.frombuffer(big_comma[:-5000], dtype=np.uint8), (5, 6))):
            d = torch.from_numpy(a.copy()).cuda()
            for md in modes:
                want = port.stage1(a, md)
                p.n_structural_indexes = O.N_SENTINEL
                rcd = p.stage1_device(d, md)
                got = O.Stage1Result(rcd, p.n_structural_indexes, p.device_index_buffer().cpu().numpy().view(np.uint32))
                assert_same(got, want, ("device filter, big", md, len(a)))
        # a batch of streams through one call (the tails of all documents are fetched together)
        docs = [np.frombuffer(bytes(corpus.multi_document(rng)), dtype=np.uint8) for _ in range(50)]
        d_bufs = [torch.from_numpy(x.copy()).cuda() for x in docs]
        d_idxs = [torch.empty(int(sj.lib().sjb200_index_words(len(x))), dtype=torch.int32, device="cuda") for x in docs]
        res = p.stage1_device_batch(d_bufs, d_idxs, 2)
        for x, di, (err, n) in zip(docs, d_idxs, res):
            want = port.stage1(x, 2)
            assert err == want.err and (not want.wrote or (n == want.n and np.array_equal(di.cpu().numpy().view(np.uint32)[: n + 3], want.words())))
        # the document table of a big NDJSON buffer and of mixed streams
        for doc in (corpus.ndjson_rows(5 << 20), np.frombuffer(bytes(corpus.tile_documents([b'{"k":[1,2,{"z":null}]}', b"[]", b"7", b'"s"', b"[[],{}]"], 1 << 20)), dtype=np.uint8)):
            d = torch.from_numpy(doc.copy()).cuda()
            assert p.stage1_device(d, 2) == 0
            n = p.n_structural_indexes
            idx = p.device_index_buffer().cpu().numpy().view(np.uint32)[:n].astype(np.int64)
            want_starts = _doc_starts(doc, idx)
            table = torch.zeros(2 * (len(want_starts) + 8), dtype=torch.int32, device="cuda")
            nd = C.c_uint32(0)
            rct = sj.lib().sjb200_document_table_dev(p._ctx, d.data_ptr(), p.device_index_buffer().data_ptr(), n, table.data_ptr(), len(want_starts) + 8, C.byref(nd), None)
            assert rct == 0 and nd.value == len(want_starts)
            t = table.cpu().numpy().view(np.uint32).reshape(-1, 2)[: nd.value]
            assert np.array_equal(t[:, 0], want_starts) and np.array_equal(t[:, 1], idx[want_starts])
            assert all(doc[b] in b'[{"0123456789-tfn' for b in t[:50, 1])
    finally:
        p.close()


# --------------------------------------------------------------------------- stage-2-lite (SURVEY.md 8(f) row 4)
def _tokens_on_device(p, doc):
    """stage 1 + sjb200_tokens_dev on a device-resident document; returns the oracle-shaped tuple"""
    a = np.frombuffer(bytes(doc), dtype=np.uint8)
    d = torch.from_numpy(a.copy()).cuda()
    rc = p.stage1_device(d, sj.REGULAR)
    return rc, d


def _tokens_tuple(res, d_type, d_payload, d_strbuf, cap):
    used = min(res.string_bytes, cap) if res.error != sj.CAPACITY else 0
    return (res.error, d_type.cpu().numpy(), d_payload.cpu().numpy().view(np.uint64), d_strbuf[:used].cpu().numpy(), res.string_bytes, res.n_strings,
            res.first_error_index)


def _same_tokens(got, want, ctx):
    assert got[0] == want[0], (ctx, got[0], want[0])
    assert bytes(got[1]) == bytes(want[1]), (ctx, "types")
    if not np.array_equal(got[2], want[2]):
        k = int(np.argmax(got[2] != want[2]))
        raise AssertionError((ctx, "payload", k, got[2][k], want[2][k], chr(want[1][k])))
    assert got[4:] == want[4:], (ctx, got[4:], want[4:])
    assert bytes(got[3]) == bytes(want[3]), (ctx, "string_buf")


def test_tokens_device_matches_oracle(port):
    import token_fuzz as TF
    rng = random.Random(corpus.SEED ^ 0x70c3)
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(32 << 20)
    assert rc == sj.SUCCESS
    try:
        docs = [bytes(corpus.random_json(rng.randrange(300, 300000), seed=5000 + i)) for i in range(8)]
        docs += [O.jsonexample(f) for f in ("twitter.json", "citm_catalog.json")]
        docs += [bytes(corpus.random_json(16 << 20, seed=31337)), b"[]", b"7", b'""', b'{"a":"b"}']
        for _ in range(40):  # documents of adversarial tokens: every scalar and string body the fuzzers produce, errors included
            parts = []
            for _ in range(rng.randrange(1, 3000)):
                if rng.random() < 0.5:
                    parts.append(b'"' + TF.string_body(rng)[0] + b'"')
                else:
                    tok = TF.scalar_token(rng)
                    if b'"' not in tok and b"\\" not in tok:
                        parts.append(tok)
            docs.append(b"[" + rng.choice([b",", b" ,\n ", b", "]).join(parts) + b"]")
        for _ in range(12):  # long strings (handled by whole warps): plain runs, dense escapes, at every phase of the 32-byte steps
            parts = [b'"' + TF.long_body(rng, rng.choice([90, 97, 200, 513, 3000, 40000]), rng.choice([0.0, 0.05, 0.3, 1.0])) + b'"' for _ in range(rng.randrange(1, 40))]
            parts += [b'"' + b"q" * rng.randrange(0, 200) + bad + b'tail"' for bad in (b"\\uD800", b"\\uDC00 ", b"\\u12", b"\\q")][: rng.randrange(0, 5)]
            rng.shuffle(parts)
            docs.append(b"[" + b" , ".join(parts) + b"]")
        docs.append(b'{"blob":"' + TF.long_body(rng, 3 << 20, 0.0) + b'","esc":"' + TF.long_body(rng, 1 << 20, 1.0) + b'"}')
        for k, doc in enumerate(docs):
            r = port.stage1(doc)
            assert r.err == 0
            rc, d = _tokens_on_device(p, doc)
            assert rc == 0 and p.n_structural_indexes == r.n
            want = port.tokens(doc, r.idx, r.n, strbuf_cap=sj.lib().sjb200_string_buf_capacity(len(doc)))
            for stage in ((1, 0) if k % 4 == 0 else (1,)):  # 0: the unstaged baseline path (every thread on global memory)
                p.set_option("tok_stage", stage)
                res, d_type, d_payload, d_strbuf = p.tokens_device(d)
                _same_tokens(_tokens_tuple(res, d_type, d_payload, d_strbuf, d_strbuf.numel()), want, ("doc", k, stage, doc[:60]))
            p.set_option("tok_stage", 1)
            if k < 4:  # unaligned document and string buffer: the staging falls back to byte copies
                du = torch.empty(len(doc) + 3, dtype=torch.uint8, device="cuda")[3:]
                du.copy_(d)
                assert p.stage1_device(du, sj.REGULAR) == 0
                cap = int(sj.lib().sjb200_string_buf_capacity(len(doc)))
                sb = torch.empty(cap + 5, dtype=torch.uint8, device="cuda")[5:]
                ty = torch.empty(r.n, dtype=torch.uint8, device="cuda")
                pl = torch.empty(r.n, dtype=torch.int64, device="cuda")
                import ctypes as C
                res2 = sj.capi.TokensResult()
                sj.lib().sjb200_tokens_dev(p._ctx, du.data_ptr(), len(doc), p.device_index_buffer().data_ptr(), r.n, ty.data_ptr(), pl.data_ptr(), sb.data_ptr(), cap,
                                           C.byref(res2), None)
                _same_tokens(_tokens_tuple(res2, ty, pl, sb, cap), want, ("unaligned", k))
        # too small a string buffer: CAPACITY, nothing written, payloads keep the lengths; and no structurals at all
        doc = docs[0]
        r = port.stage1(doc)
        rc, d = _tokens_on_device(p, doc)
        want = port.tokens(doc, r.idx, r.n, strbuf_cap=16)
        res, d_type, d_payload, d_strbuf = p.tokens_device(d, strbuf_capacity=16)
        assert res.error == sj.CAPACITY == want[0]
        _same_tokens(_tokens_tuple(res, d_type, d_payload, d_strbuf, 16), (want[0], want[1], want[2], b"", want[4], want[5], want[6]), "capacity")
        res, *_ = p.tokens_device(d, n=0)
        assert res.error == 0 and res.n_strings == 0 and res.string_bytes == 0 and res.first_error_index == 0xFFFFFFFF
    finally:
        p.close()


def test_tokens_device_matches_golden():
    """the string buffer and the tape types / payloads the reference itself produced (tests/golden/tokens.json)"""
    g = _load("tokens.json")
    rc, p = sj.get_active_implementation().create_dom_parser_implementation(4 << 20)
    assert rc == sj.SUCCESS
    try:
        for c in g["documents"]:
            doc = bytes.fromhex(c["doc"])
            rc, d = _tokens_on_device(p, doc)
            assert rc == 0
            res, d_type, d_payload, d_strbuf = p.tokens_device(d)
            assert res.error == c["err"] == 0
            types, pay = d_type.cpu().numpy(), d_payload.cpu().numpy().view(np.uint64)
            keep = [i for i, t in enumerate(types) if chr(t) not in ":,"]
            assert bytes(types[keep]) == c["types"].encode("latin1"), doc[:60]
            for i, v in c["payloads"].items():
                assert int(pay[keep][int(i)]) == int(v), (doc[:60], i)
            assert bytes(d_strbuf[: res.string_bytes].cpu().numpy()) == bytes.fromhex(c["string_buf"]), doc[:60]
        for c in g["scalars"]:
            doc = bytes.fromhex(c["doc"])
            rc, d = _tokens_on_device(p, doc)
            if rc != 0:
                assert rc == c["err"]
                continue
            res, d_type, d_payload, _sb = p.tokens_device(d)
            k = c["index"]
            if c["err"] == 0:
                assert res.error == 0 and chr(int(d_type[k])) == c["type"], doc
                if c["value"] is not None:
                    assert int(d_payload[k].cpu().numpy().view(np.uint64)) == int(c["value"]), doc
            else:
                assert int(d_type[k]) == 0 and int(d_payload[k]) == c["err"] == res.error and res.first_error_index == k, doc
        for f in g["files"]:
            doc = O.jsonexample(f["file"])
            rc, d = _tokens_on_device(p, doc)
            res, d_type, d_payload, d_strbuf = p.tokens_device(d)
            types, pay = d_type.cpu().numpy(), d_payload.cpu().numpy().view(np.uint64)
            keep = np.array([chr(t) not in ":," for t in types])
            t, pp = types[keep], pay[keep]
            assert res.error == 0 and len(t) == f["entries"] and hashlib.sha256(bytes(t)).hexdigest() == f["types_sha256"]
            assert hashlib.sha256(np.where(t == ord("d"), 0, pp).astype(np.uint64).tobytes()).hexdigest() == f["payloads_no_doubles_sha256"]
            assert res.string_bytes == f["string_buf_bytes"] and hashlib.sha256(bytes(d_strbuf[: res.string_bytes].cpu().numpy())).hexdigest() == f["string_buf_sha256"]
    finally:
        p.close()
