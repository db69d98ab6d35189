"""CPU check of the stage-2-lite per-token functions (simdjson_b200/csrc/sjb200_tokens.cuh, compiled for the host by
tests/tokens_emul.cpp in the kernels' tile decomposition) against the oracle.  The GPU run of the kernels themselves is
tests/test_gpu_parity.py::test_tokens_*."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import token_fuzz as TF
from simdjson_b200 import corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("tokemu") / "libtokemu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wall", "-I", os.path.join(ROOT, "simdjson_b200", "csrc"),
                           os.path.join(ROOT, "tests", "tokens_emul.cpp"), "-o", so])
    L = C.CDLL(so)
    L.emu_tokens.restype = C.c_int
    L.emu_tokens.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64),
                             C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    return L


def run_emu(L, doc, idx, n, cap=None):
    a = np.frombuffer(bytes(doc), dtype=np.uint8)
    ix = np.ascontiguousarray(idx[: max(n, 1)], dtype=np.uint32)
    types = np.zeros(max(n, 1), dtype=np.uint8)
    pay = np.zeros(max(n, 1), dtype=np.uint64)
    cap = (len(a) + 5 * n + 64) if cap is None else cap
    sb = np.zeros(max(cap, 1), dtype=np.uint8)
    sl, ns, fe = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0)
    err = L.emu_tokens(a.ctypes.data, len(a), ix.ctypes.data, n, types.ctypes.data, pay.ctypes.data, sb.ctypes.data, cap, C.byref(sl), C.byref(ns), C.byref(fe))
    return err, types[:n], pay[:n], sb[: min(sl.value, cap)], sl.value, ns.value, fe.value


def same(a, b):
    return a[0] == b[0] and bytes(a[1]) == bytes(b[1]) and np.array_equal(a[2], b[2]) and bytes(a[3]) == bytes(b[3]) and a[4:] == b[4:]


def test_token_functions_match_oracle(emu):
    port = O.Port()
    rng = random.Random(99)
    docs = [bytes(corpus.random_json(rng.randrange(300, 200000), seed=4000 + i)) for i in range(10)]
    docs += [O.jsonexample(f) for f in ("twitter.json", "citm_catalog.json")]
    # documents made of adversarial tokens: every scalar kind and string body the fuzzers produce, errors included
    for _ in range(60):
        parts = []
        for _ in range(rng.randrange(1, 400)):
            if rng.random() < 0.5:
                body, _bad = TF.string_body(rng)
                parts.append(b'"' + body + b'"')
            else:
                tok = TF.scalar_token(rng)
                if b'"' in tok or b"\\" in tok:
                    continue
                parts.append(tok)
        docs.append(b"[" + rng.choice([b",", b" ,\n ", b", "]).join(parts) + b"]")
    for _ in range(10):  # long strings: over the lane budget (handed to the warp on the GPU), tiles that do not fit the window
        parts = [b'"' + TF.long_body(rng, rng.choice([90, 97, 200, 513, 3000, 30000]), rng.choice([0.0, 0.05, 0.3, 1.0])) + b'"' for _ in range(rng.randrange(1, 30))]
        parts += [str(rng.randrange(10 ** 9)).encode() for _ in range(rng.randrange(0, 900))]
        rng.shuffle(parts)
        docs.append(b"[" + b" , ".join(parts) + b"]")
    for d in docs:
        r = port.stage1(d)
        assert r.err == 0
        want = port.tokens(d, r.idx, r.n)
        got = run_emu(emu, d, r.idx, r.n)
        assert same(got, want), d[:100]
    # tokens cut off by the end of the input, capacity
    for d in (b'["abc', b'[12', b'[tru', b'["\\u12', b'["\\ud800\\u', b"[-", b"[1e"):
        r = port.stage1(d, mode=O.STREAMING_PARTIAL)
        ix = np.array([1], dtype=np.uint32)
        assert same(run_emu(emu, d, ix, 1), port.tokens(d, ix, 1)), d
    d = docs[0]
    r = port.stage1(d)
    assert same(run_emu(emu, d, r.idx, r.n, cap=16), port.tokens(d, r.idx, r.n, strbuf_cap=16))


# ------------------------------------------------------------------ long strings by a whole warp (host SIMT emulation)
@pytest.fixture(scope="module")
def warp_emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("tokwarp") / "libtokwarp.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-I", os.path.join(ROOT, "simdjson_b200", "csrc"),
                           os.path.join(ROOT, "tests", "tokens_warp_emul.cpp"), "-o", so])
    L = C.CDLL(so)
    L.emu_warp_strings.restype = C.c_int
    L.emu_warp_strings.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
    return L


def test_warp_string_matches_oracle(warp_emu):
    port = O.Port()
    rng = random.Random(4242)
    cases = []  # (document bytes, position of the opening quote)
    for _ in range(120):
        body = TF.long_body(rng, rng.choice([0, 1, 30, 31, 32, 33, 64, 95, 96, 97, 200, 511, 512, 513, 1024, 3000, 9000]), rng.choice([0.0, 0.0, 0.05, 0.3, 1.0]))
        pre = b" " * rng.randrange(0, 40)
        cases.append((pre + b'"' + body + b'"' + b" ," * rng.randrange(0, 3), len(pre)))
    for _ in range(200):  # short adversarial bodies, bad escapes included, at every alignment of the 32-byte steps
        body, _bad = TF.string_body(rng, bad_rate=0.4, maxlen=rng.choice([80, 300]))
        pre = b"x" * rng.randrange(0, 33)
        cases.append((pre + b'"' + body + b'"', len(pre)))
    for bad in (b"\\uD800", b"\\uDC00", b"\\uD800\\uD800\\uDC00", b"\\uDBFF\\uDFFF\\uDC00", b"\\u12", b"\\q", b"\\ud83d\\n", b"\\ud83d\\ude00\\ude00"):
        for padn in (0, 5, 26, 27, 28, 29, 30, 31, 32, 60, 600):
            cases.append((b'"' + b"p" * padn + bad + b"tail" * 3 + b'"', 0))
    for cut in (b'"abc', b'"abc\\', b'"abc\\u12', b'"' + b"y" * 31 + b"\\", b'"' + b"y" * 600, b'"' + b"z" * 40 + b"\\ud83d\\ude", b'"\\'):  # the input ends first
        cases.append((cut, 0))
    doc = bytearray()
    pos = []
    for d, p in cases:
        pos.append(len(doc) + p)
        doc += d + b"\n"
    # strings that run to the very end of the buffer must be last: re-append the cut ones as separate buffers below
    a = np.frombuffer(bytes(doc), dtype=np.uint8)
    stride = 16384
    for win in ((0, 0), (1000, 7000)):
        posa = np.array(pos, dtype=np.uint64)
        lens = np.zeros(len(pos), dtype=np.int64)
        out = np.zeros(len(pos) * stride, dtype=np.uint8)
        assert warp_emu.emu_warp_strings(a.ctypes.data, len(a), posa.ctypes.data, len(pos), lens.ctypes.data, out.ctypes.data, stride, win[0], win[1]) == 0
        for k, p in enumerate(pos):
            wl, wb = port.parse_string(a, p)
            assert lens[k] == wl, (k, cases[k][0][:80], lens[k], wl)
            if wl > 0:
                assert bytes(out[k * stride: k * stride + wl]) == wb, (k, cases[k][0][:80])
    for cut in (b'"abc', b'"abc\\', b'"abc\\u12', b'"' + b"y" * 31 + b"\\", b'"' + b"y" * 63 + b"\\", b'"' + b"y" * 600, b'"' + b"z" * 40 + b"\\ud83d\\ude", b'"\\', b'"'):
        a2 = np.frombuffer(cut, dtype=np.uint8)
        posa = np.array([0], dtype=np.uint64)
        lens = np.zeros(1, dtype=np.int64)
        out = np.zeros(stride, dtype=np.uint8)
        assert warp_emu.emu_warp_strings(a2.ctypes.data, len(a2), posa.ctypes.data, 1, lens.ctypes.data, out.ctypes.data, stride, 0, 0) == 0
        assert lens[0] == port.parse_string(a2, 0)[0], (cut[:40], lens[0], port.parse_string(a2, 0)[0])
