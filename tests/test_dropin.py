"""Drop-in tests: the UNMODIFIED simdjson public API (dom::parser::parse / parse_many, ondemand::parser::iterate,
simdjson::minify, simdjson::validate_utf8) with the "b200" plug-in active must give what it gives with a CPU
implementation active.  The library under test is simdjson_b200/plugin/libsimdjson_b200.so (plug-in + the
reference compiled from /root/reference, built by __graft_entry__.build()); it travels to the GPU box prebuilt."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
from simdjson_b200 import corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLUGIN = os.path.join(ROOT, "simdjson_b200", "plugin", "libsimdjson_b200.so")
needs_plugin = pytest.mark.skipif(not os.path.exists(PLUGIN), reason="plug-in not built (needs the reference headers)")


class Harness:
    def __init__(self):
        L = C.CDLL(PLUGIN)
        u8, sz = C.c_void_p, C.c_size_t
        L.dropin_active_name.restype = C.c_char_p
        L.dropin_active_name.argtypes = [C.c_int]
        L.dropin_dom_roundtrip.restype = C.c_int
        L.dropin_dom_roundtrip.argtypes = [C.c_int, u8, sz, C.c_char_p, sz, C.POINTER(sz), C.POINTER(C.c_ulonglong)]
        L.dropin_parse_many.restype = C.c_long
        L.dropin_parse_many.argtypes = [C.c_int, u8, sz, sz, C.c_char_p, sz, C.POINTER(sz), C.POINTER(C.c_int), C.POINTER(C.c_ulonglong)]
        L.dropin_ondemand_roundtrip.restype = C.c_int
        L.dropin_ondemand_roundtrip.argtypes = [C.c_int, u8, sz, C.c_char_p, sz, C.POINTER(sz)]
        L.dropin_minify.restype = C.c_int
        L.dropin_minify.argtypes = [C.c_int, u8, sz, u8, C.POINTER(sz)]
        L.dropin_validate_utf8.restype = C.c_int
        L.dropin_validate_utf8.argtypes = [C.c_int, u8, sz]
        self.L = L

    @staticmethod
    def _buf(b):
        a = np.ascontiguousarray(np.frombuffer(bytes(b), dtype=np.uint8) if not isinstance(b, np.ndarray) else b)
        return a

    def dom(self, use_b200, b):
        a = self._buf(b)
        cap = 2 * len(a) + 64
        out = C.create_string_buffer(cap)
        ol, calls = C.c_size_t(0), C.c_ulonglong(0)
        err = self.L.dropin_dom_roundtrip(use_b200, a.ctypes.data, len(a), out, cap, C.byref(ol), C.byref(calls))
        return err, out.raw[: ol.value], calls.value

    def parse_many(self, use_b200, b, batch_size=1000000):
        a = self._buf(b)
        cap = 2 * len(a) + 64
        out = C.create_string_buffer(cap)
        ol, fe, calls = C.c_size_t(0), C.c_int(0), C.c_ulonglong(0)
        nd = self.L.dropin_parse_many(use_b200, a.ctypes.data, len(a), batch_size, out, cap, C.byref(ol), C.byref(fe), C.byref(calls))
        return nd, fe.value, out.raw[: ol.value], calls.value

    def ondemand(self, use_b200, b):
        a = self._buf(b)
        cap = 2 * len(a) + 64
        out = C.create_string_buffer(cap)
        ol = C.c_size_t(0)
        err = self.L.dropin_ondemand_roundtrip(use_b200, a.ctypes.data, len(a), out, cap, C.byref(ol))
        return err, out.raw[: ol.value]

    def minify(self, use_b200, b):
        a = self._buf(b)
        dst = np.zeros(len(a) + 64, dtype=np.uint8)
        dl = C.c_size_t(0)
        err = self.L.dropin_minify(use_b200, a.ctypes.data, len(a), dst.ctypes.data, C.byref(dl))
        return err, bytes(dst[: dl.value])

    def utf8(self, use_b200, b):
        a = self._buf(b)
        return bool(self.L.dropin_validate_utf8(use_b200, a.ctypes.data, len(a)))


@pytest.fixture(scope="module")
def h():
    return Harness()


def _corpora():
    docs = [b'{"a":[1,2,{"b":"c\\"d"}],"e":null,"u":"\xc3\xa9"}', bytes(corpus.random_json(200000, seed=3)), bytes(corpus.random_json(1 << 20, seed=4))]
    return docs + [O.jsonexample(name) for name in ("twitter.json", "citm_catalog.json")]


@needs_plugin
def test_plugin_loads_and_cpu_path_matches_reference(h):
    """no GPU needed: the harness with a CPU implementation active reproduces the reference build in oracle/_ref"""
    assert h.L.dropin_active_name(1) == b"b200"
    assert h.L.dropin_active_name(0) in (b"icelake", b"haswell", b"westmere", b"fallback")
    doc = _corpora()[1]
    err, out, calls = h.dom(0, doc)
    assert err == 0 and calls == 0
    if O.have_ref():
        rerr, rout = O.Ref("").dom_roundtrip(doc)
        assert (err, out) == (rerr, rout)


@needs_plugin
def test_plugin_fails_loudly_without_gpu(h):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    err, out, calls = h.dom(1, b"[1,2,3]")
    assert err == 16 and out == b""  # UNSUPPORTED_ARCHITECTURE: no silent CPU fallback
    assert h.utf8(1, b"abc") is False
    assert h.minify(1, b"[1, 2]")[0] == 16


@needs_plugin
@pytest.mark.gpu
def test_dom_parse_dropin(h):
    for doc in _corpora():
        cerr, cout, _ = h.dom(0, doc)
        gerr, gout, calls = h.dom(1, doc)
        assert (gerr, gout) == (cerr, cout)
        assert calls >= 1  # stage 1 really ran on the GPU
    for bad in (b'{"a":1', b'["a\x01b"]', b'["\xff"]', b"", b"   ", b'"abc', b"[1,2,,]"):
        assert h.dom(1, bad)[:2] == h.dom(0, bad)[:2], bad


@needs_plugin
@pytest.mark.gpu
def test_parse_many_dropin(h):
    amazon = O.jsonexample("amazon_cellphones.ndjson")
    streams = [bytes(corpus.ndjson_rows(600000, seed=9)), b'{"a":1} [1,2,3] "x" 12 {"b":[true,false]}  ', amazon]
    for s in streams:
        for batch in (4096, 100000, 1000000):
            c = h.parse_many(0, s, batch)
            g = h.parse_many(1, s, batch)
            assert g[:3] == c[:3], (len(s), batch, g[0], c[0], g[1], c[1])
            assert g[3] >= 1
    nd, fe, _, _ = h.parse_many(1, amazon)
    assert (nd, fe) == (793, 0)  # tests/dom/basictests.cpp L36, L692-708


@needs_plugin
@pytest.mark.gpu
def test_ondemand_minify_utf8_dropin(h):
    for doc in _corpora():
        assert h.ondemand(1, doc) == h.ondemand(0, doc)
        assert h.minify(1, doc) == h.minify(0, doc)
        assert h.utf8(1, doc) == h.utf8(0, doc) is True
    for s in (b'"', b'{"a" : 1 , "b":[ 1, 2 ,3 ] }', b"", b" ", b"\xff", b"\xe2\x82", b'"\\"  "  x'):
        assert h.minify(1, s) == h.minify(0, s), s
        assert h.utf8(1, s) == h.utf8(0, s), s


@needs_plugin
def test_force_implementation_by_name():
    """SIMDJSON_FORCE_IMPLEMENTATION=b200 selects the plug-in once its library is loaded (doc/implementation-selection.md;
    src/implementation.cpp L303 resolves the name against a static list an out-of-tree implementation cannot join, so the
    plug-in installs itself from a load-time constructor).  Needs no GPU: nothing is created."""
    import subprocess
    import sys
    code = ("import ctypes as C; L = C.CDLL(%r); L.dropin_default_active_name.restype = C.c_char_p; "
            "print(L.dropin_default_active_name().decode())" % PLUGIN)
    for env_value, want_b200 in (("b200", True), (None, False)):
        env = dict(os.environ)
        env.pop("SIMDJSON_FORCE_IMPLEMENTATION", None)
        if env_value:
            env["SIMDJSON_FORCE_IMPLEMENTATION"] = env_value
        out = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, text=True, timeout=120).stdout.strip()
        assert (out == "b200") == want_b200, (env_value, out)
