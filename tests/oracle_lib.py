"""ctypes bindings for the two CPU checkers under oracle/ (test infrastructure only).

  port : oracle/libsj_oracle.so    -- our byte-at-a-time C restatement (always built)
  ref  : oracle/_ref/libsj_ref.so  -- the unmodified reference compiled from its
                                      singleheader sources (may be absent)

and the reference's own sample documents (jsonexample), stored xz-compressed under tests/golden/jsonexamples/.
"""
import ctypes as C
import lzma
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
PORT_SO = os.path.join(ORACLE_DIR, "libsj_oracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libsj_ref.so")
JSONEXAMPLES = os.path.join(ROOT, "tests", "golden", "jsonexamples")


def jsonexample(name):
    """bytes of one of the reference's sample documents: twitter.json, citm_catalog.json, amazon_cellphones.ndjson"""
    with lzma.open(os.path.join(JSONEXAMPLES, name + ".xz")) as f:
        return f.read()

SUCCESS, CAPACITY, MEMALLOC, UTF8_ERROR, EMPTY, UNESCAPED_CHARS, UNCLOSED_STRING, UNEXPECTED_ERROR = 0, 1, 2, 11, 13, 14, 15, 24
REGULAR, STREAMING_PARTIAL, STREAMING_FINAL, JSON_SEQUENCE_PARTIAL, JSON_SEQUENCE_FINAL, COMMA_DELIMITED_PARTIAL, COMMA_DELIMITED_FINAL = range(7)
ALL_MODES = list(range(7))

# error codes after which the reference has written n_structural_indexes and the sentinels
# (json_structural_indexer.h L264-287): everything except the early returns.
N_SENTINEL = 0xDEADBEEF


def index_capacity(capacity):
    return ((capacity + 63) // 64) * 64 + 9


def _u8(buf):
    if isinstance(buf, (bytes, bytearray)):
        return np.frombuffer(bytes(buf), dtype=np.uint8)
    return np.ascontiguousarray(buf, dtype=np.uint8)


def _ptr(a, t=C.c_uint8):
    return a.ctypes.data_as(C.POINTER(t))


class Stage1Result:
    __slots__ = ("err", "n", "idx")

    def __init__(self, err, n, idx):
        self.err, self.n, self.idx = err, n, idx

    @property
    def wrote(self):
        """True when the call got far enough to store n and the sentinels."""
        return self.n != N_SENTINEL

    def words(self):
        """the (n+3) words the parity bar compares"""
        return self.idx[: self.n + 3]


def _build_port():
    if not os.path.exists(PORT_SO) or os.path.getmtime(PORT_SO) < os.path.getmtime(os.path.join(ORACLE_DIR, "sj_oracle.c")):
        subprocess.check_call(["make", "-C", ORACLE_DIR, os.path.join(ORACLE_DIR, "libsj_oracle.so")], stdout=subprocess.DEVNULL)


class Port:
    def __init__(self):
        _build_port()
        L = C.CDLL(PORT_SO)
        L.sjo_stage1.restype = C.c_int
        L.sjo_stage1.argtypes = [C.POINTER(C.c_uint8), C.c_size_t, C.c_size_t, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.sjo_minify.restype = C.c_int
        L.sjo_minify.argtypes = [C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_uint8), C.POINTER(C.c_size_t)]
        L.sjo_validate_utf8.restype = C.c_int
        L.sjo_validate_utf8.argtypes = [C.POINTER(C.c_uint8), C.c_size_t]
        L.sjo_trim_partial_utf8.restype = C.c_size_t
        L.sjo_trim_partial_utf8.argtypes = [C.POINTER(C.c_uint8), C.c_size_t]
        L.sjo_tokens.restype = C.c_int
        L.sjo_tokens.argtypes = [C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_uint32), C.c_uint32, C.POINTER(C.c_uint8), C.POINTER(C.c_uint64),
                                 C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.sjo_parse_string.restype = C.c_long
        L.sjo_parse_string.argtypes = [C.POINTER(C.c_uint8), C.c_size_t, C.c_size_t, C.POINTER(C.c_uint8)]
        self.L = L
        self.name = "port"

    def tokens(self, buf, idx, n, strbuf_cap=None):
        """stage-2-lite: (err, types[n], payloads[n], string_buf bytes, n_strings, first_error_index)"""
        a = _u8(buf)
        ix = np.ascontiguousarray(idx[:n], dtype=np.uint32) if n else np.zeros(1, dtype=np.uint32)
        types = np.zeros(max(n, 1), dtype=np.uint8)
        pay = np.zeros(max(n, 1), dtype=np.uint64)
        cap = (len(a) + 5 * n + 64) if strbuf_cap is None else strbuf_cap
        sb = np.zeros(max(cap, 1), dtype=np.uint8)
        sl, ns, fe = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0)
        err = self.L.sjo_tokens(_ptr(a), len(a), _ptr(ix, C.c_uint32), n, _ptr(types), _ptr(pay, C.c_uint64), _ptr(sb), cap, C.byref(sl), C.byref(ns), C.byref(fe))
        return err, types[:n], pay[:n], sb[: min(sl.value, cap)], sl.value, ns.value, fe.value

    def parse_string(self, buf, pos=0):
        """the string whose opening quote is at buf[pos]: (length or -1 / -2, bytes)"""
        a = _u8(buf)
        dst = np.zeros(len(a) + 8, dtype=np.uint8)
        r = self.L.sjo_parse_string(_ptr(a), len(a), pos, _ptr(dst))
        return r, bytes(dst[: max(r, 0)])

    def stage1(self, buf, mode=REGULAR, capacity=None):
        a = _u8(buf)
        n = len(a)
        cap = n if capacity is None else capacity
        idx = np.zeros(index_capacity(max(cap, n)), dtype=np.uint32)
        nn = C.c_uint32(N_SENTINEL)
        pa = _ptr(a) if n else C.cast(C.c_void_p(0), C.POINTER(C.c_uint8))
        err = self.L.sjo_stage1(pa, n, cap, mode, _ptr(idx, C.c_uint32), C.byref(nn))
        return Stage1Result(err, nn.value, idx)

    def minify(self, buf):
        a = _u8(buf)
        dst = np.zeros(max(len(a), 1), dtype=np.uint8)
        dl = C.c_size_t(0)
        err = self.L.sjo_minify(_ptr(a), len(a), _ptr(dst), C.byref(dl))
        return err, bytes(dst[: dl.value])

    def validate_utf8(self, buf):
        a = _u8(buf)
        return bool(self.L.sjo_validate_utf8(_ptr(a), len(a)))


class Ref:
    """the unmodified reference; impl = "icelake" | "haswell" | "westmere" | "fallback" | "" (best)."""

    def __init__(self, impl=""):
        L = C.CDLL(REF_SO)
        L.sjr_supported.restype = C.c_int
        L.sjr_supported.argtypes = [C.c_char_p]
        L.sjr_best_name.restype = C.c_char_p
        L.sjr_stage1.restype = C.c_int
        L.sjr_stage1.argtypes = [C.c_char_p, C.POINTER(C.c_uint8), C.c_size_t, C.c_size_t, C.c_int, C.POINTER(C.c_uint32), C.c_size_t, C.POINTER(C.c_uint32)]
        L.sjr_minify.restype = C.c_int
        L.sjr_minify.argtypes = [C.c_char_p, C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_uint8), C.POINTER(C.c_size_t)]
        L.sjr_validate_utf8.restype = C.c_int
        L.sjr_validate_utf8.argtypes = [C.c_char_p, C.POINTER(C.c_uint8), C.c_size_t]
        L.sjr_time.restype = C.c_double
        L.sjr_time.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_uint8), C.c_size_t, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.sjr_time_rounds.restype = C.c_int
        L.sjr_time_rounds.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_uint8), C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.sjr_dom_roundtrip.restype = C.c_int
        L.sjr_dom_roundtrip.argtypes = [C.c_char_p, C.POINTER(C.c_uint8), C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.sjr_dom_parse_many.restype = C.c_long
        L.sjr_dom_parse_many.argtypes = [C.c_char_p, C.POINTER(C.c_uint8), C.c_size_t, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
        L.sjr_parse_string.restype = C.c_long
        L.sjr_parse_string.argtypes = [C.c_char_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]
        L.sjr_dom_tape.restype = C.c_int
        L.sjr_dom_tape.argtypes = [C.c_char_p, C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_uint8), C.POINTER(C.c_uint64), C.c_size_t, C.POINTER(C.c_size_t),
                                   C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_size_t)]
        self.L = L
        self.impl = impl.encode()
        if not L.sjr_supported(self.impl):
            raise RuntimeError(f"reference implementation {impl!r} not supported on this host")
        self.name = impl or L.sjr_best_name().decode()

    def stage1(self, buf, mode=REGULAR, capacity=None):
        a = _u8(buf)
        n = len(a)
        cap = n if capacity is None else capacity
        words = index_capacity(cap)
        idx = np.zeros(words, dtype=np.uint32)
        nn = C.c_uint32(N_SENTINEL)
        # the reference may read up to SIMDJSON_PADDING bytes past len in stage 2 only; stage 1 never over-reads
        err = self.L.sjr_stage1(self.impl, _ptr(a), n, cap, mode, _ptr(idx, C.c_uint32), words, C.byref(nn))
        return Stage1Result(err, nn.value, idx)

    def minify(self, buf):
        a = _u8(buf)
        dst = np.zeros(len(a) + 64, dtype=np.uint8)
        dl = C.c_size_t(0)
        err = self.L.sjr_minify(self.impl, _ptr(a), len(a), _ptr(dst), C.byref(dl))
        return err, bytes(dst[: dl.value])

    def validate_utf8(self, buf):
        a = _u8(buf)
        return bool(self.L.sjr_validate_utf8(self.impl, _ptr(a), len(a)))

    def time(self, op, buf, mode=REGULAR, threads=1, iters=3):
        a = _u8(buf)
        err = C.c_int(0)
        s = self.L.sjr_time(self.impl, op, _ptr(a), len(a), mode, threads, iters, C.byref(err))
        return s, err.value

    def time_rounds(self, op, buf, mode=REGULAR, threads=1, warmup=1, iters=3):
        """pre-spawned threads, one private copy of the document per thread; returns (best_s, mean_s, error_code)"""
        a = _u8(buf)
        out = (C.c_double * 2)()
        err = C.c_int(0)
        rc = self.L.sjr_time_rounds(self.impl, op, _ptr(a), len(a), mode, threads, warmup, iters, out, C.byref(err))
        if rc != 0:
            raise RuntimeError(f"sjr_time_rounds failed ({rc})")
        return out[0], out[1], err.value

    def dom_roundtrip(self, buf):
        a = _u8(buf)
        cap = 4 * len(a) + 64
        out = C.create_string_buffer(cap)
        ol = C.c_size_t(0)
        err = self.L.sjr_dom_roundtrip(self.impl, _ptr(a), len(a), out, cap, C.byref(ol))
        return err, out.raw[: ol.value]

    def parse_string(self, body):
        """dom_parser_implementation::parse_string on the bytes after an opening quote (closing quote included in body)"""
        a = np.concatenate([_u8(body), np.full(128, 0x20, dtype=np.uint8)])
        dst = np.zeros(len(a) + 128, dtype=np.uint8)
        r = self.L.sjr_parse_string(self.impl, _ptr(a), _ptr(dst))
        return r, bytes(dst[: max(r, 0)])

    def dom_tape(self, buf):
        """(error_code, types, payloads, string_buf bytes) of dom::parser::parse: one entry per tape value, root words left out"""
        a = _u8(buf)
        cap = len(a) + 16
        types = np.zeros(cap, dtype=np.uint8)
        pay = np.zeros(cap, dtype=np.uint64)
        sbc = 2 * len(a) + 64
        sb = np.zeros(sbc, dtype=np.uint8)
        ne, sl = C.c_size_t(0), C.c_size_t(0)
        err = self.L.sjr_dom_tape(self.impl, _ptr(a), len(a), _ptr(types), _ptr(pay, C.c_uint64), cap, C.byref(ne), _ptr(sb), sbc, C.byref(sl))
        return err, types[: ne.value], pay[: ne.value], sb[: sl.value]

    def dom_parse_many(self, buf, batch_size=1000000):
        a = _u8(buf)
        cap = 4 * len(a) + 64
        out = C.create_string_buffer(cap)
        ol = C.c_size_t(0)
        fe = C.c_int(0)
        nd = self.L.sjr_dom_parse_many(self.impl, _ptr(a), len(a), batch_size, out, cap, C.byref(ol), C.byref(fe))
        return nd, fe.value, out.raw[: ol.value]


def have_ref():
    return os.path.exists(REF_SO)


def ref_impls():
    """reference CPU kernels usable on this host, best first"""
    if not have_ref():
        return []
    L = C.CDLL(REF_SO)
    L.sjr_supported.restype = C.c_int
    L.sjr_supported.argtypes = [C.c_char_p]
    return [n for n in ("icelake", "haswell", "westmere", "fallback") if L.sjr_supported(n.encode())]


def same_stage1(a, b):
    """the parity bar: error code, n, and the (n+3) words when they were written"""
    if a.err != b.err or a.n != b.n:
        return False
    if a.wrote:
        return bool(np.array_equal(a.words(), b.words()))
    return True
