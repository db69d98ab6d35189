"""Seeded inputs of the reference-pinning tests (tests/test_oracle_pinning.py) and the records they compare.

oracle/gen_golden_pinning.py ran these inputs through the unmodified reference and stored its records in
tests/golden/pinning.json.xz; the tests run the same inputs through the port and compare record by record, so that
the port stays pinned to the reference on machines that cannot build it.  A record holds the error code and the
length of each result and a digest of its bytes (the first 8 hex digits of their SHA-256).

The inputs are the exact byte streams of simdjson_b200/corpus.py and tests/token_fuzz.py under fixed seeds: a change
to either (or to this module) changes the inputs, and the records must then be regenerated (REGENERATE).
"""
import hashlib
import json
import lzma
import math
import os
import random

import numpy as np

import oracle_lib as O
import token_fuzz as TF
from simdjson_b200 import corpus

PINNED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pinning.json.xz")
FUZZ_IMPLS = ("icelake", "haswell")  # the reference kernels the fuzz inputs were drawn for (one seed each)
REGENERATE = ("if simdjson_b200/corpus.py, tests/token_fuzz.py or tests/pinning_cases.py changed, the inputs changed rather than the port: "
              "regenerate the records with `python oracle/gen_golden_pinning.py SIMDJSON_SOURCE_DIR`")


def load():
    with lzma.open(PINNED, "rt") as f:
        return json.load(f)


def digest(b):
    return hashlib.sha256(bytes(b)).hexdigest()[:8]


def stage1_record(r):
    """what oracle_lib.same_stage1 compares: error code, n, and the (n+3) words when they were written"""
    return [int(r.err), int(r.n), digest(r.words().tobytes()) if r.wrote else None]


def minify_record(res):
    err, out = res
    return [int(err), len(out), digest(out)]


# --------------------------------------------------------------------------- stage 1, minify, validate_utf8
def fuzz_records(impl, name):
    """4000 adversarial / multi-document inputs in all seven modes: (input, mode), record"""
    rng = random.Random(corpus.SEED + (1 if name == "haswell" else 0))
    for i in range(4000):
        kind = i % 4
        if kind == 0:
            b, mode = corpus.adversarial(rng), rng.choice(O.ALL_MODES)
        elif kind == 1:
            b, mode = corpus.multi_document(rng), rng.choice([1, 2])
        elif kind == 2:
            b, mode = b"\x1e" + corpus.multi_document(rng, sep=b"\x1e"), rng.choice([3, 4])
        else:
            b, mode = corpus.multi_document(rng, sep=b","), rng.choice([5, 6])
        rec = stage1_record(impl.stage1(b, mode))
        if kind == 0:
            rec += minify_record(impl.minify(b)) + [bool(impl.validate_utf8(b))]
        yield (b, mode), rec


def size_records(impl):
    """a document longer than the capacity, then every length 0..199 and the block boundaries: n, record"""
    doc = b'{"a":[1,2,3],"b":"xyz"}'
    yield "capacity", stage1_record(impl.stage1(doc, 0, capacity=8))
    for n in list(range(0, 200)) + [255, 256, 257, 4095, 4096, 4097]:
        b = bytes(corpus.random_json(max(n, 64)))[:n]
        u = bytes(corpus.random_utf8(max(n, 1), seed=n))[:n]
        yield n, sum((stage1_record(impl.stage1(b, mode)) for mode in (0, 1, 2)), []) + minify_record(impl.minify(b)) + [bool(impl.validate_utf8(u))]


def large_records(impl):
    """4 MiB of JSON, 2 MiB of NDJSON (whole and cut mid-row), 1 MiB of UTF-8 text with three corruptions: name, record"""
    d = corpus.random_json(4 << 20)
    yield "json", stage1_record(impl.stage1(d)) + minify_record(impl.minify(d))
    nd = corpus.ndjson_rows(2 << 20)
    for mode in (1, 2):
        yield f"ndjson mode {mode}", stage1_record(impl.stage1(nd, mode))
    cut = nd[: (1 << 20) + 123]
    r = impl.stage1(cut, 1)
    yield "ndjson cut mid-row", stage1_record(r) + [int(r.idx[r.n]) if r.wrote else None]
    u = corpus.random_utf8(1 << 20)
    yield "utf8", bool(impl.validate_utf8(u))
    for pos in (0, len(u) // 2, len(u) - 2):
        v = u.copy()
        v[pos] = 0xFF
        yield f"utf8 0xFF at {pos}", bool(impl.validate_utf8(v))


# --------------------------------------------------------------------------- stage-2-lite
def token_inputs():
    """per reference kernel: 1500 string bodies, 1500 one-scalar documents (no infinite floats: the reference rejects
    infinite VALUES in write_float and stage-2-lite does not convert floats), 12 random documents -- one seeded stream"""
    rng = random.Random(20260923)
    out = {}
    for name in FUZZ_IMPLS:
        bodies = [TF.string_body(rng, maxlen=rng.choice([80, 200]))[0] for _ in range(1500)]
        scalars = []
        for _ in range(1500):
            tok = TF.scalar_token(rng)
            try:
                if not math.isfinite(float(tok.decode("latin1"))):
                    continue
            except ValueError:
                pass
            scalars.append(TF.wrap_scalar(tok, rng))
        docs = [bytes(corpus.random_json(rng.randrange(500, 60000), seed=777 + i)) for i in range(12)]
        out[name] = (bodies, scalars, docs)
    return out


def tape_record(types, pay):
    """tape types and the payloads of strings and integers (the values stage-2-lite produces)"""
    types = np.asarray(types, dtype=np.uint8)
    keep = np.isin(types, np.frombuffer(b'"lu', dtype=np.uint8))
    return [len(types), digest(types.tobytes()), digest(np.asarray(pay, dtype=np.uint64)[keep].tobytes())]
