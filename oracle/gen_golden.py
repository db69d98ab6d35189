#!/usr/bin/env python
"""Generate tests/golden/*.json from the UNMODIFIED reference (oracle/_ref/libsj_ref.so).

Run in the build container (needs /root/reference to have been compiled by
`make -C oracle`).  The fixtures are small and committed; the GPU box and
later rounds check the oracle port and the CUDA path against them without
needing the reference.  Each vector was produced by the reference's icelake
kernel and asserted identical on haswell before being written.

    python oracle/gen_golden.py
"""
import hashlib
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import oracle_lib as O  # noqa: E402
from simdjson_b200 import corpus  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# hand-written known-answer inputs (the reference's own tests pin the same behaviours:
# tests/dom/basictests.cpp L1913-2034 minify, tests/dom/document_stream_tests.cpp L592-704
# truncation, tests/unicode_tests.cpp L187-246 utf-8 tables; SURVEY.md section 8(c) goldens)
STAGE1_KAT = [
    (b'{"a":[1,2,"x\\"y"],"b":true}', [0]),
    (b'[1,2,3]  {"1":1,"2":3,"4":4} [1,2  ', [0, 1, 2]),
    (b"", [0, 1, 2]),
    (b"   \n\t  ", [0, 1, 2]),
    (b'"', [0, 1, 2]),
    (b'"abc', [0, 1, 2]),
    (b'["a\xffb"]', [0, 1, 2]),
    (b'["a\x01b"]', [0, 1, 2]),
    (b"1\x0c2", [0]),
    (b"1\x1a2", [0]),
    (b'\\"abc"', [0, 1, 2]),
    (b'{"a":"\\\\"}', [0]),
    (b'{"a":"\\\\\\""}', [0]),
    (b"\\" * 64 + b'"', [0, 1, 2]),
    (b"\\" * 65 + b'"', [0, 1, 2]),
    (b"\\" * 127 + b'"x"', [0, 1, 2]),
    (b"\\" * 128 + b'"x"', [0, 1, 2]),
    (b'{"k":"' + b"a" * 200 + b'"}', [0]),
    (b"[" + b"1," * 100 + b"1]", [0]),
    (b'{"a":1}\n{"b":2}\n{"c":', [1, 2]),
    (b'{"a":1}\n{"b":2}\n{"c":"\xe2\x82', [1, 2]),
    (b"\xe2\x82", [1, 2]),
    (b"\xc3", [0, 1, 2]),
    (b'\x1e{"a":1}\n\x1e[1,2]\n\x1e3\n', [3, 4]),
    (b'\x1e{"a":1}\n\x1e[1,2]\n\x1e{"b"', [3, 4]),
    (b'\x1e1\x1e2\x1e"s"\x1etrue', [3, 4]),
    (b'\x1e\x1e \x1e{"a":1}', [3, 4]),
    (b'{"a":1},{"b":[1,2]},3,"s"', [5, 6]),
    (b'{"a":1},{"b":[1,2]},{"c":', [5, 6]),
    (b",,,", [5, 6]),
    (b'[1,2],[3,4', [5, 6]),
]

MINIFY_KAT = [
    b'{"a" : 1 , "b":[ 1, 2 ,3 ] }', b'  "a b  c"  ', b"[ 1 ,\n\t2 ]\r\n", b'{"k":"v\\" x"} ', b"", b" ", b'"', b'" "', b'\\" "',
    b'{ "a\\\\" : " " }', b"true false null 1 2 3", b'"\\', b"\\" * 31 + b" x", b'{"s":"' + b" " * 300 + b'"}', b" " * 1000,
]

UTF8_KAT = [
    b"", b"a", b"\xc3\xb1", b"\xe2\x82\xa1", b"\xf0\x90\x8c\xbc", b"\xc2\x80", b"\xf0\x90\x80\x80", b"\xee\x80\x80", b"\xef\xbb\xbf",
    b"\xf4\x8f\xbf\xbf", b"\xed\x9f\xbf", b"\xe0\xa0\x80",
    b"\xc3\x28", b"\xa0\xa1", b"\xe2\x28\xa1", b"\xe2\x82\x28", b"\xf0\x28\x8c\xbc", b"\xf0\x90\x28\xbc", b"\xf0\x28\x8c\x28", b"\xc0\x9f",
    b"\xf5\xff\xff\xff", b"\xed\xa0\x81", b"\xf8\x90\x80\x80\x80", b"123456789012345\xed", b"123456789012345\xf1", b"123456789012345\xc2",
    b"\xc2\x7f", b"\xce", b"\xce\xba\xe1", b"\xce\xba\xe1\xbd", b"\xce\xba\xe1\xbd\xb9\xcf", b"\xce\xba\xe1\xbd\xb9\xcf\x83\xce",
    b"\xce\xba\xe1\xbd\xb9\xcf\x83\xce\xbc\xce", b"\xdf", b"\xef\xbf", b"\x80", b"\x91\x85\x95\x9e", b"\x6c\x02\x8e\x18", b"\xc1\xbf", b"\xe0\x9f\xbf",
    b"\xf0\x8f\xbf\xbf", b"\xf4\x90\x80\x80", b"\xed\xa0\x80", b"\xed\xbf\xbf", b"\xf7\xbf\xbf\xbf", b"\xfe", b"\xff",
    b"a" * 63 + b"\xc3", b"a" * 63 + b"\xc3\xa9", b"a" * 62 + b"\xe2\x82\xac", b"a" * 61 + b"\xf0\x9f\x98\x80", b"a" * 64 + b"\x80",
    b"a" * 31 + b"\xf0\x9f\x98\x80" + b"b" * 100, b"a" * 127 + b"\xe2\x82\xac", b"\xe2\x82\xac" * 50, b"\xf0\x9f\x98\x80" * 40 + b"\xf0\x9f\x98",
    b"\xc3" + b"a" * 64, b"a" * 64 + b"\xed\xa0\x80", b"\xf0\x9f\x98\x80"[:3] + b" " * 70,
]


def hexs(b):
    return bytes(b).hex()


def main():
    if not O.have_ref():
        sys.exit("oracle/_ref/libsj_ref.so missing: run `make -C oracle` where /root/reference exists")
    ice, has = O.Ref("icelake"), O.Ref("haswell")
    os.makedirs(OUT, exist_ok=True)
    rng = random.Random(corpus.SEED)

    # ---- stage 1
    cases = []
    inputs = [(b, modes) for b, modes in STAGE1_KAT]
    for _ in range(260):
        inputs.append((corpus.adversarial(rng, 400), [rng.choice(O.ALL_MODES)]))
    for _ in range(120):
        inputs.append((corpus.multi_document(rng), [rng.choice([1, 2])]))
    for _ in range(60):
        inputs.append((b"\x1e" + corpus.multi_document(rng, sep=b"\x1e"), [rng.choice([3, 4])]))
    for _ in range(60):
        inputs.append((corpus.multi_document(rng, sep=b","), [rng.choice([5, 6])]))
    for b, modes in inputs:
        for mode in modes:
            a, h = ice.stage1(b, mode), has.stage1(b, mode)
            assert O.same_stage1(a, h), (b, mode)
            rec = {"hex": hexs(b), "mode": mode, "err": a.err, "n": a.n if a.wrote else None}
            if a.wrote:
                rec["words"] = [int(x) for x in a.words()]
            cases.append(rec)
    json.dump({"generator": "oracle/gen_golden.py", "impl": "icelake (== haswell)", "cases": cases}, open(os.path.join(OUT, "stage1.json"), "w"))

    # ---- minify
    cases = []
    inputs = list(MINIFY_KAT)
    for n in list(range(0, 130)) + [255, 256, 257, 511, 512, 513, 1023]:
        inputs.append(b"\\" * n)
        inputs.append(b'"' + b" " * n + b'"')
    for _ in range(200):
        inputs.append(corpus.adversarial(rng, 400))
    for b in inputs:
        (e1, o1), (e2, o2) = ice.minify(b), has.minify(b)
        assert (e1, o1) == (e2, o2), b
        cases.append({"hex": hexs(b), "err": e1, "out": hexs(o1)})
    json.dump({"generator": "oracle/gen_golden.py", "cases": cases}, open(os.path.join(OUT, "minify.json"), "w"))

    # ---- utf-8
    cases = []
    inputs = list(UTF8_KAT)
    base = bytes(corpus.random_utf8(4096, seed=7))
    for _ in range(300):  # random single-bit flips of valid text (tests/unicode_tests.cpp L157-185 brute force)
        n = rng.randint(1, 400)
        off = rng.randrange(0, len(base) - n)
        s = bytearray(base[off : off + n])
        if rng.random() < 0.8:
            pos = rng.randrange(n)
            s[pos] ^= 1 << rng.randrange(8)
        inputs.append(bytes(s))
    for b in inputs:
        v1, v2 = ice.validate_utf8(b), has.validate_utf8(b)
        assert v1 == v2, b
        cases.append({"hex": hexs(b), "valid": bool(v1)})
    json.dump({"generator": "oracle/gen_golden.py", "cases": cases}, open(os.path.join(OUT, "utf8.json"), "w"))

    # ---- whole-file digests for the reference's own corpora
    files = []
    for name, mode in [("twitter.json", 0), ("citm_catalog.json", 0), ("amazon_cellphones.ndjson", 2), ("twitter.json", 2)]:
        data = np.frombuffer(O.jsonexample(name), dtype=np.uint8)
        a, h = ice.stage1(data, mode), has.stage1(data, mode)
        assert O.same_stage1(a, h)
        me, mo = ice.minify(data)
        files.append({
            "file": name, "len": int(len(data)), "mode": mode, "err": a.err, "n": a.n,
            "first": [int(x) for x in a.idx[:4]], "tail": [int(x) for x in a.idx[a.n - 1 : a.n + 3]],
            "idx_sha256": hashlib.sha256(a.words().tobytes()).hexdigest(),
            "minify_err": me, "minify_len": len(mo), "minify_sha256": hashlib.sha256(mo).hexdigest(),
            "utf8": bool(ice.validate_utf8(data)),
        })
    json.dump({"generator": "oracle/gen_golden.py", "files": files}, open(os.path.join(OUT, "corpora.json"), "w"), indent=1)
    for f in ("stage1.json", "minify.json", "utf8.json", "corpora.json"):
        print(f, os.path.getsize(os.path.join(OUT, f)), "bytes")


if __name__ == "__main__":
    main()
