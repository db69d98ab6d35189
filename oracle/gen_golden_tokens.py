#!/usr/bin/env python
"""Generate tests/golden/tokens.json from the UNMODIFIED reference (oracle/_ref/libsj_ref.so): stage-2-lite vectors.

  strings   dom_parser_implementation::parse_string on seeded string bodies (valid and invalid escapes)
  scalars   dom::parser::parse of a one-value document around a seeded scalar token: error code, tape type, value
  documents dom::parser::parse of small documents: tape types / payloads / string_buf; digests for the jsonexamples files

    python oracle/gen_golden_tokens.py
"""
import hashlib
import json
import math
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import oracle_lib as O  # noqa: E402
import token_fuzz as TF  # noqa: E402
from simdjson_b200 import corpus  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "tokens.json")

DOCS = [
    b'{"a":[1,-2,3.5e3,true,false,null,"x\\n\\u00e9\\ud83d\\ude00y"],"k\\"":18446744073709551615, "z":-0, "e":""}',
    b'[]', b'{}', b'[[],{},[{}]]', b'""', b'"a"', b'0', b'-1', b'true', b'null', b'1.5',
    b'["\\\\","\\"","\\/\\b\\f\\n\\r\\t"]',
    b'{"\\u0041\\u00e9\\u20ac":"\\ud800\\udc00\\udbff\\udfff"}',
    b'[9223372036854775807,9223372036854775808,-9223372036854775808,18446744073709551615,1e5,0.0,-0.0]',
    b'  [ 1 , 2 , "a b" , { "k" : [ ] } ]  ',
]


def float_is_finite(tok):
    try:
        return math.isfinite(float(tok.decode("latin1")))
    except ValueError:
        return True  # not a float by Python's grammar: the reference decides


def main():
    ref, ref2 = O.Ref("icelake" if "icelake" in O.ref_impls() else ""), O.Ref("haswell" if "haswell" in O.ref_impls() else "")
    rng = random.Random(0x5EED1234)
    strings = []
    for _ in range(700):
        body, _bad = TF.string_body(rng)
        r, out = ref.parse_string(body + b'"')
        r2, out2 = ref2.parse_string(body + b'"')
        assert (r, out) == (r2, out2), body
        strings.append({"body": body.hex(), "len": r, "out": out.hex()})
    scalars = []
    for _ in range(900):
        tok = TF.scalar_token(rng)
        doc, k = TF.wrap_scalar(tok, rng)
        if not float_is_finite(tok):
            continue
        err, types, pay, _sb = ref.dom_tape(doc)
        err2, types2, pay2, _ = ref2.dom_tape(doc)
        assert err == err2 and bytes(types) == bytes(types2), doc
        # the value's tape entry: tape order == structural order without ':' and ','
        nth = {1: 1, 3: 2}[k] if doc.startswith(b"[") else 2
        ent = {"doc": doc.hex(), "index": k, "err": int(err)}
        if err == 0:
            ent["type"] = chr(types[nth])
            ent["value"] = str(int(pay[nth])) if chr(types[nth]) in "lu" else None
        scalars.append(ent)
    docs = []
    pieces = DOCS + [bytes(corpus.random_json(rng.randrange(200, 3000), seed=1000 + i)) for i in range(30)]
    for d in pieces:
        err, types, pay, sb = ref.dom_tape(d)
        err2, types2, pay2, sb2 = ref2.dom_tape(d)
        assert err == err2 and bytes(types) == bytes(types2) and bytes(sb) == bytes(sb2), d
        keep = [i for i, t in enumerate(types) if chr(t) in '"lu']
        docs.append({"doc": d.hex(), "err": int(err), "types": bytes(types).decode("latin1"), "payloads": {str(i): str(int(pay[i])) for i in keep},
                     "string_buf": bytes(sb).hex()})
    files = []
    for name in ("twitter.json", "citm_catalog.json"):
        d = O.jsonexample(name)
        err, types, pay, sb = ref.dom_tape(d)
        assert err == 0
        isd = np.array([chr(t) == "d" for t in types])
        files.append({"file": name, "entries": int(len(types)), "types_sha256": hashlib.sha256(bytes(types)).hexdigest(),
                      "payloads_no_doubles_sha256": hashlib.sha256(np.where(isd, 0, pay).astype(np.uint64).tobytes()).hexdigest(),
                      "string_buf_bytes": int(len(sb)), "string_buf_sha256": hashlib.sha256(bytes(sb)).hexdigest()})
    json.dump({"generator": "oracle/gen_golden_tokens.py", "impl": "icelake (== haswell)", "strings": strings, "scalars": scalars, "documents": docs,
               "files": files}, open(OUT, "w"))
    print(len(strings), "strings,", len(scalars), "scalars,", len(docs), "documents ->", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
