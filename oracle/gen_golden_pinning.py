#!/usr/bin/env python
"""Generate tests/golden/pinning.json.xz and tests/golden/jsonexamples/*.xz from the UNMODIFIED reference.

    python oracle/gen_golden_pinning.py SIMDJSON_SOURCE_DIR

Builds oracle/_ref/libsj_ref.so from SIMDJSON_SOURCE_DIR first (`make -B -C oracle REF=SIMDJSON_SOURCE_DIR ref`), so
that the records and the sample documents come from the same source tree.  The reference's sample documents
(jsonexamples/twitter.json, citm_catalog.json, amazon_cellphones.ndjson: data, not source) are stored xz-compressed.
pinning.json.xz holds the reference's records (tests/pinning_cases.py) for the seeded inputs of the pinning tests in
tests/test_oracle_pinning.py: stage 1 / minify / validate_utf8 from the icelake and haswell kernels (asserted
identical), stage-2-lite from dom::parser::parse and parse_string.  The port is asserted to match the stage-1 /
minify / validate_utf8 records before pinning.json.xz is written.
"""
import json
import lzma
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_lib as O  # noqa: E402
import pinning_cases as PC  # noqa: E402

EXAMPLES = ("twitter.json", "citm_catalog.json", "amazon_cellphones.ndjson")


def stage_jsonexamples(src):
    os.makedirs(O.JSONEXAMPLES, exist_ok=True)
    for name in EXAMPLES:
        data = open(os.path.join(src, "jsonexamples", name), "rb").read()
        with open(os.path.join(O.JSONEXAMPLES, name + ".xz"), "wb") as f:
            f.write(lzma.compress(data, preset=9 | lzma.PRESET_EXTREME))
        assert O.jsonexample(name) == data


def records(gen):
    return [rec for _ctx, rec in gen]


def token_records(ref, bodies, scalars, docs):
    strings = []
    for body in bodies:
        r, out = ref.parse_string(body + b'"')
        strings.append([int(r), PC.digest(out)])
    sc = []
    for doc, _k in scalars:
        err, types, pay, _sb = ref.dom_tape(doc)
        sc.append([int(err), bytes(types).decode("latin1"), PC.tape_record(types, pay)[2]])
    dd = []
    for doc in docs:
        err, types, pay, sb = ref.dom_tape(doc)
        dd.append([int(err)] + PC.tape_record(types, pay) + [len(sb), PC.digest(sb)])
    return {"strings": strings, "scalars": sc, "documents": dd}


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    src = os.path.abspath(sys.argv[1])
    if os.path.exists(O.REF_SO):
        os.remove(O.REF_SO)
    subprocess.check_call(["make", "-B", "-C", O.ORACLE_DIR, "REF=" + src, "ref"])
    if not O.have_ref():
        sys.exit(f"{src} holds no singleheader/simdjson.cpp: the reference could not be built")
    stage_jsonexamples(src)
    port = O.Port()
    ice, has = O.Ref("icelake"), O.Ref("haswell")
    out = {"generator": "oracle/gen_golden_pinning.py", "fuzz": {}}
    for name in PC.FUZZ_IMPLS:
        want = records(PC.fuzz_records(O.Ref(name), name))
        assert want == records(PC.fuzz_records(ice if name == "haswell" else has, name)) == records(PC.fuzz_records(port, name)), name
        out["fuzz"][name] = want
    out["sizes"] = records(PC.size_records(ice))
    assert out["sizes"] == records(PC.size_records(has)) == records(PC.size_records(port))
    out["large"] = records(PC.large_records(ice))
    assert out["large"] == records(PC.large_records(has)) == records(PC.large_records(port))
    out["tokens"] = {}
    for name, (bodies, scalars, docs) in PC.token_inputs().items():
        out["tokens"][name] = token_records(O.Ref(name), bodies, scalars, docs)
    path = PC.PINNED
    with lzma.open(path, "wt", preset=9 | lzma.PRESET_EXTREME) as f:
        json.dump(out, f, separators=(",", ":"))
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
