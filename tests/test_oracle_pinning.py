"""Pins the CPU restatement (oracle/sj_oracle.c) before anything trusts it.

 * against the committed golden vectors produced by the unmodified reference
   (tests/golden/*.json, generator oracle/gen_golden.py);
 * against what the reference (icelake AND haswell kernels) returned for
   seeded adversarial inputs in all seven stage1 modes, recorded in
   tests/golden/pinning.json.xz (generator oracle/gen_golden_pinning.py,
   inputs and records in tests/pinning_cases.py).
"""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_lib as O
import pinning_cases as PC

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def port():
    return O.Port()


def _load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def test_port_matches_golden_stage1(port):
    cases = _load("stage1.json")["cases"]
    assert len(cases) > 500
    for c in cases:
        r = port.stage1(bytes.fromhex(c["hex"]), c["mode"])
        assert r.err == c["err"], c
        if c["n"] is None:
            assert not r.wrote, c
        else:
            assert r.n == c["n"], c
            assert [int(x) for x in r.words()] == c["words"], c


def test_port_matches_golden_minify(port):
    cases = _load("minify.json")["cases"]
    assert len(cases) > 400
    for c in cases:
        err, out = port.minify(bytes.fromhex(c["hex"]))
        assert (err, out.hex()) == (c["err"], c["out"]), c


def test_port_matches_golden_utf8(port):
    cases = _load("utf8.json")["cases"]
    assert len(cases) > 300
    for c in cases:
        assert port.validate_utf8(bytes.fromhex(c["hex"])) == c["valid"], c


@pytest.fixture(scope="module")
def pinned():
    return PC.load()


def test_port_matches_golden_corpora(port):
    for f in _load("corpora.json")["files"]:
        data = np.frombuffer(O.jsonexample(f["file"]), dtype=np.uint8)
        assert len(data) == f["len"]
        r = port.stage1(data, f["mode"])
        assert (r.err, r.n) == (f["err"], f["n"])
        assert hashlib.sha256(r.words().tobytes()).hexdigest() == f["idx_sha256"]
        err, out = port.minify(data)
        assert (err, len(out), hashlib.sha256(out).hexdigest()) == (f["minify_err"], f["minify_len"], f["minify_sha256"])
        assert port.validate_utf8(data) == f["utf8"]


def test_amazon_is_793_documents(port):
    """tests/dom/basictests.cpp L36, L692-708: parse_many over amazon_cellphones.ndjson yields 793 docs;
    at stage-1 level: 793 top-level '[' ... ']' rows in streaming_final mode."""
    data = np.frombuffer(O.jsonexample("amazon_cellphones.ndjson"), dtype=np.uint8)
    r = port.stage1(data, O.STREAMING_FINAL)
    assert r.err == 0 and r.n == 15067
    # count row starts: a '[' structural that is the first structural on its line
    starts = 0
    idx = r.idx[: r.n]
    for k, pos in enumerate(idx):
        if data[pos] == ord("[") and (k == 0 or data[idx[k - 1]] == ord("]")):
            starts += 1
    assert starts == 793


def _same_records(got, want):
    got = list(got)
    assert len(got) == len(want), PC.REGENERATE
    for (ctx, g), w in zip(got, want):
        assert g == w, (ctx, g, w, PC.REGENERATE)


@pytest.mark.parametrize("impl", PC.FUZZ_IMPLS)
def test_port_matches_live_reference_fuzz(port, pinned, impl):
    """stage 1 in all seven modes, minify and validate_utf8 on the seeded inputs drawn for the reference's icelake / haswell
    kernel, against that kernel's recorded answers"""
    _same_records(PC.fuzz_records(port, impl), pinned["fuzz"][impl])


def test_port_matches_live_reference_capacity_and_sizes(port, pinned):
    """stage 1 / minify / validate_utf8 at every length 0..199 and the block boundaries, against the reference's recorded answers"""
    # len > capacity -> CAPACITY before anything is written (json_structural_indexer.h L195)
    assert pinned["sizes"][0] == [O.CAPACITY, O.N_SENTINEL, None]
    # block-boundary lengths
    _same_records(PC.size_records(port), pinned["sizes"])


def test_port_matches_live_reference_large(port, pinned):
    """MiB-sized JSON, NDJSON and UTF-8 text, against the reference's recorded answers"""
    want = pinned["large"]
    # cut an NDJSON buffer mid-row: streaming_partial must point at the last complete row
    cut = want[3]
    assert cut[0] == 0 and cut[3] < (1 << 20) + 123
    # valid UTF-8, then three corrupted copies
    assert want[4:] == [True, False, False, False]
    _same_records(PC.large_records(port), want)


# ---------------------------------------------------------------- stage-2-lite (SURVEY.md 8(f) row 4)
def _tape_view(types, pay):
    """the port's per-structural arrays in the reference's tape order: ':' and ',' have no tape entry"""
    keep = [i for i, t in enumerate(types) if chr(t) not in ":,"]
    return bytes(types[keep]), pay[keep]


def _check_doc_against(port, doc, want_err, want_types, want_pay_by_index, want_sb):
    r = port.stage1(doc)
    assert r.err == 0
    err, types, pay, sb, sl, ns, fe = port.tokens(doc, r.idx, r.n)
    assert err == 0 and fe == 0xFFFFFFFF, (doc[:80], err)
    t, p = _tape_view(types, pay)
    assert want_err == 0 and t == want_types, doc[:80]
    for i, v in want_pay_by_index.items():
        assert int(p[int(i)]) == int(v), (doc[:80], i)
    assert bytes(sb) == want_sb and sl == len(want_sb)


def test_port_tokens_match_golden(port):
    g = _load("tokens.json")
    for c in g["strings"]:
        body = bytes.fromhex(c["body"])
        r, out = port.parse_string(b'"' + body + b'"')
        assert r == c["len"] and out == bytes.fromhex(c["out"]), body
    for c in g["scalars"]:
        doc = bytes.fromhex(c["doc"])
        r = port.stage1(doc)
        if r.err != 0:  # stage 1 already fails (a quote inside the token): the reference reports the same error
            assert c["err"] == r.err, doc
            continue
        err, types, pay, *_ = port.tokens(doc, r.idx, r.n)
        k = c["index"]
        if c["err"] == 0:
            assert err == 0 and chr(types[k]) == c["type"], doc
            if c["value"] is not None:
                assert int(pay[k]) == int(c["value"]), doc
        else:
            # the reference stops at its first error; the token must be that error (it is the only scalar that can fail here)
            assert types[k] == 0 and int(pay[k]) == c["err"] and err == c["err"], (doc, err, int(pay[k]), c["err"])
    for c in g["documents"]:
        _check_doc_against(port, bytes.fromhex(c["doc"]), c["err"], c["types"].encode("latin1"), c["payloads"], bytes.fromhex(c["string_buf"]))
    for f in g["files"]:
        doc = O.jsonexample(f["file"])
        r = port.stage1(doc)
        err, types, pay, sb, sl, ns, fe = port.tokens(doc, r.idx, r.n)
        t, p = _tape_view(types, pay)
        assert err == 0 and len(t) == f["entries"] and hashlib.sha256(t).hexdigest() == f["types_sha256"]
        isd = np.frombuffer(t, dtype=np.uint8) == ord("d")
        assert hashlib.sha256(np.where(isd, 0, p).astype(np.uint64).tobytes()).hexdigest() == f["payloads_no_doubles_sha256"]
        assert sl == f["string_buf_bytes"] and hashlib.sha256(bytes(sb)).hexdigest() == f["string_buf_sha256"]


def test_port_tokens_match_live_reference(port, pinned):
    """parse_string, one-scalar documents and random documents against the recorded answers of dom::parser::parse"""
    hint = PC.REGENERATE
    for impl, (bodies, scalars, docs) in PC.token_inputs().items():
        want = pinned["tokens"][impl]
        assert (len(bodies), len(scalars), len(docs)) == tuple(len(want[k]) for k in ("strings", "scalars", "documents")), hint
        for body, w in zip(bodies, want["strings"]):
            r, out = port.parse_string(b'"' + body + b'"')
            assert [r, PC.digest(out)] == w, (body, hint)
        for (doc, k), (rerr, rtypes, rpay) in zip(scalars, want["scalars"]):
            r = port.stage1(doc)
            if r.err != 0:
                assert rerr == r.err, (doc, hint)
                continue
            err, types, pay, *_ = port.tokens(doc, r.idx, r.n)
            if rerr == 0:
                t, p = _tape_view(types, pay)
                assert err == 0 and t == rtypes.encode("latin1"), (doc, hint)
                assert PC.tape_record(np.frombuffer(t, dtype=np.uint8), p)[2] == rpay, (doc, hint)
            else:
                assert types[k] == 0 and int(pay[k]) == rerr and err == rerr, (doc, err, int(pay[k]), rerr, hint)
        for doc, (rerr, *rtape, rsb_len, rsb) in zip(docs, want["documents"]):
            r = port.stage1(doc)
            assert r.err == 0
            err, types, pay, sb, sl, ns, fe = port.tokens(doc, r.idx, r.n)
            assert err == 0 and fe == 0xFFFFFFFF, (doc[:80], err)
            t, p = _tape_view(types, pay)
            assert rerr == 0 and PC.tape_record(np.frombuffer(t, dtype=np.uint8), p) == rtape, (doc[:80], hint)
            assert [sl, PC.digest(sb)] == [rsb_len, rsb], (doc[:80], hint)
