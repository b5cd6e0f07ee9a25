"""Oracle vs outputs of the reference itself: (a) the committed golden dumps produced by
tools/make_golden.py with the unmodified reference (oracle/_ref), (b) the reference's outputs
on further seeded corpora and fuzzed inputs, kept as digests (tests/reference_outputs.py).  CPU only."""
import base64
import json
import os

import numpy as np
import pytest

from conftest import ROOT, model_bytes
from oracle import oracle_py
from reference_outputs import Reference

GOLD = os.path.join(ROOT, "tests", "golden")
SETS = [("uni32k", "en"), ("uni32k", "mixed"), ("mix_bf8k", "mixed"), ("botchan8k", "en"), ("bpe32k", "en"),
        ("mix_bpe4k", "mixed")]


@pytest.mark.parametrize("model,kind", SETS)
def test_golden_ids(model, kind, corpus_gen):
    z = np.load(os.path.join(GOLD, "ids", f"{model}__{kind}.npz"))
    buf, offs = corpus_gen.fill(kind, int(z["seed"]), int(z["n"]))
    ids, ido = oracle_py.OracleModel(model_bytes(model)).encode_batch(buf, offs)
    assert np.array_equal(ido.astype(np.uint32), z["id_offsets"])
    assert np.array_equal(ids, z["ids"])


def load_edge():
    with open(os.path.join(GOLD, "edge_cases.json")) as f:
        e = json.load(f)
    return [base64.b64decode(s) for s in e["inputs"]], e["models"]


@pytest.mark.parametrize("model", ["uni32k", "mix_bf8k", "botchan8k", "bpe32k", "mix_bpe4k"])
def test_golden_edge_cases(model):
    inputs, models = load_edge()
    g = models[model]
    om = oracle_py.OracleModel(model_bytes(model))
    for k, s in enumerate(inputs):
        ids, te = om.encode(s)
        assert ids.tolist() == g["ids"][k], (model, k, s[:40])
        nrm, n2o = om.normalize(s)
        assert nrm == base64.b64decode(g["normalized"][k]), (model, k)
        if g["n2o"][k] is not None and len(nrm):
            assert n2o == g["n2o"][k], (model, k)
        assert (int(te[-1]) if len(te) else 0) == len(nrm)


@pytest.mark.parametrize("model,kind", SETS)
def test_live_reference(model, kind, corpus_gen, request):
    mb = model_bytes(model)
    buf, offs = corpus_gen.fill(kind, 777, 3000)
    a, ao = oracle_py.OracleModel(mb).encode_batch(buf, offs)
    Reference(request).check("encode", (a, ao), lambda: oracle_py.RefModel(mb).encode_batch(buf, offs, threads=4))


@pytest.mark.parametrize("model", ["uni32k", "bpe32k"])
def test_live_reference_set_vocabulary(model, corpus_gen, request):
    """SetVocabulary flips piece types in place (Q8); UNUSED pieces are skipped by the unigram
    Viterbi and re-split by BPE (sentencepiece_processor.cc:301-340, bpe_model.cc:175-193)."""
    mb = model_bytes(model)
    om, ref = oracle_py.OracleModel(mb), Reference(request)
    rng = np.random.default_rng(5)
    pieces = om.proto["pieces"]
    keep = [p for p in pieces if rng.random() < 0.5]
    buf, offs = corpus_gen.fill("en", 778, 1500)

    def reference(reset):
        rm = oracle_py.RefModel(mb)
        rm.set_vocabulary(keep)
        if reset:
            rm.reset_vocabulary()
        return rm.encode_batch(buf, offs)
    om.set_types(om.vocabulary_types(keep))
    ref.check("restricted", om.encode_batch(buf, offs), lambda: reference(False))
    om.set_types(om.types)
    ref.check("reset", om.encode_batch(buf, offs), lambda: reference(True))


def test_live_reference_normalize_alignment(corpus_gen, request):
    mb = model_bytes("mix_bf8k")
    om = oracle_py.OracleModel(mb)
    lines = corpus_gen.lines("mixed", 779, 400)

    def normalize_all(m):
        out = [m.normalize(s) for s in lines]
        return (b"".join(n for n, _ in out), [len(n) for n, _ in out], [len(a) for _, a in out],
                np.concatenate([np.asarray(a, np.int64) for _, a in out]))
    Reference(request).check("normalize", normalize_all(om), lambda: normalize_all(oracle_py.RefModel(mb)))


@pytest.mark.parametrize("model", ["uni32k", "mix_bf8k", "bpe32k", "mix_bpe4k"])
def test_fuzz_oracle_vs_live_reference(model, request):
    """Random mixes of ASCII, runs of spaces, CJK, emoji, NFKC compatibility forms, combining marks, control bytes,
    NUL, reserved piece strings and malformed UTF-8: oracle ids (and the decoded text of those ids) == reference."""
    rng = np.random.default_rng(20260922)
    chunks = [b" ", b"  ", b"a", b"e", b"the", b"ing", "▁".encode(), "あ".encode(), "ガ".encode(), "ｗ".encode(),
              "㍿".encode(), "😀".encode(), b"\xff", b"\xc0\xaf", b"\xed\xa0\x80", b"\xe2\x82", b"\x00", b"\t", b"\n",
              "Å".encode(), b"1", "①".encode(), b".", b",", " ".encode(), "　".encode(), b"<unk>", b"<s>",
              "�".encode()]
    sents = []
    for _ in range(6000):
        parts = [chunks[int(rng.integers(0, len(chunks)))] for _ in range(int(rng.integers(0, 40)))]
        if rng.random() < 0.2:
            parts.append(bytes(rng.integers(0, 256, size=int(rng.integers(1, 12)), dtype=np.uint8)))
        sents.append(b"".join(parts))
    mb = model_bytes(model)
    om, ref = oracle_py.OracleModel(mb), Reference(request)
    buf, offs = oracle_py.pack(sents)
    a, ao = om.encode_batch(buf, offs)
    ref.check("encode", (a, ao), lambda: oracle_py.RefModel(mb).encode_batch(buf, offs, threads=8))
    ref.check("decode", om.decode_batch(a, ao), lambda: oracle_py.RefModel(mb).decode_batch(a, ao, threads=8))
