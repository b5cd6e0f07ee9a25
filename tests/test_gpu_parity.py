"""Parity of the CUDA engine (through the C ABI) with the oracle, the committed golden dumps
of the reference, and the reference's outputs on larger corpora (kept as digests, tests/reference_outputs.py).
Bit-exact ids are required everywhere (integer/index work).  Needs a B200."""
import base64
import json
import os

import numpy as np
import pytest

from conftest import ROOT, model_bytes
from oracle import modelproto as mp
from oracle import oracle_py
from reference_outputs import Reference

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
ALL_MODELS = ["uni32k", "mix_bf8k", "botchan8k", "bpe32k", "mix_bpe4k"]
SETS = [("uni32k", "en"), ("uni32k", "mixed"), ("mix_bf8k", "mixed"), ("botchan8k", "en"), ("bpe32k", "en"),
        ("mix_bpe4k", "mixed")]

_engines = {}


def engine(model):
    from sentencepiece_b200 import Engine
    if model not in _engines:
        _engines[model] = Engine(model_bytes(model))
    return _engines[model]


def assert_same(a, ao, b, bo, what=""):
    assert np.array_equal(np.asarray(ao, dtype=np.uint64), np.asarray(bo, dtype=np.uint64)), f"offsets differ {what}"
    assert np.array_equal(a, b), f"ids differ {what}"


@pytest.mark.parametrize("model,kind", SETS)
def test_golden_dumps(model, kind, corpus_gen):
    """engine == the reference's own output (committed by tools/make_golden.py)"""
    z = np.load(os.path.join(GOLD, "ids", f"{model}__{kind}.npz"))
    buf, offs = corpus_gen.fill(kind, int(z["seed"]), int(z["n"]))
    ids, ido = engine(model).encode_packed(buf, offs)
    assert_same(ids, ido, z["ids"], z["id_offsets"], f"{model}/{kind}")


@pytest.mark.parametrize("model,kind", SETS)
def test_oracle_seeded(model, kind, corpus_gen):
    buf, offs = corpus_gen.fill(kind, 4001, 20000)
    ids, ido = engine(model).encode_packed(buf, offs)
    oids, oido = oracle_py.OracleModel(model_bytes(model)).encode_batch(buf, offs)
    assert_same(ids, ido, oids, oido, f"{model}/{kind}")


@pytest.mark.parametrize("model", ALL_MODELS)
def test_edge_cases(model):
    """empty / whitespace-only / NUL / malformed UTF-8 / user symbols / long sentences that take the
    long-sentence path; as one ragged batch and one by one."""
    with open(os.path.join(GOLD, "edge_cases.json")) as f:
        e = json.load(f)
    inputs = [base64.b64decode(s) for s in e["inputs"]]
    gold = e["models"][model]["ids"]
    buf, offs = oracle_py.pack(inputs)
    ids, ido = engine(model).encode_packed(buf, offs)
    for k in range(len(inputs)):
        assert ids[int(ido[k]):int(ido[k + 1])].tolist() == gold[k], (model, k, inputs[k][:40])
    for k in (0, 1, 5, 12, 18, 28):
        b1, o1 = oracle_py.pack([inputs[k]])
        i1, io1 = engine(model).encode_packed(b1, o1)
        assert i1.tolist() == gold[k]


def test_empty_batch_and_offsets_base():
    eng = engine("uni32k")
    ids, ido = eng.encode_packed(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    assert len(ids) == 0 and ido.tolist() == [0]
    # offsets that do not start at 0 (a window into a larger buffer)
    s = [b"hello world", b"second sentence here", b"", b"third"]
    buf, offs = oracle_py.pack([b"PADDING"] + s)
    ids, ido = eng.encode_packed(buf, offs[1:])
    ref, rido = oracle_py.OracleModel(model_bytes("uni32k")).encode_batch(*oracle_py.pack(s))
    assert_same(ids, ido, ref, rido)


@pytest.mark.parametrize("model", ["uni32k", "bpe32k"])
def test_very_long_sentences(model, corpus_gen):
    """sentences far beyond the shared-memory capacity (global-scratch path), up to ~1 MB"""
    lines = corpus_gen.lines("en", 4002, 9000)
    big = [b" ".join(lines[:8]), b" ".join(lines[8:200]), b" ".join(lines[200:8200]) if model == "uni32k" else
           b" ".join(lines[200:400]), b"tail"]
    buf, offs = oracle_py.pack(big)
    ids, ido = engine(model).encode_packed(buf, offs)
    oids, oido = oracle_py.OracleModel(model_bytes(model)).encode_batch(buf, offs)
    assert_same(ids, ido, oids, oido)
    assert engine(model).info().last_deferred >= 2


@pytest.mark.parametrize("model", ["uni32k", "bpe32k"])
def test_set_vocabulary_live_types(model, corpus_gen):
    """spm_engine_set_types == SetVocabulary / ResetVocabulary (sentencepiece_processor.cc:301-340)"""
    from sentencepiece_b200 import Engine
    mb = model_bytes(model)
    eng = Engine(mb)
    om = oracle_py.OracleModel(mb)
    rng = np.random.default_rng(11)
    keep = [p for p in om.proto["pieces"] if rng.random() < 0.5]
    t = om.vocabulary_types(keep)
    buf, offs = corpus_gen.fill("en", 4003, 3000)
    # first with the full vocabulary (fills the BPE word cache, which must not survive the change of types)
    assert_same(*eng.encode_packed(buf, offs), *om.encode_batch(buf, offs), "full vocabulary")
    om.set_types(t)
    eng.set_types(t)
    assert_same(*eng.encode_packed(buf, offs), *om.encode_batch(buf, offs), "restricted vocabulary")
    om.set_types(om.types)
    eng.set_types(om.types)
    assert_same(*eng.encode_packed(buf, offs), *om.encode_batch(buf, offs), "reset vocabulary")
    eng.close()


@pytest.mark.parametrize("model,kind", [("bpe32k", "en"), ("mix_bpe4k", "mixed")])
def test_bpe_word_cache_is_transparent(model, kind, corpus_gen, monkeypatch):
    """the BPE lane kernel's word cache (bpe_lane2_kernel.cuh) only ever returns what the merge loop would: cold cache,
    warm cache (second call, other sentences with the same words), a tiny table (every slot contended) and no cache
    give the oracle's ids"""
    from sentencepiece_b200 import Engine
    mb = model_bytes(model)
    om = oracle_py.OracleModel(mb)
    b1, o1 = corpus_gen.fill(kind, 4101, 20000)
    b2, o2 = corpus_gen.fill(kind, 4102, 20000)
    want1, want2 = om.encode_batch(b1, o1), om.encode_batch(b2, o2)
    for log2 in (None, 8, 0):
        if log2 is None:
            monkeypatch.delenv("SPM_B200_BPE_CACHE", raising=False)
        else:
            monkeypatch.setenv("SPM_B200_BPE_CACHE", str(log2))
        eng = Engine(mb)
        assert_same(*eng.encode_packed(b1, o1), *want1, f"cold cache (log2 {log2})")
        assert_same(*eng.encode_packed(b2, o2), *want2, f"warm cache (log2 {log2})")
        assert_same(*eng.encode_packed(b1, o1), *want1, f"warm cache, first batch again (log2 {log2})")
        eng.close()


@pytest.mark.parametrize("flags", [dict(add_dummy_prefix=False), dict(remove_extra_whitespaces=False),
                                   dict(escape_whitespaces=False, add_dummy_prefix=False),
                                   dict(treat_whitespace_as_suffix=True),
                                   dict(escape_whitespaces=False, remove_extra_whitespaces=False)])
def test_normalizer_flag_variants(flags, corpus_gen):
    """the flag variants of src/normalizer_test.cc:77-147 on a real model and corpus"""
    from sentencepiece_b200 import Engine
    mb = mp.replace_flags(model_bytes("mix_bf8k"), **flags)
    eng = Engine(mb)
    buf, offs = corpus_gen.fill("mixed", 4004, 3000)
    assert_same(*eng.encode_packed(buf, offs), *oracle_py.OracleModel(mb).encode_batch(buf, offs), str(flags))
    eng.close()


def test_toy_models_from_reference_tests():
    """the synthetic models of unigram_model_test.cc:782-871 / bpe_model_test.cc:49-250 through the
    full engine (identity normalizer), including USER_DEFINED and UNUSED pieces"""
    from sentencepiece_b200 import Engine
    from test_oracle_kat import BASE, ENCODE_PIECES, UNUSED_PIECES
    texts = [b"abc", b"AB", b"abcd", b"abcc", b"xabcabaabcdd", "xyz東京".encode(), b"ABC", b"abABCcd",
             b"ababcdabcdcd", b"abqrcd", b"", b"  ab  cd "]
    for mt in (mp.UNIGRAM, mp.BPE):
        pcs = BASE + [(p, s, mp.NORMAL) for p, s in ENCODE_PIECES]
        for i in (9, 10, 11, 12):
            pcs[i] = (pcs[i][0], pcs[i][1], mp.USER_DEFINED)
        for unused in ((), (3,), (3, 5), (3, 4)):
            variants = [mp.build_model(pcs, model_type=mt, charsmap=b"", add_dummy_prefix=False)]
            up = BASE + [(p, s, mp.UNUSED if 3 + i in unused else mp.NORMAL) for i, (p, s) in enumerate(UNUSED_PIECES)]
            variants.append(mp.build_model(up, model_type=mt, charsmap=b"", add_dummy_prefix=False))
            for mb in variants:
                eng = Engine(mb)
                buf, offs = oracle_py.pack(texts)
                assert_same(*eng.encode_packed(buf, offs), *oracle_py.OracleModel(mb).encode_batch(buf, offs),
                            f"type={mt} unused={unused}")
                eng.close()


@pytest.mark.parametrize("model,kind", [("uni32k", "mixed"), ("mix_bf8k", "mixed"), ("bpe32k", "en")])
def test_spans_api(model, kind, corpus_gen):
    """spm_encode_spans: ids, token end offsets, normalized text and norm_to_orig alignment
    (what EncodeAsPieces / the SentencePieceText overload need), vs the oracle"""
    lines = corpus_gen.lines(kind, 4005, 600) + [b"", b"   ", b"a"]
    buf, offs = oracle_py.pack(lines)
    r = engine(model).encode_spans(buf, offs)
    om = oracle_py.OracleModel(model_bytes(model))
    for i, s in enumerate(lines):
        ids, te = om.encode(s)
        nrm, n2o = om.normalize(s)
        a, b = int(r["id_offsets"][i]), int(r["id_offsets"][i + 1])
        assert r["ids"][a:b].tolist() == ids.tolist(), i
        assert r["tok_end"][a:b].tolist() == te.tolist(), i
        na, nb = int(r["norm_offsets"][i]), int(r["norm_offsets"][i + 1])
        assert r["normalized"][na:nb] == nrm, i
        if len(nrm):
            assert r["n2o"][na + i: nb + i + 1].tolist() == n2o, i


def test_device_pointer_api(corpus_gen):
    """spm_encode_ids_device with torch-owned device buffers"""
    import torch
    buf, offs = corpus_gen.fill("en", 4006, 5000)
    dev = torch.device("cuda", 0)
    d_b = torch.from_numpy(buf.copy()).to(dev)
    d_o = torch.from_numpy(offs.astype(np.int64)).to(dev)
    cap = len(buf) + 4 * 5000 + 1024
    d_ids = torch.empty(cap, dtype=torch.int32, device=dev)
    d_ido = torch.empty(5001, dtype=torch.int64, device=dev)
    tot = engine("uni32k").encode_device(d_b.data_ptr(), d_o.data_ptr(), 5000, len(buf), d_ids.data_ptr(), cap,
                                         d_ido.data_ptr(), None)
    oids, oido = oracle_py.OracleModel(model_bytes("uni32k")).encode_batch(buf, offs)
    assert tot == len(oids)
    assert np.array_equal(d_ids[:tot].cpu().numpy(), oids)
    assert np.array_equal(d_ido.cpu().numpy().astype(np.uint64), oido)


def test_tuning_variants_agree(corpus_gen):
    """every kernel variant (tile widths, CTA sizes, the general tile kernel) gives the same ids"""
    from sentencepiece_b200 import Engine
    buf, offs = corpus_gen.fill("mixed", 4007, 4000)
    mb = model_bytes("mix_bf8k")
    ref = oracle_py.OracleModel(mb).encode_batch(buf, offs)
    for lanes, cap, thr in [(32, 256, 1024), (32, 128, 512), (8, 256, 256), (16, 192, 512), (4, 128, 128)]:
        eng = Engine(mb)
        eng.set_tuning(lanes, cap, thr)
        assert_same(*eng.encode_packed(buf, offs), *ref, f"lanes={lanes} cap={cap} threads={thr}")
        eng.close()


@pytest.mark.parametrize("workload", [("uni32k", "en"), ("bpe32k", "en")])
def test_full_size_properties(workload, corpus_gen):
    """BASELINE.json's full size (1M sentences): size-independent properties --
    determinism/idempotence, shard additivity (encode(A+B) == encode(A) ++ encode(B)),
    a checksum against the live reference on a strided sample."""
    model, kind = workload
    n = 1_000_000
    buf, offs = corpus_gen.fill(kind, 20260922, n)
    eng = engine(model)
    ids, ido = eng.encode_packed(buf, offs)
    ids2, ido2 = eng.encode_packed(buf, offs)
    assert np.array_equal(ids, ids2) and np.array_equal(ido, ido2)
    h = n // 2
    a, ao = eng.encode_packed(buf, offs[: h + 1])
    b, bo = eng.encode_packed(buf, offs[h:])
    assert np.array_equal(np.concatenate([a, b]), ids)
    assert np.array_equal(np.concatenate([ao[:-1], bo + ao[-1]]), ido)
    # every id is a valid vocab id, every non-empty sentence has at least one id
    assert ids.min() >= 0 and ids.max() < eng.info().vocab_size
    assert np.all((ido[1:] - ido[:-1])[(offs[1:] - offs[:-1]) > 0] > 0)
    # strided sample vs the oracle
    om = oracle_py.OracleModel(model_bytes(model))
    raw = buf.tobytes()
    for i in range(0, n, 9973):
        s = raw[int(offs[i]):int(offs[i + 1])]
        assert ids[int(ido[i]):int(ido[i + 1])].tolist() == om.encode(s)[0].tolist(), i


@pytest.mark.parametrize("model,kind", [("uni32k", "en"), ("mix_bf8k", "mixed"), ("bpe32k", "en")])
def test_live_reference(model, kind, corpus_gen, request):
    buf, offs = corpus_gen.fill(kind, 4008, 50000)
    Reference(request).check("encode", engine(model).encode_packed(buf, offs),
                             lambda: oracle_py.RefModel(model_bytes(model)).encode_batch(buf, offs, threads=16))
