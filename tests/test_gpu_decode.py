"""spm_decode_ids (K7, decode_kernel.cuh) against the oracle restatement of
SentencePieceProcessor::Decode(ids) and the reference's outputs (kept as digests, tests/reference_outputs.py).  Needs a B200."""
import numpy as np
import pytest

from conftest import model_bytes
from oracle import modelproto as mp
from oracle import oracle_py
from reference_outputs import Reference

pytestmark = pytest.mark.gpu
WS = "▁"


def _lists_to_packed(lists):
    ido = np.zeros(len(lists) + 1, dtype=np.uint64)
    if lists:
        ido[1:] = np.cumsum([len(x) for x in lists])
    ids = np.concatenate([np.asarray(x, dtype=np.int32) for x in lists]) if int(ido[-1]) else np.zeros(0, np.int32)
    return ids, ido


def _random_lists(om, rng, n, maxlen):
    vocab = len(om.proto["pieces"])
    special = np.nonzero(np.asarray(om.proto["types"]) != mp.NORMAL)[0]
    lists = []
    for _ in range(n):
        a = rng.integers(0, vocab, size=int(rng.integers(0, maxlen)))
        m = rng.random(len(a)) < 0.35
        if len(special) and m.any():
            a[m] = rng.choice(special, size=int(m.sum()))
        lists.append(a.astype(np.int32))
    return lists


@pytest.mark.parametrize("model,kind", [("uni32k", "en"), ("mix_bf8k", "mixed"), ("bpe32k", "en"), ("botchan8k", "en"),
                                        ("mix_bpe4k", "mixed")])
def test_decode_round_trip_and_random_lists(model, kind, corpus_gen):
    from sentencepiece_b200 import Engine
    rng = np.random.default_rng(21)
    base = model_bytes(model)
    variants = [base, mp.replace_flags(base, remove_extra_whitespaces=False),
                mp.replace_flags(base, add_dummy_prefix=False, remove_extra_whitespaces=False)]
    for vi, mb in enumerate(variants):
        eng = Engine(mb)
        om = oracle_py.OracleModel(mb)
        buf, offs = corpus_gen.fill(kind, 9201, 20000 if vi == 0 else 2000)
        ids, ido = eng.encode_packed(buf, offs)
        text, to = eng.decode_packed(ids, ido)
        otext, oto = om.decode_batch(ids, ido)
        assert np.array_equal(to, oto) and np.array_equal(text, otext), f"{model} variant {vi} round trip"
        # lists with control / unknown / byte pieces, broken UTF-8 byte runs, empty lists, > 32 and > 64 tokens
        lists = _random_lists(om, rng, 3000, 24) + _random_lists(om, rng, 200, 150) + [[], []]
        ids2, ido2 = _lists_to_packed(lists)
        text, to = eng.decode_packed(ids2, ido2)
        otext, oto = om.decode_batch(ids2, ido2)
        assert np.array_equal(to, oto) and np.array_equal(text, otext), f"{model} variant {vi} random lists"
        eng.close()


def test_decode_toy_models_and_errors():
    from sentencepiece_b200 import Engine, SentencePieceProcessor
    N, U, C, B = mp.NORMAL, mp.UNKNOWN, mp.CONTROL, mp.BYTE
    pieces = [("<unk>", 0.0, U), ("<s>", 0.0, C), ("</s>", 0.0, C), (WS + "ABC", 0.0, N), (WS + "DE", 0.0, N),
              ("F", 0.0, N), ("G" + WS + "H", 0.0, N), (WS, 0.0, N), (WS + WS, 0.0, N)]
    for kw in ({}, dict(remove_extra_whitespaces=False), dict(add_dummy_prefix=False, remove_extra_whitespaces=False)):
        mb = mp.build_model(pieces, **kw)
        eng = Engine(mb)
        om = oracle_py.OracleModel(mb)
        lists = [[1, 3, 0, 4, 5, 6, 2], [], [1, 2], [7, 7, 3, 3], [8, 5], [0, 3], [7], [8], [1, 7, 2, 8, 3]]
        ids, ido = _lists_to_packed(lists)
        text, to = eng.decode_packed(ids, ido)
        otext, oto = om.decode_batch(ids, ido)
        assert np.array_equal(to, oto) and np.array_equal(text, otext), kw
        if not kw:
            raw = text.tobytes()
            assert raw[int(to[0]):int(to[1])].decode() == "ABC ⁇  DEFG H"  # sentencepiece_processor_test.cc:590
        with pytest.raises(RuntimeError, match="Invalid id: 9"):
            eng.decode_packed(*_lists_to_packed([[3], [4, 9]]))
        with pytest.raises(RuntimeError, match="Invalid id: -1"):
            eng.decode_packed(*_lists_to_packed([[-1]]))
        eng.close()
    # byte fallback KAT, sentencepiece_processor_test.cc:843-872
    bp = [("<unk>", 0.0, U), ("<s>", 0.0, C), ("</s>", 0.0, C), ("A", 0.0, N), ("B", 0.0, N), ("C", 0.0, N)]
    bp += [("<0x%02X>" % i, 0.0, B) for i in range(256)]
    sp = SentencePieceProcessor(model_proto=mp.build_model(bp, byte_fallback=True))
    b = lambda x: 6 + x  # noqa: E731
    ids = [1, 3, 4, b(0xE3), b(0x81), b(0x82), b(0x5A), b(0xCE), b(0xA9), 5, b(0xE0), b(0x80), b(0xE3), b(0x81), b(0x84),
           b(0xEF), b(0xBF), b(0xBD)]
    assert sp.DecodeIds(ids) == "ABあZΩC��い�"
    assert sp.DecodeIds([ids, [b(0xE3), b(0x81), 3]]) == ["ABあZΩC��い�", "��A"]


def test_decode_vs_live_reference_large(corpus_gen, request):
    from sentencepiece_b200 import Engine
    ref = Reference(request)
    for model, kind in (("uni32k", "en"), ("mix_bf8k", "mixed")):
        mb = model_bytes(model)
        eng = Engine(mb)
        buf, offs = corpus_gen.fill(kind, 9202, 200000)
        ids, ido = eng.encode_packed(buf, offs)
        ref.check(f"decode_{model}", eng.decode_packed(ids, ido),
                  lambda: oracle_py.RefModel(mb).decode_batch(ids, ido, threads=16))
        eng.close()
