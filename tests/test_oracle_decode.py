"""Oracle restatement of SentencePieceProcessor::Decode(ids) (oracle/spm_oracle.c, oracle_decode_ids):
the reference's own known answers (sentencepiece_processor_test.cc DecodeTest :544-640,
ByteFallbackDecodeTest :790-900, restated over ids) and the reference's outputs (kept as digests,
tests/reference_outputs.py) on round trips, random id lists and normalizer-flag variants.  CPU only."""
import numpy as np
import pytest

from conftest import model_bytes
from oracle import modelproto as mp
from oracle import oracle_py
from reference_outputs import Reference

WS = "▁"
N, U, C, B = mp.NORMAL, mp.UNKNOWN, mp.CONTROL, mp.BYTE


def _decode(om, ids):
    ido = np.array([0, len(ids)], dtype=np.uint64)
    text, to = om.decode_batch(np.asarray(ids, dtype=np.int32), ido)
    return text.tobytes().decode("utf-8")


def _toy(**kw):
    pieces = [("<unk>", 0.0, U), ("<s>", 0.0, C), ("</s>", 0.0, C), (WS + "ABC", 0.0, N), (WS + "DE", 0.0, N),
              ("F", 0.0, N), ("G" + WS + "H", 0.0, N)]
    return oracle_py.OracleModel(mp.build_model(pieces, **kw))


def test_kat_decode_test():
    # sentencepiece_processor_test.cc:575-590 without the out-of-vocabulary piece "I"
    om = _toy()
    assert _decode(om, [1, 3, 0, 4, 5, 6, 2]) == "ABC ⁇  DEFG H"
    assert _decode(om, []) == ""
    assert _decode(om, [1, 2]) == ""
    # only the first U+2581 goes when add_dummy_prefix is set without remove_extra_whitespaces (:792-807)
    om2 = _toy(remove_extra_whitespaces=False)
    assert _decode(om2, [3, 4]) == "ABC DE"
    assert _decode(om2, [1, 3, 3]) == "ABC ABC"
    # neither flag: nothing is stripped
    om3 = _toy(add_dummy_prefix=False, remove_extra_whitespaces=False)
    assert _decode(om3, [3, 4]) == " ABC DE"


def test_kat_leading_whitespace_pieces():
    pieces = [("<unk>", 0.0, U), (WS, 0.0, N), (WS + WS, 0.0, N), (WS + "a", 0.0, N), ("b", 0.0, N)]
    rm = oracle_py.OracleModel(mp.build_model(pieces))                                   # remove_extra_whitespaces
    assert _decode(rm, [1, 1, 3, 3]) == "a a"          # every leading U+2581 goes while the text is empty
    assert _decode(rm, [2, 4]) == " b"                 # only ONE U+2581 per piece is consumed
    norm = oracle_py.OracleModel(mp.build_model(pieces, remove_extra_whitespaces=False))  # add_dummy_prefix only
    assert _decode(norm, [1, 1, 3]) == "  a"           # the first consumed U+2581 closes the state
    assert _decode(norm, [0, 3]) == " ⁇  a"


def test_kat_byte_fallback_decode():
    # sentencepiece_processor_test.cc:843-872
    pieces = [("<unk>", 0.0, U), ("<s>", 0.0, C), ("</s>", 0.0, C), ("A", 0.0, N), ("B", 0.0, N), ("C", 0.0, N)]
    pieces += [("<0x%02X>" % i, 0.0, B) for i in range(256)]
    om = oracle_py.OracleModel(mp.build_model(pieces, byte_fallback=True))
    b = lambda x: 6 + x  # noqa: E731
    ids = [1, 3, 4, b(0xE3), b(0x81), b(0x82), b(0x5A), b(0xCE), b(0xA9), 5, b(0xE0), b(0x80), b(0xE3), b(0x81), b(0x84),
           b(0xEF), b(0xBF), b(0xBD)]
    assert _decode(om, ids) == "ABあZΩC��い�"
    # a byte run is flushed before the next piece; a run that ends inside a character is invalid byte by byte
    assert _decode(om, [b(0xE3), b(0x81), 3]) == "��A"


def test_out_of_range_id_fails():
    om = _toy()
    with pytest.raises(RuntimeError):
        _decode(om, [3, 7])
    with pytest.raises(RuntimeError):
        _decode(om, [-1])


@pytest.mark.parametrize("model,kind", [("uni32k", "en"), ("mix_bf8k", "mixed"), ("bpe32k", "en"), ("mix_bpe4k", "mixed")])
def test_oracle_decode_vs_live_reference(model, kind, corpus_gen, request):
    rng = np.random.default_rng(11)
    ref = Reference(request)
    base = model_bytes(model)
    variants = [base, mp.replace_flags(base, add_dummy_prefix=False), mp.replace_flags(base, remove_extra_whitespaces=False),
                mp.replace_flags(base, add_dummy_prefix=False, remove_extra_whitespaces=False)]
    for v, mb in enumerate(variants):
        om = oracle_py.OracleModel(mb)
        buf, offs = corpus_gen.fill(kind, 9101, 1500)
        ids, ido = om.encode_batch(buf, offs)
        ref.check(f"encode{v}", (ids, ido), lambda: oracle_py.RefModel(mb).encode_batch(buf, offs, threads=4))
        ref.check(f"roundtrip{v}", om.decode_batch(ids, ido), lambda: oracle_py.RefModel(mb).decode_batch(ids, ido, threads=4))
        vocab = len(om.proto["pieces"])
        special = np.nonzero(np.asarray(om.proto["types"]) != mp.NORMAL)[0]
        lists = []
        for _ in range(1500):
            a = rng.integers(0, vocab, size=int(rng.integers(0, 24)))
            m = rng.random(len(a)) < 0.4
            if len(special) and m.any():
                a[m] = rng.choice(special, size=int(m.sum()))
            lists.append(a.astype(np.int32))
        ido2 = np.zeros(len(lists) + 1, dtype=np.uint64)
        ido2[1:] = np.cumsum([len(x) for x in lists])
        ids2 = np.concatenate(lists)
        ref.check(f"random{v}", om.decode_batch(ids2, ido2), lambda: oracle_py.RefModel(mb).decode_batch(ids2, ido2, threads=4))
