"""Config 5 (SURVEY 8a rows a7/a8): n-best lists and SampleEncode on the GPU vs the oracle
(which tests/test_oracle_nbest.py pins against the reference incl. libstdc++ heap tie order and the
mt19937 / discrete_distribution draw).  Ids bit-exact, scores bit-exact floats.  Needs a B200."""
import numpy as np
import pytest

from conftest import model_bytes
from oracle import oracle_py
from reference_outputs import Reference

pytestmark = pytest.mark.gpu


def _engine(model):
    from sentencepiece_b200 import Engine
    return Engine(model_bytes(model))


@pytest.mark.parametrize("model,kind,nbest", [("uni32k", "en", 64), ("uni32k", "en", 5), ("mix_bf8k", "mixed", 64),
                                               ("botchan8k", "en", 2), ("uni32k", "mixed", 16)])
def test_nbest_lists(model, kind, nbest, corpus_gen):
    lines = corpus_gen.lines(kind, 8101, 400) + [b"", b"   ", b"a", b"hello world"]
    buf, offs = oracle_py.pack(lines)
    eng = _engine(model)
    r = eng.nbest_encode(buf, offs, nbest)
    om = oracle_py.OracleModel(model_bytes(model))
    K = r["K"]
    for i, s in enumerate(lines):
        cands, scores = om.nbest_encode(s, nbest)
        assert int(r["n_cands"][i]) == len(cands), i
        for c, (ids, sc) in enumerate(zip(cands, scores)):
            a, b = int(r["cand_offsets"][i * K + c]), int(r["cand_offsets"][i * K + c + 1])
            assert r["ids"][a:b].tolist() == ids.tolist(), (i, c)
            assert np.float32(r["scores"][i * K + c]).view(np.uint32) == np.float32(sc).view(np.uint32), (i, c)
    eng.close()


def test_nbest_size_one_is_viterbi(corpus_gen):
    buf, offs = corpus_gen.fill("en", 8102, 500)
    eng = _engine("uni32k")
    r = eng.nbest_encode(buf, offs, 1)
    ids, ido = eng.encode_packed(buf, offs)
    assert np.array_equal(r["ids"], ids) and np.array_equal(r["cand_offsets"], ido)
    assert np.all(r["scores"] == 0) and np.all(r["n_cands"] == 1)
    eng.close()


@pytest.mark.parametrize("model,kind,nbest,alpha", [("uni32k", "en", 64, 0.5), ("mix_bf8k", "mixed", 8, 0.1),
                                                     ("uni32k", "en", 2, 1.0)])
def test_sample_encode_seeded(model, kind, nbest, alpha, corpus_gen):
    """SampleEncode(nbest_size, alpha) with SetRandomGeneratorSeed: the draw sequence is defined for one
    generator consumed in sentence order (two 32-bit draws per sentence with >= 2 candidates)."""
    lines = corpus_gen.lines(kind, 8103, 1500) + [b"", b"  ", b"x"]
    buf, offs = oracle_py.pack(lines)
    eng = _engine(model)
    om = oracle_py.OracleModel(model_bytes(model))
    for seed in (1, 12345):
        eng.set_random_seed(seed)
        ids, ido = eng.sample_encode(buf, offs, nbest, alpha)
        oids, oido = om.sample_encode_batch(buf, offs, nbest, alpha, seed)
        assert np.array_equal(ido, oido) and np.array_equal(ids, oids), seed
    # sampling must actually deviate from the Viterbi path for some sentences
    v, vo = eng.encode_packed(buf, offs)
    assert not (np.array_equal(v, ids) and np.array_equal(vo, ido))
    # nbest_size 0 / 1 is the plain encode (sentencepiece_processor.cc:695-698)
    p, po = eng.sample_encode(buf, offs, 1, alpha)
    assert np.array_equal(p, v) and np.array_equal(po, vo)
    eng.close()


def test_sample_encode_vs_live_reference(corpus_gen, request):
    lines = corpus_gen.lines("en", 8104, 3000)
    buf, offs = oracle_py.pack(lines)
    mb = model_bytes("uni32k")
    eng = _engine("uni32k")
    eng.set_random_seed(777)
    Reference(request).check("sample", eng.sample_encode(buf, offs, 64, 0.5),
                             lambda: oracle_py.RefModel(mb).sample_encode_batch(buf, offs, 64, 0.5, 777))
    eng.close()


def test_nbest_error_behaviour(corpus_gen):
    buf, offs = corpus_gen.fill("en", 8105, 10)
    bpe = _engine("bpe32k")
    with pytest.raises(RuntimeError, match="NBestEncode is not available"):
        bpe.nbest_encode(buf, offs, 4)
    bpe.close()
    uni = _engine("uni32k")
    with pytest.raises(RuntimeError, match="nbest_size <= 512"):
        uni.sample_encode(buf, offs, 513, 0.5)
    with pytest.raises(RuntimeError, match="wor / include_best"):
        uni.sample_encode_and_score(buf, offs, 3, 0.5, wor=True)
    uni.close()
    # BPE: SampleEncode is BPE-dropout whatever nbest_size is (sentencepiece_processor.cc:689-693); only alpha <= 0
    # equals Encode, alpha > 0 is refused rather than silently returning the deterministic encode
    bpe = _engine("bpe32k")
    with pytest.raises(RuntimeError, match="BPE-dropout"):
        bpe.sample_encode(buf, offs, 1, 0.1)
    a, ao = bpe.sample_encode(buf, offs, 64, 0.0)
    b, bo = bpe.encode_packed(buf, offs)
    assert np.array_equal(a, b) and np.array_equal(ao, bo)
    with pytest.raises(RuntimeError, match="CalculateEntropy is not available"):
        bpe.calculate_entropy(buf, offs, 0.5)
    bpe.close()


@pytest.mark.parametrize("nbest", [512, 1024])
def test_nbest_large(nbest, corpus_gen):
    """nbest 512 / 1024 (the clamp of unigram_model.cc:701): on ~130-byte sentences the agenda passes 10,000 entries and
    is shrunk to min(512, 10 * nbest) (:481-505); hypothesis pools overflow the first attempt's capacity and the batch is
    redone with roomy slabs."""
    lines = corpus_gen.lines("en", 8106, 24) + [b"a", b""]
    buf, offs = oracle_py.pack(lines)
    eng = _engine("uni32k")
    r = eng.nbest_encode(buf, offs, nbest)
    om = oracle_py.OracleModel(model_bytes("uni32k"))
    K = r["K"]
    assert K == nbest
    for i, s in enumerate(lines):
        cands, scores = om.nbest_encode(s, nbest)
        assert int(r["n_cands"][i]) == len(cands), i
        for c, (ids, sc) in enumerate(zip(cands, scores)):
            a, b = int(r["cand_offsets"][i * K + c]), int(r["cand_offsets"][i * K + c + 1])
            assert r["ids"][a:b].tolist() == ids.tolist(), (i, c)
            assert np.float32(r["scores"][i * K + c]).view(np.uint32) == np.float32(sc).view(np.uint32), (i, c)
    eng.close()


def test_nbest_and_sampling_long_sentences(corpus_gen):
    """Sentences beyond the 512 normalized bytes of the fast slabs (up to ~8 KB) are redone with roomy slabs instead of
    being refused: n-best lists, seeded n-best sampling and seeded lattice sampling against the oracle."""
    short = corpus_gen.lines("en", 8107, 40)
    long1 = b" ".join(corpus_gen.lines("en", 8108, 12))            # ~1.6 KB
    long2 = " ".join(l.decode("utf8", "replace") for l in corpus_gen.lines("mixed", 8109, 10)).encode()
    lines = short[:20] + [long1] + short[20:] + [long2, b"x"]
    buf, offs = oracle_py.pack(lines)
    assert max(len(x) for x in lines) > 1500
    eng = _engine("uni32k")
    om = oracle_py.OracleModel(model_bytes("uni32k"))
    r = eng.nbest_encode(buf, offs, 8)
    K = r["K"]
    for i, s in enumerate(lines):
        cands, scores = om.nbest_encode(s, 8)
        assert int(r["n_cands"][i]) == len(cands), i
        for c, (ids, sc) in enumerate(zip(cands, scores)):
            a, b = int(r["cand_offsets"][i * K + c]), int(r["cand_offsets"][i * K + c + 1])
            assert r["ids"][a:b].tolist() == ids.tolist(), (i, c)
            assert np.float32(r["scores"][i * K + c]).view(np.uint32) == np.float32(sc).view(np.uint32), (i, c)
    for nb in (8, -1):
        eng.set_random_seed(31337)
        ids, ido = eng.sample_encode(buf, offs, nb, 0.3)
        oids, oido = om.sample_encode_batch(buf, offs, nb, 0.3, 31337)
        assert np.array_equal(ido, oido) and np.array_equal(ids, oids), nb
    ent = eng.calculate_entropy(buf, offs, 0.3)
    np.testing.assert_allclose(ent, om.entropy_batch(buf, offs, 0.3), rtol=2e-5, atol=2e-5)
    eng.close()
