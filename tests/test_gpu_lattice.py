"""Full-lattice operations (SURVEY 8f item 1) through the C ABI: SampleEncode with nbest_size < 0 (forward-filtering /
backward-sampling), SampleEncodeAndScore(wor=False) and CalculateEntropy, against the oracle (pinned against the
reference in tests/test_oracle_lattice.py) and the reference's outputs (kept as digests, tests/reference_outputs.py).  Sampled ids bit-exact under a seed (one generator,
sentence order); sample scores and entropies within float rounding (1e-5 relative: the device's exp/log differ from
glibc's in the last place).  Needs a B200."""
import numpy as np
import pytest

from conftest import model_bytes
from oracle import oracle_py
from reference_outputs import Reference

pytestmark = pytest.mark.gpu
EDGE = [b"", b"   ", b"x", b"hello world", "こんにちは \U0001F600\U0001F600 ok".encode(), b"\xff\xfe broken"]


def _engine(model):
    from sentencepiece_b200 import Engine
    return Engine(model_bytes(model))


@pytest.mark.parametrize("model,kind,alpha", [("uni32k", "en", 0.5), ("uni32k", "en", 0.0), ("mix_bf8k", "mixed", 0.2),
                                              ("botchan8k", "mixed", 1.0)])
def test_sample_lattice_seeded(model, kind, alpha, corpus_gen):
    lines = corpus_gen.lines(kind, 9201, 3000) + EDGE
    buf, offs = oracle_py.pack(lines)
    eng = _engine(model)
    om = oracle_py.OracleModel(model_bytes(model))
    for seed in (5, 20260922):
        eng.set_random_seed(seed)
        ids, ido = eng.sample_encode(buf, offs, -1, alpha)
        oids, oido = om.sample_encode_batch(buf, offs, -1, alpha, seed)
        assert np.array_equal(ido, oido) and np.array_equal(ids, oids), seed
    v, vo = eng.encode_packed(buf, offs)
    assert not (np.array_equal(v, ids) and np.array_equal(vo, ido))  # it does sample
    eng.close()


def test_sample_lattice_vs_live_reference(corpus_gen, request):
    lines = corpus_gen.lines("en", 9202, 40000)   # spans two chunks of the engine's lattice path
    buf, offs = oracle_py.pack(lines)
    mb = model_bytes("uni32k")
    eng = _engine("uni32k")
    eng.set_random_seed(4711)
    Reference(request).check("sample", eng.sample_encode(buf, offs, -1, 0.5),
                             lambda: oracle_py.RefModel(mb).sample_encode_batch(buf, offs, -1, 0.5, 4711))
    eng.close()


@pytest.mark.parametrize("model,kind,alpha", [("uni32k", "en", 0.5), ("mix_bf8k", "mixed", 0.1), ("botchan8k", "en", 1.0)])
def test_entropy(model, kind, alpha, corpus_gen):
    lines = corpus_gen.lines(kind, 9203, 2000) + EDGE
    buf, offs = oracle_py.pack(lines)
    eng = _engine(model)
    ent = eng.calculate_entropy(buf, offs, alpha)
    exp = oracle_py.OracleModel(model_bytes(model)).entropy_batch(buf, offs, alpha)
    assert ent.shape == exp.shape and np.all(np.isfinite(ent))
    np.testing.assert_allclose(ent, exp, rtol=2e-5, atol=2e-5)
    eng.close()


@pytest.mark.parametrize("model,kind,samples,alpha", [("uni32k", "en", 4, 0.5), ("mix_bf8k", "mixed", 3, 0.2)])
def test_sample_encode_and_score(model, kind, samples, alpha, corpus_gen):
    lines = corpus_gen.lines(kind, 9204, 1500) + [b"x", b"hello world"]
    buf, offs = oracle_py.pack(lines)
    eng = _engine(model)
    eng.set_random_seed(99)
    ids, co, sc = eng.sample_encode_and_score(buf, offs, samples, alpha)
    oids, oco, osc = oracle_py.OracleModel(model_bytes(model)).sample_score_batch(buf, offs, samples, alpha, 99)
    assert np.array_equal(co, oco) and np.array_equal(ids, oids)
    np.testing.assert_allclose(sc, osc, rtol=2e-5, atol=2e-5)
    eng.close()
