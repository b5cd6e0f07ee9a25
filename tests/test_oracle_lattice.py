"""Pins the oracle's full-lattice restatement (SURVEY 8f item 1) against the reference's outputs (kept as digests,
tests/reference_outputs.py): SampleEncode with
nbest_size < 0 (forward-filtering / backward-sampling, unigram_model.cc:511-542), SampleEncodeAndScore with
wor = false (:741-855) and CalculateEntropy (:266-291).  Sampled ids and sample scores bit for bit under a fixed seed
(one generator, sentences in order); entropies bit for bit as well (same libm as the reference's run).  CPU only."""
import numpy as np
import pytest

from conftest import model_bytes
from oracle import oracle_py
from reference_outputs import Reference

EDGE = [b"", b"   ", b"x", b"hello world", "こんにちは \U0001F600\U0001F600 ok".encode(), b"\xff\xfe broken"]


@pytest.mark.parametrize("model,kind,alpha", [("uni32k", "en", 0.5), ("uni32k", "en", 0.0), ("mix_bf8k", "mixed", 0.2),
                                              ("botchan8k", "mixed", 1.0)])
def test_sample_lattice_vs_reference(model, kind, alpha, corpus_gen, request):
    mb = model_bytes(model)
    lines = corpus_gen.lines(kind, 911, 500) + EDGE
    buf, offs = oracle_py.pack(lines)
    for seed in (3, 20260922):
        Reference(request).check(f"seed{seed}", oracle_py.OracleModel(mb).sample_encode_batch(buf, offs, -1, alpha, seed),
                                 lambda: oracle_py.RefModel(mb).sample_encode_batch(buf, offs, -1, alpha, seed))


@pytest.mark.parametrize("model,kind,alpha", [("uni32k", "en", 0.5), ("mix_bf8k", "mixed", 0.1), ("botchan8k", "en", 1.0)])
def test_entropy_vs_reference(model, kind, alpha, corpus_gen, request):
    mb = model_bytes(model)
    lines = corpus_gen.lines(kind, 912, 400) + EDGE
    buf, offs = oracle_py.pack(lines)
    a = oracle_py.OracleModel(mb).entropy_batch(buf, offs, alpha)
    Reference(request).check("entropy", (a,), lambda: (oracle_py.RefModel(mb).entropy_batch(buf, offs, alpha),))
    assert np.all(np.isfinite(a)) and a[len(lines) - len(EDGE)] == 0.0  # the empty sentence


@pytest.mark.parametrize("model,kind,samples,alpha", [("uni32k", "en", 4, 0.5), ("mix_bf8k", "mixed", 3, 0.2)])
def test_sample_score_vs_reference(model, kind, samples, alpha, corpus_gen, request):
    mb = model_bytes(model)
    lines = corpus_gen.lines(kind, 913, 300) + [b"x", b"hello world"]  # (the reference fails on empty input here)
    buf, offs = oracle_py.pack(lines)
    Reference(request).check("sample_score", oracle_py.OracleModel(mb).sample_score_batch(buf, offs, samples, alpha, 77),
                             lambda: oracle_py.RefModel(mb).sample_score_batch(buf, offs, samples, alpha, 77))
