"""Pins the oracle's n-best / sampling restatement (SURVEY 8a rows a7/a8) against the reference's outputs
(kept as digests, tests/reference_outputs.py):
candidate ids, float scores bit for bit (the order among ties is libstdc++'s heap order), the agenda
shrink path (nbest 512 on long sentences) and the seeded SampleEncode draw.  CPU only."""
import numpy as np
import pytest

from conftest import model_bytes
from oracle import modelproto as mp
from oracle import oracle_py
from reference_outputs import Reference


def nbest_all(m, lines, nbest_size):
    """n-best lists of every line, flattened: (candidates per line, ids per candidate, ids, float32 scores)"""
    out = [m.nbest_encode(s, nbest_size) for s in lines]
    cands = [c for cs, _ in out for c in cs]
    return ([len(cs) for cs, _ in out], [len(c) for c in cands], np.concatenate([np.zeros(0, np.int32)] + cands),
            np.concatenate([np.zeros(0, np.float32)] + [np.asarray(sc, np.float32) for _, sc in out]))


@pytest.mark.parametrize("model,kind", [("uni32k", "en"), ("mix_bf8k", "mixed"), ("botchan8k", "en")])
def test_nbest_vs_reference(model, kind, corpus_gen, request):
    mb = model_bytes(model)
    om, ref = oracle_py.OracleModel(mb), Reference(request)
    lines = corpus_gen.lines(kind, 321, 250) + [b"", b"   ", b"a", b"hello world"]
    ref.check("nbest64", nbest_all(om, lines, 64), lambda: nbest_all(oracle_py.RefModel(mb), lines, 64))
    for nb in (1, 2, 5, 512, 2000):  # 512 on these sentences goes through the agenda shrink (:481-505)
        ref.check(f"nbest{nb}", nbest_all(om, lines[:6], nb), lambda: nbest_all(oracle_py.RefModel(mb), lines[:6], nb))


@pytest.mark.parametrize("model,kind,nbest,alpha", [("uni32k", "en", 64, 0.5), ("mix_bf8k", "mixed", 8, 0.1)])
def test_sample_encode_vs_reference(model, kind, nbest, alpha, corpus_gen, request):
    mb = model_bytes(model)
    lines = corpus_gen.lines(kind, 322, 400) + [b"", b"  ", b"x"]
    buf, offs = oracle_py.pack(lines)
    for seed in (7, 4242):
        Reference(request).check(f"seed{seed}", oracle_py.OracleModel(mb).sample_encode_batch(buf, offs, nbest, alpha, seed),
                                 lambda: oracle_py.RefModel(mb).sample_encode_batch(buf, offs, nbest, alpha, seed))


# src/unigram_model_test.cc:195-238 (Viterbi / NBest on a hand-made lattice): the 2-best of "ABC" with
# pieces A,B,C,AB,BC,ABC scored so that the best paths are known
def test_nbest_hand_lattice():
    base = [("<unk>", 0.0, mp.UNKNOWN), ("<s>", 0.0, mp.CONTROL), ("</s>", 0.0, mp.CONTROL)]
    pcs = base + [("A", 0.0, mp.NORMAL), ("B", 0.0, mp.NORMAL), ("C", 0.0, mp.NORMAL), ("AB", 2.0, mp.NORMAL),
                  ("BC", 5.0, mp.NORMAL), ("ABC", 10.0, mp.NORMAL)]
    m = oracle_py.OracleModel(mp.build_model(pcs, charsmap=b"", add_dummy_prefix=False))
    cands, scores = m.nbest_encode(b"ABC", 10)
    assert [c.tolist() for c in cands] == [[8], [3, 7], [6, 5], [3, 4, 5]]  # ABC | A BC | AB C | A B C
    assert scores.tolist() == [10.0, 5.0, 2.0, 0.0]


def test_sample_pick_against_numpy_mt19937():
    """The draw restated in the oracle (std::mt19937 + generate_canonical<double,53> + the cumulative table of
    std::discrete_distribution) vs an independent emulation on numpy's legacy MT19937 (same init_genrand
    seeding as std::mt19937(seed))."""
    import ctypes
    import math
    lib = ctypes.CDLL(oracle_py.build_oracle())

    class G(ctypes.Structure):
        _fields_ = [("mt", ctypes.c_uint32 * 624), ("idx", ctypes.c_int)]
    lib.oracle_sample_pick.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_float]
    rng = np.random.default_rng(3)
    for seed in (1, 5489, 20260922):
        g = G()
        lib.oracle_mt_seed(ctypes.byref(g), seed)
        rs = np.random.RandomState(seed)
        for _ in range(300):
            k = int(rng.integers(1, 9))
            scores = (-rng.random(k) * 30).astype(np.float32)
            alpha = np.float32(rng.choice([0.1, 0.5, 1.0]))
            got = lib.oracle_sample_pick(ctypes.byref(g), scores.ctypes.data, k, float(alpha))
            if k < 2:
                assert got == 0
                continue
            x0, x1 = (int(v) for v in rs.randint(0, 2 ** 32, size=2, dtype=np.uint64))
            u = (float(x0) + float(x1) * 4294967296.0) / 18446744073709551616.0
            lp = [float(np.float32(alpha * s)) for s in scores]
            z = lp[0]
            for v in lp[1:]:
                a, b = (z, v) if z <= v else (v, z)
                z = b + math.log1p(math.exp(a - b))
            pr = [math.exp(v - z) for v in lp]
            tot = sum(pr)
            run, cp = 0.0, []
            for v in pr:
                run += v / tot
                cp.append(run)
            cp[-1] = 1.0
            exp_pick = next(i for i, c in enumerate(cp) if not c < u)
            assert got == exp_pick
