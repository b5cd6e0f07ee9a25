"""Edges of the unigram lane kernel's whole-word shortcut (lane_kernel.cuh, engine.cu upload_word_safe): a word that
is one piece is retired as a whole.  The ids must be the oracle's for words of 10 to 15 bytes after the U+2581 (the
end of the text window the walk keeps in registers), runs of whole words, a word at the end of the text or followed
by punctuation, sentences near the kernel's 512-byte capacity, live type changes (SetVocabulary, a frequent word
piece turned UNUSED or USER_DEFINED), models without the shortcut and the normalizer flag variants.  Needs a B200."""
import numpy as np
import pytest

from conftest import model_bytes
from oracle import modelproto as mp
from oracle import oracle_py

pytestmark = pytest.mark.gpu
WS = "▁".encode()
KEY_MAX = 12  # the words around this length reach past the 13-byte register window


@pytest.fixture(autouse=True)
def whole_word_kernel(monkeypatch):
    # the engine picks the whole-word instantiation from a sample of each batch; these batches must take it
    monkeypatch.setenv("SPM_B200_FASTWORDS", "1")


def word_pieces(mb):
    """NORMAL pieces '▁' + lower-case ASCII letters, by key length"""
    m = mp.parse_model(mb)
    out = {}
    for p, t in zip(m["pieces"], m["types"]):
        if t == mp.NORMAL and p.startswith(WS) and len(p) > 3 and p[3:].isalpha() and p[3:].islower():
            out.setdefault(len(p) - 3, []).append(p[3:])
    return out


def check(mb, lines, what=""):
    from sentencepiece_b200 import Engine
    buf, offs = oracle_py.pack(lines)
    eng = Engine(mb)
    ids, ido = eng.encode_packed(buf, offs)
    eng.close()
    oids, oido = oracle_py.OracleModel(mb).encode_batch(buf, offs)
    assert np.array_equal(ido, oido), f"offsets differ {what}"
    assert np.array_equal(ids, oids), f"ids differ {what}"


def test_key_lengths_around_capacity():
    mb = model_bytes("uni32k")
    wp = word_pieces(mb)
    rng = np.random.default_rng(1)
    lines = []
    for L in range(KEY_MAX - 2, KEY_MAX + 4):
        words = wp.get(L, [])
        assert L > KEY_MAX or words, L
        for w in words[:40]:
            filler = [rng.choice(wp[3]).decode() for _ in range(3)]
            lines += [w, b"a " + w, (" ".join(filler) + " ").encode() + w + b" " + w, w + b"s", w + b"x"]
        # words that are no piece, longer than any key: the walk from the U+2581 node takes them
        lines.append(b" ".join(w + w for w in words[:10]))
    check(mb, lines, "key lengths")


def test_runs_end_of_text_and_punctuation(corpus_gen):
    mb = model_bytes("uni32k")
    wp = word_pieces(mb)
    rng = np.random.default_rng(2)
    short = [w for L in (1, 2, 3, 4, 5, 6) for w in wp.get(L, [])]
    lines = []
    for _ in range(400):  # runs of retired words, one of them last in the text
        lines.append(b" ".join(rng.choice(short, size=int(rng.integers(1, 40)))))
    for w in short[:300]:  # a word followed by punctuation instead of U+2581, and at the very end
        lines += [w + b".", w + b", " + w, b"(" + w + b")", w + b"-" + w, w + b"\xe2\x80\x94" + w, w + b" \xc3\xa9",
                  w + b"  " + w, b"  " + w + b"  "]
    lines += corpus_gen.lines("en", 4301, 3000)
    check(mb, lines, "runs / punctuation")


def test_sentences_near_lane_capacity():
    mb = model_bytes("uni32k")
    wp = word_pieces(mb)
    rng = np.random.default_rng(3)
    words = [w for L in range(1, KEY_MAX + 1) for w in wp.get(L, [])]
    lines = []
    for target in (480, 500, 505, 508, 509, 510, 511, 512, 513, 516, 530):
        for _ in range(20):
            s = b""
            while True:  # normalized length ~ 3 bytes per space + the letters
                w = rng.choice(words)
                if len(s) + len(w) + 1 + 2 * (s.count(b" ") + 2) > target:
                    break
                s += (b" " if s else b"") + w
            lines.append(s)
    check(mb, lines, "near 512 bytes")


@pytest.mark.parametrize("kind", [mp.UNUSED, mp.USER_DEFINED])
def test_live_types_drop_whole_words(kind, corpus_gen):
    """a frequent word piece turned UNUSED / USER_DEFINED must no longer be retired as a whole word; then back to
    the full vocabulary"""
    from sentencepiece_b200 import Engine
    mb = model_bytes("uni32k")
    om = oracle_py.OracleModel(mb)
    pieces = om.proto["pieces"]
    targets = [WS + w for w in (b"the", b"of", b"and", b"to", b"in", b"is", b"was")]
    t = om.types.copy()
    for p in targets:
        t[pieces.index(p)] = kind
    lines = corpus_gen.lines("en", 4302, 3000) + [b" ".join(p[3:] for p in targets) * 4]
    buf, offs = oracle_py.pack(lines)
    eng = Engine(mb)
    want = om.encode_batch(buf, offs)
    got = eng.encode_packed(buf, offs)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), "full vocabulary"
    om.set_types(t)
    eng.set_types(t)
    want2 = om.encode_batch(buf, offs)
    got2 = eng.encode_packed(buf, offs)
    assert not np.array_equal(want2[0], want[0])
    assert np.array_equal(got2[0], want2[0]) and np.array_equal(got2[1], want2[1]), f"types {kind}"
    om.set_types(om.types)
    eng.set_types(om.types)
    got3 = eng.encode_packed(buf, offs)
    assert np.array_equal(got3[0], want[0]) and np.array_equal(got3[1], want[1]), "reset"
    # SetVocabulary: a random half of the pieces
    rng = np.random.default_rng(12)
    tv = om.vocabulary_types([p for p in pieces if rng.random() < 0.5])
    om.set_types(tv)
    eng.set_types(tv)
    want4 = om.encode_batch(buf, offs)
    got4 = eng.encode_packed(buf, offs)
    assert np.array_equal(got4[0], want4[0]) and np.array_equal(got4[1], want4[1]), "SetVocabulary"
    eng.close()


@pytest.mark.parametrize("flags", [dict(treat_whitespace_as_suffix=True), dict(escape_whitespaces=False)])
def test_ineligible_model(flags, corpus_gen):
    """whitespace as suffix / unescaped whitespace: no whole-word shortcut, same ids"""
    check(mp.replace_flags(model_bytes("uni32k"), **flags), corpus_gen.lines("en", 4303, 3000), str(flags))


# With remove_extra_whitespaces off, sentences with two spaces in a row come out differently from the oracle on this
# model and corpus with either lane kernel instantiation (SPM_B200_FASTWORDS=0 or 1): the divergence is in the
# normalized text (K1), not in the segmentation.
KNOWN_K1 = pytest.mark.xfail(strict=True, reason="lane kernel K1 with remove_extra_whitespaces off and a double space")


@pytest.mark.parametrize("flags", [dict(add_dummy_prefix=False),
                                   pytest.param(dict(remove_extra_whitespaces=False), marks=KNOWN_K1),
                                   dict(escape_whitespaces=False, add_dummy_prefix=False),
                                   dict(treat_whitespace_as_suffix=True),
                                   dict(escape_whitespaces=False, remove_extra_whitespaces=False)])
def test_normalizer_flag_variants(flags, corpus_gen):
    lines = corpus_gen.lines("en", 4304, 3000) + [b"  two  spaces  ", b"end ", b" start", b"a  b   c"]
    check(mp.replace_flags(model_bytes("uni32k"), **flags), lines, str(flags))


def test_ws_piece_unused(corpus_gen):
    """the piece "▁" itself UNUSED: a walk that starts on its node relaxes nothing there and the U+2581 is an UNK
    edge, as in the reference"""
    from sentencepiece_b200 import Engine
    mb = model_bytes("uni32k")
    om = oracle_py.OracleModel(mb)
    t = om.types.copy()
    t[om.proto["pieces"].index(WS)] = mp.UNUSED
    lines = corpus_gen.lines("en", 4305, 3000) + [b"a  b", b"x", b"\xe2\x96\x81 \xe2\x96\x81q"]
    buf, offs = oracle_py.pack(lines)
    eng = Engine(mb)
    om.set_types(t)
    eng.set_types(t)
    want = om.encode_batch(buf, offs)
    got = eng.encode_packed(buf, offs)
    eng.close()
    assert np.array_equal(got[1], want[1]) and np.array_equal(got[0], want[0])
