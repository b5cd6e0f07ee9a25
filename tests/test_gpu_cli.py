"""The drop-in caller: spm_encode_b200 (C++ host layer over the C ABI) must print exactly what the
reference's spm_encode prints for --output_format=id / piece (BASELINE.json config 1 plumbing:
train-on-botchan model, encode a text file, compare by md5 with the reference's output, kept in
tests/golden/reference_md5.json).  Needs a B200."""
import os
import subprocess

import pytest

from conftest import ROOT, MODELS_DIR
from reference_outputs import Reference

pytestmark = pytest.mark.gpu
CLI = os.path.join(ROOT, "sentencepiece_b200", "lib", "spm_encode_b200")
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "spm_encode")


def run_reference(args):
    return subprocess.run([REF_CLI] + args, capture_output=True, check=True).stdout


@pytest.mark.parametrize("model,kind,fmt,extra", [("botchan8k", "en", "id", ""), ("botchan8k", "en", "piece", ""),
                                                  ("mix_bf8k", "mixed", "id", ""), ("mix_bf8k", "mixed", "piece", ""),
                                                  ("uni32k", "mixed", "piece", "bos:eos"), ("uni32k", "mixed", "piece", "unk"),
                                                  ("bpe32k", "en", "id", "reverse:eos"), ("bpe32k", "en", "piece", "")])
def test_cli_matches_reference(model, kind, fmt, extra, corpus_gen, tmp_path, request):
    assert os.path.exists(CLI), "spm_encode_b200 has not been built (__graft_entry__.build())"
    path = str(tmp_path / "in.txt")
    n = 3000
    # text files cannot carry newlines inside a sentence; the generator never emits them
    corpus_gen.write_file(path, kind, 5151, n)
    mpath = os.path.join(MODELS_DIR, model + ".model")
    args = [f"--model={mpath}", f"--output_format={fmt}", f"--input={path}"]
    if extra:
        args.append(f"--extra_options={extra}")
    ours = subprocess.run([CLI, "--batch_lines=1000"] + args, capture_output=True, check=True).stdout
    Reference(request).check("stdout", (ours,), lambda: (run_reference(args),))


@pytest.mark.parametrize("model,kind,fmt,flags", [
    ("uni32k", "en", "nbest_id", ["--nbest_size=5"]),
    ("uni32k", "mixed", "nbest_piece", ["--nbest_size=4"]),
    ("botchan8k", "mixed", "nbest_piece", ["--nbest_size=3", "--extra_options=bos:eos"]),
    ("uni32k", "en", "sample_id", ["--nbest_size=8", "--alpha=0.5", "--random_seed=12345"]),
    ("botchan8k", "mixed", "sample_piece", ["--nbest_size=6", "--alpha=0.2", "--random_seed=7"]),
    ("mix_bf8k", "mixed", "sample_id", ["--nbest_size=4", "--alpha=1.0", "--random_seed=99", "--extra_options=reverse"]),
    ("uni32k", "en", "id", ["--vocabulary=VOCAB", "--vocabulary_threshold=3"]),
    ("bpe32k", "en", "piece", ["--vocabulary=VOCAB", "--vocabulary_threshold=2"]),
    ("botchan8k", "en", "piece", ["--generate_vocabulary"]),
])
def test_cli_formats_match_reference(model, kind, fmt, flags, corpus_gen, tmp_path, request):
    """The other formats of spm_encode (src/spm_encode_main.cc:102-157): n-best lists, seeded sampling (the draws of a
    batch are taken in line order on one generator, like the reference's single-threaded loop), vocabulary
    restriction (:83-92) and --generate_vocabulary (:102-110,166-172)."""
    assert os.path.exists(CLI), "spm_encode_b200 has not been built (__graft_entry__.build())"
    ref = Reference(request)
    path = str(tmp_path / "in.txt")
    n = 1500
    corpus_gen.write_file(path, kind, 6262, n)
    mpath = os.path.join(MODELS_DIR, model + ".model")
    if any("VOCAB" in f for f in flags):
        # a vocabulary file in the format --generate_vocabulary writes, the same as the reference's own
        vpath = str(tmp_path / "vocab.tsv")
        gen = [f"--model={mpath}", "--generate_vocabulary", f"--input={path}"]
        vocab = subprocess.run([CLI] + gen, capture_output=True, check=True).stdout
        ref.check("vocabulary", (vocab,), lambda: (run_reference(gen),))
        with open(vpath, "wb") as f:
            f.write(vocab)
        flags = [f.replace("VOCAB", vpath) for f in flags]
    args = [f"--model={mpath}", f"--output_format={fmt}", f"--input={path}"] + flags
    ours = subprocess.run([CLI, "--batch_lines=400"] + args, capture_output=True, check=True).stdout
    assert len(ours) > 0
    ref.check("stdout", (ours,), lambda: (run_reference(args),))
