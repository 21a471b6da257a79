"""Parity of hot path (b): batch encode_as_ids on the GPU (through the C ABI) against the oracle
given the SAME model file — ids bit-exact (stress_test.cpp:468-469), batch == one by one
(:387), BPE-dropout bit-exact against the oracle's Philox stream — plus the Python surface
round trips of test_python_api.py:17-51."""
import numpy as np
import pytest

import _cases
import _refgolden as R
from _bind import _pack, read_model, tmp_model_path
from _gpu import GpuEncoder, gpu_train
from youtokentome_b200 import synth

pytestmark = pytest.mark.gpu

KW = [dict(), dict(bos=True, eos=True), dict(reverse=True, eos=True), dict(bos=True, reverse=True)]


def _model(oracle, text, vocab, cov=1.0):
    m = tmp_model_path("orc")
    oracle.train(text, m, vocab, cov)
    return m


@pytest.mark.parametrize("seed", range(30))
def test_stress(product, oracle, seed):
    text, vocab, cov, sents = _cases.stress_case(seed)
    try:
        m = _model(oracle, text, vocab, cov)
    except ValueError:
        return
    g, o = GpuEncoder(m), oracle.encoder(m)
    sents = sents + _cases.EDGE_SENTENCES
    for kw in KW:
        assert g.encode(sents, **kw) == o.encode(sents, **kw)
    # batch == sentence by sentence (parallel_test, stress_test.cpp:351-389)
    assert [g.encode([s])[0] for s in sents[:6]] == g.encode(sents[:6])


@pytest.mark.parametrize("name", sorted(synth.GOLDEN_TEXTS))
def test_manual_corpora(product, oracle, name):
    train, test, vocab = synth.GOLDEN_TEXTS[name]
    m = _model(oracle, train.encode(), vocab)
    assert GpuEncoder(m).encode([test.encode()]) == oracle.encoder(m).encode([test.encode()])


@pytest.mark.parametrize("cov", [1.0, 0.9])
def test_zipf_unicode(product, oracle, cov):
    m = _model(oracle, _cases.dirty_zipf_text(), 1500, cov)
    sents = _cases.zipf_sentences(2000) + _cases.EDGE_SENTENCES
    g, o = GpuEncoder(m), oracle.encoder(m)
    for kw in KW[:2]:
        assert g.encode(sents, **kw) == o.encode(sents, **kw)


def test_long_words_and_sentences(product, oracle):
    m = _model(oracle, _cases.dirty_zipf_text(), 1500)
    zc = _cases.zipf()
    long_sent = b" ".join(zc.sentences(300, 100, seed=5))             # 30 KB sentence
    long_word = b"".join(zc.sentences(40, 60, seed=6)).replace(b" ", b"")  # one ~2 KB word
    sents = [long_sent, long_word, b"a" * 3000, long_word + b" " + long_sent, b""]
    assert GpuEncoder(m).encode(sents) == oracle.encoder(m).encode(sents)


@pytest.mark.parametrize("p", [0.1, 0.5, 1.0])
def test_dropout_matches_oracle_stream(product, oracle, p):
    """dropout > 0: "parity unpinned" w.r.t. the reference (global unsynchronised mt19937,
    bpe.cpp:1415); pinned instead to the oracle's restatement of DropoutQueue with the same
    counter-based generator."""
    m = _model(oracle, _cases.dirty_zipf_text(), 1500)
    sents = _cases.zipf_sentences(500)
    g, o = GpuEncoder(m), oracle.encoder(m)
    a = g.encode(sents, dropout=p, seed=1234)
    assert a == o.encode(sents, dropout=p, seed=1234, first_index=0)
    # the stream continues across calls like the reference's global generator does
    b = g.encode(sents, dropout=p)
    assert b == o.encode(sents, dropout=p, seed=1234, first_index=len(sents))
    if p < 1.0:
        assert a != b
    # invariants (SURVEY.md §7.2-6): more tokens than dropout 0, same text back
    base = g.encode(sents)
    assert sum(map(len, a)) >= sum(map(len, base))


def test_dropout_distribution_vs_reference(product, oracle):
    """mean tokens / sentence at p = 0.1 within 2 % of the reference's own DropoutQueue (its total recorded, see
    _refgolden)."""
    m = _model(oracle, _cases.dirty_zipf_text(), 1500)
    sents = _cases.zipf_sentences(3000)
    r = R.want("encode_gpu/dropout_total_ids",
               lambda: sum(map(len, R.reference().encoder(m, n_threads=1).encode(sents, dropout=0.1))))
    g = sum(map(len, GpuEncoder(m).encode(sents, dropout=0.1, seed=99)))
    assert abs(g - r) / r < 0.02


def check_space_id_zero(oracle, special):
    import os
    text = _cases.zipf().text(60_000) + b" zab zab ab z zz z q"
    n_chars = len(set(text.decode().replace("\n", " ").replace(" ", "")))
    m = tmp_model_path("orc")
    oracle.train(text, m, n_chars + 5 + 25, 1.0, **special)
    long_word = b"".join(_cases.zipf().sentences(12, 60, seed=6)).replace(b" ", b"")
    sents = _cases.zipf_sentences(300) + list(_cases.EDGE_SENTENCES) + [b"zab", b"z", b"q z zz", long_word, b"q" + long_word]
    g, o = GpuEncoder(m), oracle.encoder(m)
    kws = [dict(), dict(reverse=True), dict(dropout=0.3, seed=5)]
    if special["bos"] != -1:
        kws.append(dict(bos=True, eos=True))
    for plain in (False, True):
        if plain:
            os.environ["YTTM_ENC_PLAIN"] = "1"
        try:
            for kw in kws:
                assert g.encode(sents, **kw) == o.encode(sents, **kw), (plain, kw)
        finally:
            os.environ.pop("YTTM_ENC_PLAIN", None)


@pytest.mark.parametrize("special", [dict(pad=-1, unk=1, bos=2, eos=3), dict(pad=-1, unk=5, bos=-1, eos=-1)])
def test_space_token_with_id_zero(product, oracle, special):
    """The reference's id-0 quirk (bpe.cpp:1591-1596) on the GPU kernels, see check_space_id_zero."""
    check_space_id_zero(oracle, special)


def test_bos_eos_errors(product, oracle):
    m = tmp_model_path("orc")
    oracle.train(synth.readme_corpus(n_lines=200), m, 100, 1.0, pad=-1, unk=0, bos=-1, eos=-1)
    g = GpuEncoder(m)
    with pytest.raises(ValueError, match="Can't add <BOS> token"):
        g.encode([b"ab"], bos=True)
    with pytest.raises(ValueError, match="Can't add <EOS> token"):
        g.encode([b"ab"], eos=True)
    assert g.encode([]) == []


def test_python_api_roundtrip(product, tmp_path):
    """test_python_api.py:17-51 of the reference against the new package."""
    import youtokentome_b200 as yttm
    import random
    rnd = random.Random(19)
    train = tmp_path / "train.txt"
    lines = ["".join(rnd.choice("abcd ") for _ in range(100)) for _ in range(2000)]
    train.write_text("\n".join(lines) + "\n")
    test_lines = ["".join(rnd.choice("abcde ") for _ in range(100)).strip() for _ in range(200)]
    model = str(tmp_path / "m.yttm")
    bpe = yttm.BPE.train(data=str(train), model=model, vocab_size=1200, coverage=0.999, bos_id=2, eos_id=3)
    norm = [" ".join(l.split()) for l in test_lines]
    ids = bpe.encode(test_lines, output_type=yttm.OutputType.ID, bos=True, eos=True)
    dec = bpe.decode(ids, ignore_ids=[2, 3])
    import re
    # "e" is not in the alphabet: a maximal run of e inside a word is one <UNK> (bpe.cpp:1513-1533)
    assert dec == [re.sub("e+", "<UNK>", n) for n in norm]
    sub = bpe.encode(test_lines, output_type=yttm.OutputType.SUBWORD)
    assert ["".join(s).replace("▁", " ").strip() for s in sub] == norm
    vocab = bpe.vocab()
    assert len(vocab) == bpe.vocab_size() == len(set(vocab))
    assert all(bpe.subword_to_id(v) == i for i, v in enumerate(vocab))
    assert isinstance(bpe.encode("ab cd"), list) and isinstance(bpe.encode("ab cd")[0], int)
    with pytest.raises(TypeError):
        bpe.encode(["a"], output_type="id")
    with pytest.raises(ValueError):
        bpe.encode(["a"], dropout_prob=1.5)
    import pickle
    assert pickle.loads(pickle.dumps(bpe)).encode(test_lines[:5]) == bpe.encode(test_lines[:5])


def test_config2_shape_vs_reference(product):
    """BASELINE config 2 shape at 1/20 scale: 50k x 128-byte Zipf sentences, vocab 8000 model
    trained on the GPU == the reference's; ids identical to the reference (8 threads; recorded, see _refgolden)."""
    zc = synth.ZipfCorpus(n_words=50_000, seed=11)
    text = zc.text(6_000_000)
    sents = zc.sentences(50_000, 128, seed=77)
    want_model = R.want("encode_gpu/config2/model", lambda: R.model(text, 8000, 1.0, threads=8))
    want_ids = R.want("encode_gpu/config2/ids",
                      lambda: R.reference().encoder(R.train(text, 8000, 1.0, threads=8), n_threads=8).encode(sents))
    m = gpu_train(text, 8000, 1.0)
    assert R.canon(read_model(m)) == want_model
    assert R.canon(GpuEncoder(m).encode(sents)) == want_ids


def test_chunked_h2d_pipeline(product, oracle, monkeypatch):
    """yttm_enc_run pipelines the batch in chunks (H2D / kernels / D2H overlapped, two buffer
    sets): force 1 MB chunks so that several chunks and both buffer sets are exercised; the
    result must not depend on the chunking (incl. the dropout stream, keyed by sentence index)."""
    m = _model(oracle, _cases.dirty_zipf_text(), 1500)
    zc = _cases.zipf()
    sents = zc.sentences(30_000, 120, seed=21) + _cases.EDGE_SENTENCES + [b" ".join(zc.sentences(2000, 100, seed=5))]
    o = oracle.encoder(m)
    want = o.encode(sents, bos=True, eos=True)
    want_drop = o.encode(sents, dropout=0.2, seed=77)
    for mb in ("1", "64"):
        monkeypatch.setenv("YTTM_ENC_CHUNK_MB", mb)
        g = GpuEncoder(m)
        assert g.encode(sents, bos=True, eos=True) == want
        assert g.encode(sents, dropout=0.2, seed=77) == want_drop


def test_cli_bpe_encode_roundtrip(product, tmp_path):
    """test_cli.py of the reference in miniature: `yttm bpe`, `yttm encode --output_type id --bos --eos`
    (ids separated by a blank, trailing blank before the newline, utils.h:92-103), `yttm decode`."""
    import random
    import subprocess
    import sys
    from _bind import ROOT
    rnd = random.Random(19)
    lines = ["".join(rnd.choice("abcd ") for _ in range(100)) for _ in range(1500)]
    data = tmp_path / "train.txt"
    data.write_text("\n".join(lines) + "\n")
    model = str(tmp_path / "cli.yttm")
    base = [sys.executable, "-m", "youtokentome_b200.yttm_cli"]
    subprocess.run(base + ["bpe", "--data", str(data), "--model", model, "--vocab_size", "900", "--coverage", "0.999"],
                   cwd=ROOT, check=True, capture_output=True)
    test_lines = ["".join(rnd.choice("abcd ") for _ in range(60)).strip() for _ in range(50)]
    enc = subprocess.run(base + ["encode", "--model", model, "--output_type", "id", "--bos", "--eos"],
                         input="\n".join(test_lines) + "\n", capture_output=True, text=True, cwd=ROOT, check=True).stdout
    rows = enc.split("\n")[:-1]
    assert len(rows) == len(test_lines) and all(r.endswith(" ") for r in rows)
    assert all(r.split()[0] == "2" and r.split()[-1] == "3" for r in rows)
    dec = subprocess.run(base + ["decode", "--model", model, "--ignore_ids", "2,3"], input=enc, capture_output=True,
                         text=True, cwd=ROOT, check=True).stdout
    assert dec.split("\n")[:-1] == [" ".join(l.split()) for l in test_lines]


def check_pieces_with_u0001(tmp_path):
    """U+0001 is an ordinary alphabet character: piece lists travel length-framed, never split on a separator."""
    import youtokentome_b200 as yttm
    train = tmp_path / "t.txt"
    train.write_bytes(b"a\x01b a\x01b ab \x01\x01 a\x01b ab\n" * 20)
    bpe = yttm.BPE.train(data=str(train), model=str(tmp_path / "m.yttm"), vocab_size=12)
    vocab = bpe.vocab()
    assert len(vocab) == bpe.vocab_size() == 12 and all(vocab) and len(set(vocab)) == 12
    assert any("\x01" in v for v in vocab)
    sub = bpe.encode(["a\x01b ab", "\x01", ""], output_type=yttm.OutputType.SUBWORD)
    assert ["".join(s).replace("\u2581", " ").strip() for s in sub] == ["a\x01b ab", "\x01", ""]
    ids = bpe.encode(["a\x01b ab", "\x01"])
    assert bpe.decode(ids) == ["a\x01b ab", "\x01"]
    assert [bpe.id_to_subword(i) for i in range(12)] == vocab


def check_shared_handle_between_threads(oracle):
    """Two host threads share one BPE object (ctypes releases the GIL during foreign calls): results never mix."""
    import threading
    import youtokentome_b200 as yttm
    m = _model(oracle, _cases.dirty_zipf_text(), 1200)
    bpe = yttm.BPE(m)
    batches = [[s.decode(errors="ignore") for s in _cases.zipf_sentences(40 + 17 * k)[k:]] for k in range(4)]
    want = [bpe.encode(b) for b in batches]
    want_sub = [bpe.encode(b, output_type=yttm.OutputType.SUBWORD) for b in batches]
    errs = []

    def body(k):
        try:
            for _ in range(6):
                assert bpe.encode(batches[k]) == want[k]
                assert bpe.encode(batches[k], output_type=yttm.OutputType.SUBWORD) == want_sub[k]
                assert bpe.decode(want[k]) == bpe.decode(want[k])
        except BaseException as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=body, args=(k,)) for k in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs[0]


def test_pieces_with_u0001(product, tmp_path):
    check_pieces_with_u0001(tmp_path)


def test_shared_handle_between_threads(product, oracle):
    check_shared_handle_between_threads(oracle)


def test_encode_packed_outputs(product, oracle):
    """encode_packed(out=...): numpy / torch / cuda give the same ids; device input stays on the device (SURVEY 8f-1)."""
    import torch
    import youtokentome_b200 as yttm
    m = _model(oracle, _cases.dirty_zipf_text(), 1200)
    bpe = yttm.BPE(m)
    sents = _cases.zipf_sentences(500) + list(_cases.EDGE_SENTENCES)
    buf, offs = _pack(sents)
    want, woo = oracle.encoder(m).encode_packed(buf, offs, bos=True)
    ids, oo = bpe.encode_packed(buf, offs, bos=True)
    assert np.array_equal(ids, want) and np.array_equal(oo, woo)
    t_ids, t_oo = bpe.encode_packed(buf, offs, bos=True, out="torch")
    assert t_ids.dtype == torch.int32 and np.array_equal(t_ids.numpy(), want) and np.array_equal(t_oo.numpy(), woo.astype(np.int64))
    d_bytes = torch.frombuffer(bytearray(buf), dtype=torch.uint8).cuda()
    d_offs = torch.from_numpy(offs.astype(np.int64)).cuda()
    c_ids, c_oo = bpe.encode_packed(d_bytes, d_offs, bos=True, out="cuda")
    assert c_ids.is_cuda and c_oo.is_cuda and np.array_equal(c_ids.cpu().numpy(), want) and np.array_equal(c_oo.cpu().numpy(), woo.astype(np.int64))
    h_ids, _ = bpe.encode_packed(buf, offs, bos=True, out="cuda")
    assert h_ids.is_cuda and np.array_equal(h_ids.cpu().numpy(), want)
