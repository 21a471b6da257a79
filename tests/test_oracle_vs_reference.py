"""Pins the oracle (oracle/bpe_oracle.cpp) to the unmodified reference built with
-DDETERMINISTIC_QUEUE (recorded in tests/golden/reference/outputs.json, see _refgolden): same rules + char2id
(stress_test.cpp:433-434), same ids (:468-469), the manual case (:313-337) and the corpora of test_manual.py:7-75."""
import pytest

import _cases
import _refgolden as R
from _bind import read_model, tmp_model_path
from youtokentome_b200 import synth


def _train_both(key, oracle, text, vocab, cov, threads=4, **special):
    """The oracle's model (or error text) == the reference's; returns the oracle's model path, None after an error."""
    m = tmp_model_path("orc")
    try:
        oracle.train(text, m, vocab, cov, **special)
        got = read_model(m)
    except ValueError as e:
        got, m = {"error": str(e)}, None
    assert R.canon(got) == R.want(key + "/model", lambda: R.model(text, vocab, cov, threads, **special))
    return m


def _encode_both(key, oracle, m, text, vocab, cov, threads, sents, kw, **special):
    got = oracle.encoder(m).encode(sents, **kw)
    assert R.canon(got) == R.want(key, lambda: R.encoder(text, vocab, cov, threads, **special).encode(sents, **kw))
    return got


@pytest.mark.parametrize("seed", range(60))
def test_stress_train_and_encode(oracle, seed):
    text, vocab, cov, sents = _cases.stress_case(seed)
    key = "oracle_vs_reference/stress/%d" % seed
    threads = 1 + seed % 8
    m = _train_both(key, oracle, text, vocab, cov, threads=threads)
    if m is None:
        return
    sents = sents + _cases.EDGE_SENTENCES
    for i, kw in enumerate([dict(), dict(bos=True, eos=True), dict(reverse=True, eos=True)]):
        _encode_both("%s/ids%d" % (key, i), oracle, m, text, vocab, cov, threads, sents, kw)


def test_manual_case(oracle):
    key = "oracle_vs_reference/manual"
    m = _train_both(key, oracle, b"baba baaab", 9, 1.0, threads=1)
    _encode_both(key + "/ids", oracle, m, b"baba baaab", 9, 1.0, 1, [b"d d"], {})


@pytest.mark.parametrize("name", sorted(synth.GOLDEN_TEXTS))
def test_manual_corpora(oracle, name):
    train, test, vocab = synth.GOLDEN_TEXTS[name]
    key = "oracle_vs_reference/manual_corpora/" + name
    m = _train_both(key, oracle, train.encode(), vocab, 1.0)
    _encode_both(key + "/ids", oracle, m, train.encode(), vocab, 1.0, 4, [test.encode()], {})


@pytest.mark.parametrize("cov", [1.0, 0.98, 0.9])
def test_dirty_unicode(oracle, cov):
    text = _cases.dirty_zipf_text()
    if cov == 1.0:
        # with nothing removed the reference keeps invalid bytes and dies in char2id.at()
        # (bpe.cpp:410, SURVEY.md §5); compare on the cleaned text instead
        text = _cases.zipf().text(200_000)
    key = "oracle_vs_reference/dirty_unicode/%g" % cov
    m = _train_both(key, oracle, text, 1500, cov)
    _encode_both(key + "/ids", oracle, m, text, 1500, cov, 4, _cases.zipf_sentences(), {})


@pytest.mark.parametrize("special", [dict(pad=-1, unk=1, bos=2, eos=3), dict(pad=-1, unk=5, bos=-1, eos=-1)])
def test_space_token_with_id_zero(oracle, special):
    """No special token at id 0 => U+2581 gets final id 0, and the reference drops a word-initial, never merged "▁" from
    its output (it starts at the first node whose id is not 0, bpe.cpp:1591-1596).  Few merges, so most words keep it."""
    text = _cases.zipf().text(60_000) + b" zab zab ab z zz z q"
    n_chars = len(set(text.decode().replace("\n", " ").replace(" ", "")))
    vocab = n_chars + 5 + 25
    key = "oracle_vs_reference/space_id_zero/unk%d" % special["unk"]
    m = _train_both(key, oracle, text, vocab, 1.0, threads=1, **special)
    assert read_model(m)[0][9601] == 0
    sents = _cases.zipf_sentences(400) + list(_cases.EDGE_SENTENCES) + [b"zab", b"z", b"q z zz", "▁▁z".encode()]
    kws = [dict(), dict(reverse=True)]
    if special["bos"] != -1:
        kws.append(dict(bos=True, eos=True))
    for i, kw in enumerate(kws):
        _encode_both("%s/ids%d" % (key, i), oracle, m, text, vocab, 1.0, 1, sents, kw, **special)
    # the quirk really fires: a one-letter word whose ("▁", letter) pair has no rule comes out as ONE id
    c2i, rules, _ = read_model(m)
    merged_with_space = {y for x, y, _ in rules if x == 0}
    lone = [cp for cp, i in c2i.items() if cp != 9601 and i not in merged_with_space]
    assert lone
    got = _encode_both(key + "/lone", oracle, m, text, vocab, 1.0, 1, [chr(lone[0]).encode()], {}, **special)
    assert got == [[c2i[lone[0]]]]


def test_vocab_too_small(oracle):
    _train_both("oracle_vs_reference/vocab_too_small", oracle, b"abcdefgh ijkl", 6, 1.0)


def test_readme_config(oracle):
    """BASELINE config 1: 10k x 100 chars over "abcd ", vocab 5000 (README.md:41-69)."""
    text = synth.readme_corpus()
    assert len(text) == 1_010_000
    _train_both("oracle_vs_reference/readme", oracle, text, 5000, 1.0)
    assert oracle.last_stats["n_merges"] == 4991
    assert oracle.last_stats["n_unique"] == 43814 and oracle.last_stats["n_tokens"] == 499544
