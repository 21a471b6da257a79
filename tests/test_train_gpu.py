"""Parity of hot path (a): the CUDA trainer (through the C ABI) against the oracle — rules and
char2id bit-exact (the assertion of stress_test.cpp:433-434) — and against the unmodified reference
(its outputs recorded in tests/golden/reference/outputs.json, see _refgolden).  All tests need a GPU."""
import ctypes as C

import numpy as np
import pytest

import _cases
import _refgolden as R
from _bind import read_model, tmp_model_path
from _gpu import gpu_train
from youtokentome_b200 import synth

pytestmark = pytest.mark.gpu


def _same(oracle, text, vocab, cov=1.0, **special):
    m_o = tmp_model_path("orc")
    try:
        oracle.train(text, m_o, vocab, cov, **special)
    except ValueError as e:
        with pytest.raises(ValueError) as ei:
            gpu_train(text, vocab, cov, **special)
        assert str(ei.value) == str(e)
        return None
    m_g = gpu_train(text, vocab, cov, **special)
    a, b = read_model(m_o), read_model(m_g)
    assert a[0] == b[0], "char2id differs"
    assert a[2] == b[2], "special tokens differ"
    if a[1] != b[1]:
        k = next(i for i, (p, q) in enumerate(zip(a[1], b[1])) if p != q) if len(a[1]) == len(b[1]) or True else -1
        raise AssertionError("rules differ: %d vs %d rules, first difference at %s" % (len(a[1]), len(b[1]), k))
    return m_g


@pytest.mark.parametrize("seed", range(40))
def test_stress(product, oracle, seed):
    text, vocab, cov, _ = _cases.stress_case(seed)
    _same(oracle, text, vocab, cov)


def test_manual(product, oracle):
    _same(oracle, b"baba baaab", 9)


@pytest.mark.parametrize("name", sorted(synth.GOLDEN_TEXTS))
def test_manual_corpora(product, oracle, name):
    train, _, vocab = synth.GOLDEN_TEXTS[name]
    _same(oracle, train.encode(), vocab)


@pytest.mark.parametrize("cov", [1.0, 0.98, 0.9])
def test_dirty_unicode(product, oracle, cov):
    """invalid bytes, U+2581 separators, 2/3/4-byte scripts, rare-char removal."""
    _same(oracle, _cases.dirty_zipf_text(), 1500, cov)


def test_long_runs(product, oracle):
    """floor(L/2) counting and greedy pairing inside long runs of one token (SURVEY.md §7.2-3)."""
    _same(oracle, b"a" * 500 + b" " + b"ab" * 300 + b" aaa aaaa aaaaa " + b"b" * 1001, 40)


def test_edge_inputs(product, oracle):
    _same(oracle, b"", 10)
    _same(oracle, b"   \n\t ", 10)
    _same(oracle, b"a", 10)
    _same(oracle, b"\xff\xfe", 10)
    _same(oracle, b"abcdefgh ijkl", 6)          # vocab too small -> same error text
    _same(oracle, b"ab ab ab", 1000)            # merges run out ("merged only")


def test_special_ids(product, oracle):
    text = synth.readme_corpus(n_lines=300)
    _same(oracle, text, 300, 1.0, pad=-1, unk=5, bos=29, eos=-1)
    _same(oracle, text, 300, 0.999, pad=7, unk=0, bos=3, eos=299)


def test_readme_config(product, oracle):
    """BASELINE config 1 at full size; also against the unmodified reference."""
    text = synth.readme_corpus()
    want = R.want("train_gpu/readme", lambda: R.model(text, 5000, 1.0, threads=4))
    m = _same(oracle, text, 5000)
    assert R.canon(read_model(m)) == want


def test_zipf_medium_vs_reference(product):
    """8 MB multi-script Zipf corpus, vocab 8000: too slow for the oracle, checked against the reference."""
    zc = synth.ZipfCorpus(n_words=50_000, seed=11)
    text = zc.text(8_000_000)
    want = R.want("train_gpu/zipf_medium", lambda: R.model(text, 8000, 0.9995, threads=8))
    m_g = gpu_train(text, 8000, 0.9995)
    assert R.canon(read_model(m_g)) == want


def test_initial_pair_table(product, oracle):
    """The pair-count scan kernel alone: table after build == counts recomputed in numpy."""
    from youtokentome_b200 import _lib
    L = _lib.lib()
    text = _cases.zipf().text(100_000)
    ctx = C.c_void_p()
    assert L.yttm_ctx_create(0, C.byref(ctx)) == 0
    try:
        dl, nd = C.c_uint64(0), C.c_uint64(0)
        assert L.yttm_train_load_corpus(ctx, C.cast(C.c_char_p(text), C.c_void_p), len(text), 0) == 0
        assert L.yttm_train_char_hist(ctx, C.byref(dl), C.byref(nd)) == 0
        cps = np.zeros(nd.value, dtype=np.uint32)
        cnt = np.zeros(nd.value, dtype=np.uint64)
        L.yttm_train_get_char_hist(ctx, cps.ctypes.data, cnt.ctypes.data)
        # reference-free check of the histogram
        import collections
        want = collections.Counter(ch for ch in text.decode() if not ch.isspace())
        assert {chr(c): int(n) for c, n in zip(cps, cnt)} == dict(want)
        assert dl.value == len(text.decode())
        ids = np.arange(5, 5 + len(cps), dtype=np.uint32)
        kc = np.concatenate([cps, [9601]]).astype(np.uint32)
        ki = np.concatenate([ids, [4]]).astype(np.uint32)
        assert L.yttm_train_set_alphabet(ctx, kc.ctypes.data, ki.ctypes.data, len(kc), 4) == 0
        st = _lib.TrainStats()
        assert L.yttm_train_build(ctx, C.byref(st)) == 0, L.yttm_last_error(ctx)
        keys = np.zeros(st.n_pairs + 16, dtype=np.uint64)
        cts = np.zeros(st.n_pairs + 16, dtype=np.uint64)
        n = C.c_uint64(0)
        assert L.yttm_train_dump_pairs(ctx, keys.ctypes.data, cts.ctypes.data, len(keys), C.byref(n)) == 0
        got = {int(k): int(c) for k, c in zip(keys[:n.value], cts[:n.value])}
        cp2id = {int(c): int(i) for c, i in zip(kc, ki)}
        want = collections.Counter()
        for w in text.decode().split():
            t = [4] + [cp2id[ord(ch)] for ch in w]
            i = 0
            while i < len(t):
                j = i
                while j < len(t) and t[j] == t[i]:
                    j += 1
                if j - i >= 2:
                    want[(t[i] << 32) | t[i]] += (j - i) // 2
                if j < len(t):
                    want[(t[i] << 32) | t[j]] += 1
                i = j
        assert got == dict(want)
        assert st.n_words == len(text.decode().split())
        assert st.n_unique == len(set(w for w in text.decode().split()))
    finally:
        L.yttm_ctx_destroy(ctx)


@pytest.mark.parametrize("q", ["64", "1000"])
def test_streaming_tiles(product, oracle, monkeypatch, q):
    """The STREAMING mode of the merge loop (token buffer larger than shared memory) forced on
    small inputs: many tiny tiles, words straddling tile windows, write-through to HBM."""
    monkeypatch.setenv("YTTM_FORCE_STREAM", "1")
    monkeypatch.setenv("YTTM_STREAM_Q", q)
    for seed in range(8):
        text, vocab, cov, _ = _cases.stress_case(seed)
        _same(oracle, text, vocab, cov)
    _same(oracle, _cases.dirty_zipf_text(), 1500, 0.98)
    _same(oracle, b"a" * 500 + b" " + b"ab" * 300 + b" aaa aaaa aaaaa " + b"b" * 1001, 40)
    _same(oracle, synth.readme_corpus(n_lines=1500), 1200)


def test_oversized_word_direct_path(product, oracle):
    """One word longer than the shared-memory tile buffer (60k tokens): the loop leaves resident
    mode and handles that tile straight on global memory."""
    rng = np.random.default_rng(5)
    long_word = bytes(rng.choice(list(b"abc"), size=60_000).tolist())
    text = synth.readme_corpus(n_lines=300) + long_word + b" " + synth.readme_corpus(n_lines=50, seed=3)
    _same(oracle, text, 400)


def test_words_of_33_plus_tokens(product, oracle):
    """Words longer than a warp (scalar lane-0 path inside a tile) next to short ones."""
    rng = np.random.default_rng(9)
    words = [bytes(rng.choice(list(b"abcd"), size=int(n)).tolist()) for n in rng.integers(1, 90, size=3000)]
    _same(oracle, b" ".join(words), 600)


def test_zz_model_file_bytes_equal_the_reference(product):
    """SURVEY.md §8f-4: the model FILE (not only its parsed content) equals the one the unmodified reference
    (DETERMINISTIC_QUEUE build) writes — char2id lines in flat_hash_map slot order (tests/test_dump_order.py
    pins that order on the CPU).  Kept last: everything above compares parsed models."""
    cases = [(synth.readme_corpus(n_lines=800), 600, 1.0), (_cases.zipf().text(300_000), 3000, 1.0),
             (_cases.dirty_zipf_text(), 2500, 0.995)]
    wants = [(R.want("train_gpu/model_file/%d/model" % k, lambda: R.model(text, vocab, cov, threads=2)),
              R.want("train_gpu/model_file/%d/sha256" % k, lambda: R.file_sha256(R.train(text, vocab, cov, threads=2))))
             for k, (text, vocab, cov) in enumerate(cases)]
    for (text, vocab, cov), (want_model, want_sha) in zip(cases, wants):
        m_g = gpu_train(text, vocab, cov)
        assert R.canon(read_model(m_g)) == want_model
        assert R.file_sha256(m_g) == want_sha, "model file differs in bytes although its content is equal"
