"""Byte-identical model dump (SURVEY.md §8f-4): the char2id lines of a model written by the reference
come in ska::flat_hash_map slot order (utils.cpp:57-59).  `yttm_api_dump_order` replays that order
from the insertion sequence alone; checked here against model files the UNMODIFIED reference writes
(DETERMINISTIC_QUEUE build, recorded in tests/golden/reference/outputs.json, see _refgolden) — CPU only, no GPU needed."""
import ctypes as C
import os

import numpy as np
import pytest

import _bind
import _refgolden as R
from _cases import dirty_zipf_text, stress_case, zipf
from youtokentome_b200 import _lib, synth


def file_order(path):
    with open(path) as f:
        n, _ = map(int, f.readline().split())
        rows = [tuple(map(int, f.readline().split())) for _ in range(n)]
    return [r[0] for r in rows], dict(rows)


def replay(char2id):
    filled = np.array(sorted(char2id, key=lambda cp: char2id[cp]), dtype=np.uint32)
    out = np.zeros(len(filled), dtype=np.uint32)
    L = _lib.lib()
    L.yttm_api_dump_order.restype = C.c_int
    L.yttm_api_dump_order.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    assert L.yttm_api_dump_order(filled.ctypes.data, len(filled), out.ctypes.data) == 0
    return out.tolist()


def check(key, text, vocab, coverage=1.0, **special):
    """replay() of the char2id of this training == the code point order of the reference's model file."""
    path = _bind.tmp_model_path("dumporder")
    try:
        _bind.Oracle().train(text, path, vocab, coverage, **special)
        order = replay(_bind.read_model(path)[0])
        assert R.canon(order) == R.want("dump_order/" + key,
                                        lambda: file_order(R.train(text, vocab, coverage, **special))[0])
        return len(order)
    finally:
        if os.path.exists(path):
            os.remove(path)


@pytest.mark.parametrize("seed", range(12))
def test_stress_alphabets(seed):
    text, vocab, cov, _ = stress_case(seed)
    check("stress/%d" % seed, text, vocab, cov)


def test_readme_alphabet():
    assert check("readme", synth.readme_corpus(200), 300) == 5


def test_multiscript_alphabets():
    # thousands of code points: several doublings of the table, robin-hood displacement chains
    n = check("multiscript", zipf().text(400_000), 4000)
    assert n > 300
    check("dirty", dirty_zipf_text(), 3500, 0.999)


def test_coverage_and_special_ids():
    t = zipf().text(150_000)
    check("coverage", t, 3500, 0.98)
    check("special_ids", t, 3500, 1.0, pad=-1, bos=-1, eos=7, unk=0)


def test_wide_code_point_range():
    # 4-byte code points next to ASCII: the multiplicative hash spreads them over the whole table
    rng = np.random.default_rng(5)
    cps = np.concatenate([rng.integers(0x21, 0x7f, 40), rng.integers(0x400, 0x500, 60), rng.integers(0x4e00, 0x9fff, 700),
                          rng.integers(0x1f300, 0x1f700, 200)])
    words = ["".join(chr(int(c)) for c in rng.choice(cps, int(rng.integers(1, 7)))) for _ in range(6000)]
    check("wide_range", " ".join(words).encode(), len(set(cps.tolist())) + 50)


# ---- the replay against the reference's own container on arbitrary key sets ---------------------
def ref_order(keys):
    lib = R.reference().lib
    lib.ref_char2id_order.restype = C.c_int
    lib.ref_char2id_order.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    keys = np.ascontiguousarray(keys, dtype=np.uint32)
    out = np.zeros(len(keys), dtype=np.uint32)
    assert lib.ref_char2id_order(keys.ctypes.data, len(keys), out.ctypes.data) == 0
    return out.tolist()


def our_order(keys):
    keys = np.ascontiguousarray(keys, dtype=np.uint32)
    out = np.zeros(len(keys), dtype=np.uint32)
    L = _lib.lib()
    L.yttm_api_dump_order.restype = C.c_int
    L.yttm_api_dump_order.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    assert L.yttm_api_dump_order(keys.ctypes.data, len(keys), out.ctypes.data) == 0
    return out.tolist()


@pytest.mark.parametrize("n", [0, 1, 2, 3, 4, 5, 7, 8, 9, 16, 17, 31, 33, 100, 1000, 4097, 50_000])
def test_random_keys_match_the_reference_container(n):
    rng = np.random.default_rng(n)
    for hi in (0x80, 0x3000, 0x110000, 2 ** 32 - 1):
        keys = rng.permutation(np.unique(rng.integers(0, hi, n + 8)))[:n]
        if len(keys) < n:
            continue
        assert R.canon(our_order(keys)) == R.want("dump_order/random/%d/%x" % (n, hi), lambda: ref_order(keys))


def test_clustered_home_slots_force_regrowth():
    """Keys picked so that many share one home slot at every table size: walks hit max_lookups and the
    table doubles long before the load-factor rule — the `swap back, grow, retry` path (flat_hash_map.h:862-866)."""
    FIB = 11400714819323198485
    rng = np.random.default_rng(11)
    cand = rng.permutation(1 << 20).astype(np.uint64)
    top = (cand * np.uint64(FIB)) >> np.uint64(52)          # 12 leading bits of the product
    for n in (6, 12, 40, 200):
        clustered = cand[top == top[0]][:n]                  # same home slot in every table up to 4096 buckets
        mixed = np.concatenate([clustered, cand[:n]])
        for j, keys in enumerate((clustered, rng.permutation(np.unique(mixed)))):
            assert R.canon(our_order(keys)) == R.want("dump_order/clustered/%d/%d" % (n, j), lambda: ref_order(keys))


def test_sequential_and_strided_keys():
    for j, keys in enumerate((np.arange(0, 3000), np.arange(0, 300000, 97), np.arange(2 ** 32 - 2000, 2 ** 32 - 1),
                              (np.arange(1, 2000, dtype=np.uint64) * 2654435769 % 2 ** 32))):
        assert R.canon(our_order(keys)) == R.want("dump_order/sequential/%d" % j, lambda: ref_order(keys))


# ---- the product's BPEState::dump writes the reference's bytes -----------------------------------
def _redump_sha256(path):
    L = _lib.lib()
    L.yttm_api_redump.restype = C.c_int
    L.yttm_api_redump.argtypes = [C.c_char_p, C.c_char_p]
    out = path + ".redump"
    try:
        assert L.yttm_api_redump(path.encode(), out.encode()) == 0
        return R.file_sha256(out)
    finally:
        if os.path.exists(out):
            os.remove(out)


@pytest.mark.parametrize("case", ["readme", "zipf", "dirty_cov", "stress3", "special_ids"])
def test_product_dump_is_byte_identical_to_the_reference_file(case):
    text, vocab, cov, special = {
        "readme": (synth.readme_corpus(300), 400, 1.0, {}),
        "zipf": (zipf().text(300_000), 3000, 1.0, {}),
        "dirty_cov": (dirty_zipf_text(), 2500, 0.995, {}),
        "stress3": stress_case(3)[:3] + ({},),
        "special_ids": (zipf().text(100_000), 2000, 1.0, dict(pad=-1, bos=-1, eos=5, unk=0)),
    }[case]
    path = _bind.tmp_model_path("orcdump")
    try:
        _bind.Oracle().train(text, path, vocab, cov, **special)
        assert _redump_sha256(path) == R.want("dump_order/redump/" + case,
                                              lambda: R.file_sha256(R.train(text, vocab, cov, **special)))
    finally:
        if os.path.exists(path):
            os.remove(path)


def test_redump_missing_file():
    L = _lib.lib()
    L.yttm_api_redump.restype = C.c_int
    L.yttm_api_redump.argtypes = [C.c_char_p, C.c_char_p]
    assert L.yttm_api_redump(b"/nonexistent/model.yttm", b"/tmp/never_written.yttm") == 1
