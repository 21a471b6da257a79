"""CPU-side checks of the boundary: the C-ABI library loads and exports every symbol that
include/*.h declares; without a GPU every hot-path entry fails loudly (no CPU fallback); the
host-only parts of the mirrored surface (model I/O, decode, vocab, id<->subword) agree with the
reference (its outputs recorded in tests/golden/reference/outputs.json, see _refgolden)."""
import ctypes as C
import os
import re

import pytest

import _refgolden as R
from _bind import ROOT, tmp_model_path
from youtokentome_b200 import synth


def _declared(header):
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(yttm_[a-z0-9_]+)\s*\(", src)))


def test_exports_every_declared_symbol(product):
    names = _declared("yttm_b200.h") + _declared("yttm_b200_api.h")
    assert len(names) > 40
    for n in names:
        assert hasattr(product, n), "libyttm_b200.so does not export " + n


def test_oracle_is_not_linked_into_product():
    """The product library must not reference the checkers."""
    import subprocess
    from youtokentome_b200 import _lib
    out = subprocess.run(["nm", "-D", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "orc_" not in out and "ref_train" not in out
    ldd = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in ldd and "yttm_ref" not in ldd


def _no_gpu(product):
    return product.yttm_device_count() == 0


def test_fails_loudly_without_gpu(product, oracle):
    if not _no_gpu(product):
        pytest.skip("a GPU is present")
    import youtokentome_b200 as yttm
    ctx = C.c_void_p()
    assert product.yttm_ctx_create(0, C.byref(ctx)) != 0
    assert b"no CPU fallback" in product.yttm_last_error(None)
    m = tmp_model_path()
    oracle.train(b"ab ab abc", m, 12)
    bpe = yttm.BPE(m)                       # model tables load on the host
    with pytest.raises(ValueError, match="no CUDA device"):
        bpe.encode(["ab"])
    with pytest.raises(ValueError, match="no CUDA device"):
        yttm.BPE.train(m, m + ".out", 12)


def test_null_encoder_handle_is_an_error_not_a_crash(product):
    """yttm_enc_run / yttm_enc_run_device on a null handle (what yttm_api_device_encoder returns when no device context
    could be created): error code + message, on any box."""
    n, p1, p2 = C.c_uint64(7), C.c_void_p(), C.c_void_p()
    assert product.yttm_enc_run_device(None, None, None, 0, 0, 0, 0, 0, 0.0, 0, 0, C.byref(p1), C.byref(p2), C.byref(n)) == 1
    assert b"null encoder handle" in product.yttm_last_error(None)
    assert product.yttm_enc_run(None, None, None, 0, 0, 0, 0, 0.0, 0, 0, None, 0, None, C.byref(n)) == 1
    assert b"null encoder handle" in product.yttm_last_error(None)


def test_host_surface_matches_reference(product, oracle):
    """decode / vocab / id_to_subword / subword_to_id / error texts vs the unmodified reference."""
    import youtokentome_b200 as yttm
    m = tmp_model_path()
    train, test, vocab = synth.GOLDEN_TEXTS["russian"]
    oracle.train(train.encode(), m, vocab)
    bpe = yttm.BPE(m)
    assert bpe.vocab_size() == R.want("abi/host_surface/vocab_size", lambda: R.reference().encoder(m).vocab_size()) == vocab
    sents = [test.encode(), b"ab", b""]
    ids = oracle.encoder(m).encode(sents, bos=True, eos=True)
    assert R.canon(ids) == R.want("abi/host_surface/ids",
                                  lambda: R.reference().encoder(m).encode(sents, bos=True, eos=True))
    assert R.canon(bpe.decode(ids)) == R.want("abi/host_surface/decode",
                                              lambda: [R.reference().encoder(m).decode(s) for s in ids])
    assert bpe.decode(ids, ignore_ids=[2, 3]) != bpe.decode(ids)
    assert R.canon(bpe.decode(ids[0])) == R.want("abi/host_surface/decode0",
                                                 lambda: [R.reference().encoder(m).decode(ids[0])])
    v = bpe.vocab()
    assert v[:4] == ["<PAD>", "<UNK>", "<BOS>", "<EOS>"] and v[4] == "▁"
    assert all(bpe.subword_to_id(s) == i for i, s in enumerate(v))
    assert bpe.subword_to_id("definitely-not-a-piece") == 1
    with pytest.raises(ValueError, match="id must be in the range"):
        bpe.id_to_subword(vocab)
    with pytest.raises(TypeError):
        bpe.decode("1 2 3")
    with pytest.raises(TypeError):
        bpe.decode([1], ignore_ids=5)
    with pytest.raises(ValueError, match="Can not open file with model"):
        yttm.BPE("/nonexistent/model")


def test_train_argument_errors_match_reference(product):
    """check_config (bpe.cpp:1295-1350) runs before any device work: same texts as the reference."""
    import youtokentome_b200 as yttm
    path = tmp_model_path("txt")
    open(path, "w").write("ab ab abc\n")
    cases = [dict(coverage=0.0), dict(coverage=1.5), dict(unk_id=-1), dict(unk_id=50), dict(pad_id=-2),
             dict(bos_id=100), dict(eos_id=77), dict(pad_id=1, unk_id=1)]
    def ref_error(args):
        with pytest.raises(ValueError) as e_ref:
            R.reference().train_file(path, path + ".m", 20, args["coverage"], 1, args["pad_id"], args["unk_id"],
                                     args["bos_id"], args["eos_id"])
        return str(e_ref.value)

    for i, kw in enumerate(cases):
        args = dict(coverage=1.0, pad_id=0, unk_id=1, bos_id=2, eos_id=3)
        args.update(kw)
        with pytest.raises(ValueError) as e_new:
            yttm.BPE.train(path, path + ".m", 20, **args)
        assert str(e_new.value) == R.want("abi/train_errors/%d" % i, lambda: ref_error(args))
    with pytest.raises(ValueError, match="Failed to open file"):
        yttm.BPE.train("/nonexistent/file", path + ".m", 20)


def test_cli_host_commands_match_reference_format(product, oracle):
    """`yttm vocab [--verbose]` and `yttm decode [--ignore_ids]` (host-only paths, no GPU needed):
    stdout framing of the reference (bpe.cpp:1896-1940, 2016-2028)."""
    import subprocess
    import sys
    m = tmp_model_path()
    train, test, vocab = synth.GOLDEN_TEXTS["english"]
    oracle.train(train.encode(), m, vocab)
    base = [sys.executable, "-m", "youtokentome_b200.yttm_cli"]
    out = subprocess.run(base + ["vocab", "--model", m], capture_output=True, text=True, cwd=ROOT, check=True).stdout
    lines = out.rstrip("\n").split("\n")
    import youtokentome_b200 as yttm
    assert len(lines) == yttm.BPE(m).vocab_size() and lines[0] == "0\t<PAD>" and lines[4] == "4\t▁"
    verbose = subprocess.run(base + ["vocab", "--model", m, "--verbose"], capture_output=True, text=True, cwd=ROOT,
                             check=True).stdout
    assert "=" in verbose and "+" in verbose
    sents = [test.encode(), b"chrono"]
    ids = oracle.encoder(m).encode(sents, bos=True, eos=True)
    assert R.canon(ids) == R.want("abi/cli/ids", lambda: R.reference().encoder(m).encode(sents, bos=True, eos=True))
    stdin = "\n".join(" ".join(map(str, s)) for s in ids) + "\n"
    dec = subprocess.run(base + ["decode", "--model", m, "--ignore_ids", "2,3"], input=stdin, capture_output=True,
                         text=True, cwd=ROOT, check=True).stdout
    assert R.canon(dec.split("\n")[:-1]) == R.want(
        "abi/cli/decode", lambda: [R.reference().encoder(m).decode([i for i in s if i not in (2, 3)]) for s in ids])
