"""Recorded outputs of the original YouTokenToMe, so that the tests comparing with it run without it.

The original's C++ core, built with -DDETERMINISTIC_QUEUE (oracle/Makefile -> oracle/_ref), is what the oracle and the
CUDA product are pinned to.  Each comparison states the original's computation as a callable and asks
`want(key, compute)` for its result, which comes from tests/golden/reference/outputs.json.  With
YTTM_RECORD_REFERENCE=1 (and oracle/_ref built) `want` runs the callable instead and records what it returns:
    YTTM_RECORD_REFERENCE=1 python -m pytest tests -k <tests to record>
`canon` turns a value into what is stored: the value itself when its JSON is short, its SHA-256 otherwise."""
import hashlib
import json
import os

import _bind

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "outputs.json")
RECORD = os.environ.get("YTTM_RECORD_REFERENCE") == "1"
_data = None
_models = {}


def canon(value):
    text = json.dumps(value, sort_keys=True, separators=(",", ":"), default=lambda o: o.tolist())
    return json.loads(text) if len(text) <= 200 else "sha256:" + hashlib.sha256(text.encode()).hexdigest()


def want(key, compute):
    global _data
    if _data is None:
        _data = {}
        if os.path.exists(PATH):
            with open(PATH) as f:
                _data = json.load(f)
    if RECORD:
        _data[key] = canon(compute())
        with open(PATH, "w") as f:
            json.dump(_data, f, indent=0, sort_keys=True)
            f.write("\n")
    assert key in _data, "no recorded output of the original for " + key
    return _data[key]


def file_sha256(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


# ---- the original's side of the comparisons (called only while recording) ----------------------
def reference():
    return _bind.Reference("det")


def train(text, vocab, cov=1.0, threads=1, **special):
    """Model file the original writes for these arguments (trained once per argument set)."""
    key = (hashlib.sha256(text).hexdigest(), vocab, cov, threads, tuple(sorted(special.items())))
    if key not in _models:
        m = _bind.tmp_model_path("ref")
        reference().train(text, m, vocab, cov, n_threads=threads, **special)
        _models[key] = m
    return _models[key]


def model(text, vocab, cov=1.0, threads=1, **special):
    """The original's parsed model, or its error text."""
    try:
        return _bind.read_model(train(text, vocab, cov, threads, **special))
    except ValueError as e:
        return {"error": str(e)}


def encoder(text, vocab, cov=1.0, threads=1, **special):
    return reference().encoder(train(text, vocab, cov, threads, **special))
