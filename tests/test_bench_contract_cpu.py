"""bench.py's control flow and the JSON-line contract, checked without a GPU: tools/bench_dryrun_emulated.py runs
bench.main() unchanged on the CPU emulator build of the kernels (torch.cuda stubbed, workload shrunk).  The numbers are
meaningless here; the keys, their types and the internal consistency of the line are what the driver depends on."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from _bind import ROOT, have_reference


def test_bench_line_contract_on_the_emulator(tmp_path):
    env = dict(os.environ, YTTM_BENCH_CACHE=str(tmp_path / "cache"))
    for k in [k for k in env if k.startswith(("YTTM_ENC_", "YTTM_LOOP_"))]:
        env.pop(k)
    dump = tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_dryrun_emulated.py"), "--dump-outputs", str(dump)],
                       cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-2000:]
    lines = [ln for ln in r.stdout.decode().splitlines() if ln.strip()]
    assert len(lines) == 1, "stdout must carry exactly ONE line"
    d = json.loads(lines[0])
    for k, t in (("metric", str), ("value", float), ("unit", str), ("n_gpus", int), ("steps", int), ("warmup", int),
                 ("ms_per_step", float), ("higher_is_better", bool), ("scaling", str), ("dtype", str), ("data", str),
                 ("config", dict), ("e2e", dict), ("gpu_launches", int), ("clocks", dict), ("roofline", dict),
                 ("cpu_baseline", dict)):
        assert isinstance(d[k], t), (k, d[k])
    assert d["vs_baseline"] is None and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] >= 3 and d["gpu_launches"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and d["e2e"]["h2d_bytes_per_step"] > 0
    rf = d["roofline"]
    assert set(rf) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and rf["bound"] == "hbm"
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    cb = d["cpu_baseline"]
    assert set(cb) >= {"value", "unit", "cores", "kind", "sample"} and cb["kind"] in ("reference", "port") and cb["ids_equal_on_sample"]
    assert abs(d["ms_per_step"] * d["value"] / 1e3 - d["config"]["sentences_per_gpu"] / 1e6) < 1e-6   # value = S / t
    # hot path (a) travels in keys the driver keeps: config.train.* and roofline.train_*
    tr = d["config"]["train"]
    chk = "reference" if have_reference("det") else "oracle"     # what the GPU models are checked against
    assert set(tr) >= {"config1", "config3", "config5"}
    for key in ("config3", "config5"):
        leg = tr[key]
        assert leg["gpus"] == 1 and leg["merges"] > 0 and leg["GBps"] > 0 and leg["us_per_merge"] > 0 and len(leg["model_sha1"]) == 12
        assert leg["parity_chunk0"]["equals_" + chk] is True
    assert tr["config1"]["equals_" + chk] is True
    assert set(rf["train_scan"]) >= {"heavy", "light", "algorithmic_bytes_per_merge"} and rf["train_scan"]["heavy"]["frac"] > 0
    assert set(rf["train_front"]) >= {"char_hist_GBps", "word_count_GBps"}
    e4 = d["config"]["encode_config4"]
    assert e4["dropout"] == 0.1 and e4["ids_equal_oracle_on_sample"] is True and e4["Msent_s_device"] > 0
    # train_1GB_8thr times the reference's own (multi-threaded) trainer: only where it is built
    assert d["e2e"]["pageable_value"] > 0 and set(cb) >= {"n_threads_1"} | ({"train_1GB_8thr"} if cb["kind"] == "reference" else set())
    assert len(lines[0]) < 8000, "the line must stay small enough for the driver's retained tail"
    # --dump-outputs: the offsets of every sentence and the ids of the sampled ones, in float
    offs, ids, pick = (np.load(dump / (n + ".npy")) for n in ("offsets", "ids_sample", "ids_sample_sentences"))
    assert offs.dtype == pick.dtype == np.float64 and ids.dtype == np.float32
    assert len(offs) == d["config"]["sentences_per_gpu"] + 1 and offs[0] == 0 and offs[-1] == d["config"]["ids_per_gpu"]
    assert np.all(np.diff(offs) >= 0) and np.all(np.diff(pick) > 0)
    p = pick.astype(np.int64)
    assert len(ids) == (offs[p + 1] - offs[p]).sum() > 0 and ids.min() >= 0


@pytest.mark.skipif(not have_reference("prod"), reason="oracle/_ref not built")
def test_reference_arm_line_contract(tmp_path):
    """`bench.py --impl reference` (the unmodified reference's CPU encode_as_ids from oracle/_ref, no GPU involved)."""
    env = dict(os.environ, YTTM_BENCH_CACHE=str(tmp_path / "cache"))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-2000:]
    lines = [ln for ln in r.stdout.decode().splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Msent/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"] == "encode throughput, 1M x 128 B synthetic sentences, vocab 32k"
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert cb["steps_s"]["min"] <= cb["steps_s"]["median"] <= cb["steps_s"]["max"]
    assert d["config"]["workload"] == "configs[1]: encode 1M synthetic 128-byte sentences, vocab 32k"
