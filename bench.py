#!/usr/bin/env python
"""bench.py — measurement of the two BPE hot paths on B200 (contract: task statement ④; BASELINE.json metric
"GB/s BPE-train scan + Msent/s encode at 1/2/4/8 B200 vs ref CPU n_threads").

The JSON line's `value` / `e2e` are hot path (b), BASELINE configs[1]: batch encode_as_ids of 1 M synthetic 128-byte
sentences, vocab 32 000 (one "step" = one pass over the batch; the model is trained by this framework's own GPU
trainer outside the timed region).
  value   Msent/s, whole job, inputs already resident in HBM (yttm_enc_run_device)
  e2e     the same through the host-buffer C-ABI call (yttm_enc_run): pinned host input, H2D + kernels + D2H of ids and
          offsets inside the timed region; `pageable_value`: the same call from pageable numpy buffers
Hot path (a), training, travels in keys the driver keeps (`config.train`, `roofline.train_*`):
  config.train.config1   BASELINE configs[0] (README, 1 MB, vocab 5000): seconds and us / merge
  config.train.config3   configs[2]: 1 GB Zipf corpus, vocab 32 000, on `n_gpus` GPUs (strong scaling: the corpus is
                         eight independently seeded 125 MB chunks, rank r trains on its 8 / N chunks)
  config.train.config5   configs[4] shape: multilingual corpus, vocab 64 000, coverage 0.9999, 1.25 GB per GPU
                         (weak scaling: 10 GB on 8 GPUs)
  config.encode_config4  configs[3] shape: lognormal sentences of mean 512 B, dropout 0.1 (Philox; parity unpinned by
                         the reference), ids == oracle on a sample
  roofline.train_scan    per-merge scan of a packed token buffer >> L2 (STREAMING tiles through the TMA ring), the
                         kernel BASELINE.json's 70 % target names; roofline.train_front: the two byte passes
  cpu_baseline           the unmodified reference (oracle/_ref prod build) on the host: encode_as_ids with 1 / 8 / all
                         threads, train_bpe with 8 threads (its cap) on the 1 GB corpus and 1 thread on a 125 MB chunk
`--impl reference` times the reference's own CPU encode_as_ids (all host threads) on the same workload.
`--dump-outputs DIR` writes what the last timed step of `value` returned (ids and offsets, see dump_outputs) as .npy
files, so that two builds can be compared output for output on the same seeded inputs.
N > 1 (torchrun): sentences shard by rank (no collective); training runs through distributed.train_distributed (words
hash-partitioned across ranks, per-merge count exchange by peer stores inside the merge-loop kernel).
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CACHE = os.environ.get("YTTM_BENCH_CACHE", "/tmp/yttm_b200_bench_cache")
N_SENT, SENT_LEN, VOCAB = 1_000_000, 128, 32_000
TRAIN_BYTES = 100_000_000          # corpus of the encode model
CHUNK = 125_000_000                # training corpora come in independently seeded chunks of this size
VOCAB5, CFG1_LINES, CFG1_VOCAB, N_SENT4, TRAIN_RUNS = 64_000, 10_000, 5000, 250_000, 2   # (the CPU dry run of this file shrinks these)
DUMP_SENTENCES = 65_536            # --dump-outputs: ids of this many sentences (at most 130 ids each: <= 34 MB)
WORKLOAD = "configs[1]: encode 1M synthetic 128-byte sentences, vocab 32k"
METRIC = "encode throughput, 1M x 128 B synthetic sentences, vocab 32k"
T_START = time.time()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except (OSError, KeyError, ValueError, TypeError):  # absent or of another shape: the recipe's stated fallback
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(kernel, n_sent):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu --set full capture of
    this very workload (profiles/r02_traffic.json, written from the .ncu-rep by tools/ncu_summary.py); None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            t = json.load(f)
        if t.get("n_sent") == n_sent and kernel in t.get("kernels", {}):
            return int(t["kernels"][kernel]["dram_bytes"]), t.get("source")
    except (OSError, ValueError, KeyError, TypeError):
        pass
    return None, None


def workload(rank, n_sent, train_bytes):
    """(train text, sentence bytes, uint64 offsets) — cached on local disk between the two arms."""
    from youtokentome_b200 import synth
    os.makedirs(CACHE, exist_ok=True)
    tp = os.path.join(CACHE, "train_%d.bin" % train_bytes)
    sp = os.path.join(CACHE, "sent_%d_%d_r%d" % (n_sent, SENT_LEN, rank))
    fz = None
    if os.path.exists(tp):
        text = open(tp, "rb").read()
    else:
        fz = synth.FastZipf(n_words=200_000, s=1.07, seed=1234)
        text = fz.text(train_bytes)
        if rank == 0:
            with open(tp + ".tmp%d" % os.getpid(), "wb") as f:
                f.write(text)
            os.replace(tp + ".tmp%d" % os.getpid(), tp)
    if os.path.exists(sp + ".bin") and os.path.exists(sp + ".npy"):
        buf = open(sp + ".bin", "rb").read()
        offs = np.load(sp + ".npy")
    else:
        fz = fz or synth.FastZipf(n_words=200_000, s=1.07, seed=1234)
        buf, offs = fz.packed_sentences(n_sent, SENT_LEN, seed=4321 + rank)
        with open(sp + ".bin.tmp%d" % os.getpid(), "wb") as f:
            f.write(buf)
        os.replace(sp + ".bin.tmp%d" % os.getpid(), sp + ".bin")
        np.save(sp + ".npy", offs)
    return text, buf, offs


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.rows, self.proc = [], None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_reference_encode(model, buf, offs, cores, max_sent, reps=1):
    """The unmodified reference (prod build) encode_as_ids with `cores` threads on a bounded sample; returns
    (row, ids).  value = sample / MEDIAN seconds over `reps` calls (a shared host makes single calls noisy)."""
    import _bind
    kind = "reference" if _bind.have_reference("prod") else "port"
    n = min(len(offs) - 1, max_sent)
    o = np.ascontiguousarray(offs[:n + 1])
    secs = []
    if kind == "reference":
        enc = _bind.Reference("prod").encoder(model, n_threads=cores)
    else:
        enc, cores = _bind.Oracle().encoder(model), 1
    for _ in range(reps):
        ids, _ = enc.encode_packed(buf, o)
        secs.append(enc.last_seconds)
    sec = statistics.median(secs)
    return {"value": n / sec / 1e6, "unit": "Msent/s", "cores": cores, "kind": kind,
            "sample": "%d of the %d sentences (%.0f MB), encode_as_ids only, median %.3f s / min %.3f s of %d call(s)" %
                      (n, len(offs) - 1, float(o[-1]) / 1e6, sec, min(secs), reps)}, ids


def cpu_train(text, model, vocab, coverage):
    """Single-threaded CPU training the GPU models are checked against: the unmodified reference (DETERMINISTIC_QUEUE
    build) when oracle/_ref is built, else the oracle, which the tests pin to the reference.  Returns (kind, seconds)."""
    import _bind
    if _bind.have_reference("det"):
        return "reference", _bind.Reference("det").train(text, model, vocab, coverage, n_threads=1)
    return "oracle", _bind.Oracle().train(text, model, vocab, coverage)


def device_array(ptr, n, typestr):
    """Host copy of n elements (numpy typestr) of device memory at ptr, read through __cuda_array_interface__."""
    import torch
    cai = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3, "strides": None}
    return torch.as_tensor(type("DeviceBuffer", (), {"__cuda_array_interface__": cai})(), device="cuda").cpu().numpy()


def dump_outputs(out_dir, d_ids, d_offs, n_ids, n_sent):
    """What one call of the timed path returns: ids (int32, on the device) and the n_sent + 1 offsets of each
    sentence's ids.  Writes out_dir/offsets.npy (all offsets, float64), ids_sample.npy (float32, exact: ids < 2^24)
    with the ids of DUMP_SENTENCES sentences drawn with a fixed seed, and ids_sample_sentences.npy (their indices)."""
    ids = device_array(d_ids, n_ids, "<i4")
    offs = device_array(d_offs, n_sent + 1, "<i8")
    pick = np.sort(np.random.default_rng(0).choice(n_sent, min(n_sent, DUMP_SENTENCES), replace=False))
    sample = np.concatenate([ids[offs[i]:offs[i + 1]] for i in pick] + [np.zeros(0, np.int32)])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "offsets.npy"), offs.astype(np.float64))
    np.save(os.path.join(out_dir, "ids_sample.npy"), sample.astype(np.float32))
    np.save(os.path.join(out_dir, "ids_sample_sentences.npy"), pick.astype(np.float64))


def ref_train_isolated(build, chunk_files, model, vocab, coverage, threads, timeout=600):
    """The reference's train_bpe (build "det" / "prod") or the oracle's (build "oracle", single-threaded) in a CHILD
    process, on the concatenation of cached corpus chunks.  The reference's multi-threaded trainer is racy (SURVEY 4):
    on a 128-core host the assert of BigObjectQueue::top (bpe.cpp:232) has fired on the config-5 corpus and would take
    the bench line with it.  Returns seconds, or a string saying what happened (e.g. the timeout)."""
    who = "oracle" if build == "oracle" else "reference"
    call = ("_bind.Oracle().train(data, %r, %d, %r)" % (model, vocab, coverage) if build == "oracle" else
            "_bind.Reference(%r).train(data, %r, %d, %r, n_threads=%d)" % (build, model, vocab, coverage, threads))
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import _bind\n"
            "data = b''.join(open(f, 'rb').read() for f in %r)\n"
            "sec = %s\n"
            "print('REF_SECONDS', sec)\n") % (ROOT, os.path.join(ROOT, "tests"), list(chunk_files), call)
    try:
        r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=timeout)
    except subprocess.TimeoutExpired:
        return "%s timed out after %d s" % (who, timeout)
    for ln in r.stdout.decode(errors="replace").splitlines():
        if ln.startswith("REF_SECONDS"):
            return float(ln.split()[1])
    tail = r.stderr.decode(errors="replace").strip().splitlines()[-1:] or ["no output"]
    return "%s died (rc %d): %s" % (who, r.returncode, tail[0][-160:])


def chunk_files(kind, ids):
    return [os.path.join(CACHE, "%s_%d_%d.bin" % (kind, CHUNK, k)) for k in ids]


def reference_model(text):
    """The 32k model of the reference arm, trained with the reference itself (DETERMINISTIC_QUEUE build = the tie-break
    order both implementations are pinned to), cached on disk."""
    import _bind
    model = os.path.join(CACHE, "model_ref_%d.yttm" % VOCAB)
    if not os.path.exists(model):
        if _bind.have_reference("det"):
            _bind.Reference("det").train(text, model, VOCAB, 1.0, n_threads=min(8, os.cpu_count() or 1))
        else:
            _bind.Oracle().train(text, model, VOCAB, 1.0)
    return model


def reference_arm(args, rank, world):
    """--impl reference: the reference's CPU encode_as_ids on the same workload, all host threads."""
    if rank != 0:
        return
    import _bind
    _bind.build_checkers()
    cores = os.cpu_count() or 1
    text, buf, offs = workload(0, N_SENT, TRAIN_BYTES)
    model = reference_model(text)
    times = []
    sample = min(N_SENT, max(50_000, 40_000 * cores))
    base = None
    for it in range(args.warmup + args.steps):
        base, _ = cpu_reference_encode(model, buf, offs, cores, sample)
        if it >= args.warmup:
            times.append(sample / (base["value"] * 1e6))
    sec = sum(times) / len(times)          # the line's value: mean over the timed steps, as for the GPU arm
    val = sample / sec / 1e6
    base["value"] = val
    base["steps_s"] = {"min": min(times), "median": statistics.median(times), "max": max(times)}
    for th in (1, 8):                      # SURVEY 8d: n_threads rows that make the ratio interpretable
        if th < cores:
            row, _ = cpu_reference_encode(model, buf, offs, th, 50_000 * th, reps=3)
            base["n_threads_%d" % th] = {"value": row["value"], "sample": row["sample"]}
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Msent/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32", "data": "synthetic",
           "config": {"workload": WORKLOAD,
                      "step": "reference encode_as_ids on %d sentences, %d threads" % (sample, cores)},
           "cpu_baseline": base,
           "e2e": {"value": val, "unit": "Msent/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


_REAL_STDOUT = None


def quiet_stdout():
    """stdout must carry the ONE JSON line and nothing else, but libraries write to fd 1 behind
    Python's back (NCCL prints its version banner there): point fd 1 at stderr for the whole run
    and keep a private duplicate of the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(out):
    line = (json.dumps(out) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, line)
    else:
        os.write(_REAL_STDOUT, line)


def r3(x):
    return None if x is None else float("%.4g" % x)


# ---------------------------------------------------------------------------------------------------------------
# training legs (hot path a) — every world size runs the same code: distributed.train_distributed
# ---------------------------------------------------------------------------------------------------------------
def train_leg(comm, device, kind, chunk_ids, vocab, coverage, tag, runs=None, cache=True):
    """Train on this rank's chunks of corpus `kind`; wall = max over ranks, from host memory to the rules on the host.
    Returns the summary of the fastest of `runs` runs (the first one pays context creation and allocations)."""
    import torch
    from youtokentome_b200 import distributed as D, synth
    t0 = time.perf_counter()
    shard = b"".join(synth.corpus_chunks(kind, chunk_ids, CHUNK, cache_dir=CACHE if cache else None))
    gen_s = time.perf_counter() - t0
    model = os.path.join(CACHE, "model_%s_w%d.yttm" % (tag, comm.world))
    best = None
    walls = []
    for _ in range(runs or TRAIN_RUNS):
        st = {}
        comm.barrier()
        t0 = time.perf_counter()
        D.train_distributed(shard, model, vocab, coverage, comm=comm, device=device, sharded=True, stats_out=st)
        wall = time.perf_counter() - t0
        if comm.world > 1:
            t = torch.tensor([wall], dtype=torch.float64, device="cuda")
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            wall = float(t.item())
        walls.append(wall)
        if best is None or wall < best[0]:
            best = (wall, st)
    wall, st = best
    total = len(shard)
    uniq, toks = st["n_unique"], st["n_tokens"]
    if comm.world > 1:
        t = torch.tensor([total, uniq, toks], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(t)
        total, uniq, toks = (int(x) for x in t.tolist())
    sha = None
    if comm.rank == 0:
        with open(model, "rb") as f:
            sha = hashlib.sha1(f.read()).hexdigest()[:12]
    fm = st["front_ms"]
    return {"bytes": total, "gpus": comm.world, "wall_s": r3(wall), "GBps": r3(total / wall / 1e9), "walls_s": [r3(w) for w in walls],
            "merges": st["n_merges"], "us_per_merge": r3(st["merge_loop_ms"] * 1e3 / max(st["n_merges"], 1)),
            "merge_loop_ms": r3(st["merge_loop_ms"]), "launches": int(st["launches"]), "U": uniq, "T": toks,
            "front_ms_rank0": {k: r3(v) for k, v in fm.items()},
            "phase_us": {k.replace("loop_", ""): r3(v) for k, v in st["phase_us_per_iter"].items()},
            "host_ms_rank0": {k: r3(v) for k, v in st.get("host_ms", {}).items()},
            "model_sha1": sha, "gen_s": r3(gen_s)}, shard, model


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-legs", action="store_true", help="encode only (profiling runs)")
    ap.add_argument("--scan-tokens", type=int, default=256 * 1024 * 1024)
    ap.add_argument("--budget-s", type=float, default=420.0, help="optional legs are skipped once the run is this old")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) as .npy files")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from youtokentome_b200 import _lib, distributed as D
    from _gpu import gpu_train
    torch.cuda.set_device(local)
    os.environ["YTTM_DEVICE"] = str(local)
    os.environ.setdefault("YTTM_TRAIN_KEEP_CACHE", "1")   # the encode model is trained several times: reuse the context
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    L = _lib.lib()
    hbm_peak, peak_src = peaks()
    old = lambda: time.time() - T_START > args.budget_s
    notes = []

    text, buf, offs = workload(rank, N_SENT, TRAIN_BYTES)
    n_sent, n_bytes = len(offs) - 1, int(offs[-1])

    # ---- model of the encode leg: this framework's GPU trainer (hot path a), outside the timed region
    model = os.path.join(CACHE, "model_gpu_%d_r%d.yttm" % (VOCAB, rank))
    gpu_train(text, VOCAB, 1.0, model=model)           # cold: first CUDA work of the process
    L.yttm_api_release_training_cache()

    # ---- encoder handle + device-resident inputs
    h = L.yttm_api_open(model.encode(), 1)
    assert h, L.yttm_api_last_error(None)
    ctx, enc = L.yttm_api_device_context(h), L.yttm_api_device_encoder(h)
    host_bytes = torch.frombuffer(bytearray(buf), dtype=torch.uint8).pin_memory()
    host_offs = torch.from_numpy(offs.astype(np.int64)).pin_memory()
    d_bytes, d_offs = host_bytes.cuda(), host_offs.cuda()
    out_cap = n_bytes + 3 * n_sent + 16
    host_ids = torch.empty(out_cap, dtype=torch.int32).pin_memory()
    host_oo = torch.empty(n_sent + 1, dtype=torch.int64).pin_memory()
    page_bytes = np.frombuffer(buf, dtype=np.uint8)     # pageable caller: plain numpy buffers
    page_offs = offs.astype(np.uint64)
    page_ids = np.empty(out_cap, dtype=np.int32)
    page_oo = np.empty(n_sent + 1, dtype=np.uint64)

    last = {}

    def step_device():
        out_n = C.c_uint64(0)
        p1, p2 = C.c_void_p(), C.c_void_p()
        rc = L.yttm_enc_run_device(enc, d_bytes.data_ptr(), d_offs.data_ptr(), n_bytes, n_sent, 0, 0, 0, 0.0, 0, 0,
                                   C.byref(p1), C.byref(p2), C.byref(out_n))
        assert rc == 0, L.yttm_last_error(ctx)
        last.update(ids=p1.value, offsets=p2.value)
        return out_n.value

    def step_host():
        out_n = C.c_uint64(0)
        rc = L.yttm_enc_run(enc, host_bytes.data_ptr(), host_offs.data_ptr(), n_sent, 0, 0, 0, 0.0, 0, 0,
                            host_ids.data_ptr(), out_cap, host_oo.data_ptr(), C.byref(out_n))
        assert rc == 0, L.yttm_last_error(ctx)
        return out_n.value

    def step_pageable():
        out_n = C.c_uint64(0)
        rc = L.yttm_enc_run(enc, page_bytes.ctypes.data, page_offs.ctypes.data, n_sent, 0, 0, 0, 0.0, 0, 0,
                            page_ids.ctypes.data, out_cap, page_oo.ctypes.data, C.byref(out_n))
        assert rc == 0, L.yttm_last_error(ctx)
        return out_n.value

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    STAGES = ["enc_find", "enc_words", "enc_dedup", "enc_rep", "enc_copy", "enc_count", "enc_gather", "enc_scan"]

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            n_ids = fn()
        barrier()
        l0 = L.yttm_launch_count(ctx)
        kern = {k: 0.0 for k in STAGES}
        t0 = time.perf_counter()
        for _ in range(steps):
            n_ids = fn()
            for k in kern:
                kern[k] += max(L.yttm_stage_ms(ctx, k.encode()), 0.0)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        launches = L.yttm_launch_count(ctx) - l0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        return sec, n_ids, {k: v / steps for k, v in kern.items()}, launches

    # clocks / throttle reasons are sampled (100 ms period) from before the warm-up of the first timed
    # loop to the end of the last one: the timed regions themselves last only tens of milliseconds
    sampler = ClockSampler(local) if rank == 0 else None
    time.sleep(0.3 if rank == 0 else 0.0)
    sec_d, n_ids, kern, launches = timed(step_device, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:      # the results stay valid until the encoder's next call
        dump_outputs(args.dump_outputs, last["ids"], last["offsets"], n_ids, n_sent)
    sec_h, n_ids_h, _, _ = timed(step_host, args.steps, args.warmup)
    sec_p, n_ids_p, _, _ = timed(step_pageable, args.steps, 2)
    for _ in range(20):                       # keep the GPU busy long enough for a few more samples
        step_device()
    clocks = sampler.stop() if sampler else None
    assert n_ids == n_ids_h == n_ids_p

    value = world * n_sent * args.steps / sec_d / 1e6
    e2e = world * n_sent * args.steps / sec_h / 1e6
    e2e_page = world * n_sent * args.steps / sec_p / 1e6
    algo = n_bytes + 4 * n_ids + 16 * n_sent
    # enc_words is the sum of its three launches in the dedup path: the roofline kernel is a single launch
    single = {k: v for k, v in kern.items() if v > 0 and not (k == "enc_words" and kern["enc_dedup"] > 0)}
    dom = max(single, key=lambda k: single[k])
    names = {"enc_words": "encode_words_kernel", "enc_find": "find_words_vec_kernel", "enc_gather": "emit_ids_kernel",
             "enc_count": "sentence_ids_kernel",
             "enc_scan": "scan", "enc_dedup": "dedup_words_kernel", "enc_rep": "encode_rep_words_kernel",
             "enc_copy": "copy_word_ids_kernel"}
    ach = algo / (single[dom] * 1e-3) / 1e9
    traffic, traffic_src = measured_traffic(names[dom], n_sent)
    roofline = {"bound": "hbm", "kernel": names[dom], "achieved": r3(ach), "peak": hbm_peak, "unit": "GB/s",
                "frac": r3(ach / hbm_peak), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo, "kernel_ms": {k: r3(v) for k, v in kern.items() if v > 0},
                "step_frac_of_peak": r3(algo / (sec_d / args.steps) / 1e9 / hbm_peak)}

    cfg_train, cpu, enc4 = {}, None, None
    comm = D.TorchComm() if world > 1 else D.LocalComm()
    L.yttm_api_close(h)
    h = None
    torch.cuda.empty_cache()

    if not args.no_train_legs:
        # ---- BASELINE configs[2]: 1 GB Zipf, vocab 32k, strong scaling over the ranks (8 / N chunks each)
        per = 8 // world if world in (1, 2, 4, 8) else 1
        c3, shard3, model3 = train_leg(comm, local, "zipf", range(rank * per, (rank + 1) * per), VOCAB, 1.0, "cfg3")
        c3["scaling"] = "strong (1 GB total)"
        cfg_train["config3"] = c3
        fm = c3["front_ms_rank0"]
        if rank == 0:
            nb = len(shard3)
            piped = fm["char_hist"] <= 0   # both byte passes ran per piece behind the H2D copy (train.cu: pipelined_load)
            roofline["train_front"] = {"bytes_rank0": nb, "h2d_GBps": r3(nb / fm["h2d"] / 1e6),
                                       "char_hist_GBps": None if piped else r3(nb / fm["char_hist"] / 1e6),
                                       "word_count_GBps": None if piped else r3(nb / fm["word_count"] / 1e6),
                                       "note": ("char_hist + word split run per 32 MB piece on a second stream while the next piece is "
                                                "copied: their time is inside h2d (kernel rates: profiles/r02_prof_front.raw.csv, "
                                                "57 / 25 GB/s)") if piped else None,
                                       "algorithmic_bytes": "B per pass (SURVEY 8d)"}
        del shard3
        # ---- BASELINE configs[4] shape: multilingual, vocab 64k, coverage 0.9999, 1.25 GB per GPU (weak)
        if not old():
            c5, shard5, _ = train_leg(comm, local, "multilingual", range(rank * 10, rank * 10 + 10), VOCAB5, 0.9999, "cfg5",
                                      cache=(world == 1))
            c5["scaling"] = "weak (1.25 GB per GPU)"
            cfg_train["config5"] = c5
        else:
            notes.append("config5 skipped: run older than --budget-s")
            shard5 = None

    if rank == 0 and world == 1 and not args.no_train_legs:
        import _bind
        _bind.build_checkers()
        cores = os.cpu_count() or 1
        from youtokentome_b200 import synth
        # ---- BASELINE configs[0]: the README example (latency-bound: us / merge is the figure, not a roofline fraction)
        readme = synth.readme_corpus(n_lines=CFG1_LINES)
        st = {}
        walls = []
        m1 = os.path.join(CACHE, "model_cfg1.yttm")
        for _ in range(TRAIN_RUNS + 1):
            t0 = time.perf_counter()
            D.train_distributed(readme, m1, CFG1_VOCAB, 1.0, comm=comm, device=local, sharded=True, stats_out=st)
            walls.append(time.perf_counter() - t0)
        cfg_train["config1"] = {"bytes": len(readme), "wall_s": r3(min(walls)), "merges": st["n_merges"],
                                "us_per_merge": r3(st["merge_loop_ms"] * 1e3 / max(st["n_merges"], 1)),
                                "U": st["n_unique"], "T": st["n_tokens"]}
        if not args.no_cpu_baseline:
            mo = os.path.join(CACHE, "model_cfg1_ref.yttm")
            chk, sec = cpu_train(readme, mo, CFG1_VOCAB, 1.0)
            cfg_train["config1"]["equals_" + chk] = _bind.read_model(mo) == _bind.read_model(m1)
            cfg_train["config1"]["cpu_%s_1thr_s" % chk] = r3(sec)

        # ---- parity + CPU baselines of configs 3 / 5 on their first chunk (the reference needs ~10 s per 100 MB)
        if not args.no_cpu_baseline and not old():
            for key, kind, vocab, cov in (("config3", "zipf", VOCAB, 1.0), ("config5", "multilingual", VOCAB5, 0.9999)):
                if key not in cfg_train or old():
                    continue
                chunk = synth.corpus_chunks(kind, [0], CHUNK, cache_dir=CACHE)[0]
                mg = os.path.join(CACHE, "model_%s_chunk0_gpu.yttm" % key)
                mr = os.path.join(CACHE, "model_%s_chunk0_ref.yttm" % key)
                D.train_distributed(chunk, mg, vocab, cov, comm=comm, device=local, sharded=True)
                chk = "reference" if _bind.have_reference("det") else "oracle"   # the oracle runs under the same timeout
                sec = ref_train_isolated("det" if chk == "reference" else "oracle", chunk_files(kind, [0]), mr, vocab, cov, 1)
                ok = isinstance(sec, float) and _bind.read_model(mg) == _bind.read_model(mr)
                cfg_train[key]["parity_chunk0"] = {"bytes": len(chunk), "equals_" + chk: ok if isinstance(sec, float) else None,
                                                   ("reference_det_1thr_s" if chk == "reference" else "oracle_1thr_s"):
                                                       r3(sec) if isinstance(sec, float) else sec}

        # ---- hot path (a) on a buffer >> L2: the per-merge scan in STREAMING mode (TMA-staged tiles).  Algorithmic
        # bytes 4T + 4U per merge (frequencies are read for rewritten words only); time = device-side timers of the
        # apply phase incl. its closing grid barrier.
        if args.scan_tokens > 0 and not old():
            def scan_probe(log2_first):
                c2 = C.c_void_p()
                assert L.yttm_ctx_create(local, C.byref(c2)) == 0
                wl, alpha, iters = 8, 2000, 12
                n_w = args.scan_tokens // wl
                rc = L.yttm_train_synth_words(c2, n_w, wl, alpha | (log2_first << 24), 7)
                assert rc == 0, L.yttm_last_error(c2)
                rules = np.zeros(3 * iters, dtype=np.uint32)
                fr = np.zeros(iters, dtype=np.uint64)
                nd = C.c_uint32(0)
                assert L.yttm_train_run(c2, 4 + (1 << log2_first) + alpha, iters, rules.ctypes.data, fr.ctypes.data,
                                        C.byref(nd)) == 0, L.yttm_last_error(c2)
                g = lambda k: L.yttm_stage_ms(c2, k.encode())
                it = max(g("loop_iters"), 1.0)
                t_scan = (g("loop_apply") + g("loop_partition") + g("loop_drain")) / it          # ms per merge
                ab = 4 * args.scan_tokens + 4 * n_w
                a_ = ab / (t_scan * 1e-3) / 1e9
                ms, ab2 = C.c_double(0), C.c_uint64(0)
                L.yttm_train_scan_once(c2, C.byref(ms), C.byref(ab2))
                out = {"achieved": r3(a_), "frac": r3(a_ / hbm_peak), "ms_per_merge_scan": r3(t_scan),
                       "ms_per_merge_all": r3(sum(g(k) for k in ("loop_elect", "loop_apply", "loop_partition", "loop_drain")) / it),
                       "resident": int(g("loop_resident")),
                       "pair_hist_GBps": r3(ab2.value / (ms.value * 1e-3) / 1e9)}
                L.yttm_ctx_destroy(c2)
                return out, ab
            heavy, ab = scan_probe(0)     # every merge rewrites ~17 000 words
            light, _ = scan_probe(10)     # a merge rewrites a few dozen words (the bulk of a long training run)
            roofline["train_scan"] = {"kernel": "merge_loop_kernel apply phase, STREAMING (TMA ring)", "tokens": args.scan_tokens,
                                      "algorithmic_bytes_per_merge": ab, "heavy": heavy, "light": light, "peak": hbm_peak}

        # ---- BASELINE configs[3] shape: lognormal sentences of mean 512 B, dropout 0.1
        if not old():
            fz = synth.FastZipf(n_words=200_000, s=1.07, seed=1234)
            n4 = N_SENT4
            b4, o4 = fz.packed_sentences(n4, 512, seed=4321, lognormal=True)
            h4 = L.yttm_api_open(model.encode(), 1)
            ctx4, enc4h = L.yttm_api_device_context(h4), L.yttm_api_device_encoder(h4)
            hb = torch.frombuffer(bytearray(b4), dtype=torch.uint8).pin_memory()
            ho = torch.from_numpy(o4.astype(np.int64)).pin_memory()
            db, do = hb.cuda(), ho.cuda()
            cap4 = len(b4) + 3 * n4 + 16
            hid = torch.empty(cap4, dtype=torch.int32).pin_memory()
            hoo = torch.empty(n4 + 1, dtype=torch.int64).pin_memory()

            def run4(host, dropout):
                out_n = C.c_uint64(0)
                if host:
                    rc = L.yttm_enc_run(enc4h, hb.data_ptr(), ho.data_ptr(), n4, 0, 0, 0, dropout, 77, 0, hid.data_ptr(), cap4,
                                        hoo.data_ptr(), C.byref(out_n))
                else:
                    p1, p2 = C.c_void_p(), C.c_void_p()
                    rc = L.yttm_enc_run_device(enc4h, db.data_ptr(), do.data_ptr(), len(b4), n4, 0, 0, 0, dropout, 77, 0,
                                               C.byref(p1), C.byref(p2), C.byref(out_n))
                assert rc == 0, L.yttm_last_error(ctx4)
                return out_n.value

            def t4(host, dropout, reps=5):
                run4(host, dropout)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(reps):
                    run4(host, dropout)
                torch.cuda.synchronize()
                return n4 * reps / (time.perf_counter() - t0) / 1e6
            enc4 = {"sentences": n4, "bytes": len(b4), "dropout": 0.1, "Msent_s_device": r3(t4(False, 0.1)),
                    "Msent_s_e2e": r3(t4(True, 0.1)), "Msent_s_device_dropout0": r3(t4(False, 0.0)),
                    "note": "dropout parity unpinned by the reference (its RNG is a racy global mt19937): ids == the oracle's Philox stream"}
            run4(True, 0.1)
            k = min(3000, n4)
            oo = np.ascontiguousarray(o4[:k + 1])
            want, _ = _bind.Oracle().encoder(model).encode_packed(b4, oo, dropout=0.1, seed=77)
            enc4["ids_equal_oracle_on_sample"] = bool(np.array_equal(hid[:len(want)].numpy(), want))
            enc4["sample"] = "%d sentences vs oracle" % k
            L.yttm_api_close(h4)

        # ---- CPU baselines: the unmodified reference on the host cores
        if not args.no_cpu_baseline:
            hm = L.yttm_api_open(model.encode(), 1)
            enc_m = L.yttm_api_device_encoder(hm)
            cpu, ref_ids = cpu_reference_encode(model, buf, offs, cores, min(n_sent, max(50_000, 40_000 * cores)), reps=3)
            out_n = C.c_uint64(0)
            rc = L.yttm_enc_run(enc_m, host_bytes.data_ptr(), host_offs.data_ptr(), n_sent, 0, 0, 0, 0.0, 0, 0,
                                host_ids.data_ptr(), out_cap, host_oo.data_ptr(), C.byref(out_n))
            assert rc == 0
            assert np.array_equal(host_ids[:len(ref_ids)].numpy(), ref_ids), "bench: GPU ids differ from the reference"
            cpu["ids_equal_on_sample"] = True
            L.yttm_api_close(hm)
            for th in (1, 8):
                if th < cores:
                    row, _ = cpu_reference_encode(model, buf, offs, th, 50_000 * th, reps=3)
                    cpu["n_threads_%d" % th] = {"value": r3(row["value"]), "sample": row["sample"]}
            if _bind.have_reference("prod") and "config3" in cfg_train and not old():
                nb = cfg_train["config3"]["bytes"]
                sec8 = ref_train_isolated("prod", chunk_files("zipf", range(8)), os.path.join(CACHE, "model_refprod.yttm"), VOCAB, 1.0,
                                          min(8, cores))
                sec1 = ref_train_isolated("prod", chunk_files("zipf", [0]), os.path.join(CACHE, "model_refprod1.yttm"), VOCAB, 1.0, 1)
                cpu["train_1GB_8thr"] = {"seconds": r3(sec8), "GBps": r3(nb / sec8 / 1e9)} if isinstance(sec8, float) else {"error": sec8}
                cpu["train_125MB_1thr"] = {"seconds": r3(sec1), "GBps": r3(nb / 8 / sec1 / 1e9)} if isinstance(sec1, float) else {"error": sec1}
                if isinstance(sec8, float):
                    cfg_train["config3"]["speedup_vs_reference_8thr"] = r3(sec8 / cfg_train["config3"]["wall_s"])

    if rank == 0:
        config = {"workload": WORKLOAD, "sharding": "per GPU: the workload above on every rank (weak scaling), no collective",
                  "sentences_per_gpu": n_sent, "bytes_per_gpu": n_bytes, "ids_per_gpu": n_ids,
                  "l2": "inputs + slot buffers (%.0f MB) exceed the 126 MB L2" % ((5 * n_bytes) / 1e6),
                  "train": cfg_train}
        if enc4:
            config["encode_config4"] = enc4
        if notes:
            config["notes"] = notes
        out = {"metric": METRIC, "value": value, "unit": "Msent/s", "n_gpus": args.gpus, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": sec_d / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "u8/u32", "data": "synthetic", "config": config,
               "e2e": {"value": e2e, "unit": "Msent/s", "h2d_bytes_per_step": n_bytes + 8 * (n_sent + 1),
                       "d2h_bytes_per_step": 4 * n_ids + 8 * (n_sent + 1), "ms_per_step": sec_h / args.steps * 1e3,
                       "host_buffers": "pinned", "pageable_value": r3(e2e_page)},
               "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
               "wall_s": r3(time.time() - T_START)}
        emit(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
