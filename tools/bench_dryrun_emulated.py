"""TEST HARNESS: bench.py's whole control flow on a box without a GPU.  torch.cuda is stubbed to no-ops, the library is
the CPU SIMT emulator build of the product's kernels (tests/emul/simt: its "device" memory is host memory), the workload
constants are shrunk (3 000 sentences, vocab 3 000, 300 KB of training text, 30 KB corpus chunks) and bench.main() runs
as it is: model training, the device-resident / pinned / pageable timed loops, the training legs of configs 1, 3 and 5
through distributed.train_distributed with their reference parity checks, the scan probes, the dropout leg of config 4
with its oracle check, the CPU baselines with the id comparison and the ONE JSON line.
The numbers mean nothing; the point is that a slip in bench.py shows up here and not on the driver's GPU box.
    python tools/bench_dryrun_emulated.py [extra bench.py flags]  > line.json"""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ.setdefault("YT_EMU_SMS", "2")
os.environ.setdefault("YTTM_BENCH_CACHE", "/tmp/yttm_b200_bench_dryrun_cache")

import numpy as np  # noqa: E402
import torch  # noqa: E402
from _emu import emu_lib  # noqa: E402
from youtokentome_b200 import _lib  # noqa: E402

_lib._lib = emu_lib()
torch.cuda.set_device = lambda *a, **k: None
torch.cuda.synchronize = lambda *a, **k: None
torch.cuda.is_available = lambda: False
torch.cuda.empty_cache = lambda *a, **k: None
torch.Tensor.cuda = lambda self, *a, **k: self
torch.Tensor.pin_memory = lambda self, *a, **k: self

import bench  # noqa: E402

bench.N_SENT, bench.VOCAB, bench.TRAIN_BYTES = 3000, 3000, 300_000
bench.CHUNK, bench.VOCAB5, bench.CFG1_LINES, bench.CFG1_VOCAB, bench.N_SENT4, bench.TRAIN_RUNS = 30_000, 4200, 200, 200, 300, 1


class _NoClocks:
    def __init__(self, index):
        pass

    def stop(self):
        return {"sm_mhz": 0.0, "sm_max_mhz": 0.0, "reasons": [], "samples": 0}


bench.ClockSampler = _NoClocks
# the emulator's "device" memory is host memory
bench.device_array = lambda ptr, n, typestr: np.frombuffer((C.c_char * (n * np.dtype(typestr).itemsize)).from_address(ptr),
                                                           dtype=typestr).copy()
sys.argv = ["bench.py", "--steps", "2", "--warmup", "3", "--scan-tokens", "131072"] + sys.argv[1:]
bench.main()
