"""The reference's OWN stress test (tests/unit_tests/stress_test.cpp: learn_bpe_slow / decode_slow specs, seeds,
manual case, batch == single) run against the product's kernels under the SIMT emulator (tests/emul/simt; test harness
only).  The binary is oracle/_ref/ref_stress_b200, which build() compiles (oracle/Makefile) from the unmodified source
against this repo's drop-in headers (include/compat) where the reference's sources are present; it is linked with
libyttm_b200.so, and here the emulator build takes that name on LD_LIBRARY_PATH, which its RUNPATH gives way to.
tests/test_zz_reference_stress_gpu.py runs the same binary with the real library on the B200."""
import os
import subprocess

import pytest

from _bind import ROOT

BIN = os.path.join(ROOT, "oracle", "_ref", "ref_stress_b200")
pytestmark = pytest.mark.skipif(not os.path.exists(BIN), reason="oracle/_ref/ref_stress_b200 not built")


@pytest.fixture(scope="module")
def emulated_lib_dir(tmp_path_factory):
    """A directory where libyttm_b200.so is the emulator build of the kernels."""
    from _emu import emu_lib
    emu_lib()  # builds tests/emul/simt/_gen/libyttm_emu.so
    d = tmp_path_factory.mktemp("emulated_lib")
    os.symlink(os.path.join(ROOT, "tests", "emul", "simt", "_gen", "libyttm_emu.so"), d / "libyttm_b200.so")
    return str(d)


@pytest.mark.parametrize("args", [["manual"], ["base", "60"], ["parallel", "6"]])
def test_reference_stress_test_passes_on_the_emulated_kernels(emulated_lib_dir, tmp_path, args):
    env = dict(os.environ, YT_EMU_SMS="2", LD_LIBRARY_PATH=emulated_lib_dir)
    r = subprocess.run([BIN] + args, cwd=tmp_path, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE,
                       timeout=900)
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-2000:]
