"""k_fft_tiles' cross-phase bin map (csrc/fft_tile_core.cuh tile_bin_parity), emulated on the host: every bin below
N/2 taken once, accumulators bit-equal to reading all four operands from shared memory, conflict-free 64-bit loads."""
import shutil
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.skipif(shutil.which("nvcc") is None, reason="needs nvcc (host compile only)")
def test_tile_cross_bin_map(tmp_path):
    exe = tmp_path / "fft_tile_cross_emul"
    subprocess.run(["nvcc", "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "-I",
                    str(ROOT / "tdoa-geolocation_b200" / "csrc"), "-o", str(exe),
                    str(ROOT / "tests" / "native" / "fft_tile_cross_emul.cu")], check=True)
    res = subprocess.run([str(exe)], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout
    vals = {l.split()[0]: int(l.split()[1]) for l in res.stdout.splitlines()}
    assert vals == {"bins_not_taken_once": 0, "accumulators_differing": 0, "conflicted_loads": 0}
