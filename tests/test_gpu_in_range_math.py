"""GPU: the guard-free square root and division of csrc/s2d_math.cuh (sqrt_in_range, div_in_range, atan2_deg<true>),
which check_episode uses when in_range_vector holds, give the bits of the IEEE operators over the domains that predicate
proves: every float of [2^-40, 2^40] for the square root; for the division every 64th divisor of [2^-21, 2^22] and both
ends, each with numerator +0, +-divisor, the floats next to it, +-2^-100 and random numerators; 2^28 random vectors,
with components down to subnormals, through check_episode's selection for atan2 and the distance.
tests/in_range_math_check.cu is compiled with the library's flags into a temporary directory and run."""
import os
import shutil
import subprocess
import tempfile

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gym-soccer-2d-env_b200", "csrc")


def nvcc():
    for c in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc"), shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found (CUDA_HOME or PATH): the check has to be compiled for sm_100a")


def test_in_range_sqrt_and_division_equal_ieee():
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "in_range_math_check")
        subprocess.run([nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "--fmad=false", "-std=c++17",
                        "-I", CSRC, "-o", exe, os.path.join(ROOT, "tests", "in_range_math_check.cu")],
                       check=True, capture_output=True, text=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    print(out)
    rows = {line.split()[0]: line.split()[1:] for line in out.splitlines() if not line.startswith(" ")}
    assert {"sqrt", "div", "atan2", "div_outside_domain", "atan2_fast"} <= set(rows), out
    assert int(rows["sqrt"][0]) == (80 << 23) + 1  # every float of [2^-40, 2^40]
    assert int(rows["div"][0]) == 32 * ((43 << 23) // 64 + 2) and int(rows["atan2"][0]) == 1 << 28
    assert int(rows["atan2_fast"][0]) > 1 << 26  # most vectors take the guard-free forms, tiny components do not
    assert [int(rows[k][1]) for k in ("sqrt", "div", "atan2")] == [0, 0, 0], out
