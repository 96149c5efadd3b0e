"""gvpm::quotient_negative (gvpm_device.cuh) replaces the strictly rounded division of the side tests, whose quotient was
only read for its sign.  It must give the sign test's answer for every input: +-0, +-inf, NaN, subnormals and random
pairs with |b| < 2, against the host's IEEE division and against __fdiv_rn on the device."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "quotient_sign_check")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-o", exe,
                           os.path.join(ROOT, "tests", "quotient_sign_check.cu")])
    return exe


def _run(exe, mode):
    r = subprocess.run([exe, mode], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    assert " 0 mismatches" in r.stdout


def test_quotient_negative_host(tmp_path):
    _run(_build(tmp_path), "host")


@pytest.mark.gpu
def test_quotient_negative_device(tmp_path):
    _run(_build(tmp_path), "device")
