"""The C++ host example (examples/train_c_abi.cc) compiles against include/*.h alone, links to the in-tree library
and behaves as documented: a full training run on a GPU box, a loud YGG_ERR_NO_DEVICE without one."""
import os
import shutil
import subprocess

import pytest

import ydf_b200

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "yggdrasil-decision-forests_b200")


def _build(tmp_path):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no g++")
    ydf_b200.lib()  # makes sure the library is built
    exe = str(tmp_path / "train_c_abi")
    subprocess.check_call([cxx, "-std=c++17", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "train_c_abi.cc"), "-L", PKG, "-lygg_b200",
                           f"-Wl,-rpath,{PKG}", "-o", exe])
    return exe


def test_example_reports_abi_4_and_fails_loudly_without_a_device(tmp_path):
    if ydf_b200.device_count() > 0:
        pytest.skip("a CUDA device is present")
    r = subprocess.run([_build(tmp_path), "1000", "4", "5"], capture_output=True, text=True)
    assert r.returncode == 2                                        # YGG_ERR_NO_DEVICE
    assert "no CPU fallback" in r.stderr and "ABI 4" in r.stdout


@pytest.mark.gpu
def test_example_trains(tmp_path):
    r = subprocess.run([_build(tmp_path), "60000", "6", "40"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "trees kept" in r.stdout and "tree 0:" in r.stdout
    # 10 % of the rows are held out and the validation loss is reported
    assert "valid loss" in r.stdout
