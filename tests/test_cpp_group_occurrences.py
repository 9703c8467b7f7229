"""The occurrence records on the sharded table from a plain C++ host (tests/cpp/test_group_occurrences.cpp over
include/apgk.h): single-process group on one GPU, and -- where the box has two GPUs -- one process per GPU with NCCL
+ CUDA IPC.  Both compare every shard row with one context's apgk_build_occurrences over all the reads."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp_path):
    exe = str(tmp_path / "test_group_occurrences")
    libdir = os.path.join(ROOT, "allpathslg_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_group_occurrences.cpp"), "-L" + libdir, "-lapgk",
                           "-Wl,-rpath," + libdir, "-o", exe])
    return exe


def test_cpp_group_occurrences_compiles(tmp_path, apgk_lib):
    _build(tmp_path)


@pytest.mark.gpu
def test_cpp_group_occurrences_single_process(tmp_path, apgk_lib):
    r = subprocess.run([_build(tmp_path), "local", "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr + r.stdout
    assert "OCCURRENCES OK" in r.stdout


@pytest.mark.gpu
def test_cpp_group_occurrences_one_process_per_gpu(tmp_path, apgk_lib):
    r = subprocess.run([_build(tmp_path), "procs", "2"], capture_output=True, text=True, timeout=300)
    if r.returncode == 77:
        pytest.skip(r.stdout.strip())
    assert r.returncode == 0, r.stderr + r.stdout
    assert "OCCURRENCES OK" in r.stdout
