"""The affix records from a plain C++ host (tests/cpp/test_affixes.cpp over include/apgk_adapters.hpp):
KmerFreqAffixes<K> and KmerParcelsBuilder::Affixes against the hand vectors and each other."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp_path):
    exe = str(tmp_path / "test_affixes")
    libdir = os.path.join(ROOT, "allpathslg_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_affixes.cpp"), "-L" + libdir, "-lapgk",
                           "-Wl,-rpath," + libdir, "-o", exe])
    return exe


def test_cpp_affixes_compiles(tmp_path, apgk_lib):
    _build(tmp_path)


@pytest.mark.gpu
def test_cpp_affixes_on_gpu(tmp_path, apgk_lib):
    r = subprocess.run([_build(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr + r.stdout
    assert "AFFIXES OK" in r.stdout
