"""The C++ mirror of zoe's interface (include/zoe_cuda.hpp): compiles and links on CPU; runs on the GPU box."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(out_dir):
    """Compile tests/cpp/test_hpp.cpp into `out_dir` (the source tree may be read-only); returns the executable."""
    from zoe_b200.build import build
    lib = build()
    exe = os.path.join(str(out_dir), "test_hpp")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_hpp.cpp"), "-o", exe, lib, f"-Wl,-rpath,{os.path.dirname(lib)}"]
    subprocess.check_call(cmd)
    return exe


def test_cpp_mirror_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_cpp_mirror_known_answers(tmp_path):
    exe = _build(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr + out.stdout
    assert "cpp mirror ok" in out.stdout
