"""The source-compatible C++ facade (include/ufomap_b200/ufomap.hpp) compiles with a plain
host compiler against the C ABI and behaves like the reference on a device."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(out_dir):
    """Compiles tests/cpp/facade_smoke.cpp into out_dir (the source tree may be read-only)."""
    exe = os.path.join(str(out_dir), "facade_smoke")
    lib_dir = os.path.join(ROOT, "ufomap_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "facade_smoke.cpp"), "-o", exe,
                           "-L" + lib_dir, "-lufomap_b200", "-Wl,-rpath," + lib_dir])
    return exe


def test_facade_compiles_and_validates_arguments(tmp_path):
    exe = _build(tmp_path)
    out = subprocess.run([exe, "--no-device"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr


@pytest.mark.gpu
def test_facade_on_device(tmp_path):
    exe = _build(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and "facade ok" in out.stdout, (out.returncode, out.stdout, out.stderr)
