"""include/snn_b200.hpp — the C++17 mirror of the reference's Rust API above the C ABI (the reference's host language has no
toolchain in this image).  CPU: the header and its test program compile with -Wall -Wextra and link against libsnn_b200.so, and
without a device populate() reports GPUError::GetDeviceFailure instead of falling back.  GPU: the program replays the reference's
own integration tests (tests/cpp/host_mirror.cpp lists them) through the mirror."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "spiking-neural-networks_b200")
SRC = os.path.join(ROOT, "tests", "cpp", "host_mirror.cpp")


def build(out_dir):
    """Compiles the test program into `out_dir` (the repository tree may be read-only)."""
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if cxx is None:
        pytest.skip("no host C++ compiler")
    if not os.path.exists(os.path.join(PKG, "libsnn_b200.so")):
        pytest.fail("libsnn_b200.so is not built (python -c 'import __graft_entry__ as g; g.build()')")
    exe = str(out_dir / "host_mirror")
    cmd = [cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), SRC, "-o", exe,
           "-L", PKG, "-lsnn_b200", f"-Wl,-rpath,{PKG}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_cpp_mirror_compiles_links_and_has_no_cpu_fallback(tmp_path):
    exe = build(tmp_path)
    r = subprocess.run([exe, "--no-gpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cpp_mirror_replays_reference_integration_tests(tmp_path):
    exe = build(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "HOST_MIRROR_OK" in r.stdout, r.stdout + r.stderr
