"""spiking-neural-networks_b200/csrc/step_spec.h — dispatch_step, the map from a run's kernel specialisation (model, chemg, ntrel,
stdp, net) to the template arguments of every step kernel.  CPU: tests/cpp/step_dispatch.cpp walks every input the engine can
produce and checks the instantiation it reaches, and that an unknown model is refused."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "step_dispatch.cpp")

# 9 models x (chemg 0: 8 inputs, chemg 1: 2 single-lattice inputs, chemg 3: 4) + 3 out-of-range models
N_INPUTS = 9 * 14 + 3


def test_dispatch_step_reaches_the_normalised_specialisation(tmp_path):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if cxx is None:
        pytest.skip("no host C++ compiler")
    exe = str(tmp_path / "step_dispatch")
    cmd = [cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "spiking-neural-networks_b200", "csrc"),
           SRC, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and r.stdout.strip() == f"STEP_DISPATCH_OK {N_INPUTS}", r.stdout + r.stderr
