"""tests/cpp/leaves_example.cpp: getVoxelCenters / getOccupiedVoxelIndices / isEmpty of the C++ shim compile against the C ABI
and link with libb200tsdf.so; on a GPU box the example runs (getOccupiedVoxelIndices appends, getVoxelCenters () gives the
8^4 level-4 cells at 2048^3 / 10 m)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "leaves_example.cpp")
CXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def build(engine_lib, out_dir):
    libdir = os.path.dirname(engine_lib)
    exe = os.path.join(str(out_dir), "leaves_example")
    subprocess.run([CXX, "-std=c++17", "-O1", "-Wall", SRC, "-o", exe, f"-L{libdir}", "-lb200tsdf", f"-Wl,-rpath,{libdir}",
                    "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"], check=True)
    return exe


def test_leaves_example_compiles_and_reports_missing_device(engine_lib, tmp_path):
    exe = build(engine_lib, tmp_path)
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("device present: covered by the gpu test")
    except ImportError:
        pass
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3, r.stdout + r.stderr


@pytest.mark.gpu
def test_leaves_example_runs(engine_lib, tmp_path):
    exe = build(engine_lib, tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "leaves ok" in r.stdout
