"""The C++ host class's subset overloads (include/SdrBatch.hpp) build against the C ABI and link to the product library."""
import os
import subprocess

from audiosdr_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cpp_subset_overloads_build_and_link(tmp_path):
    lib = api.lib_path()
    assert os.path.exists(lib), "libsdr_batch.so missing: __graft_entry__.build() builds it"
    exe = str(tmp_path / "subset_class_smoke")
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", os.path.join(ROOT, "tests", "cpp", "subset_class_smoke.cpp"), "-o", exe,
                    "-L" + os.path.dirname(lib), "-lsdr_batch", "-Wl,-rpath," + os.path.dirname(lib)], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "NO_DEVICE" in r.stdout or "GPU_OK" in r.stdout
