"""The grabber's process overloads with per-pair snapshots and spectra (include/SdrAux.hpp) build against the C ABI and link
to the product library; on a GPU machine the program also runs them."""
import os
import subprocess

from audiosdr_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cpp_grabber_snapshot_overloads_build_and_link(tmp_path):
    lib = build.build_aux_library()  # nvcc cross-compiles sm_100a without a GPU
    exe = str(tmp_path / "grabber_snapshots_smoke")
    cuda = os.path.dirname(os.path.dirname(build._nvcc()))
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", os.path.join(ROOT, "tests", "cpp", "grabber_snapshots_smoke.cpp"), "-o", exe,
                    "-I" + os.path.join(cuda, "include"), "-L" + os.path.dirname(lib), "-lsdr_aux", "-L" + os.path.join(cuda, "lib64"),
                    "-lcudart", "-Wl,-rpath," + os.path.dirname(lib) + ":" + os.path.join(cuda, "lib64")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "NO_DEVICE" in r.stdout or "GPU_OK" in r.stdout
