"""The streamed receiver graph's C++ wrapper (include/SdrGraph.hpp) builds against the C ABI and links to the product
libraries; on a GPU machine the program also runs it."""
import os
import subprocess

from audiosdr_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cpp_graph_builds_and_links(tmp_path):
    lib = build.build_graph_library()  # nvcc cross-compiles sm_100a without a GPU
    exe = str(tmp_path / "graph_smoke")
    here = os.path.dirname(lib)
    cuda = os.path.dirname(os.path.dirname(build._nvcc()))
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", os.path.join(ROOT, "tests", "cpp", "graph_smoke.cpp"), "-o", exe,
                    "-I" + os.path.join(cuda, "include"), "-L" + here, "-lsdr_graph", "-lsdr_batch", "-lsdr_aux",
                    "-Wl,-rpath," + here], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "NO_DEVICE" in r.stdout or "GPU_OK" in r.stdout
