"""The waterfall's C++ wrappers (include/SdrAux.hpp WaterfallBatch and the grabber overload, include/SdrGraph.hpp's
_waterfall calls) build against the C ABI and link to the product libraries; on a GPU machine the program also runs them."""
import os
import subprocess

from audiosdr_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cpp_waterfall_builds_and_links(tmp_path):
    lib = build.build_graph_library()  # nvcc cross-compiles sm_100a without a GPU
    exe = str(tmp_path / "waterfall_smoke")
    here = os.path.dirname(lib)
    cuda = os.path.dirname(os.path.dirname(build._nvcc()))
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", os.path.join(ROOT, "tests", "cpp", "waterfall_smoke.cpp"), "-o", exe,
                    "-I" + os.path.join(cuda, "include"), "-L" + here, "-lsdr_graph", "-lsdr_batch", "-lsdr_aux",
                    "-L" + os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + here + ":" + os.path.join(cuda, "lib64")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "NO_DEVICE" in r.stdout or "GPU_OK" in r.stdout
