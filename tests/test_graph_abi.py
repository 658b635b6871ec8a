"""CPU tier: include/sdr_graph.h, libsdr_graph.so and audiosdr_b200/graph.py agree, and the library cross-compiles and links
without a device (no compute calls)."""
import ctypes
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    src = open(os.path.join(ROOT, "include", "sdr_graph.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sdr_graph_\w+)\s*\(", src)))


def test_header_declares_the_graph():
    f = declared_functions()
    for name in ("sdr_graph_create", "sdr_graph_destroy", "sdr_graph_submit_host", "sdr_graph_process_host", "sdr_graph_host_ticket",
                 "sdr_graph_wait_host", "sdr_graph_wait_host_ticket"):
        assert name in f


def test_library_exports_every_declared_symbol_and_links_its_members_by_origin():
    from audiosdr_b200 import build, graph
    path = build.build_graph_library()  # nvcc cross-compiles sm_100a without a GPU
    lib = ctypes.CDLL(path)
    for name in declared_functions():
        assert hasattr(lib, name), name
    assert set(graph.EXPORTS) == set(declared_functions())
    assert b"sm_100a" in ctypes.cast(lib.sdr_graph_version, ctypes.CFUNCTYPE(ctypes.c_char_p))()
    dyn = subprocess.run(["readelf", "-d", path], capture_output=True, text=True, check=True).stdout
    assert "[libsdr_batch.so]" in dyn and "[libsdr_aux.so]" in dyn and "$ORIGIN" in dyn


def test_the_graph_uses_the_members_accessors():
    """The handle checks (one device, one channel count) rest on accessors both member libraries export."""
    from audiosdr_b200 import api, aux, build
    for path, names, exports in ((build.build_library(), ["sdr_batch_get_desc"], api.EXPORTS),
                                 (build.build_aux_library(), ["sdr_preproc_get_info", "sdr_iqgen_get_info", "sdr_grabber_get_info"], aux.EXPORTS)):
        lib = ctypes.CDLL(path)
        for n in names:
            assert hasattr(lib, n) and n in exports, n


def test_structs_match_the_header():
    from audiosdr_b200 import graph
    assert ctypes.sizeof(graph.GraphDesc) == 4 * ctypes.sizeof(ctypes.c_void_p)
    assert ctypes.sizeof(graph.GraphOutputs) == 5 * ctypes.sizeof(ctypes.c_void_p)
    src = open(os.path.join(ROOT, "include", "sdr_graph.h")).read()
    desc = src[src.index("typedef struct {"):src.index("} sdr_graph_desc;")]
    outs = src[src.rindex("typedef struct {"):src.index("} sdr_graph_outputs;")]
    field = re.compile(r"\*(\w+);")
    assert [f for f in field.findall(re.sub(r"/\*.*?\*/", "", desc, flags=re.S))] == [n for n, _ in graph.GraphDesc._fields_]
    assert [f for f in field.findall(re.sub(r"/\*.*?\*/", "", outs, flags=re.S))] == [n for n, _ in graph.GraphOutputs._fields_]


NO_DEVICE_CHILD = """
import sys
sys.path.insert(0, %(root)r)
from audiosdr_b200 import graph
graph.load_library()
try:
    graph.load_library("/nonexistent/libsdr_graph.so")
except graph.GraphError:
    print("REFUSED")
"""


def test_library_loads_without_a_device_and_a_missing_one_raises():
    from audiosdr_b200 import build
    build.build_graph_library()
    r = subprocess.run([sys.executable, "-c", NO_DEVICE_CHILD % {"root": ROOT}], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "REFUSED" in r.stdout
