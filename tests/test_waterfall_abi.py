"""CPU tier: the waterfall's C ABI (include/sdr_aux.h, include/sdr_graph.h) is exported by the libraries and mirrored by the
Python wrappers, and rejects bad arguments before any device work."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["sdr_waterfall_create", "sdr_waterfall_destroy", "sdr_waterfall_get_info", "sdr_waterfall_state_bytes", "sdr_waterfall_export_state",
         "sdr_waterfall_import_state", "sdr_grabber_process_device_waterfall", "sdr_grabber_process_device_waterfall_at"]
GRAPH_NAMES = ["sdr_graph_attach_waterfall", "sdr_graph_submit_host_waterfall", "sdr_graph_process_host_waterfall"]


def _declared(header):
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", header)).read(), flags=re.S)
    return set(re.findall(r"\b(sdr_\w+)\s*\(", src))


def test_symbols_declared_exported_and_mirrored():
    from audiosdr_b200 import aux, build, graph
    lib = C.CDLL(build.build_aux_library())
    glib = C.CDLL(build.build_graph_library())
    for n in NAMES:
        assert n in _declared("sdr_aux.h") and hasattr(lib, n) and n in aux.EXPORTS + aux.WATERFALL_EXPORTS, n
    assert set(aux.WATERFALL_EXPORTS) == {n for n in _declared("sdr_aux.h") if n.startswith("sdr_waterfall_")}
    for n in GRAPH_NAMES:
        assert n in _declared("sdr_graph.h") and hasattr(glib, n) and n in graph.EXPORTS, n
    import audiosdr_b200
    assert audiosdr_b200.WaterfallBatch is aux.WaterfallBatch


def test_argument_errors_before_device_work():
    from audiosdr_b200 import aux, graph
    L = aux.load_library()
    G = graph.load_library()
    h = C.c_void_p()
    assert L.sdr_waterfall_create(C.byref(h), 4, 0, 0) == -1 and h.value is None  # K == 0
    assert b"K >= 1" in L.sdr_aux_last_error()
    assert L.sdr_waterfall_create(C.byref(h), 0, 0, 4) == -1 and h.value is None  # no channels
    assert L.sdr_waterfall_create(None, 4, 0, 4) == -1
    assert L.sdr_waterfall_state_bytes() == 16 + 256 * 4  # tag, version, K, held, partial sum
    assert L.sdr_waterfall_get_info(None, None, None, None) == -1
    assert L.sdr_waterfall_export_state(None, None, 1, None) == -1
    assert L.sdr_waterfall_import_state(None, None, 1, None) == -1
    buf = C.create_string_buffer(4096)
    assert L.sdr_grabber_process_device_waterfall(None, None, None, 1, buf, buf, 128, 1, buf, None, None) == -1
    assert L.sdr_grabber_process_device_waterfall_at(None, None, None, 1, buf, buf, 128, 1, buf, 1, None, None, None) == -1
    assert G.sdr_graph_attach_waterfall(None, None) != 0
    assert G.sdr_graph_submit_host_waterfall(None, None, 1, buf, buf, 128, buf, 128, 0, 1, None, buf, None) != 0
    assert G.sdr_graph_process_host_waterfall(None, None, 1, buf, buf, 128, buf, 128, 0, 1, None, buf, None) != 0

