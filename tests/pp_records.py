"""tests/pp_records.py -- TEST INFRASTRUCTURE for the pre-processor's per-block status records (SDR_PP_BS_*).

  oracle_records(I, Q, events)  the oracle's getters after every block (tests/pp_records_oracle.c, which compiles
                                oracle/sdr_aux_oracle.c unchanged and drives it as ora_aux_run does)
  emu_records()                 pp_emu_run_records of tests/emu/pp_emu_records.cpp: what the records instantiations of the
                                kernels compute, run on the host from sdr_aux_core.cuh

Both libraries are compiled once per process into a temporary directory (the tree may be read-only).
events: list of (channel | None, block, setter name[, arg]), as for oracle/aux_lib.py."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import aux_lib as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NF = len(A.PP_STATUS)
FLAGS = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared"]
_libs = {}


def _build(kind):
    if kind not in _libs:
        d = tempfile.mkdtemp(prefix="pp_records_")
        so = os.path.join(d, "lib%s.so" % kind)
        if kind == "oracle":  # the flags of oracle/Makefile
            cmd = ["gcc"] + FLAGS + ["-std=c11", "-Wall", os.path.join(ROOT, "tests", "pp_records_oracle.c"), "-o", so, "-lm", "-lpthread"]
        else:  # the flags of tests/test_emu_pp_edges.py's emulator build
            cmd = ["g++"] + FLAGS + ["-std=gnu++17", "-Wno-unused-function", os.path.join(ROOT, "tests", "emu", "pp_emu_records.cpp"), "-o", so]
        subprocess.run(cmd, check=True)
        _libs[kind] = C.CDLL(so)
    return _libs[kind]


def oracle_records(I, Q, events=()):
    """Returns (out I, out Q, status [C, 8] int32, records [n_blocks, 6, C] int32: the PP_STATUS fields of each channel right
    after its update() for block b)."""
    f = _build("oracle").ora_pp_run_records
    f.restype = C.c_int
    f.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32] + [C.c_void_p] * 6
    I = np.ascontiguousarray(I, np.int16); Q = np.ascontiguousarray(Q, np.int16)
    nch, ns = I.shape
    assert ns % A.N_BLOCK == 0
    o0, o1 = np.empty_like(I), np.empty_like(Q)
    st = np.zeros((nch, 8), np.int32)
    rec = np.empty((ns // A.N_BLOCK, NF, nch), np.int32)
    blob, nev = A._pack_events("pp", events)
    buf = C.create_string_buffer(blob, len(blob)) if nev else None
    assert f(nch, ns // A.N_BLOCK, C.cast(buf, C.c_void_p) if nev else None, nev, I.ctypes.data, Q.ctypes.data, o0.ctypes.data,
             o1.ctypes.data, rec.ctypes.data, st.ctypes.data) == 0
    return o0, o1, st, rec


def emu_records():
    """pp_emu_run_records(n_channels, n_blocks, events, n_events, I, Q, out I, out Q, status [C][8] in/out, records)."""
    f = _build("emu").pp_emu_run_records
    f.restype = C.c_int
    f.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32] + [C.c_void_p] * 6
    return f
