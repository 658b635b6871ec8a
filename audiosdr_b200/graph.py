"""audiosdr_b200/graph.py -- the shipped sketch's receiver graph streamed from host memory, over the C ABI of
include/sdr_graph.h (audiosdr_b200/libsdr_graph.so; CUDA only, no CPU fallback).

  GraphBatch(receiver, preproc=None, iqgen=None, grabber=None, waterfall=None)

runs  front (PreProcessorBatch or IQGeneratorBatch or none) -> GrabberBatch tap (optional) -> SdrBatch  on int16 host
planes: one call copies the input I/Q (or X) up, runs every block's device entry point on the same ids and copies the audio
(and the optional records, spectra and snapshots) down, chunk by chunk on three streams.  The result is bit for bit the
composition of the blocks' device calls over the whole call; the member handles stay usable and see every submitted call
once wait_host() has returned (drive a member directly only after wait_host()).  With a waterfall (aux.WaterfallBatch on the
grabber), calls take `lines=` and return the lines written per row in place of the grabber's slot counts."""
import ctypes as C
import os

import numpy as np

from .api import BS_FIELDS, FMT_F32, FMT_I16, N_BLOCK
from .aux import PP_BS_FIELDS

HERE = os.path.dirname(os.path.abspath(__file__))
EXPORTS = ["sdr_graph_create", "sdr_graph_destroy", "sdr_graph_submit_host", "sdr_graph_process_host", "sdr_graph_host_ticket",
           "sdr_graph_wait_host", "sdr_graph_wait_host_ticket", "sdr_graph_last_error", "sdr_graph_version",
           "sdr_graph_attach_waterfall", "sdr_graph_submit_host_waterfall", "sdr_graph_process_host_waterfall"]


class GraphError(RuntimeError):
    pass


class GraphDesc(C.Structure):
    _fields_ = [("rx", C.c_void_p), ("pp", C.c_void_p), ("gen", C.c_void_p), ("grabber", C.c_void_p)]


class GraphOutputs(C.Structure):
    _fields_ = [("rx_status", C.c_void_p), ("pp_status", C.c_void_p), ("power", C.c_void_p), ("snapshots", C.c_void_p),
                ("counts", C.c_void_p)]


def lib_path():
    return os.path.join(HERE, "libsdr_graph.so")


_LIB = None


def load_library(path=None):
    """Loads libsdr_graph.so; raises GraphError when it is missing (there is no other implementation to fall back to)."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    p = path or lib_path()
    if not os.path.exists(p):
        raise GraphError("CUDA library %s not built: run `python -m audiosdr_b200.build` (nvcc, sm_100a)" % p)
    L = C.CDLL(p)
    vp, u32, sz = C.c_void_p, C.c_uint32, C.c_size_t
    L.sdr_graph_create.argtypes = [C.POINTER(vp), C.POINTER(GraphDesc)]
    L.sdr_graph_destroy.argtypes = [vp]; L.sdr_graph_destroy.restype = None
    L.sdr_graph_submit_host.argtypes = [vp, vp, u32, vp, vp, sz, vp, sz, C.c_int, u32, C.POINTER(GraphOutputs)]
    L.sdr_graph_process_host.argtypes = L.sdr_graph_submit_host.argtypes
    if hasattr(L, "sdr_graph_attach_waterfall"):
        L.sdr_graph_attach_waterfall.argtypes = [vp, vp]
        L.sdr_graph_submit_host_waterfall.argtypes = L.sdr_graph_submit_host.argtypes + [vp, vp]
        L.sdr_graph_process_host_waterfall.argtypes = L.sdr_graph_submit_host_waterfall.argtypes
    L.sdr_graph_host_ticket.argtypes = [vp]; L.sdr_graph_host_ticket.restype = C.c_uint64
    L.sdr_graph_wait_host.argtypes = [vp]
    L.sdr_graph_wait_host_ticket.argtypes = [vp, C.c_uint64]
    L.sdr_graph_last_error.restype = C.c_char_p
    L.sdr_graph_version.restype = C.c_char_p
    if path is None:
        _LIB = L
    return L


def _fmt(a):
    if a.dtype == np.int16:
        return FMT_I16
    if a.dtype == np.float32:
        return FMT_F32
    raise GraphError("audio must be int16 or float32, got %s" % a.dtype)


class GraphBatch:
    """front -> grabber tap -> receiver over existing handles (api.SdrBatch, aux.PreProcessorBatch / IQGeneratorBatch,
    aux.GrabberBatch), all on one device with the same channel count.  The graph does not own them: close it first."""

    def __init__(self, receiver, preproc=None, iqgen=None, grabber=None, waterfall=None, _lib=None):
        self.L = _lib or load_library()
        self.receiver, self.preproc, self.iqgen, self.grabber, self.waterfall = receiver, preproc, iqgen, grabber, waterfall
        self.n_channels = receiver.n_channels
        d = GraphDesc(receiver.h.value, preproc.h.value if preproc is not None else None, iqgen.h.value if iqgen is not None else None,
                      grabber.h.value if grabber is not None else None)
        self.h = C.c_void_p()
        self._check(self.L.sdr_graph_create(C.byref(self.h), C.byref(d)))
        if waterfall is not None:
            self._check(self.L.sdr_graph_attach_waterfall(self.h, waterfall.h))

    def _check(self, rc):
        if rc != 0:
            raise GraphError(self.L.sdr_graph_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.sdr_graph_destroy(self.h)
            self.h = None

    __del__ = close

    def _call(self, fn, I, Q, audio, n_blocks, channels, block_status, pp_block_status, power, snapshots, lines=None):
        if channels is None:
            ids, rows = None, self.n_channels
        else:
            ids = np.ascontiguousarray(np.atleast_1d(np.asarray(channels)).astype(np.uint32))
            rows = ids.size
        n_blocks = int(n_blocks if n_blocks is not None else I.shape[1] // N_BLOCK)
        assert I.dtype == np.int16 and I.shape[0] == rows and I.strides[1] == 2, "I (or X): int16 [rows, >= 128 n_blocks], unit stride"
        if Q is not None:
            assert Q.dtype == np.int16 and Q.shape == I.shape and Q.strides == I.strides, "Q: as I"
        assert audio.shape[0] == rows and audio.strides[1] == audio.itemsize
        S = (n_blocks + 1) // 2
        o = GraphOutputs()
        for field, a, shape, dt in (("rx_status", block_status, (n_blocks, BS_FIELDS, rows), None),
                                    ("pp_status", pp_block_status, (n_blocks, PP_BS_FIELDS, rows), np.int32),
                                    ("power", power, (rows, S, 256), np.float32), ("snapshots", snapshots, (rows, S, 512), np.int16)):
            if a is None:
                continue
            assert isinstance(a, np.ndarray) and a.flags.c_contiguous and a.shape == shape and (a.dtype == dt if dt else a.itemsize == 4), \
                "%s: a C-contiguous numpy array %r%s" % (field, shape, "" if dt is None else " of " + np.dtype(dt).name)
            setattr(o, field, a.ctypes.data)
        counts = np.zeros(rows, np.uint32) if self.grabber is not None else None
        args = (self.h, ids.ctypes.data if ids is not None else None, rows, I.ctypes.data, Q.ctypes.data if Q is not None else None,
                I.strides[0] // 2, audio.ctypes.data, audio.strides[0] // audio.itemsize, _fmt(audio), n_blocks, C.byref(o))
        if self.waterfall is not None:
            shape = (rows, self.waterfall.line_slots(n_blocks), 256)
            assert isinstance(lines, np.ndarray) and lines.dtype == np.float32 and lines.flags.c_contiguous and lines.shape == shape, \
                "lines: a C-contiguous numpy float32 array %r" % (shape,)
            self._check(fn[1](*args, lines.ctypes.data, counts.ctypes.data))
            return counts
        assert lines is None, "lines need GraphBatch(..., waterfall=)"
        if counts is not None:
            o.counts = counts.ctypes.data
        self._check(fn[0](*args))
        return counts

    def submit_host(self, I, Q, audio, n_blocks=None, channels=None, block_status=None, pp_block_status=None, power=None, snapshots=None,
                    lines=None):
        """Queues one call and returns (ticket, counts).  Host numpy planes, int16 [rows, >= 128 n_blocks] with unit stride
        (pinned for asynchronous copies): I and Q, or the real input X as I with Q=None for the I/Q generator front.  audio:
        int16 or float32 [rows, >= 128 n_blocks].  channels: the ids the rows belong to (None: every channel).  Optional
        outputs, C-contiguous numpy arrays: block_status [n_blocks, BS_FIELDS, rows] (the receiver's records, 4-byte words),
        pp_block_status int32 [n_blocks, PP_BS_FIELDS, rows], power float32 [rows, S, 256] and snapshots int16 [rows, S, 512]
        with S = (n_blocks + 1) // 2 (the grabber's).  counts: uint32 [rows], the slots written per row (None without a
        grabber), valid on return.  Inputs must stay unchanged and outputs unread until wait_host(ticket).
        With a waterfall: lines, float32 [rows, waterfall.line_slots(n_blocks), 256], receives each row's lines of the call
        (later slots keep what they held) and counts are the lines per row; power, snapshots are not available."""
        fn = (self.L.sdr_graph_submit_host, getattr(self.L, "sdr_graph_submit_host_waterfall", None))
        counts = self._call(fn, I, Q, audio, n_blocks, channels, block_status, pp_block_status, power, snapshots, lines)
        return int(self.L.sdr_graph_host_ticket(self.h)), counts

    def process_host(self, I, Q, audio=None, out_fmt=FMT_F32, n_blocks=None, channels=None, block_status=None, pp_block_status=None,
                     power=None, snapshots=None, lines=None):
        """submit_host + wait for that call; returns (audio, counts).  audio=None: a new array of out_fmt."""
        if audio is None:
            nb = int(n_blocks if n_blocks is not None else I.shape[1] // N_BLOCK)
            audio = np.empty((I.shape[0], nb * N_BLOCK), np.float32 if out_fmt == FMT_F32 else np.int16)
        fn = (self.L.sdr_graph_process_host, getattr(self.L, "sdr_graph_process_host_waterfall", None))
        counts = self._call(fn, I, Q, audio, n_blocks, channels, block_status, pp_block_status, power, snapshots, lines)
        return audio, counts

    def wait_host(self, ticket=None):
        """Everything submitted so far (ticket None), or the call submit_host returned `ticket` for (later calls stay in flight)."""
        if ticket is None:
            self._check(self.L.sdr_graph_wait_host(self.h))
        else:
            self._check(self.L.sdr_graph_wait_host_ticket(self.h, int(ticket)))
