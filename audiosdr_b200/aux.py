"""audiosdr_b200/aux.py -- Python mirrors of the two blocks either side of the receiver chain, over the C ABI of
include/sdr_aux.h (audiosdr_b200/libsdr_aux.so; CUDA only, no CPU fallback):

  PreProcessorBatch  <-  class AudioSDRpreProcessor    (AudioSDRpreProcessor.h:49-73): same method names, channel selector first
  IQGeneratorBatch   <-  class AudioIQgenerator        (AudioIQgenerator.h:49-107)
  GrabberBatch       <-  class AudioGrabberComplex256  (AudioGrabberComplex256.h:46-64)
  WaterfallBatch     averaged waterfall lines per channel over the grabber's per-pair spectra (sdr_waterfall_*)

Channel selector: None = every channel, an int, or a sequence of ints.  Planes are int16 [n_channels, >= 128*n_blocks].

`channels=` on process / process_host advances only the listed channels (the reference's update() returns untouched when
an input block is missing): the planes then have len(channels) rows, row i belonging to channels[i], and every other
channel is left as it is (sdr_*_process_*_subset).  `block_status=` on PreProcessorBatch.process / process_host receives the
getters after every block, int32 [n_blocks, PP_BS_FIELDS, rows] (sdr_preproc_process_*_status).  export_state / import_state move channels' whole state between
handles as opaque blobs, uint8 [n, state_bytes]."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
N_BLOCK = 128
PP_SETTERS = dict(startAutoI2SerrorDetection=1, stopAutoI2SerrorDetection=2, setI2SerrorCompensation=3, swapIQ=4)
EXPORTS = ["sdr_preproc_create", "sdr_preproc_destroy", "sdr_preproc_set", "sdr_preproc_get_status", "sdr_preproc_process_device",
           "sdr_preproc_process_host", "sdr_preproc_launch_count", "sdr_iqgen_create", "sdr_iqgen_destroy",
           "sdr_iqgen_set_gain_balance", "sdr_iqgen_process_device", "sdr_iqgen_process_host", "sdr_iqgen_launch_count",
           "sdr_grabber_create", "sdr_grabber_destroy", "sdr_grabber_process_device", "sdr_grabber_new_data_available",
           "sdr_grabber_grab", "sdr_grabber_grab_device", "sdr_grabber_spectrum", "sdr_grabber_spectrum_device", "sdr_aux_last_error",
           "sdr_aux_version",
           "sdr_preproc_process_device_subset", "sdr_preproc_process_host_subset", "sdr_preproc_state_bytes", "sdr_preproc_export_state",
           "sdr_preproc_import_state", "sdr_iqgen_process_device_subset", "sdr_iqgen_process_host_subset", "sdr_iqgen_state_bytes",
           "sdr_iqgen_export_state", "sdr_iqgen_import_state", "sdr_grabber_process_device_subset", "sdr_grabber_state_bytes",
           "sdr_grabber_export_state", "sdr_grabber_import_state", "sdr_grabber_process_device_snapshots",
           "sdr_preproc_process_device_status", "sdr_preproc_process_host_status",
           "sdr_preproc_get_info", "sdr_iqgen_get_info", "sdr_grabber_get_info", "sdr_grabber_process_device_waterfall",
           "sdr_grabber_process_device_waterfall_at"]
# the waterfall handle's own functions (sdr_waterfall_*)
WATERFALL_EXPORTS = ["sdr_waterfall_create", "sdr_waterfall_destroy", "sdr_waterfall_get_info", "sdr_waterfall_state_bytes",
                     "sdr_waterfall_export_state", "sdr_waterfall_import_state"]
# per-block status records of the pre-processor (include/sdr_aux.h, SDR_PP_BS_*): int32 [n_blocks, PP_BS_FIELDS, rows], the
# fields in the order of sdr_preproc_status
(PP_BS_AUTO_DETECT, PP_BS_CORRECTION, PP_BS_FAILURE_COUNT, PP_BS_SUCCESS_COUNT, PP_BS_SAVED_SAMPLE, PP_BS_SWAP,
 PP_BS_FIELDS) = range(7)


class AuxError(RuntimeError):
    pass


class PreprocStatus(C.Structure):
    _fields_ = [("auto_detect", C.c_int32), ("correction", C.c_int32), ("failure_count", C.c_int32),
                ("success_count", C.c_int32), ("saved_sample", C.c_int32), ("swap", C.c_int32)]


def lib_path():
    return os.path.join(HERE, "libsdr_aux.so")


_LIB = None


def load_library(path=None):
    """Loads libsdr_aux.so; raises AuxError when it is missing (there is no other implementation to fall back to)."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    p = path or lib_path()
    if not os.path.exists(p):
        raise AuxError("CUDA library %s not built: run `python -m audiosdr_b200.build` (nvcc, sm_100a)" % p)
    L = C.CDLL(p)
    vp, u32, sz = C.c_void_p, C.c_uint32, C.c_size_t
    L.sdr_preproc_create.argtypes = [C.POINTER(vp), u32, C.c_int]
    L.sdr_preproc_destroy.argtypes = [vp]; L.sdr_preproc_destroy.restype = None
    L.sdr_preproc_set.argtypes = [vp, vp, u32, u32, C.c_int32]
    L.sdr_preproc_get_status.argtypes = [vp, vp, u32, vp]
    L.sdr_preproc_process_device.argtypes = [vp, vp, vp, sz, vp, vp, sz, u32, vp]
    L.sdr_preproc_process_host.argtypes = [vp, vp, vp, sz, vp, vp, sz, u32]
    L.sdr_preproc_launch_count.argtypes = [vp]; L.sdr_preproc_launch_count.restype = C.c_uint64
    L.sdr_iqgen_create.argtypes = [C.POINTER(vp), u32, C.c_int]
    L.sdr_iqgen_destroy.argtypes = [vp]; L.sdr_iqgen_destroy.restype = None
    L.sdr_iqgen_set_gain_balance.argtypes = [vp, vp, u32, C.c_float]
    L.sdr_iqgen_process_device.argtypes = [vp, vp, sz, vp, vp, sz, u32, vp]
    L.sdr_iqgen_process_host.argtypes = [vp, vp, sz, vp, vp, sz, u32]
    L.sdr_iqgen_launch_count.argtypes = [vp]; L.sdr_iqgen_launch_count.restype = C.c_uint64
    L.sdr_grabber_create.argtypes = [C.POINTER(vp), u32, C.c_int]
    L.sdr_grabber_destroy.argtypes = [vp]; L.sdr_grabber_destroy.restype = None
    L.sdr_grabber_process_device.argtypes = [vp, vp, vp, sz, u32, vp]
    L.sdr_grabber_new_data_available.argtypes = [vp, u32]
    L.sdr_grabber_grab.argtypes = [vp, vp, u32, vp]
    L.sdr_grabber_grab_device.argtypes = [vp, vp, vp]
    L.sdr_grabber_spectrum.argtypes = [vp, vp, u32, vp]
    L.sdr_grabber_spectrum_device.argtypes = [vp, vp, u32, vp, vp]
    if hasattr(L, "sdr_preproc_process_device_subset"):  # absent from builds older than the subset calls (benchmark comparisons)
        L.sdr_preproc_process_device_subset.argtypes = [vp, vp, u32, vp, vp, sz, vp, vp, sz, u32, vp]
        L.sdr_preproc_process_host_subset.argtypes = [vp, vp, u32, vp, vp, sz, vp, vp, sz, u32]
        L.sdr_iqgen_process_device_subset.argtypes = [vp, vp, u32, vp, sz, vp, vp, sz, u32, vp]
        L.sdr_iqgen_process_host_subset.argtypes = [vp, vp, u32, vp, sz, vp, vp, sz, u32]
        L.sdr_grabber_process_device_subset.argtypes = [vp, vp, u32, vp, vp, sz, u32, vp]
        for k in ("preproc", "iqgen", "grabber"):
            getattr(L, "sdr_%s_state_bytes" % k).restype = sz
            getattr(L, "sdr_%s_state_bytes" % k).argtypes = []
            getattr(L, "sdr_%s_export_state" % k).argtypes = [vp, vp, u32, vp]
            getattr(L, "sdr_%s_import_state" % k).argtypes = [vp, vp, u32, vp]
    if hasattr(L, "sdr_grabber_process_device_snapshots"):
        L.sdr_grabber_process_device_snapshots.argtypes = [vp, vp, u32, vp, vp, sz, u32, vp, vp, vp, vp]
    if hasattr(L, "sdr_preproc_process_device_status"):
        L.sdr_preproc_process_device_status.argtypes = [vp, vp, u32, vp, vp, sz, vp, vp, sz, u32, vp, vp]
        L.sdr_preproc_process_host_status.argtypes = [vp, vp, u32, vp, vp, sz, vp, vp, sz, u32, vp]
    if hasattr(L, "sdr_waterfall_create"):
        L.sdr_waterfall_create.argtypes = [C.POINTER(vp), u32, C.c_int, u32]
        L.sdr_waterfall_destroy.argtypes = [vp]; L.sdr_waterfall_destroy.restype = None
        L.sdr_waterfall_get_info.argtypes = [vp, vp, vp, vp]
        L.sdr_waterfall_state_bytes.argtypes = []; L.sdr_waterfall_state_bytes.restype = sz
        L.sdr_waterfall_export_state.argtypes = [vp, vp, u32, vp]
        L.sdr_waterfall_import_state.argtypes = [vp, vp, u32, vp]
        L.sdr_grabber_process_device_waterfall.argtypes = [vp, vp, vp, u32, vp, vp, sz, u32, vp, vp, vp]
        L.sdr_grabber_process_device_waterfall_at.argtypes = [vp, vp, vp, u32, vp, vp, sz, u32, vp, sz, vp, vp, vp]
    L.sdr_aux_last_error.restype = C.c_char_p
    L.sdr_aux_version.restype = C.c_char_p
    if path is None:
        _LIB = L
    return L


def _sel(channels):
    if channels is None:
        return None, 0, None
    arr = np.atleast_1d(np.asarray(channels, dtype=np.uint32))
    return arr.ctypes.data, len(arr), arr


def _check_dev(n_rows, *ts):
    for t in ts:
        assert t.shape[0] == n_rows and t.stride(1) == 1 and str(t.dtype) == "torch.int16" and t.is_cuda


def _ids(channels, n_channels):
    """(pointer, n_ids, keep-alive array, rows) of a subset call's id list; channels=None: every channel (NULL)."""
    if channels is None:
        return None, n_channels, None, n_channels
    arr = np.ascontiguousarray(np.atleast_1d(np.asarray(channels)).astype(np.uint32))
    return arr.ctypes.data, len(arr), arr, len(arr)


class _Base:
    _kind = None

    def _check(self, rc):
        if rc != 0:
            raise AuxError(self.L.sdr_aux_last_error().decode())

    @property
    def state_bytes(self):
        return int(getattr(self.L, "sdr_%s_state_bytes" % self._kind)())

    def export_state(self, channels=None):
        """uint8 [n, state_bytes]: one opaque blob per channel (None: every channel)."""
        p, n, keep = _sel(channels)
        cnt = n if channels is not None else self.n_channels
        out = np.zeros((cnt, self.state_bytes), np.uint8)
        self._check(getattr(self.L, "sdr_%s_export_state" % self._kind)(self.h, p, cnt, out.ctypes.data))
        return out

    def import_state(self, channels, blobs):
        """Loads blobs of export_state (of any handle of this library version) into the channels (None: 0..len(blobs)-1)."""
        b = np.ascontiguousarray(blobs, np.uint8).reshape(-1, self.state_bytes)
        p, n, keep = _sel(channels)
        if channels is not None:
            assert n == b.shape[0]
        self._check(getattr(self.L, "sdr_%s_import_state" % self._kind)(self.h, p, b.shape[0], b.ctypes.data))


class PreProcessorBatch(_Base):
    _kind = "preproc"

    def __init__(self, n_channels, device=0, _lib=None):
        self.L = _lib or load_library()
        self.n_channels = int(n_channels)
        self.h = C.c_void_p()
        self._check(self.L.sdr_preproc_create(C.byref(self.h), self.n_channels, int(device)))

    def close(self):
        if getattr(self, "h", None):
            self.L.sdr_preproc_destroy(self.h)
            self.h = None

    __del__ = close

    def _set(self, channels, name, arg=0):
        p, n, keep = _sel(channels)
        self._check(self.L.sdr_preproc_set(self.h, p, n, PP_SETTERS[name], int(arg)))

    # ---- the reference's public functions (AudioSDRpreProcessor.h:54-59)
    def startAutoI2SerrorDetection(self, channels=None):
        self._set(channels, "startAutoI2SerrorDetection")

    def stopAutoI2SerrorDetection(self, channels=None):
        self._set(channels, "stopAutoI2SerrorDetection")

    def setI2SerrorCompensation(self, channels, correction):
        self._set(channels, "setI2SerrorCompensation", correction)

    def swapIQ(self, channels, swap):
        self._set(channels, "swapIQ", 1 if swap else 0)

    def getAutoI2SerrorDetectionStatus(self, channel):
        return bool(self.status(channel)[0].auto_detect)

    def getI2SerrorCompensation(self, channel):
        return int(self.status(channel)[0].correction)

    def status(self, channels=None):
        p, n, keep = _sel(channels)
        cnt = n if channels is not None else self.n_channels
        out = (PreprocStatus * cnt)()
        self._check(self.L.sdr_preproc_get_status(self.h, p, n, out))
        return list(out)

    # ---- update() for every channel (or the listed ones), n_blocks times
    def process(self, I, Q, I_out, Q_out, n_blocks=None, stream=None, channels=None, block_status=None):
        """`block_status`: optional CUDA int32 tensor [n_blocks, PP_BS_FIELDS, rows], contiguous, that receives the getters
        after every block on the same stream as the planes (sdr_preproc_process_device_status)."""
        n_blocks = int(n_blocks if n_blocks is not None else I.shape[1] // N_BLOCK)
        p, n, keep, rows = _ids(channels, self.n_channels)
        _check_dev(rows, I, Q, I_out, Q_out)
        assert I.stride(0) == Q.stride(0) and I_out.stride(0) == Q_out.stride(0)
        sp = C.c_void_p(stream.cuda_stream) if stream is not None else None
        args = (I.data_ptr(), Q.data_ptr(), I.stride(0), I_out.data_ptr(), Q_out.data_ptr(), I_out.stride(0), n_blocks)
        if block_status is not None:
            t = block_status
            assert t.is_cuda and str(t.dtype) == "torch.int32" and t.is_contiguous() and tuple(t.shape) == (n_blocks, PP_BS_FIELDS, rows), \
                "block_status: a contiguous CUDA int32 tensor [%d, %d, %d]" % (n_blocks, PP_BS_FIELDS, rows)
            self._check(self.L.sdr_preproc_process_device_status(self.h, p, n, *args, t.data_ptr(), sp))
        elif channels is None:
            self._check(self.L.sdr_preproc_process_device(self.h, *args, sp))
        else:
            self._check(self.L.sdr_preproc_process_device_subset(self.h, p, n, *args, sp))

    def process_host(self, I, Q, I_out, Q_out, n_blocks=None, channels=None, block_status=None):
        """`block_status`: optional numpy int32 array [n_blocks, PP_BS_FIELDS, rows], C-contiguous, filled before the call
        returns (sdr_preproc_process_host_status)."""
        n_blocks = int(n_blocks if n_blocks is not None else I.shape[1] // N_BLOCK)
        p, n, keep, rows = _ids(channels, self.n_channels)
        for a in (I, Q, I_out, Q_out):
            assert a.dtype == np.int16 and a.shape[0] == rows and a.strides[1] == 2
        assert I.strides[0] == Q.strides[0] and I_out.strides[0] == Q_out.strides[0]
        args = (I.ctypes.data, Q.ctypes.data, I.strides[0] // 2, I_out.ctypes.data, Q_out.ctypes.data, I_out.strides[0] // 2, n_blocks)
        if block_status is not None:
            t = block_status
            assert isinstance(t, np.ndarray) and t.dtype == np.int32 and t.flags.c_contiguous and t.shape == (n_blocks, PP_BS_FIELDS, rows), \
                "block_status: a C-contiguous numpy int32 array [%d, %d, %d]" % (n_blocks, PP_BS_FIELDS, rows)
            self._check(self.L.sdr_preproc_process_host_status(self.h, p, n, *args, t.ctypes.data))
        elif channels is None:
            self._check(self.L.sdr_preproc_process_host(self.h, *args))
        else:
            self._check(self.L.sdr_preproc_process_host_subset(self.h, p, n, *args))

    @property
    def launch_count(self):
        return int(self.L.sdr_preproc_launch_count(self.h))


class IQGeneratorBatch(_Base):
    _kind = "iqgen"

    def __init__(self, n_channels, device=0, _lib=None):
        self.L = _lib or load_library()
        self.n_channels = int(n_channels)
        self.h = C.c_void_p()
        self._check(self.L.sdr_iqgen_create(C.byref(self.h), self.n_channels, int(device)))

    def close(self):
        if getattr(self, "h", None):
            self.L.sdr_iqgen_destroy(self.h)
            self.h = None

    __del__ = close

    def setGainBalance(self, channels, balance):
        """AudioIQgenerator::setGainBalance (AudioIQgenerator.h:56-60)"""
        p, n, keep = _sel(channels)
        self._check(self.L.sdr_iqgen_set_gain_balance(self.h, p, n, float(balance)))

    def process(self, X, I_out, Q_out, n_blocks=None, stream=None, channels=None):
        n_blocks = int(n_blocks if n_blocks is not None else X.shape[1] // N_BLOCK)
        p, n, keep, rows = _ids(channels, self.n_channels)
        _check_dev(rows, X, I_out, Q_out)
        assert I_out.stride(0) == Q_out.stride(0)
        sp = C.c_void_p(stream.cuda_stream) if stream is not None else None
        args = (X.data_ptr(), X.stride(0), I_out.data_ptr(), Q_out.data_ptr(), I_out.stride(0), n_blocks, sp)
        if channels is None:
            self._check(self.L.sdr_iqgen_process_device(self.h, *args))
        else:
            self._check(self.L.sdr_iqgen_process_device_subset(self.h, p, n, *args))

    def process_host(self, X, I_out, Q_out, n_blocks=None, channels=None):
        n_blocks = int(n_blocks if n_blocks is not None else X.shape[1] // N_BLOCK)
        p, n, keep, rows = _ids(channels, self.n_channels)
        for a in (X, I_out, Q_out):
            assert a.dtype == np.int16 and a.shape[0] == rows and a.strides[1] == 2
        assert I_out.strides[0] == Q_out.strides[0]
        args = (X.ctypes.data, X.strides[0] // 2, I_out.ctypes.data, Q_out.ctypes.data, I_out.strides[0] // 2, n_blocks)
        if channels is None:
            self._check(self.L.sdr_iqgen_process_host(self.h, *args))
        else:
            self._check(self.L.sdr_iqgen_process_host_subset(self.h, p, n, *args))

    @property
    def launch_count(self):
        return int(self.L.sdr_iqgen_launch_count(self.h))


class GrabberBatch(_Base):
    """AudioGrabberComplex256 for n_channels: process() = update() x n_blocks, grab() = the last complete 256-sample snapshot.
    Each channel is one reference object: after calls on subsets, some channels may have a snapshot while others have none
    yet; grab() and spectrum() then write only the rows of channels that have one (pass `out=` to keep the other rows)."""
    _kind = "grabber"

    def __init__(self, n_channels, device=0, _lib=None):
        self.L = _lib or load_library()
        self.n_channels = int(n_channels)
        self.h = C.c_void_p()
        self._check(self.L.sdr_grabber_create(C.byref(self.h), self.n_channels, int(device)))

    def close(self):
        if getattr(self, "h", None):
            self.L.sdr_grabber_destroy(self.h)
            self.h = None

    __del__ = close

    def process(self, I, Q, n_blocks=None, stream=None, channels=None, snapshots=None, power=None, waterfall=None, lines=None):
        """update() x n_blocks on every channel (or the listed ones).  snapshots (CUDA int16 [rows, S, 512]) and/or power
        (CUDA float32 [rows, S, 256]), S = (n_blocks + 1) // 2: every snapshot the call publishes and its spectrum, slot k of
        row i = the k-th pair the call completes for that row's channel (sdr_grabber_process_device_snapshots).  Then returns
        counts, numpy uint32 [rows]: the slots written per row.
        waterfall (a WaterfallBatch) with lines (CUDA float32 [rows, waterfall.line_slots(n_blocks), 256]): the call also
        advances the waterfall and writes the lines it completes (sdr_grabber_process_device_waterfall); counts are then the
        lines written per row.  Not combined with snapshots / power."""
        n_blocks = int(n_blocks if n_blocks is not None else I.shape[1] // N_BLOCK)
        p, n, keep, rows = _ids(channels, self.n_channels)
        _check_dev(rows, I, Q)
        assert I.stride(0) == Q.stride(0)
        sp = C.c_void_p(stream.cuda_stream) if stream is not None else None
        if waterfall is not None:
            assert snapshots is None and power is None, "waterfall lines and per-slot outputs are separate calls"
            t = lines
            assert t is not None and t.is_cuda and str(t.dtype) == "torch.float32" and t.is_contiguous() and \
                tuple(t.shape) == (rows, waterfall.line_slots(n_blocks), 256), "lines: a contiguous CUDA float32 tensor [rows, Lmax, 256]"
            counts = np.zeros(rows, np.uint32)
            self._check(self.L.sdr_grabber_process_device_waterfall(self.h, waterfall.h, p, rows, I.data_ptr(), Q.data_ptr(), I.stride(0),
                                                                    n_blocks, t.data_ptr(), counts.ctypes.data, sp))
            return counts
        if snapshots is not None or power is not None:
            S = (n_blocks + 1) // 2
            for t, dt, w in ((snapshots, "torch.int16", 512), (power, "torch.float32", 256)):
                assert t is None or (t.is_cuda and str(t.dtype) == dt and tuple(t.shape) == (rows, S, w) and t.is_contiguous())
            counts = np.zeros(rows, np.uint32)
            self._check(self.L.sdr_grabber_process_device_snapshots(
                self.h, p, rows, I.data_ptr(), Q.data_ptr(), I.stride(0), n_blocks, snapshots.data_ptr() if snapshots is not None else None,
                power.data_ptr() if power is not None else None, counts.ctypes.data, sp))
            return counts
        if channels is None:
            self._check(self.L.sdr_grabber_process_device(self.h, I.data_ptr(), Q.data_ptr(), I.stride(0), n_blocks, sp))
        else:
            self._check(self.L.sdr_grabber_process_device_subset(self.h, p, n, I.data_ptr(), Q.data_ptr(), I.stride(0), n_blocks, sp))

    def newDataAvailable(self, channel):
        r = self.L.sdr_grabber_new_data_available(self.h, int(channel))
        if r < 0:
            self._check(r)
        return bool(r)

    def spectrum(self, channels=None, out=None):
        """float32 [n, 256]: power per bin of the 256-point FFT of each channel's snapshot (natural bin order), or None while
        no listed channel has a snapshot.  Rows of channels without one are not written (zeros, or what `out` held).  A view
        of the snapshot: the new-data flags stay as they are."""
        p, n, keep = _sel(channels)
        cnt = n if channels is not None else self.n_channels
        if out is None:
            out = np.zeros((cnt, 256), np.float32)
        assert out.dtype == np.float32 and out.shape == (cnt, 256) and out.flags.c_contiguous
        r = self.L.sdr_grabber_spectrum(self.h, p, n, out.ctypes.data)
        if r < 0:
            self._check(r)
        return out if r > 0 else None

    def spectrum_device(self, power, stream=None):
        """All channels into a CUDA float32 tensor [n_channels, 256]; returns False while no snapshot is valid."""
        assert power.is_cuda and tuple(power.shape) == (self.n_channels, 256) and power.is_contiguous()
        sp = C.c_void_p(stream.cuda_stream) if stream is not None else None
        r = self.L.sdr_grabber_spectrum_device(self.h, None, 0, power.data_ptr(), sp)
        if r < 0:
            self._check(r)
        return r > 0

    def grab(self, channels=None, out=None):
        """int16 [n, 512] (re, im interleaved) or None while no listed channel has completed a pair of blocks.  The reference's
        grab() leaves the destination untouched before the first complete pair: rows of such channels are not written
        (zeros, or what `out` held).  Clears the listed channels' new-data flags."""
        p, n, keep = _sel(channels)
        cnt = n if channels is not None else self.n_channels
        if out is None:
            out = np.zeros((cnt, 512), np.int16)
        assert out.dtype == np.int16 and out.shape == (cnt, 512) and out.flags.c_contiguous
        r = self.L.sdr_grabber_grab(self.h, p, n, out.ctypes.data)
        if r < 0:
            self._check(r)
        return out if r > 0 else None


class WaterfallBatch(_Base):
    """Averaged waterfall lines per channel (include/sdr_aux.h, sdr_waterfall_*): the grabber's per-pair power spectra
    averaged K at a time in pair order, across calls, bit for bit the same however the stream is cut into calls.  Driven by
    GrabberBatch.process(..., waterfall=, lines=) and GraphBatch(..., waterfall=)."""
    _kind = "waterfall"

    def __init__(self, n_channels, K, device=0, _lib=None):
        self.L = _lib or load_library()
        self.n_channels, self.K = int(n_channels), int(K)
        self.h = C.c_void_p()
        self._check(self.L.sdr_waterfall_create(C.byref(self.h), self.n_channels, int(device), self.K))

    def close(self):
        if getattr(self, "h", None):
            self.L.sdr_waterfall_destroy(self.h)
            self.h = None

    __del__ = close

    def line_slots(self, n_blocks):
        """Lmax: the line slots per row of a call of n_blocks blocks."""
        return (self.K - 1 + (int(n_blocks) + 1) // 2) // self.K
