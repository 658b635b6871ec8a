"""audiosdr_b200/api.py -- Python mirror of the reference class's public interface over the C ABI.

`SdrBatch` exposes the reference's setter names (AudioSDR.h:88-152) with a leading channel selector
(None = every channel, an int, or a sequence of ints), the getters as `status()`, and the hot path as
`process()` (device tensors) / `process_host()` (host arrays).  ctypes only: no torch types cross the ABI.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

LSB, USB, CW_LSB, CW_USB, AM, SAM, WSPR = range(7)
(AUDIO_AM, AUDIO_CW, AUDIO_WSPR, AUDIO_2100, AUDIO_2300, AUDIO_2500, AUDIO_2700, AUDIO_2900, AUDIO_3100, AUDIO_3300,
 AUDIO_BYPASS) = range(11)
AGC_OFF, AGC_FAST, AGC_MEDIUM, AGC_SLOW = range(4)
FMT_I16, FMT_F32 = 0, 1
N_BLOCK = 128

SETTERS = dict(
    setMute=1, setInputGain=2, setIQgainBalance=3, setDemodMode=4, enableAudioFilter=5, disableAudioFilter=6,
    setOutputGain=7, setAudioFilter=8, enableALSfilter=9, disableALSfilter=10, setALSfilterNotch=11,
    setALSfilterPeak=12, setALSfilterAdaptive=13, setALSfilterStatic=14, setALSfilterParams=15, enableAGC=16,
    disableAGC=17, setAGCthreshold=18, setAGCslope=19, setAGCmode=20, setAGCkneeWidth=21, setAGCattackTime=22,
    setAGCreleaseTime=23, setAGChangTime=24, setAGCstaticGain=25, enableNoiseBlanker=26, disableNoiseBlanker=27,
    setNoiseBlankerThreshold=28, setNoiseBlankerThresholdDb=29, init=30)

EXPORTS = ["sdr_batch_create", "sdr_batch_destroy", "sdr_batch_set", "sdr_batch_configure", "sdr_batch_process_device",
           "sdr_batch_process_host", "sdr_batch_get_status", "sdr_batch_get_agc_lookup", "sdr_batch_peek_state",
           "sdr_batch_get_role_profile", "sdr_batch_launch_count", "sdr_batch_last_error", "sdr_batch_version",
           "sdr_batch_process", "sdr_batch_state_bytes", "sdr_batch_export_state", "sdr_batch_import_state",
           "sdr_batch_submit_host", "sdr_batch_wait_host", "sdr_batch_host_ticket", "sdr_batch_wait_host_ticket",
           "sdr_batch_process_device_status", "sdr_batch_process_host_status", "sdr_batch_submit_host_status",
           "sdr_batch_process_device_subset", "sdr_batch_process_host_subset", "sdr_batch_submit_host_subset",
           "sdr_batch_get_desc", "sdr_batch_release_stream"]

# per-block status records (include/sdr_batch.h, SDR_BS_*): array [n_blocks, BS_FIELDS, n_channels] of 32-bit words
(BS_AGC_GAIN, BS_AGC_ACTIVE, BS_AM_CARRIER, BS_SAM_FREQUENCY, BS_SAM_LOCKED, BS_NB_AVERAGE, BS_NB_DETECTED,
 BS_FIELDS) = range(8)
BS_NAMES = ["agc_gain", "agc_active", "am_carrier", "sam_frequency", "sam_locked", "nb_average", "nb_detected"]
_BS_FLAGS = (BS_AGC_ACTIVE, BS_SAM_LOCKED, BS_NB_DETECTED)


def block_status_fields(records):
    """Named views of a per-block status record array [n_blocks, BS_FIELDS, n_channels] (numpy, any 4-byte dtype, or a torch
    tensor, which is copied to the host): {name: [n_blocks, n_channels]}, float32 for the levels, bool for the three flags
    (AGCisActive, getSAMphaseLockStatus, NoiseBlankerDetection)."""
    if hasattr(records, "detach"):
        records = records.detach().cpu().numpy()
    r = np.asarray(records)
    assert r.ndim == 3 and r.shape[1] == BS_FIELDS and r.dtype.itemsize == 4, "expected [n_blocks, %d, n_channels] 32-bit words" % BS_FIELDS
    return {name: (r[:, f, :].view(np.uint32) != 0) if f in _BS_FLAGS else r[:, f, :].view(np.float32)
            for f, name in enumerate(BS_NAMES)}


class SdrError(RuntimeError):
    pass


class Desc(C.Structure):
    _fields_ = [("n_channels", C.c_uint32), ("device", C.c_int32), ("max_blocks_per_call", C.c_uint32),
                ("flags", C.c_uint32)]


class SetterCall(C.Structure):
    _fields_ = [("channel", C.c_uint32), ("setter", C.c_uint32), ("a0", C.c_float), ("a1", C.c_float), ("a2", C.c_float)]


class ChannelStatus(C.Structure):
    _fields_ = [("tuning_offset", C.c_float), ("bpf_lower", C.c_float), ("bpf_upper", C.c_float),
                ("sam_frequency", C.c_float), ("am_carrier", C.c_float), ("agc_gain", C.c_float),
                ("nb_average", C.c_float), ("mode", C.c_int32), ("audio_filter", C.c_int32), ("muted", C.c_uint8),
                ("agc_enabled", C.c_uint8), ("agc_active", C.c_uint8), ("nb_enabled", C.c_uint8),
                ("nb_detected", C.c_uint8), ("sam_locked", C.c_uint8), ("als_enabled", C.c_uint8),
                ("als_notch", C.c_uint8), ("als_adaptive", C.c_uint8), ("audio_filter_enabled", C.c_uint8),
                ("pad", C.c_uint8 * 2)]


def lib_path():
    """audiosdr_b200/libsdr_batch.so; SDR_LIB names another build of the same sources for A/B experiments (tools/build_variants.py)."""
    return os.environ.get("SDR_LIB") or os.path.join(HERE, "libsdr_batch.so")


def _bind(L):
    L.sdr_batch_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(Desc)]
    L.sdr_batch_destroy.argtypes = [C.c_void_p]
    L.sdr_batch_destroy.restype = None
    L.sdr_batch_set.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float]
    L.sdr_batch_configure.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    L.sdr_batch_process_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                           C.c_size_t, C.c_int, C.c_uint32, C.c_void_p]
    L.sdr_batch_process_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                         C.c_size_t, C.c_int, C.c_uint32]
    L.sdr_batch_submit_host.argtypes = L.sdr_batch_process_host.argtypes
    L.sdr_batch_wait_host.argtypes = [C.c_void_p]
    L.sdr_batch_host_ticket.argtypes = [C.c_void_p]
    L.sdr_batch_host_ticket.restype = C.c_uint64
    L.sdr_batch_wait_host_ticket.argtypes = [C.c_void_p, C.c_uint64]
    L.sdr_batch_get_status.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.sdr_batch_get_agc_lookup.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    L.sdr_batch_peek_state.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_float)]
    L.sdr_batch_process.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.sdr_batch_state_bytes.restype = C.c_size_t
    L.sdr_batch_export_state.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.sdr_batch_import_state.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.sdr_batch_get_role_profile.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.sdr_batch_launch_count.argtypes = [C.c_void_p]
    L.sdr_batch_launch_count.restype = C.c_uint64
    L.sdr_batch_last_error.restype = C.c_char_p
    L.sdr_batch_version.restype = C.c_char_p
    if hasattr(L, "sdr_batch_process_device_status"):  # (a build older than the per-block records binds without them)
        L.sdr_batch_process_device_status.argtypes = L.sdr_batch_process_device.argtypes[:-1] + [C.c_void_p, C.c_void_p]
        L.sdr_batch_process_host_status.argtypes = L.sdr_batch_process_host.argtypes + [C.c_void_p]
        L.sdr_batch_submit_host_status.argtypes = L.sdr_batch_process_host_status.argtypes
    if hasattr(L, "sdr_batch_process_device_subset"):
        ids = [C.c_void_p, C.c_uint32]
        L.sdr_batch_process_device_subset.argtypes = [C.c_void_p] + ids + L.sdr_batch_process_device_status.argtypes[1:]
        L.sdr_batch_process_host_subset.argtypes = [C.c_void_p] + ids + L.sdr_batch_process_host_status.argtypes[1:]
        L.sdr_batch_submit_host_subset.argtypes = L.sdr_batch_process_host_subset.argtypes
    return L


_LIB = None


def load_library(path=None):
    """Loads the CUDA library (building is the job of audiosdr_b200.build / __graft_entry__.build())."""
    global _LIB
    if path is None and _LIB is not None:
        return _LIB
    p = path or lib_path()
    if not os.path.exists(p):
        raise SdrError("CUDA library %s is missing: run `python -m audiosdr_b200.build` (there is no CPU fallback)" % p)
    L = _bind(C.CDLL(p))
    if path is None:
        _LIB = L
    return L


def _fmt_of(dtype_name):
    if "int16" in dtype_name:
        return FMT_I16
    if "float32" in dtype_name:
        return FMT_F32
    raise SdrError("planes must be int16 or float32, got %s" % dtype_name)


class SdrBatch:
    """n_channels independent AudioSDR receivers on one GPU (one handle of include/sdr_batch.h)."""

    def __init__(self, n_channels, device=0, max_blocks_per_call=0, _lib=None, contract=False):
        self.L = _lib if _lib is not None else load_library()
        self.n_channels = int(n_channels)
        self.device = int(device)
        self.h = C.c_void_p()
        d = Desc(self.n_channels, self.device, int(max_blocks_per_call), 1 if contract else 0)  # flags: SDR_BATCH_CONTRACT
        self._check(self.L.sdr_batch_create(C.byref(self.h), C.byref(d)))

    # ---- plumbing
    def _check(self, rc):
        if rc != 0:
            raise SdrError("sdr_batch error %d: %s" % (rc, (self.L.sdr_batch_last_error() or b"").decode()))

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.L.sdr_batch_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ids(self, channels):
        if channels is None:
            return None, 0
        a = np.atleast_1d(np.asarray(channels, dtype=np.uint32))
        return a, a.size

    def set(self, channels, setter, a0=0.0, a1=0.0, a2=0.0):
        op = SETTERS[setter] if isinstance(setter, str) else int(setter)
        ids, n = self._ids(channels)
        self._check(self.L.sdr_batch_set(self.h, ids.ctypes.data if ids is not None else None, n, op,
                                         float(a0), float(a1), float(a2)))

    def configure(self, calls):
        """calls: iterable of (channel|None, setter, a0?, a1?, a2?) applied in order."""
        arr = []
        for k in calls:
            k = tuple(k) + (0.0,) * (5 - len(k))
            ch = 0xFFFFFFFF if k[0] is None else int(k[0])
            op = SETTERS[k[1]] if isinstance(k[1], str) else int(k[1])
            arr.append(SetterCall(ch, op, float(k[2]), float(k[3]), float(k[4])))
        buf = (SetterCall * max(len(arr), 1))(*arr)
        self._check(self.L.sdr_batch_configure(self.h, C.cast(buf, C.c_void_p), len(arr)))

    # ---- the reference's setter names (AudioSDR.h:88-152), channel selector first
    def setMute(self, ch, muted): self.set(ch, "setMute", 1.0 if muted else 0.0)
    def setInputGain(self, ch, g): self.set(ch, "setInputGain", g)
    def setIQgainBalance(self, ch, b): self.set(ch, "setIQgainBalance", b)
    def setDemodMode(self, ch, mode):
        self.set(ch, "setDemodMode", mode)
        return {LSB: 8390.0, USB: 5390.0, CW_LSB: 7390.0, CW_USB: 6390.0, AM: 6890.0, SAM: 6890.0, WSPR: 5390.0}[int(mode)]
    def enableAudioFilter(self, ch=None): self.set(ch, "enableAudioFilter")
    def disableAudioFilter(self, ch=None): self.set(ch, "disableAudioFilter")
    def setOutputGain(self, ch, g): self.set(ch, "setOutputGain", g)
    def setAudioFilter(self, ch, f): self.set(ch, "setAudioFilter", f)
    def enableALSfilter(self, ch=None): self.set(ch, "enableALSfilter")
    def disableALSfilter(self, ch=None): self.set(ch, "disableALSfilter")
    def setALSfilterNotch(self, ch=None): self.set(ch, "setALSfilterNotch")
    def setALSfilterPeak(self, ch=None): self.set(ch, "setALSfilterPeak")
    def setALSfilterAdaptive(self, ch=None): self.set(ch, "setALSfilterAdaptive")
    def setALSfilterStatic(self, ch=None): self.set(ch, "setALSfilterStatic")
    def setALSfilterParams(self, ch, m, lam, delay): self.set(ch, "setALSfilterParams", m, lam, delay)
    def enableAGC(self, ch=None): self.set(ch, "enableAGC")
    def disableAGC(self, ch=None): self.set(ch, "disableAGC")
    def setAGCthreshold(self, ch, v): self.set(ch, "setAGCthreshold", v)
    def setAGCslope(self, ch, v): self.set(ch, "setAGCslope", v)
    def setAGCmode(self, ch, m): self.set(ch, "setAGCmode", m)
    def setAGCkneeWidth(self, ch, v): self.set(ch, "setAGCkneeWidth", v)
    def setAGCattackTime(self, ch, v): self.set(ch, "setAGCattackTime", v)
    def setAGCreleaseTime(self, ch, v): self.set(ch, "setAGCreleaseTime", v)
    def setAGChangTime(self, ch, v): self.set(ch, "setAGChangTime", v)
    def setAGCstaticGain(self, ch, v): self.set(ch, "setAGCstaticGain", v)
    def enableNoiseBlanker(self, ch=None): self.set(ch, "enableNoiseBlanker")
    def disableNoiseBlanker(self, ch=None): self.set(ch, "disableNoiseBlanker")
    def setNoiseBlankerThreshold(self, ch, v): self.set(ch, "setNoiseBlankerThreshold", v)
    def setNoiseBlankerThresholdDb(self, ch, v): self.set(ch, "setNoiseBlankerThresholdDb", v)
    def init(self, ch=None): self.set(ch, "init")

    # ---- getters
    def status(self, channels=None):
        ids, n = self._ids(channels)
        if ids is None:
            n = self.n_channels
        out = (ChannelStatus * n)()
        self._check(self.L.sdr_batch_get_status(self.h, ids.ctypes.data if ids is not None else None, n,
                                                C.cast(out, C.c_void_p)))
        return list(out)

    def getAGClookup(self, channel):
        out = np.zeros(129, np.float32)
        self._check(self.L.sdr_batch_get_agc_lookup(self.h, int(channel), out.ctypes.data))
        return out

    def peek_state(self, channel, word):
        v = C.c_float()
        self._check(self.L.sdr_batch_peek_state(self.h, int(channel), int(word), C.byref(v)))
        return v.value

    # ---- checkpoint / migration
    def export_state(self, channels=None):
        """Opaque per-channel blobs (uint8 array [n, sdr_batch_state_bytes()]): configuration + carry-over state."""
        ids, n = self._ids(channels)
        if ids is None:
            n = self.n_channels
        out = np.zeros((n, int(self.L.sdr_batch_state_bytes())), np.uint8)
        self._check(self.L.sdr_batch_export_state(self.h, ids.ctypes.data if ids is not None else None, n, out.ctypes.data))
        return out

    def import_state(self, channels, blobs):
        """Installs blobs from export_state (of any handle of the same library version) into the given channels."""
        ids, n = self._ids(channels)
        blobs = np.ascontiguousarray(blobs, dtype=np.uint8)
        if ids is None:
            n = self.n_channels
        assert blobs.shape == (n, int(self.L.sdr_batch_state_bytes()))
        self._check(self.L.sdr_batch_import_state(self.h, ids.ctypes.data if ids is not None else None, n, blobs.ctypes.data))

    def role_profile(self):
        """Per-stage busy fraction of the pipeline kernel (needs SDR_ROLE_PROFILE=1 at construction)."""
        busy = np.zeros(28, np.uint64); total = np.zeros(2, np.uint64); groups = np.zeros(2, np.uint64)
        self._check(self.L.sdr_batch_get_role_profile(self.h, busy.ctypes.data, total.ctypes.data, groups.ctypes.data))
        names = [["in", "nb_scan", "if_i", "if_q", "nco", "hil0", "hil1", "hil2", "hil3", "aud", "agc", "als_out", "envl", "nb_out"],
                 ["in", "nb_scan", "if_i", "if_q", "pll", "nco2", "img_i", "img_q", "mag", "aud", "agc", "als_out", "envl", "nb_out"]]
        out = {}
        for cls, cname in enumerate(("ssb", "env")):
            if total[cls]:
                out[cname] = {n: float(busy[cls * 14 + w]) / float(total[cls]) for w, n in enumerate(names[cls])}
                out[cname]["cta_cycles_per_launch"] = float(total[cls]) / float(groups[cls])
        return out

    @property
    def launch_count(self):
        return int(self.L.sdr_batch_launch_count(self.h))

    # ---- hot path
    def _rows(self, channels):
        """(ids array or None, row count) of a call: channels None = every channel; otherwise the ids whose rows the planes
        hold, in that order (kept alive by the caller until the call returns)."""
        if channels is None:
            return None, self.n_channels
        ids = np.ascontiguousarray(np.atleast_1d(np.asarray(channels)).astype(np.uint32))
        return ids, ids.size

    def _records(self, block_status, n_blocks, on_device, rows=None):
        """Address of a per-block status record buffer (None: no records): [n_blocks, BS_FIELDS, rows] (rows: the call's
        channel count), 4-byte elements, contiguous; a CUDA tensor for process(), a numpy array for the host paths."""
        if block_status is None:
            return None
        want = (n_blocks, BS_FIELDS, self.n_channels if rows is None else rows)
        if on_device:
            assert block_status.is_cuda and block_status.is_contiguous() and block_status.element_size() == 4, \
                "block_status: a contiguous CUDA tensor of 4-byte elements"
            assert tuple(block_status.shape) == want, "block_status: shape %r, want %r" % (tuple(block_status.shape), want)
            return block_status.data_ptr()
        assert isinstance(block_status, np.ndarray) and block_status.flags.c_contiguous and block_status.itemsize == 4, \
            "block_status: a C-contiguous numpy array of 4-byte elements"
        assert block_status.shape == want, "block_status: shape %r, want %r" % (block_status.shape, want)
        return block_status.ctypes.data

    def process(self, I, Q, audio, n_blocks=None, stream=None, block_status=None, channels=None):
        """Device tensors (torch, CUDA, 2-D [n_channels, >= 128*n_blocks], contiguous rows); asynchronous.  `block_status`:
        optional CUDA tensor [n_blocks, BS_FIELDS, n_channels] (4-byte dtype) that receives the getters after every block
        (block_status_fields() names them), on the same stream as the audio.  `channels`: run only these channel ids (distinct,
        any order); the planes then have one row per listed channel, row i for channels[i], and the records
        [n_blocks, BS_FIELDS, len(channels)]; every other channel skips the call untouched (sdr_batch_process_device_subset)."""
        n_blocks = int(n_blocks if n_blocks is not None else I.shape[1] // N_BLOCK)
        ids, rows = self._rows(channels)
        assert I.shape[0] == rows and Q.shape == I.shape and audio.shape[0] == rows
        assert I.stride(1) == 1 and Q.stride(1) == 1 and audio.stride(1) == 1 and I.stride(0) == Q.stride(0)
        sp = C.c_void_p(stream.cuda_stream) if stream is not None else None
        args = (self.h, I.data_ptr(), Q.data_ptr(), I.stride(0), _fmt_of(str(I.dtype)), audio.data_ptr(), audio.stride(0),
                _fmt_of(str(audio.dtype)), n_blocks)
        if ids is not None:
            self._check(self.L.sdr_batch_process_device_subset(args[0], ids.ctypes.data, rows, *args[1:],
                                                               self._records(block_status, n_blocks, True, rows), sp))
        elif block_status is None:
            self._check(self.L.sdr_batch_process_device(*args, sp))
        else:
            self._check(self.L.sdr_batch_process_device_status(*args, self._records(block_status, n_blocks, True), sp))

    def process_host(self, I, Q, audio=None, out_fmt=FMT_F32, n_blocks=None, block_status=None, channels=None):
        """Host numpy arrays [n_channels, S]; copies in, runs, copies out; returns the audio array.  `block_status`: optional
        numpy array [n_blocks, BS_FIELDS, n_channels] (4-byte dtype) that receives the getters after every block.
        `channels`: run only these channel ids, as in process() (planes [len(channels), S], records [.., len(channels)])."""
        I = np.ascontiguousarray(I)
        Q = np.ascontiguousarray(Q)
        ids, rows = self._rows(channels)
        assert I.shape == Q.shape and I.dtype == Q.dtype and I.shape[0] == rows
        n_blocks = int(n_blocks if n_blocks is not None else I.shape[1] // N_BLOCK)
        if audio is None:
            audio = np.empty((rows, n_blocks * N_BLOCK), np.float32 if out_fmt == FMT_F32 else np.int16)
        assert audio.shape[0] == rows
        args = (self.h, I.ctypes.data, Q.ctypes.data, I.strides[0] // I.itemsize, _fmt_of(str(I.dtype)), audio.ctypes.data,
                audio.strides[0] // audio.itemsize, _fmt_of(str(audio.dtype)), n_blocks)
        if ids is not None:
            self._check(self.L.sdr_batch_process_host_subset(args[0], ids.ctypes.data, rows, *args[1:],
                                                             self._records(block_status, n_blocks, False, rows)))
        elif block_status is None:
            self._check(self.L.sdr_batch_process_host(*args))
        else:
            self._check(self.L.sdr_batch_process_host_status(*args, self._records(block_status, n_blocks, False)))
        return audio

    def submit_host(self, I, Q, audio, n_blocks=None, block_status=None, channels=None):
        """Streaming form of process_host: queues the call and returns; `wait_host()` completes everything queued.  The arrays
        must be C-contiguous rows (they are used in place: no copy is made) and should be pinned; I, Q must stay unchanged
        and `audio` (and `block_status`, the optional per-block records as in process_host) unread until wait_host() -- or
        wait_host(ticket) with the ticket this returns -- has returned.  `channels`: as in process_host (the id list is
        copied by the library before this returns)."""
        ids, rows = self._rows(channels)
        assert I.shape == Q.shape and I.dtype == Q.dtype and I.shape[0] == rows and audio.shape[0] == rows
        assert I.strides[1] == I.itemsize and Q.strides == I.strides and audio.strides[1] == audio.itemsize
        n_blocks = int(n_blocks if n_blocks is not None else I.shape[1] // N_BLOCK)
        args = (self.h, I.ctypes.data, Q.ctypes.data, I.strides[0] // I.itemsize, _fmt_of(str(I.dtype)), audio.ctypes.data,
                audio.strides[0] // audio.itemsize, _fmt_of(str(audio.dtype)), n_blocks)
        if ids is not None:
            self._check(self.L.sdr_batch_submit_host_subset(args[0], ids.ctypes.data, rows, *args[1:],
                                                            self._records(block_status, n_blocks, False, rows)))
        elif block_status is None:
            self._check(self.L.sdr_batch_submit_host(*args))
        else:
            self._check(self.L.sdr_batch_submit_host_status(*args, self._records(block_status, n_blocks, False)))
        return int(self.L.sdr_batch_host_ticket(self.h))

    def wait_host(self, ticket=None):
        """Everything submitted so far (ticket None), or the call `submit_host` returned `ticket` for (later calls stay in flight)."""
        if ticket is None:
            self._check(self.L.sdr_batch_wait_host(self.h))
        else:
            self._check(self.L.sdr_batch_wait_host_ticket(self.h, int(ticket)))
