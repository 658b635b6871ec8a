"""tests/waterfall_oracle.py -- the authority for the waterfall (sdr_waterfall_*, sdr_grabber_process_device_waterfall):

  Channel(K)                       one channel's waterfall state (held pairs, partial sum), carried across calls and
                                   movable between channels like an exported blob
  Channel.run(snaps)               the lines a run of the channel's snapshots completes (tests/waterfall_oracle.c)
  waterfall_expected(I, Q, calls, K)  what each call (ids, n_blocks) of a grabber + waterfall returns, from each channel's
                                   own pairs (grabber_snapshots_oracle.grab_snapshots)

The C file is compiled once per process into a temporary directory (the tree may be read-only)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from aux_subset_harness import positions
from grabber_snapshots_oracle import grab_snapshots

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_lib = []


def _run_fn():
    if not _lib:
        d = tempfile.mkdtemp(prefix="waterfall_oracle_")
        so = os.path.join(d, "libwaterfall_oracle.so")
        subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-std=c11", "-Wall",
                        os.path.join(ROOT, "tests", "waterfall_oracle.c"), "-o", so, "-lm"], check=True)
        f = C.CDLL(so).ora_wf_run
        f.restype = C.c_int
        f.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.append(f)
    return _lib[0]


def line_slots(K, n_blocks):
    """Lmax of a call of n_blocks blocks"""
    return (K - 1 + (n_blocks + 1) // 2) // K


class Channel:
    def __init__(self, K):
        self.K = int(K)
        self.held = C.c_uint32(0)
        self.acc = np.zeros(256, np.float32)

    def run(self, snaps):
        """float32 [n_lines, 256]: the lines that the snapshots int16 [n, 512] complete, in order."""
        snaps = np.ascontiguousarray(snaps, np.int16).reshape(-1, 512)
        out = np.empty((len(snaps) // self.K + 1, 256), np.float32)
        nl = _run_fn()(self.K, len(snaps), snaps.ctypes.data, C.byref(self.held), self.acc.ctypes.data, out.ctypes.data)
        return out[:nl]


def waterfall_expected(I, Q, calls, K, chans=None):
    """[(lines float32 [n_ids, Lmax, 256], counts uint32 [n_ids]) per call]; slots past counts are zero.  chans: the
    channels' Channel objects (state carried in from earlier calls; None: fresh), updated in place."""
    nch = I.shape[0]
    pos = positions(nch, calls)
    chans = chans if chans is not None else [Channel(K) for _ in range(nch)]
    own = [grab_snapshots(I[c:c + 1, :int(pos[-1][c]) * 128], Q[c:c + 1, :int(pos[-1][c]) * 128])[0] for c in range(nch)]
    out = []
    for j, (ids, nb) in enumerate(calls):
        lines = np.zeros((len(ids), line_slots(K, nb), 256), np.float32)
        counts = np.zeros(len(ids), np.uint32)
        for i, c in enumerate(ids):
            a, b = int(pos[j][c]) // 2, int(pos[j + 1][c]) // 2
            got = chans[c].run(own[c][a:b])
            counts[i] = len(got)
            lines[i, :len(got)] = got
        out.append((lines, counts))
    return out
