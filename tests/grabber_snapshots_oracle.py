"""tests/grabber_snapshots_oracle.py -- the authority for sdr_grabber_process_device_snapshots: every snapshot an
AudioGrabberComplex256 publishes, and the rows a call on chosen channels must return.

AudioGrabberComplex256::update() (GR.cpp:50-72) has no arithmetic: it appends the block as interleaved (re, im) int16 to a
two-block buffer and, when the buffer fills, copies it to outBuffer, the moment newDataAvailable() turns true.  grab_snapshots
steps that block by block from a fresh object and records outBuffer each time it is published; the C restatement's
ora_grab_run (the last snapshot) and ora_grab_spectrum (the spectrum tap) check and extend it."""
import numpy as np

from aux_subset_harness import positions

N_BLOCK = 128


def grab_snapshots(I, Q):
    """int16 [C, n_blocks // 2, 512]: [c, m] = outBuffer when channel c's m-th pair of blocks completed."""
    I = np.asarray(I, np.int16); Q = np.asarray(Q, np.int16)
    nch, ns = I.shape
    nb = ns // N_BLOCK
    buffer = np.zeros((nch, 512), np.int16)
    out = np.empty((nch, nb // 2, 512), np.int16)
    start, m = 0, 0
    for b in range(nb):  # GR.cpp:58-69, with the interleave of GR.cpp:39-47
        z = slice(b * N_BLOCK, (b + 1) * N_BLOCK)
        buffer[:, start:start + 256:2] = I[:, z]
        buffer[:, start + 1:start + 256:2] = Q[:, z]
        start = (start + 256) % 512
        if start == 0:
            out[:, m] = buffer
            m += 1
    return out


def grab_snapshots_expected(I, Q, calls):
    """What each call (ids, n_blocks) returns: (snaps int16 [n_ids, S, 512], power float32 [n_ids, S, 256], counts uint32
    [n_ids]), rows in call order, S = (n_blocks + 1) // 2.  Row i holds the snapshots and spectra of its channel's own pairs
    m in [before // 2, after // 2) (the channel's blocks processed before and after the call) in slots 0 .. counts[i] - 1;
    later slots are zero (the call does not write them)."""
    from oracle import aux_lib as A
    nch = I.shape[0]
    pos = positions(nch, calls)
    own = {}
    for c in range(nch):
        n = int(pos[-1][c])
        s = grab_snapshots(I[c:c + 1, :n * N_BLOCK], Q[c:c + 1, :n * N_BLOCK])[0]
        own[c] = (s, A.grab_spectrum(s) if len(s) else np.zeros((0, 256), np.float32))
    out = []
    for j, (ids, nb) in enumerate(calls):
        S = (nb + 1) // 2
        snaps, power = np.zeros((len(ids), S, 512), np.int16), np.zeros((len(ids), S, 256), np.float32)
        counts = np.zeros(len(ids), np.uint32)
        for i, c in enumerate(ids):
            a, b = int(pos[j][c]) // 2, int(pos[j + 1][c]) // 2
            counts[i] = b - a
            snaps[i, :b - a], power[i, :b - a] = own[c][0][a:b], own[c][1][a:b]
        out.append((snaps, power, counts))
    return out
