"""tests/aux_subset_harness.py -- the authority for calls on chosen subsets of the channels of the pre-processor, the I/Q
generator and the grabber (sdr_*_process_*_subset): the oracle stepped over each channel's OWN blocks only.

A channel's input is its own stream: its k-th processed block is samples [128 k, 128 (k + 1)) of its row of the input
planes, whatever calls it skipped.  `calls` is a list of (ids, n_blocks) (subset_harness.random_calls makes them);
`setters` maps a call index to setter events (channel | None, name, arg...) made before that call, to listed and unlisted
channels alike: the reference object gets them between two update() calls, so they take effect at the channel's next
processed block, i.e. at the channel's own block index at the moment they were made.  Index len(calls) holds setters
made after the last call."""
import numpy as np

from subset_harness import gather_rows, random_calls  # noqa: F401  (re-exported for the tests)

N_BLOCK = 128


def _own_events(nch, calls, ev0, setters):
    """Per channel: [(own block, call index it was made before, name, args...)], ev0 = (channel | None, 0, name, args...)."""
    setters = setters or {}
    ev = {c: [] for c in range(nch)}
    for e in ev0:
        assert e[1] == 0, "initial events are at block 0"
        for c in (range(nch) if e[0] is None else [e[0]]):
            ev[c].append((0, -1, e[2]) + tuple(e[3:]))
    pos = np.zeros(nch, np.int64)
    for j in range(len(calls) + 1):
        for e in setters.get(j, []):
            for c in (range(nch) if e[0] is None else [e[0]]):
                ev[c].append((int(pos[c]), j, e[1]) + tuple(e[2:]))
        if j < len(calls):
            ids, nb = calls[j]
            pos[np.asarray(ids)] += nb
    return ev


def positions(nch, calls):
    """[pos before call j] + [pos after the last call]: each channel's own blocks processed."""
    pos = np.zeros(nch, np.int64)
    out = [pos.copy()]
    for ids, nb in calls:
        pos[np.asarray(ids)] += nb
        out.append(pos.copy())
    return out


def _run_one(kind, planes, c, n_blocks, events):
    from oracle import aux_lib as A
    ns = n_blocks * N_BLOCK
    pl = tuple(np.ascontiguousarray(p[c:c + 1, :ns]) for p in planes)
    return A.run(kind, pl, [(0, e[0], e[2]) + tuple(e[3:]) for e in events], threads=1)


def pp_expected(I, Q, ev0, calls, setters=None):
    """[(I_out, Q_out int16 [n_ids, 128 nb] in the call's row order, status int32 [n_channels, 6] of EVERY channel after the
    call)] for the pre-processor; status fields as sdr_preproc_status."""
    nch = I.shape[0]
    ev = _own_events(nch, calls, ev0, setters)
    pos = positions(nch, calls)
    full = {c: _run_one("pp", (I, Q), c, int(pos[-1][c]), ev[c]) for c in range(nch)}
    cache = {}

    def status(c, n, j):
        use = [e for e in ev[c] if e[1] <= j]
        key = (c, n, len(use))
        if key not in cache:
            cache[key] = _run_one("pp", (I, Q), c, n, use)[2][0, :6]
        return cache[key]

    out = []
    for j, (ids, nb) in enumerate(calls):
        rows = [slice(int(pos[j][c]) * N_BLOCK, int(pos[j + 1][c]) * N_BLOCK) for c in ids]
        oi = np.stack([full[c][0][0, z] for c, z in zip(ids, rows)])
        oq = np.stack([full[c][1][0, z] for c, z in zip(ids, rows)])
        st = np.stack([status(c, int(pos[j + 1][c]), j) for c in range(nch)])
        out.append((oi, oq, st))
    return out


def pp_final_status(I, Q, ev0, calls, setters=None):
    """status [n_channels, 6] after every call and every setter (including setters[len(calls)])."""
    nch = I.shape[0]
    ev = _own_events(nch, calls, ev0, setters)
    pos = positions(nch, calls)[-1]
    return np.stack([_run_one("pp", (I, Q), c, int(pos[c]), ev[c])[2][0, :6] for c in range(nch)])


def iq_expected(X, ev0, calls, setters=None):
    """[(I_out, Q_out int16 [n_ids, 128 nb])] for the I/Q generator."""
    nch = X.shape[0]
    ev = _own_events(nch, calls, ev0, setters)
    pos = positions(nch, calls)
    full = {c: _run_one("iq", (X,), c, int(pos[-1][c]), ev[c]) for c in range(nch)}
    out = []
    for j, (ids, nb) in enumerate(calls):
        rows = [slice(int(pos[j][c]) * N_BLOCK, int(pos[j + 1][c]) * N_BLOCK) for c in ids]
        out.append((np.stack([full[c][0][0, z] for c, z in zip(ids, rows)]), np.stack([full[c][1][0, z] for c, z in zip(ids, rows)])))
    return out


def grab_expected(I, Q, calls):
    """After every call: (snap int32 [n_channels, 512], -1 where the channel has no snapshot yet; valid bool [n_channels];
    completed bool [n_channels] = the call completed a pair of the channel, which sets its new-data flag)."""
    from oracle import aux_lib as A
    nch = I.shape[0]
    pos = positions(nch, calls)
    out = []
    for j in range(len(calls)):
        snap = np.empty((nch, 512), np.int32)
        valid = np.zeros(nch, bool)
        for p in np.unique(pos[j + 1]):
            cs = np.flatnonzero(pos[j + 1] == p)
            s, f = A.grab_run(I[cs, :p * N_BLOCK], Q[cs, :p * N_BLOCK])
            snap[cs], valid[cs] = s, f[:, 1] != 0
        before, after = pos[j] // 2, pos[j + 1] // 2
        out.append((snap, valid, after > before))
    return out


class FreshModel:
    """newDataAvailable() per channel: set when a call completes a pair of the channel, cleared by grab() of it."""

    def __init__(self, nch):
        self.f = np.zeros(nch, bool)

    def after_call(self, completed):
        self.f |= completed

    def grab(self, channels=None):
        if channels is None:
            self.f[:] = False
        else:
            self.f[np.asarray(channels)] = False
