"""tests/subset_harness.py -- drive a batch through calls on chosen subsets of its channels (sdr_batch_process_*_subset), and
the authority for them: oracle_lib.Channel stepped over each channel's OWN blocks only.

A channel's input is its own stream: its k-th processed block is samples [128 k, 128 (k + 1)) of its row of I / Q, whatever
the calls it skipped.  `calls` is a list of (ids, n_blocks); `setters` maps a call index to setter events (channel, op, args...)
applied before that call, to listed and unlisted channels alike (the reference object gets them between two ISRs, and they
take effect at its next processed block)."""
import numpy as np

import audiosdr_b200 as A
from test_emu_block_status import FLAGS, ORA_INDEX, status_words

N_BLOCK = 128
BS = A.BS_FIELDS


def random_calls(rng, nch, n_calls, own_blocks, sizes=(1, 2, 3, 5, 1, 2, 4, 7)):
    """n_calls calls, each on a random 10-90 % of the channels in random row order, ragged n_blocks (1 and 2 included, so
    channels fall behind the handle's clock by 1 and 2 mod 3); no channel runs past `own_blocks` blocks of its own."""
    used = np.zeros(nch, np.int64)
    calls = []
    for j in range(n_calls):
        nb = int(sizes[j % len(sizes)])
        cand = np.flatnonzero(used + nb <= own_blocks)
        if len(cand) == 0:
            break
        k = max(1, min(len(cand), int(round(rng.uniform(0.1, 0.9) * nch))))
        ids = rng.permutation(cand)[:k].astype(np.uint32)
        used[ids] += nb
        calls.append((ids, nb))
    return calls


def batch_status_words(b, channels=None):
    """sdr_batch_get_status of the channels as record words [BS_FIELDS, n]."""
    st = b.status(channels)
    return np.stack([status_words([s.tuning_offset, s.mode, s.agc_active, s.nb_detected, s.sam_frequency, s.sam_locked,
                                   s.am_carrier, 0, 0, 0, 0, 0, 0, 0, s.agc_gain, s.nb_average]) for s in st], 1)


def _events_by_channel(ev0):
    out = {}
    for e in ev0:
        assert e[1] == 0, "initial events are at block 0"
        out.setdefault(e[0], []).append((e[2],) + tuple(e[3:]))
    return out


def oracle_calls(I, Q, ev0, calls, setters=None):
    """What each call must return: [(audio float32 [n, 128 nb], pcm int16 [n, 128 nb], records uint32 [nb, BS, n],
    status words of EVERY channel after the call [BS, n_channels])]."""
    from oracle import oracle_lib
    setters = setters or {}
    nch = I.shape[0]
    first = _events_by_channel(ev0)
    chans = []
    for c in range(nch):
        ch = oracle_lib.Channel()
        for e in first.get(c, []) + first.get(0xFFFFFFFF, []):
            ch.apply(*e)
        chans.append(ch)
    pos = np.zeros(nch, np.int64)
    out = []
    for j, (ids, nb) in enumerate(calls):
        for e in setters.get(j, []):
            targets = range(nch) if e[0] is None else [e[0]]
            for c in targets:
                chans[c].apply(e[1], *e[2:])
        n = len(ids)
        audio, pcm, rec = np.empty((n, nb * N_BLOCK), np.float32), np.empty((n, nb * N_BLOCK), np.int16), np.empty((nb, BS, n), np.uint32)
        for i, c in enumerate(ids):
            for b in range(nb):
                s = slice((pos[c] + b) * N_BLOCK, (pos[c] + b + 1) * N_BLOCK)
                a, p = chans[c].update(I[c, s], Q[c, s])
                audio[i, b * N_BLOCK:(b + 1) * N_BLOCK], pcm[i, b * N_BLOCK:(b + 1) * N_BLOCK] = a, p
                rec[b, :, i] = status_words(chans[c].status())
            pos[c] += nb
        st = np.stack([status_words(chans[c].status()) for c in range(nch)], 1)
        out.append((audio, pcm, rec, st))
    return out


def gather_rows(X, ids, pos, nb):
    return np.ascontiguousarray(np.stack([X[c, pos[c] * N_BLOCK:(pos[c] + nb) * N_BLOCK] for c in ids]))


def lib_calls(lib, I, Q, ev0, calls, setters=None, path="host", device=None, out_dtype=np.float32, batch=None, pos=None):
    """The same calls on a batch of `lib` (a new one unless `batch` is given; `pos`: each channel's blocks already processed).
    path "host" (process_host), "device" (process on `device`), "submit" (submit_host, two calls in flight, each drained by
    its ticket while the next is queued).  Returns [(audio, records, status words after the call)] and the batch."""
    setters = setters or {}
    nch = I.shape[0]
    b = batch or A.SdrBatch(nch, _lib=lib)
    if batch is None:
        b.configure([(None if e[0] == 0xFFFFFFFF else e[0], e[2]) + tuple(e[3:]) for e in ev0])
    pos = np.zeros(nch, np.int64) if pos is None else pos
    out, pending = [], []
    for j, (ids, nb) in enumerate(calls):
        if setters.get(j):
            b.configure(setters[j])
        i, q = gather_rows(I, ids, pos, nb), gather_rows(Q, ids, pos, nb)
        pos[ids] += nb
        if path == "host":
            rec = np.full((nb, BS, len(ids)), 0x7FC0DEAD, np.uint32)
            a = np.empty((len(ids), nb * N_BLOCK), out_dtype)
            b.process_host(i, q, a, block_status=rec, channels=ids)
            out.append((a, rec, batch_status_words(b)))
        elif path == "submit":
            rec = np.full((nb, BS, len(ids)), 0x7FC0DEAD, np.uint32)
            a = np.empty((len(ids), nb * N_BLOCK), out_dtype)
            t = b.submit_host(i, q, a, block_status=rec, channels=ids)
            pending.append((t, i, q, a, rec))
            out.append(None)
            if len(pending) == 2:
                t0, _, _, a0, r0 = pending.pop(0)
                b.wait_host(t0)
                out[out.index(None)] = (a0, r0, None)
        else:
            import torch
            di, dq = torch.from_numpy(i).to(device), torch.from_numpy(q).to(device)
            da = torch.empty((len(ids), nb * N_BLOCK), dtype=torch.float32 if out_dtype == np.float32 else torch.int16, device=device)
            dr = torch.full((nb, BS, len(ids)), 0x7FC0DEAD, dtype=torch.int32, device=device)
            b.process(di, dq, da, n_blocks=nb, block_status=dr, channels=ids)
            out.append((da.cpu().numpy(), dr.cpu().numpy().view(np.uint32), batch_status_words(b)))
    for t0, _, _, a0, r0 in pending:
        b.wait_host(t0)
        out[out.index(None)] = (a0, r0, None)
    return out, b


def compare(got, want, out_dtype=np.float32):
    """Bit-for-bit: audio (or pcm), records and every channel's status after each call."""
    for j, (g, w) in enumerate(zip(got, want)):
        ga, gr, gs = g
        wa, wp, wr, ws = w
        ref = wa if out_dtype == np.float32 else wp
        assert ga.shape == ref.shape, (j, ga.shape, ref.shape)
        if not np.array_equal(ga.view(np.uint32 if out_dtype == np.float32 else np.uint16), ref.view(np.uint32 if out_dtype == np.float32 else np.uint16)):
            bad = np.argwhere(ga != ref)
            raise AssertionError("call %d: audio differs in %d samples, first row %d sample %d: got %r want %r"
                                 % (j, len(bad), bad[0][0], bad[0][1], ga[tuple(bad[0])], ref[tuple(bad[0])]))
        if not np.array_equal(gr, wr):
            bad = np.argwhere(gr != wr)
            raise AssertionError("call %d: %d record words differ, first block %d %s row %d" % (j, len(bad), bad[0][0], A.BS_NAMES[bad[0][1]], bad[0][2]))
        if gs is not None and not np.array_equal(gs, ws):
            bad = np.argwhere(gs != ws)
            raise AssertionError("call %d: status differs, first %s of channel %d" % (j, A.BS_NAMES[bad[0][0]], bad[0][1]))


__all__ = ["random_calls", "oracle_calls", "lib_calls", "compare", "batch_status_words", "gather_rows", "FLAGS", "ORA_INDEX"]
