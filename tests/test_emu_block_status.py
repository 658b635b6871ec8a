"""CPU tier: per-block status records (include/sdr_batch.h, SDR_BS_*) through the host emulation of the kernel source.

A process call can return, next to the audio, the reference's dynamic getters after EVERY block -- what a sketch polling
`AGCisActive()`, `getSAMfrequency()`, `NoiseBlankerDetection()` ... between two update() calls sees.  The authority is the C
restatement's `status()` after each block (oracle_lib.Channel, pinned to the reference through tests/golden): every record
word must equal it bit for bit, on every plan, across setters between calls, through the host paths' chunking.
"""
import ctypes
import os
import shutil
import subprocess
import tempfile
from multiprocessing.pool import ThreadPool

import numpy as np
import pytest

import audiosdr_b200 as A
import harness
import signals as S
from test_emu_pipeline import every_bucket_case, set_plan

N_BLOCK = 128
BS = A.BS_FIELDS
# oracle status vector index of each record field (oracle/ref_client.py STATUS_FIELDS)
ORA_INDEX = {A.BS_AGC_GAIN: 14, A.BS_AGC_ACTIVE: 2, A.BS_AM_CARRIER: 6, A.BS_SAM_FREQUENCY: 4, A.BS_SAM_LOCKED: 5,
             A.BS_NB_AVERAGE: 15, A.BS_NB_DETECTED: 3}
FLAGS = (A.BS_AGC_ACTIVE, A.BS_SAM_LOCKED, A.BS_NB_DETECTED)
POISON = 0x7FC0DEAD  # a NaN pattern no field ever takes: a word left unwritten shows up


def status_words(s):
    """One oracle status vector -> the BS_FIELDS record words."""
    w = np.zeros(BS, np.uint32)
    for f, k in ORA_INDEX.items():
        w[f] = np.uint32(s[k] != 0) if f in FLAGS else np.float32(s[k]).view(np.uint32)
    return w


def oracle_block_status(I, Q, events, channels=None, threads=8):
    """The restatement's getters after every block: [n_blocks, BS_FIELDS, len(channels)] uint32.  Each listed channel is
    stepped block by block with its events applied before the block they name, in list order within a block (as the
    oracle's batch runner applies them); channels run in parallel threads (the ctypes calls release the interpreter)."""
    from oracle import oracle_lib
    nch, ns = I.shape
    nb = ns // N_BLOCK
    chans = list(range(nch)) if channels is None else list(channels)
    out = np.zeros((nb, BS, len(chans)), np.uint32)
    order = sorted(range(len(events)), key=lambda i: (events[i][1], i))

    def one(k):
        c = chans[k]
        mine = [events[i] for i in order if events[i][0] == c or events[i][0] == 0xFFFFFFFF]
        ch, ei = oracle_lib.Channel(), 0
        for b in range(nb):
            while ei < len(mine) and mine[ei][1] <= b:
                e = mine[ei]
                ch.apply(e[2], *e[3:])
                ei += 1
            ch.update(I[c, b * N_BLOCK:(b + 1) * N_BLOCK], Q[c, b * N_BLOCK:(b + 1) * N_BLOCK])
            out[b, :, k] = status_words(ch.status())

    with ThreadPool(threads) as p:
        p.map(one, range(len(chans)))
    return out


def run_records(lib, I, Q, events, chunks=(7, 1, 13), path="host", device=None, out_dtype=np.float32):
    """harness.run_batch with records: returns (audio, records [n_blocks, BS_FIELDS, n_channels] uint32, batch).
    path: "host" (process_host), "device" (process on `device`)."""
    nch, ns = I.shape
    b = A.SdrBatch(nch, _lib=lib)
    ev = sorted(events, key=lambda e: e[1])
    nb_total = ns // N_BLOCK
    outs, recs, pos, ei, k = [], [], 0, 0, 0
    if path == "device":
        import torch
        dI, dQ = torch.from_numpy(np.ascontiguousarray(I)).to(device), torch.from_numpy(np.ascontiguousarray(Q)).to(device)
        dO = torch.empty((nch, ns), dtype=torch.float32 if out_dtype == np.float32 else torch.int16, device=device)
    while pos < nb_total:
        calls = []
        while ei < len(ev) and ev[ei][1] <= pos:
            e = ev[ei]
            calls.append((None if e[0] == 0xFFFFFFFF else e[0], e[2]) + tuple(e[3:]))
            ei += 1
        if calls:
            b.configure(calls)
        nxt = ev[ei][1] if ei < len(ev) else nb_total
        sz = min(chunks[k % len(chunks)], nb_total - pos, max(nxt - pos, 1))
        k += 1
        a, z = pos * N_BLOCK, (pos + sz) * N_BLOCK
        if path == "host":
            rec = np.full((sz, BS, nch), POISON, np.uint32)
            out = np.empty((nch, sz * N_BLOCK), out_dtype)
            b.process_host(I[:, a:z], Q[:, a:z], out, block_status=rec)
            outs.append(out)
            recs.append(rec)
        else:
            import torch
            rec = torch.full((sz, BS, nch), POISON, dtype=torch.int32, device=device)
            b.process(dI[:, a:z], dQ[:, a:z], dO[:, a:z], n_blocks=sz, block_status=rec)
            recs.append(rec)
        pos += sz
    if path == "device":
        import torch
        torch.cuda.synchronize()
        return dO.cpu().numpy(), np.concatenate([r.cpu().numpy().view(np.uint32) for r in recs], 0), b
    return np.concatenate(outs, 1), np.concatenate(recs, 0), b


def last_record_matches_status(rec, batch):
    """The last record of the call equals sdr_batch_get_status after it."""
    st = batch.status()
    want = np.stack([status_words([s.tuning_offset, s.mode, s.agc_active, s.nb_detected, s.sam_frequency, s.sam_locked,
                                   s.am_carrier, 0, 0, 0, 0, 0, 0, 0, s.agc_gain, s.nb_average]) for s in st], 1)
    return np.array_equal(rec[-1], want)


def describe(got, want):
    bad = np.argwhere(got != want)
    if len(bad) == 0:
        return "identical"
    b, f, c = bad[0]
    return "%d words differ (fields %s, blocks %d..%d); first: block %d %s channel %d: got %#x want %#x" % (
        len(bad), sorted(set(A.BS_NAMES[i] for i in bad[:, 1])), bad[:, 0].min(), bad[:, 0].max(), b, A.BS_NAMES[f], c,
        got[b, f, c], want[b, f, c])


def check_case(lib, I, Q, ev, chunks=(7, 1, 13), want=None):
    """Records bit for bit against the restatement, every word written, audio the same as the call without records."""
    if want is None:
        want = oracle_block_status(I, Q, ev)
    a, rec, b = run_records(lib, I, Q, ev, chunks=chunks)
    assert not np.any(rec == POISON), "record words left unwritten"
    assert np.array_equal(rec, want), describe(rec, want)
    assert last_record_matches_status(rec, b)
    plain = harness.run_batch(lib, I, Q, ev, chunks=chunks)
    assert harness.bits_equal(a, plain), harness.describe_mismatch(a, plain)
    return rec


@pytest.mark.parametrize("cfg,nch,nblk", [(1, 1, 40), (2, 40, 30), (3, 6, 30), (4, 70, 24), (5, 5, 30)])
def test_records_match_oracle_every_block(oracle, emu_lib, cfg, nch, nblk):
    I, Q, ev = S.make(cfg, list(range(nch)), nblk)
    check_case(emu_lib, I, Q, ev)


def test_records_with_impulses_see_every_detection(oracle, emu_lib):
    """Config 2's impulses (one every 11 025 samples per channel): the per-block detections are all there, and the status
    after each ragged call would have seen only some of them."""
    I, Q, ev = S.make(2, list(range(33)), 200)
    rec = check_case(emu_lib, I, Q, ev, chunks=(23, 17, 31))
    det = A.block_status_fields(rec)["nb_detected"]
    assert det.sum() > 0


@pytest.mark.parametrize("sched", ["lockstep", "consumers", "random:5/late"])
@pytest.mark.parametrize("tile,ctas,merge", [(16, 2, 0), (8, 2, 0), (8, 3, 1), (16, 2, 1)])
@pytest.mark.parametrize("cfg,nch,nblk", [(3, 6, 30), (5, 5, 20), (1, 2, 16)])
def test_records_on_short_tile_plans(oracle, emu_lib, monkeypatch, cfg, nch, nblk, tile, ctas, merge, sched):
    from test_emu_pipeline import set_schedule
    set_schedule(monkeypatch, sched)
    set_plan(monkeypatch, tile, ctas, merge)
    I, Q, ev = S.make(cfg, list(range(nch)), nblk)
    check_case(emu_lib, I, Q, ev)


@pytest.mark.parametrize("split", ["0", "1"])
def test_records_of_both_als_forms(oracle, emu_lib, monkeypatch, split):
    """One launch, or the chain launch + ALS post-pass (the chain's AGC writes the records), also when the scratch plane
    holds only a slice of the call (the records of each slice land at its offset)."""
    monkeypatch.setenv("SDR_ALS_SPLIT", split)
    monkeypatch.setenv("SDR_ALS_SCRATCH_MB", "1")  # 3 groups: 48 KB per block -> 21-block slices
    I, Q, ev = S.make(4, list(range(70)), 48)
    check_case(emu_lib, I, Q, ev, chunks=(48, 7))


@pytest.mark.parametrize("split", ["0", "1"])
def test_records_every_bucket_kind_in_one_handle(oracle, emu_lib, monkeypatch, split):
    monkeypatch.setenv("SDR_ALS_SPLIT", split)
    I, Q, ev = every_bucket_case(nblk=20)
    check_case(emu_lib, I, Q, ev, chunks=(5, 7))


def test_records_across_setters_between_calls(oracle, emu_lib):
    """init, setDemodMode (across classes: the channel changes bucket), enableNoiseBlanker, setNoiseBlankerThresholdDb and
    disableAGC between calls: the records follow the reference block by block (a disabled AGC keeps its gain and flag, a
    channel that leaves the SAM class keeps its frequency and lock, ...)."""
    nch = 12
    I, Q, ev = S.make(4, list(range(nch)), 40)
    for c in range(nch):
        ev += [(c, 5 + c % 3, "disableAGC"), (c, 9, "setDemodMode", (S.SAM, S.USB, S.AM)[c % 3]),
               (c, 14, "enableNoiseBlanker"), (c, 17, "setNoiseBlankerThresholdDb", 6.0 + c), (c, 21, "enableAGC"),
               (c, 26, "init"), (c, 30, "setDemodMode", (S.AM, S.SAM, S.LSB)[c % 3]), (c, 33, "disableNoiseBlanker")]
    check_case(emu_lib, I, Q, ev, chunks=(3, 4, 2))


def test_records_under_setter_fuzz(oracle, emu_lib):
    rng = np.random.default_rng(77)
    I, Q, ev = S.make(4, list(range(40)), 36)
    ev += harness.fuzz_events(rng, 40, 36, 400)
    check_case(emu_lib, I, Q, ev, chunks=(5, 2, 9))


def test_records_track_sam_lock_and_unlock(oracle, emu_lib):
    """The SAM frequency and lock flag follow the carrier through loss of lock and back, block by block."""
    I, Q, ev = S.sam_lock_unlock_case(8, 60)
    rec = check_case(emu_lib, I, Q, ev, chunks=(7, 11))
    locked = A.block_status_fields(rec)["sam_locked"]
    for c in range(8):  # each channel is locked somewhere and unlocked somewhere, and comes back
        runs = np.flatnonzero(np.diff(locked[:, c].astype(np.int8)))
        assert locked[:, c].any() and not locked[:, c].all() and len(runs) >= 2, c


def fresh_emu(tmp, env):
    """A separate instance of the emulation library (a copy under another name), so that switches it reads once per process
    (SDR_HOST_CHUNKS, SDR_HOST_MIN_CHUNK) take the values of `env`."""
    from audiosdr_b200 import api
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
    subprocess.run(["make", "-s", "-C", d], check=True)
    dst = os.path.join(tmp, "libsdr_emu_chunks.so")
    shutil.copy(os.path.join(d, "libsdr_emu.so"), dst)
    return api._bind(ctypes.CDLL(dst))


def test_host_paths_with_chunk_boundaries_inside_calls(oracle, monkeypatch):
    """process_host and submit_host cut a call into time chunks; each chunk's records are copied to their place in the
    caller's buffer.  Five chunks per call, blocks of at least one: boundaries fall inside every call."""
    monkeypatch.setenv("SDR_HOST_CHUNKS", "5")
    monkeypatch.setenv("SDR_HOST_MIN_CHUNK", "1")
    I, Q, ev = S.make(4, list(range(40)), 36)
    want = oracle_block_status(I, Q, ev)
    with tempfile.TemporaryDirectory() as tmp:
        lib = fresh_emu(tmp, os.environ)
        check_case(lib, I, Q, ev, chunks=(13, 9, 14), want=want)
        # submit_host: two calls in flight, call n drained by its ticket while call n + 1 is queued
        b = A.SdrBatch(40, _lib=lib)
        b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
        got = np.full((36, BS, 40), POISON, np.uint32)
        audio = np.empty((40, 36 * N_BLOCK), np.float32)
        sizes, pos, pending = (11, 13, 12), 0, []
        for sz in sizes:
            a, z = pos * N_BLOCK, (pos + sz) * N_BLOCK
            i, q = np.ascontiguousarray(I[:, a:z]), np.ascontiguousarray(Q[:, a:z])
            out, rec = np.empty((40, sz * N_BLOCK), np.float32), np.full((sz, BS, 40), POISON, np.uint32)
            t = b.submit_host(i, q, out, block_status=rec)
            pending.append((t, pos, sz, i, q, out, rec))
            pos += sz
            if len(pending) == 2:
                t0, p0, s0, _, _, o0, r0 = pending.pop(0)
                b.wait_host(t0)
                got[p0:p0 + s0] = r0; audio[:, p0 * N_BLOCK:(p0 + s0) * N_BLOCK] = o0
        for t0, p0, s0, _, _, o0, r0 in pending:
            b.wait_host(t0)
            got[p0:p0 + s0] = r0; audio[:, p0 * N_BLOCK:(p0 + s0) * N_BLOCK] = o0
        assert np.array_equal(got, want), describe(got, want)
        assert last_record_matches_status(got, b)


def test_record_fields_helper():
    rec = np.zeros((3, BS, 2), np.uint32)
    rec[1, A.BS_NB_DETECTED, 1] = 1
    rec[2, A.BS_AGC_GAIN, 0] = np.float32(0.25).view(np.uint32)
    f = A.block_status_fields(rec)
    assert set(f) == set(A.BS_NAMES)
    assert f["nb_detected"].dtype == bool and f["nb_detected"][1, 1] and f["nb_detected"].sum() == 1
    assert f["agc_gain"].dtype == np.float32 and f["agc_gain"][2, 0] == 0.25


def test_misaligned_records_are_rejected_before_anything_is_queued(oracle, emu_lib):
    """A record buffer that is not 16-byte aligned: SDR_ERR_ARG from all three entry points, no launch, no block consumed
    (the next call still continues the stream bit for bit)."""
    nch, nblk = 6, 8
    I, Q, ev = S.make(4, list(range(nch)), nblk)
    want = oracle_block_status(I, Q, ev)
    b = A.SdrBatch(nch, _lib=emu_lib)
    b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
    raw = np.zeros(nblk * BS * nch + 8, np.uint32)
    base = raw.ctypes.data
    bad = base + (4 if (base + 4) % 16 else 8)
    out = np.empty((nch, nblk * N_BLOCK), np.float32)
    n0 = b.launch_count
    pitch = nblk * N_BLOCK
    L = emu_lib
    assert L.sdr_batch_process_host_status(b.h, I.ctypes.data, Q.ctypes.data, pitch, A.FMT_I16, out.ctypes.data, pitch,
                                           A.FMT_F32, nblk, bad) == -1
    assert L.sdr_batch_submit_host_status(b.h, I.ctypes.data, Q.ctypes.data, pitch, A.FMT_I16, out.ctypes.data, pitch,
                                          A.FMT_F32, nblk, bad) == -1
    # the device form on "device" memory of the emulation (host memory)
    assert L.sdr_batch_process_device_status(b.h, I.ctypes.data, Q.ctypes.data, pitch, A.FMT_I16, out.ctypes.data, pitch,
                                             A.FMT_F32, nblk, bad, None) == -1
    assert b.launch_count == n0 and int(L.sdr_batch_host_ticket(b.h)) == 0
    rec = np.full((nblk, BS, nch), POISON, np.uint32)
    b.process_host(I, Q, out, block_status=rec)
    assert np.array_equal(rec, want), describe(rec, want)
