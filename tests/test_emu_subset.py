"""CPU tier: calls on a chosen subset of the channels (sdr_batch_process_*_subset) through the host emulation of the kernel
source.

The reference's update() returns without touching anything when an input block is missing (AudioSDR.cpp:48-56): in a graph,
some objects skip a block period while others run.  The authority is oracle_lib.Channel stepped over each channel's own
blocks only, with setters applied before that channel's next processed block: audio, pcm, per-block records and every
channel's status after each call must match it bit for bit, on every plan."""
import ctypes
import os
import tempfile

import numpy as np
import pytest

import audiosdr_b200 as A
import edge_signals as E
import harness
import signals as S
from subset_harness import batch_status_words, compare, gather_rows, lib_calls, oracle_calls, random_calls
from test_emu_block_status import fresh_emu
from test_emu_pipeline import SHORT_PLANS, every_bucket_case, set_plan, set_schedule

N_BLOCK = 128
BS = A.BS_FIELDS


def config4(nch=40, nblk=48):
    I, Q, ev = S.make(4, list(range(nch)), nblk)
    return I, Q, ev


def clustered_case(nblk=48):
    """Every mode with the blanker on at each threshold, ALS on every third row, bursts of impulses in blocks 8..29 of each
    channel's own stream, so that the gaps of the subset calls fall across them."""
    return E.clustered(n_blocks=nblk)


def check_sequence(lib, I, Q, ev, calls, setters=None, path="host", out_dtype=np.float32, device=None):
    want = oracle_calls(I, Q, ev, calls, setters)
    got, b = lib_calls(lib, I, Q, ev, calls, setters, path=path, device=device, out_dtype=out_dtype)
    compare(got, want, out_dtype)
    return got, want, b


def test_null_and_every_id_in_order_are_the_plain_call(oracle, emu_lib):
    """channel_ids == NULL and the list 0..n-1 give the plain call's audio, records, status and launch count."""
    nch, nblk = 40, 24
    I, Q, ev = config4(nch, nblk)
    res = []
    for form in ("plain", "null", "ids"):
        b = A.SdrBatch(nch, _lib=emu_lib)
        b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
        audio, recs = [], []
        for a, z in ((0, 7), (7, 8), (8, 24)):
            i, q = np.ascontiguousarray(I[:, a * N_BLOCK:z * N_BLOCK]), np.ascontiguousarray(Q[:, a * N_BLOCK:z * N_BLOCK])
            out, rec = np.empty((nch, (z - a) * N_BLOCK), np.float32), np.zeros((z - a, BS, nch), np.uint32)
            if form == "plain":
                b.process_host(i, q, out, block_status=rec)
            elif form == "null":
                pitch = (z - a) * N_BLOCK
                assert emu_lib.sdr_batch_process_host_subset(b.h, None, nch, i.ctypes.data, q.ctypes.data, pitch, A.FMT_I16,
                                                             out.ctypes.data, pitch, A.FMT_F32, z - a, rec.ctypes.data) == 0
            else:
                b.process_host(i, q, out, block_status=rec, channels=np.arange(nch))
            audio.append(out); recs.append(rec)
        res.append((np.concatenate(audio, 1), np.concatenate(recs, 0), batch_status_words(b), b.launch_count))
    for r in res[1:]:
        assert harness.bits_equal(r[0], res[0][0]) and np.array_equal(r[1], res[0][1]) and np.array_equal(r[2], res[0][2])
        assert r[3] == res[0][3]


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("case", ["config4", "clustered"])
def test_random_subset_sequences(oracle, emu_lib, case, seed):
    I, Q, ev = config4() if case == "config4" else clustered_case()
    rng = np.random.default_rng(seed)
    calls = random_calls(rng, I.shape[0], 12, I.shape[1] // N_BLOCK)
    assert len(calls) >= 8
    check_sequence(emu_lib, I, Q, ev, calls)


def test_random_subset_sequence_int16_output(oracle, emu_lib):
    I, Q, ev = config4(24, 40)
    calls = random_calls(np.random.default_rng(9), 24, 10, 40)
    check_sequence(emu_lib, I, Q, ev, calls, out_dtype=np.int16)


@pytest.mark.parametrize("split", ["0", "1"])
def test_random_subset_sequences_every_bucket_kind(oracle, emu_lib, monkeypatch, split):
    """USB / AM / SAM x blanker x ALS in one handle (12 buckets), the ALS filter in one launch or split into chain + post-pass."""
    monkeypatch.setenv("SDR_ALS_SPLIT", split)
    I, Q, ev = every_bucket_case(nblk=40)
    calls = random_calls(np.random.default_rng(4), I.shape[0], 12, 40)
    check_sequence(emu_lib, I, Q, ev, calls)


@pytest.mark.parametrize("sched", ["lockstep", "consumers", "random:5/late"])
@pytest.mark.parametrize("tile,ctas,merge", SHORT_PLANS)
def test_random_subset_sequences_on_short_tile_plans(oracle, emu_lib, monkeypatch, tile, ctas, merge, sched):
    set_schedule(monkeypatch, sched)
    set_plan(monkeypatch, tile, ctas, merge)
    I, Q, ev = clustered_case(40)
    calls = random_calls(np.random.default_rng(tile + ctas + merge), I.shape[0], 9, 40)
    check_sequence(emu_lib, I, Q, ev, calls)


def test_setters_on_unlisted_channels_take_effect_at_their_next_block(oracle, emu_lib):
    """setDemodMode (across classes), enableNoiseBlanker, setNoiseBlankerThreshold and init on channels the next calls do not
    list: each lands before that channel's next processed block."""
    I, Q, ev = clustered_case(40)
    nch = I.shape[0]
    calls = random_calls(np.random.default_rng(11), nch, 12, 40)
    setters = {}
    for j in range(1, len(calls)):
        skip = sorted(set(range(nch)) - set(calls[j][0].tolist()))
        if not skip:
            continue
        c = skip[j % len(skip)]
        setters[j] = [(c, "setDemodMode", (S.SAM, S.USB, S.AM, S.LSB)[j % 4]), (skip[-1], "enableNoiseBlanker"),
                      (skip[0], "setNoiseBlankerThreshold", 1.5 + 0.1 * j)]
        if j % 3 == 0:
            setters[j].append((skip[len(skip) // 2], "init"))
    assert len(setters) >= 6
    check_sequence(emu_lib, I, Q, ev, calls, setters)


def test_sam_keeps_lock_across_gaps(oracle, emu_lib):
    """SAM channels that skip calls: their status stays as it was, and their PLL continues locked where it left off."""
    I, Q, ev = S.sam_lock_unlock_case(8, 60)
    rng = np.random.default_rng(5)
    calls = random_calls(rng, 8, 14, 60, sizes=(3, 1, 2, 4))
    got, want, b = check_sequence(emu_lib, I, Q, ev, calls)
    locked_across = 0
    for j in range(1, len(calls)):
        ids = set(calls[j][0].tolist())
        st_before = want[j - 1][3][A.BS_SAM_LOCKED]
        for i, c in enumerate(calls[j][0]):
            if st_before[c] and not all(c in set(calls[k][0].tolist()) for k in range(max(0, j - 1), j)):
                locked_across += int(want[j][2][0, A.BS_SAM_LOCKED, i] == 1)
        for c in set(range(8)) - ids:  # unlisted: the getters are untouched
            assert np.array_equal(want[j][3][:, c], want[j - 1][3][:, c])
    assert locked_across > 0


def test_export_of_a_lagging_channel_continues_in_another_handle(oracle, emu_lib):
    """A channel that has skipped calls (its blanker slots lag the handle's clock) is exported and imported into a handle
    whose clock differs from both; it continues bit for bit there."""
    I, Q, ev = clustered_case(48)
    nch = I.shape[0]
    calls = random_calls(np.random.default_rng(21), nch, 8, 24)
    want_all = oracle_calls(I, Q, ev, calls + [(np.arange(nch, dtype=np.uint32), 8)])
    got, b = lib_calls(emu_lib, I, Q, ev, calls)
    compare(got, want_all[:-1])
    pos = np.zeros(nch, np.int64)
    for ids, nb in calls:
        pos[ids] += nb
    blobs = b.export_state()
    for other in (1, 2, 3):  # the new handle's clock, mod 3: each of the three
        b2 = A.SdrBatch(nch, _lib=emu_lib)
        Z = np.zeros((nch, other * N_BLOCK), np.int16)
        b2.process_host(Z, Z, np.empty((nch, other * N_BLOCK), np.float32))
        b2.import_state(None, blobs)
        ids = np.random.default_rng(other).permutation(nch).astype(np.uint32)
        i, q = gather_rows(I, ids, pos, 8), gather_rows(Q, ids, pos, 8)
        out, rec = np.empty((nch, 8 * N_BLOCK), np.float32), np.zeros((8, BS, nch), np.uint32)
        b2.process_host(i, q, out, block_status=rec, channels=ids)
        wa, _, wr, _ = want_all[-1]
        assert harness.bits_equal(out, wa[ids]), harness.describe_mismatch(out, wa[ids])
        assert np.array_equal(rec, wr[:, :, ids])


def test_host_paths_two_subsets_in_flight_with_chunks(oracle):
    """process_host_subset and submit_host_subset cut each call into time chunks (several per call here); two submitted
    calls that list different subsets are in flight at once, each drained by its ticket."""
    I, Q, ev = clustered_case(48)
    calls = random_calls(np.random.default_rng(31), I.shape[0], 10, 48, sizes=(5, 7, 3, 6, 9))
    want = oracle_calls(I, Q, ev, calls)
    old = {k: os.environ.get(k) for k in ("SDR_HOST_CHUNKS", "SDR_HOST_MIN_CHUNK")}
    os.environ["SDR_HOST_CHUNKS"], os.environ["SDR_HOST_MIN_CHUNK"] = "3", "1"
    try:
        with tempfile.TemporaryDirectory() as tmp:
            lib = fresh_emu(tmp, os.environ)
            for path in ("host", "submit"):
                got, _ = lib_calls(lib, I, Q, ev, calls, path=path)
                compare(got, want)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def test_bad_id_lists_are_rejected_before_anything_is_queued(oracle, emu_lib):
    """Duplicate id, id >= n, n_ids == 0, NULL with a wrong n_ids, a misaligned record buffer: SDR_ERR_ARG from every entry
    point, no launch, no block consumed -- the next call gives the bits of an untouched handle."""
    nch, nblk = 12, 6
    I, Q, ev = config4(nch, nblk)
    calls = [(np.array([3, 1, 7], np.uint32), nblk)]
    want = oracle_calls(I, Q, ev, calls)
    b = A.SdrBatch(nch, _lib=emu_lib)
    b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
    L = emu_lib
    pitch = nblk * N_BLOCK
    out = np.empty((nch, pitch), np.float32)
    raw = np.zeros(nblk * BS * nch + 8, np.uint32)
    good = raw.ctypes.data + (-raw.ctypes.data) % 16
    bad_rec = good + 4
    cases = [([3, 3], good), ([1, nch], good), ([], good), (None, good), ([0, 1, 2], bad_rec)]
    n0 = b.launch_count
    for ids, rec in cases:
        arr = np.array(ids if ids else [0], np.uint32)
        ptr, n = (None, nch - 1) if ids is None else (arr.ctypes.data, len(ids))
        args = (I.ctypes.data, Q.ctypes.data, pitch, A.FMT_I16, out.ctypes.data, pitch, A.FMT_F32, nblk, rec)
        assert L.sdr_batch_process_host_subset(b.h, ptr, n, *args) == -1, ids
        assert L.sdr_batch_submit_host_subset(b.h, ptr, n, *args) == -1, ids
        assert L.sdr_batch_process_device_subset(b.h, ptr, n, *args, None) == -1, ids
    assert b.launch_count == n0 and int(L.sdr_batch_host_ticket(b.h)) == 0
    got, _ = lib_calls(emu_lib, I, Q, ev, calls, batch=b)
    compare(got, want)


def test_python_channels_argument_checks_shapes(emu_lib):
    b = A.SdrBatch(6, _lib=emu_lib)
    I = np.zeros((3, N_BLOCK), np.int16)
    with pytest.raises(AssertionError):
        b.process_host(I, I, channels=[0, 1])  # 3 rows for 2 ids
    with pytest.raises(A.SdrError):
        b.process_host(I, I, channels=[0, 1, 1])
    out = b.process_host(I, I, channels=[5, 0, 2])
    assert out.shape == (3, N_BLOCK)
