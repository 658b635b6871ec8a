"""GPU tier: per-block status records (include/sdr_batch.h, SDR_BS_*) of the CUDA library, bit for bit against the C
restatement's getters after every block (the CPU tier, test_emu_block_status.py, checks the same logic in emulation)."""
import ctypes
import os
import shutil
import tempfile

import numpy as np
import pytest

import audiosdr_b200 as A
import harness
import signals as S
from test_emu_block_status import (BS, POISON, check_case, describe, last_record_matches_status, oracle_block_status,
                                   run_records)
from test_emu_pipeline import every_bucket_case, set_plan

pytestmark = pytest.mark.gpu
N_BLOCK = 128


@pytest.fixture(scope="module")
def dev():
    import torch
    return torch.device("cuda:0")


def check_device(lib, dev, I, Q, ev, chunks=(7, 1, 13), want=None):
    """The device path: records bit for bit, every word written, audio equal to the call without records."""
    if want is None:
        want = oracle_block_status(I, Q, ev)
    a, rec, b = run_records(lib, I, Q, ev, chunks=chunks, path="device", device=dev)
    assert not np.any(rec == POISON), "record words left unwritten"
    assert np.array_equal(rec, want), describe(rec, want)
    assert last_record_matches_status(rec, b)
    plain = harness.run_batch(lib, I, Q, ev, chunks=chunks, device=dev)
    assert harness.bits_equal(a, plain), harness.describe_mismatch(a, plain)
    return rec


@pytest.mark.parametrize("cfg,nch,nblk", [(1, 3, 40), (2, 64, 40), (3, 40, 30), (4, 96, 24), (5, 40, 30)])
def test_gpu_records_match_oracle(oracle, cuda_lib, dev, cfg, nch, nblk):
    I, Q, ev = S.make(cfg, list(range(nch)), nblk)
    want = oracle_block_status(I, Q, ev)
    check_device(cuda_lib, dev, I, Q, ev, want=want)
    check_case(cuda_lib, I, Q, ev, chunks=(9, 2, 13), want=want)  # process_host


@pytest.mark.parametrize("tile,ctas,merge", [(32, 1, 0), (16, 2, 0), (8, 2, 0), (16, 3, 1)])
def test_gpu_records_sam_on_every_plan(oracle, cuda_lib, dev, monkeypatch, tile, ctas, merge):
    """The SAM lock / unlock case on the 32-sample plan and on the short-tile plans (11 warps; 7 warps with the envelope
    path merged into one warp, where the carrier of a block without envelope comes from the pass-through)."""
    set_plan(monkeypatch, tile, ctas, merge)
    I, Q, ev = S.sam_lock_unlock_case(40, 60)
    rec = check_device(cuda_lib, dev, I, Q, ev, chunks=(7, 11))
    locked = A.block_status_fields(rec)["sam_locked"]
    assert locked.any() and not locked.all()


@pytest.mark.parametrize("split", ["0", "1"])
def test_gpu_records_every_bucket_kind_and_als_forms(oracle, cuda_lib, dev, monkeypatch, split):
    monkeypatch.setenv("SDR_ALS_SPLIT", split)
    I, Q, ev = every_bucket_case(nblk=20)
    check_device(cuda_lib, dev, I, Q, ev, chunks=(5, 7))
    monkeypatch.setenv("SDR_ALS_SCRATCH_MB", "1")  # the split form in slices (3 groups: 48 KB per block -> 21-block slices)
    I, Q, ev = S.make(4, list(range(70)), 48)
    check_device(cuda_lib, dev, I, Q, ev, chunks=(48, 7))


def test_gpu_records_setter_fuzz(oracle, cuda_lib, dev):
    rng = np.random.default_rng(99)
    I, Q, ev = S.make(4, list(range(64)), 36)
    ev += harness.fuzz_events(rng, 64, 36, 500)
    check_device(cuda_lib, dev, I, Q, ev, chunks=(5, 2, 9))


def test_gpu_records_config2_full_size_every_detection(oracle, cuda_lib, dev):
    """BASELINE config 2 at full size: 4 096 channels, calls of 256 blocks (the benchmark's step).  On the sampled
    channels every per-block blanker detection equals the restatement's -- and the status after each call alone (what the
    getters gave before) would have missed most of them."""
    import torch
    import bench
    nch, nblk, calls = 4096, 256, 2
    I, Q, setters = bench.synth_planes(dev, 0, nch, calls * nblk * N_BLOCK, 0x5D120002, 2)
    b = A.SdrBatch(nch, _lib=cuda_lib)
    b.configure(setters)
    out = torch.empty((nch, nblk * N_BLOCK), dtype=torch.float32, device=dev)
    rec = torch.full((calls * nblk, BS, nch), POISON, dtype=torch.int32, device=dev)
    for k in range(calls):
        s = slice(k * nblk * N_BLOCK, (k + 1) * nblk * N_BLOCK)
        b.process(I[:, s], Q[:, s], out, n_blocks=nblk, block_status=rec[k * nblk:(k + 1) * nblk])
    torch.cuda.synchronize()
    picks = S.sample_channels(2, nch, 32)
    got = rec.cpu().numpy().view(np.uint32)
    assert not np.any(got == POISON), "record words left unwritten"
    got = got[:, :, picks]
    ev = []
    for row, c in enumerate(picks):
        ev += S.channel_events(2, c, row)
    want = oracle_block_status(I[picks].cpu().numpy(), Q[picks].cpu().numpy(), ev)
    assert np.array_equal(got, want), describe(got, want)
    det = A.block_status_fields(want)["nb_detected"]
    seen_at_end = det[nblk - 1::nblk].sum()
    assert det.sum() >= 2 * len(picks), det.sum()  # an impulse every 11 025 samples: about 6 per channel over 512 blocks
    assert seen_at_end < det.sum() / 2, (seen_at_end, det.sum())


def test_gpu_records_on_a_side_stream(oracle, cuda_lib, dev):
    """The device path on a non-default stream: records land on that stream with the audio."""
    import torch
    I, Q, ev = S.make(2, list(range(64)), 24)
    want = oracle_block_status(I, Q, ev)
    b = A.SdrBatch(64, _lib=cuda_lib)
    b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
    st = torch.cuda.Stream()
    dI, dQ = torch.from_numpy(I).to(dev), torch.from_numpy(Q).to(dev)
    out = torch.empty((64, 24 * N_BLOCK), dtype=torch.float32, device=dev)
    rec = torch.full((24, BS, 64), POISON, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        for b0, nb in ((0, 10), (10, 14)):
            b.process(dI[:, b0 * N_BLOCK:(b0 + nb) * N_BLOCK], dQ[:, b0 * N_BLOCK:(b0 + nb) * N_BLOCK],
                      out[:, b0 * N_BLOCK:(b0 + nb) * N_BLOCK], n_blocks=nb, stream=st, block_status=rec[b0:b0 + nb])
    st.synchronize()
    got = rec.cpu().numpy().view(np.uint32)
    assert np.array_equal(got, want), describe(got, want)


def test_gpu_streamed_host_records_complete_at_ticket(oracle, cuda_lib, monkeypatch):
    """submit_host with records, two calls in flight: at call n's ticket its records (and audio) are complete while call
    n + 1 is queued; chunk boundaries inside every call (a separate library instance reads SDR_HOST_CHUNKS once)."""
    import torch
    from audiosdr_b200 import api
    monkeypatch.setenv("SDR_HOST_CHUNKS", "4")
    monkeypatch.setenv("SDR_HOST_MIN_CHUNK", "1")
    nch, sizes = 96, (12, 16, 9, 13)
    I, Q, ev = S.make(4, list(range(nch)), sum(sizes))
    want = oracle_block_status(I, Q, ev)
    with tempfile.TemporaryDirectory() as tmp:
        dst = os.path.join(tmp, "libsdr_batch_chunks.so")
        shutil.copy(api.lib_path(), dst)
        lib = api._bind(ctypes.CDLL(dst))
        b = A.SdrBatch(nch, _lib=lib)
        b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
        pos, pending, got = 0, [], np.zeros_like(want)
        for sz in sizes:
            a, z = pos * N_BLOCK, (pos + sz) * N_BLOCK
            i = torch.from_numpy(np.ascontiguousarray(I[:, a:z])).pin_memory().numpy()
            q = torch.from_numpy(np.ascontiguousarray(Q[:, a:z])).pin_memory().numpy()
            out = torch.empty((nch, sz * N_BLOCK), dtype=torch.float32).pin_memory().numpy()
            rec = torch.full((sz, BS, nch), POISON, dtype=torch.int32).pin_memory().numpy()
            t = b.submit_host(i, q, out, block_status=rec)
            pending.append((t, pos, sz, i, q, out, rec))
            pos += sz
            if len(pending) == 2:
                t0, p0, s0, _, _, _, r0 = pending.pop(0)
                b.wait_host(t0)
                got[p0:p0 + s0] = r0.view(np.uint32)
                assert np.array_equal(got[p0:p0 + s0], want[p0:p0 + s0]), describe(got[p0:p0 + s0], want[p0:p0 + s0])
        for t0, p0, s0, _, _, _, r0 in pending:
            b.wait_host(t0)
            got[p0:p0 + s0] = r0.view(np.uint32)
        assert np.array_equal(got, want), describe(got, want)
        assert last_record_matches_status(got, b)
        del b


def test_gpu_contracting_build_records(oracle, cuda_lib, dev):
    """The contracting build (SDR_BATCH_CONTRACT) writes records too; its last record equals its own status (its values
    are within tolerance of the reference, not bit-identical, so they are compared with themselves)."""
    import torch
    I, Q, ev = S.make(4, list(range(70)), 20)
    b = A.SdrBatch(70, _lib=cuda_lib, contract=True)
    b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
    dI, dQ = torch.from_numpy(I).to(dev), torch.from_numpy(Q).to(dev)
    out = torch.empty((70, 20 * N_BLOCK), dtype=torch.float32, device=dev)
    rec = torch.full((20, BS, 70), POISON, dtype=torch.int32, device=dev)
    b.process(dI, dQ, out, block_status=rec)
    torch.cuda.synchronize()
    got = rec.cpu().numpy().view(np.uint32)
    assert not np.any(got == POISON)
    assert last_record_matches_status(got, b)
