"""GPU tier: calls on a chosen subset of the channels (sdr_batch_process_*_subset) on the CUDA library, device and host paths,
bit for bit against oracle_lib.Channel stepped over each channel's own blocks; and one pool of 16 384 channels at size."""
import numpy as np
import pytest

import audiosdr_b200 as A
import harness
import signals as S
from subset_harness import compare, gather_rows, lib_calls, oracle_calls, random_calls
from test_emu_block_status import status_words
from test_emu_pipeline import every_bucket_case
from test_emu_subset import clustered_case, config4

N_BLOCK = 128
BS = A.BS_FIELDS
pytestmark = pytest.mark.gpu


def dev():
    import torch
    return torch.device("cuda:0")


@pytest.mark.parametrize("path", ["device", "host", "submit"])
@pytest.mark.parametrize("case", ["config4", "clustered", "every_bucket"])
def test_random_subset_sequences(oracle, cuda_lib, case, path):
    I, Q, ev = {"config4": config4, "clustered": clustered_case, "every_bucket": lambda: every_bucket_case(nblk=40)}[case]()
    calls = random_calls(np.random.default_rng(7), I.shape[0], 12, I.shape[1] // N_BLOCK)
    want = oracle_calls(I, Q, ev, calls)
    got, _ = lib_calls(cuda_lib, I, Q, ev, calls, path=path, device=dev())
    compare(got, want)


@pytest.mark.parametrize("split", ["0", "1"])
def test_random_subset_sequences_both_als_forms(oracle, cuda_lib, monkeypatch, split):
    monkeypatch.setenv("SDR_ALS_SPLIT", split)
    I, Q, ev = every_bucket_case(nblk=40)
    calls = random_calls(np.random.default_rng(4), I.shape[0], 12, 40)
    got, _ = lib_calls(cuda_lib, I, Q, ev, calls, path="device", device=dev())
    compare(got, oracle_calls(I, Q, ev, calls))


def test_setters_on_unlisted_channels(oracle, cuda_lib):
    I, Q, ev = clustered_case(40)
    nch = I.shape[0]
    calls = random_calls(np.random.default_rng(11), nch, 12, 40)
    setters = {}
    for j in range(1, len(calls)):
        skip = sorted(set(range(nch)) - set(calls[j][0].tolist()))
        if skip:
            setters[j] = [(skip[j % len(skip)], "setDemodMode", (S.SAM, S.USB, S.AM, S.LSB)[j % 4]), (skip[-1], "enableNoiseBlanker"),
                          (skip[0], "setNoiseBlankerThreshold", 1.5 + 0.1 * j)] + ([(skip[len(skip) // 2], "init")] if j % 3 == 0 else [])
    got, _ = lib_calls(cuda_lib, I, Q, ev, calls, setters, path="device", device=dev())
    compare(got, oracle_calls(I, Q, ev, calls, setters))


def test_sam_across_gaps(oracle, cuda_lib):
    I, Q, ev = S.sam_lock_unlock_case(8, 60)
    calls = random_calls(np.random.default_rng(5), 8, 14, 60, sizes=(3, 1, 2, 4))
    got, _ = lib_calls(cuda_lib, I, Q, ev, calls, path="device", device=dev())
    compare(got, oracle_calls(I, Q, ev, calls))


def test_export_of_a_lagging_channel_continues_in_another_handle(oracle, cuda_lib):
    I, Q, ev = clustered_case(48)
    nch = I.shape[0]
    calls = random_calls(np.random.default_rng(21), nch, 8, 24)
    want = oracle_calls(I, Q, ev, calls + [(np.arange(nch, dtype=np.uint32), 8)])
    got, b = lib_calls(cuda_lib, I, Q, ev, calls, path="device", device=dev())
    compare(got, want[:-1])
    pos = np.zeros(nch, np.int64)
    for ids, nb in calls:
        pos[ids] += nb
    blobs = b.export_state()
    for other in (1, 2, 3):
        b2 = A.SdrBatch(nch, _lib=cuda_lib)
        Z = np.zeros((nch, other * N_BLOCK), np.int16)
        b2.process_host(Z, Z)
        b2.import_state(None, blobs)
        ids = np.random.default_rng(other).permutation(nch).astype(np.uint32)
        out, rec = np.empty((nch, 8 * N_BLOCK), np.float32), np.zeros((8, BS, nch), np.uint32)
        b2.process_host(gather_rows(I, ids, pos, 8), gather_rows(Q, ids, pos, 8), out, block_status=rec, channels=ids)
        assert harness.bits_equal(out, want[-1][0][ids]) and np.array_equal(rec, want[-1][2][:, :, ids])


def test_bad_id_lists_are_rejected(oracle, cuda_lib):
    import torch
    nch, nblk = 12, 6
    I, Q, ev = config4(nch, nblk)
    calls = [(np.array([3, 1, 7], np.uint32), nblk)]
    b = A.SdrBatch(nch, _lib=cuda_lib)
    b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
    dI = torch.from_numpy(np.ascontiguousarray(I)).to(dev())
    out = torch.empty((nch, nblk * N_BLOCK), dtype=torch.float32, device=dev())
    rec = torch.zeros((nblk * BS * nch + 8,), dtype=torch.int32, device=dev())
    pitch = nblk * N_BLOCK
    n0 = b.launch_count
    for ids, r in (([3, 3], rec.data_ptr()), ([1, nch], rec.data_ptr()), ([], rec.data_ptr()), (None, rec.data_ptr()),
                   ([0, 1, 2], rec.data_ptr() + 4)):
        arr = np.array(ids if ids else [0], np.uint32)
        ptr, n = (None, nch - 1) if ids is None else (arr.ctypes.data, len(ids))
        assert cuda_lib.sdr_batch_process_device_subset(b.h, ptr, n, dI.data_ptr(), dI.data_ptr(), pitch, A.FMT_I16, out.data_ptr(),
                                                        pitch, A.FMT_F32, nblk, r, None) == -1, ids
    assert b.launch_count == n0
    got, _ = lib_calls(cuda_lib, I, Q, ev, calls, path="device", device=dev(), batch=b)
    compare(got, oracle_calls(I, Q, ev, calls))


def test_pool_of_16384_channels_at_size(oracle, cuda_lib):
    """16 384 channels of config 4's mix; 32 calls, each on a random 1/8 to 1/2 of the channels for 1 to 64 blocks.  72
    channels are checked against the oracle: 8 of every mode and the 16 with the longest gaps between their calls."""
    import torch
    from oracle import oracle_lib
    nch, n_calls, P, LT = 16384, 32, 256, 72
    rng = np.random.default_rng(2026)
    calls = []
    for _ in range(n_calls):
        k = int(nch * rng.uniform(1 / 8, 1 / 2))
        calls.append((rng.permutation(nch)[:k].astype(np.uint32), int(rng.integers(1, 65))))
    listed = np.zeros((n_calls, nch), bool)
    for j, (ids, _) in enumerate(calls):
        listed[j, ids] = True
    gap = np.zeros(nch, np.int64)  # longest run of consecutive calls a channel skips, in blocks of the handle's clock
    run = np.zeros(nch, np.int64)
    for j, (_, nb) in enumerate(calls):
        run = np.where(listed[j], 0, run + nb)
        gap = np.maximum(gap, run)
    modes = np.array([S.channel_mode(4, c) for c in range(nch)])
    sampled = set(np.argsort(-gap, kind="stable")[:16].tolist())
    for m in range(7):
        sampled |= set(rng.choice(np.flatnonzero(modes == m), 8, replace=False).tolist())
    sampled = np.array(sorted(sampled))
    assert len(sampled) >= 64 and set(modes[sampled]) == set(range(7))
    own = np.zeros(nch, np.int64)
    for ids, nb in calls:
        own[ids] += nb
    Is, Qs, ev_s = S.make(4, sampled.tolist(), int(own[sampled].max()))
    slot = {c: i for i, c in enumerate(sampled)}
    T_I, T_Q, _ = S.make(4, list(range(P)), LT)  # the other channels read rows of this pool
    _, _, ev = S.make(4, list(range(nch)), 1)
    b = A.SdrBatch(nch, _lib=cuda_lib)
    b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
    pos = np.zeros(nch, np.int64)
    got_audio = {c: [] for c in sampled}
    got_rec = {c: [] for c in sampled}
    for ids, nb in calls:
        i = np.empty((len(ids), nb * N_BLOCK), np.int16); q = np.empty_like(i)
        start = pos[ids] % (LT - 64)
        for s in np.unique(start):
            r = np.flatnonzero(start == s)
            i[r] = T_I[ids[r] % P, s * N_BLOCK:(s + nb) * N_BLOCK]
            q[r] = T_Q[ids[r] % P, s * N_BLOCK:(s + nb) * N_BLOCK]
        mine = [(r, int(c)) for r, c in enumerate(ids) if int(c) in slot]
        for r, c in mine:
            i[r] = Is[slot[c], pos[c] * N_BLOCK:(pos[c] + nb) * N_BLOCK]
            q[r] = Qs[slot[c], pos[c] * N_BLOCK:(pos[c] + nb) * N_BLOCK]
        pos[ids] += nb
        di, dq = torch.from_numpy(i).to(dev()), torch.from_numpy(q).to(dev())
        da = torch.empty((len(ids), nb * N_BLOCK), dtype=torch.float32, device=dev())
        dr = torch.empty((nb, BS, len(ids)), dtype=torch.int32, device=dev())
        b.process(di, dq, da, n_blocks=nb, block_status=dr, channels=ids)
        if mine:
            rows = torch.tensor([r for r, _ in mine], device=dev())
            a, rc = da.index_select(0, rows).cpu().numpy(), dr.index_select(2, rows).cpu().numpy().view(np.uint32)
            for k, (_, c) in enumerate(mine):
                got_audio[c].append(a[k]); got_rec[c].append(rc[:, :, k])
    torch.cuda.synchronize()
    bad = []
    for c in sampled:
        ch = oracle_lib.Channel()
        for e in ev_s:
            if e[0] == slot[c]:
                ch.apply(e[2], *e[3:])
        wa, wr = [], []
        for k in range(int(own[c])):
            a, _ = ch.update(Is[slot[c], k * N_BLOCK:(k + 1) * N_BLOCK], Qs[slot[c], k * N_BLOCK:(k + 1) * N_BLOCK])
            wa.append(a); wr.append(status_words(ch.status()))
        ga, gr = np.concatenate(got_audio[c]), np.concatenate(got_rec[c], 0)
        if not (np.array_equal(ga.view(np.uint32), np.concatenate(wa).view(np.uint32)) and np.array_equal(gr, np.stack(wr))):
            bad.append(int(c))
    assert not bad, "channels differing from the oracle: %s" % bad[:10]
